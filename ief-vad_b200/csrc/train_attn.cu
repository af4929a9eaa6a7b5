// Training-mode attention (row N3), head sizes 32, 64, 96 and 128: softmax(q k^T / sqrt(dh)) v with the dropout of
// nn.MultiheadAttention's train() path (model/imf_vad.py:53,70; torch/nn/functional.py:6643-6647) from a counter-based
// Philox4x32-10 mask, the library's own or PyTorch's (philox.cuh).  Forward (with the log-sum-exp the backward needs) and
// the two backward kernels (dq | dk, dv) on the tensor cores, flash style: no [T, T] tensor ever reaches memory, the mask
// is regenerated, never stored.  Also here: the backward's row term delta = out . dout, the mask itself as a tensor (the
// parity-test surface) and the host functions of train.cuh that launch all of them.
//
// Warp-level mma.sync m16n8k8 TF32 with fp32 accumulation (fp32's exponent range - gradients span 1e-8 .. 1e+1, which rules
// the 16-bit tcgen05 kinds of the inference kernels out without a scaling scheme), every product as 3xTF32
// (a_hi b_hi + a_lo b_hi + a_hi b_lo with hi = rna(x), lo = rna(x - hi): ~21 mantissa bits).  Plain TF32 is not enough here:
// the absolute error of a score becomes a RELATIVE error of the weight through exp(s - lse); the rows of dS = P (dP - delta)
// sum to zero only if delta (= out . dout, from the forward's P v) and dP (= dout . v) are computed consistently - and the
// gradient of the key bias IS that cancellation (measured with single-TF32 weight products: 2.9e-3 of the tensor's scale
// against the test's 1e-3 bound).  The kernels are bound by their shared-memory staging, not by the MMA count, so the two
// extra MMAs per product cost nothing measurable.
//
// Fragment layout of mma.m16n8k8 (g = lane / 4, t = lane % 4):  A: a0 (g, t) a1 (g + 8, t) a2 (g, t + 4) a3 (g + 8, t + 4);
// B: b0 (k = t, n = g) b1 (k = t + 4, n = g);  C: c0 (g, 2t) c1 (g, 2t + 1) c2 (g + 8, 2t) c3 (g + 8, 2t + 1).
// A product's C tile becomes the next product's A tile WITHOUT a shuffle by renaming the contraction index: k = t stands for
// column 2t and k = t + 4 for column 2t + 1, and the B fragment reads its rows in the same order.
// Shared-memory tiles have a row pitch of DH + 4 words (= 4 mod 32): every fragment load is conflict-free.
#include "common.cuh"
#include "operand.cuh"     // blocks_for
#include "philox.cuh"
#include "train.cuh"

namespace iefvad {

namespace {

constexpr int kWarps = 4;
constexpr int kThreads = 32 * kWarps;
constexpr int BQ = 16 * kWarps;      // rows owned by a CTA (16 per warp)
constexpr int BC = 32;               // columns streamed per iteration

__device__ __forceinline__ uint32_t to_tf32(float x) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return r;
}
__device__ __forceinline__ void mma_tf32(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

// rows [r0, r0 + nrows) of one [*, DH] slice of a row-major matrix -> fp32 words in shared memory (rows past `limit`: zero)
template <int DH>
__device__ __forceinline__ void load_tile(uint32_t* dst, const float* src, long long row_stride, int r0, int nrows, int limit,
                                          float scale) {
  constexpr int P = DH + 4;
  for (int i = threadIdx.x; i < nrows * DH; i += kThreads) {
    const int r = i / DH, d = i - r * DH;
    const int t = r0 + r;
    dst[r * P + d] = (t < limit) ? __float_as_uint(src[(long long)t * row_stride + d] * scale) : 0u;
  }
}

// the same through cp.async (16-byte pieces, zero-filled past `limit`): the next block's tiles travel while this one computes
template <int DH>
__device__ __forceinline__ void load_tile_async(uint32_t* dst, const float* src, long long row_stride, int r0, int nrows, int limit) {
  constexpr int P = DH + 4, C4 = DH / 4;
  for (int i = threadIdx.x; i < nrows * C4; i += kThreads) {
    const int r = i / C4, c = i - r * C4;
    const int t = r0 + r;
    const float* g = src + (long long)(t < limit ? t : 0) * row_stride + c * 4;
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(smem_u32(dst + r * P + c * 4)), "l"(g), "r"(t < limit ? 16 : 0)
                 : "memory");
  }
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// fp32 word -> (hi, lo) TF32 pair
__device__ __forceinline__ void split_tf32(uint32_t w, uint32_t& hi, uint32_t& lo) {
  const float x = __uint_as_float(w);
  hi = to_tf32(x);
  lo = to_tf32(x - __uint_as_float(hi));
}

// acc[nt] (16 x 8 each, nt < 4) += A(rows of tile_a) . B(rows [8 nt, 8 nt + 8) of tile_b)^T, contraction over the DH columns;
// 3xTF32: both operands as (hi, lo) pairs, the lo . lo term dropped
template <int DH>
__device__ __forceinline__ void mma_rows(float (&acc)[4][4], const uint32_t* tile_a, int ra, const uint32_t* tile_b, int g, int t) {
  constexpr int P = DH + 4;
#pragma unroll
  for (int kk = 0; kk < DH / 8; ++kk) {
    uint32_t ah[4], al[4];
    split_tf32(tile_a[(ra + g) * P + kk * 8 + t], ah[0], al[0]);
    split_tf32(tile_a[(ra + g + 8) * P + kk * 8 + t], ah[1], al[1]);
    split_tf32(tile_a[(ra + g) * P + kk * 8 + t + 4], ah[2], al[2]);
    split_tf32(tile_a[(ra + g + 8) * P + kk * 8 + t + 4], ah[3], al[3]);
#pragma unroll
    for (int nt = 0; nt < 4; ++nt) {
      uint32_t bh0, bl0, bh1, bl1;
      split_tf32(tile_b[(nt * 8 + g) * P + kk * 8 + t], bh0, bl0);
      split_tf32(tile_b[(nt * 8 + g) * P + kk * 8 + t + 4], bh1, bl1);
      mma_tf32(acc[nt], al, bh0, bh1);
      mma_tf32(acc[nt], ah, bl0, bl1);
      mma_tf32(acc[nt], ah, bh0, bh1);
    }
  }
}

// out[nd] (16 x 8 each, nd < DH / 8) += W . X, W = four C tiles (16 x 32, contraction index renamed as above), X = rows of a
// shared-memory tile [32, DH]
// XSPLIT = false: X as single TF32 values - measured on the backward products (dq, dk, dv): 0.9 ms of the step faster, but the
// full-size gradient test then fails its 1e-3 bound, so every call site keeps the (hi, lo) pairs
template <int DH, bool XSPLIT = true>
__device__ __forceinline__ void mma_cols(float (&out)[DH / 8][4], const float (&w)[4][4], const uint32_t* tile_x, int g, int t) {
  constexpr int P = DH + 4;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    // the weights as (hi, lo) pairs: sums over a row of dS cancel to zero (that is what makes the gradient of the key
    // bias vanish), which single-TF32 weights would only do to 2^-11
    uint32_t ah[4], al[4];
    split_tf32(__float_as_uint(w[j][0]), ah[0], al[0]);
    split_tf32(__float_as_uint(w[j][2]), ah[1], al[1]);
    split_tf32(__float_as_uint(w[j][1]), ah[2], al[2]);
    split_tf32(__float_as_uint(w[j][3]), ah[3], al[3]);
#pragma unroll
    for (int nd = 0; nd < DH / 8; ++nd) {
      if (XSPLIT) {
        uint32_t bh0, bl0, bh1, bl1;
        split_tf32(tile_x[(j * 8 + 2 * t) * P + nd * 8 + g], bh0, bl0);
        split_tf32(tile_x[(j * 8 + 2 * t + 1) * P + nd * 8 + g], bh1, bl1);
        mma_tf32(out[nd], al, bh0, bh1);
        mma_tf32(out[nd], ah, bl0, bl1);
        mma_tf32(out[nd], ah, bh0, bh1);
      } else {
        const uint32_t b0 = to_tf32(__uint_as_float(tile_x[(j * 8 + 2 * t) * P + nd * 8 + g]));
        const uint32_t b1 = to_tf32(__uint_as_float(tile_x[(j * 8 + 2 * t + 1) * P + nd * 8 + g]));
        mma_tf32(out[nd], al, b0, b1);
        mma_tf32(out[nd], ah, b0, b1);
      }
    }
  }
}

// ---------------------------------------------------------------- forward: out, lse
template <int DH>
__global__ void __launch_bounds__(kThreads)
attn_fwd_mma_kernel(const float* __restrict__ qkv, float* __restrict__ out, float* __restrict__ lse, int T, int H, int D,
                    float qscale, DropoutDesc drop) {
  constexpr int P = DH + 4;
  extern __shared__ uint32_t sm[];
  uint32_t* Qs = sm;                 // [BQ][P]
  uint32_t* KV = Qs + BQ * P;        // [2 buffers][K: BC x P | V: BC x P]
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  const int h = blockIdx.y, b = blockIdx.z, bh = b * H + h;
  const int q0 = blockIdx.x * BQ;
  const float* base = qkv + (long long)b * T * 3 * D + h * DH;
  load_tile_async<DH>(KV, base + D, 3 * D, 0, BC, T);
  load_tile_async<DH>(KV + BC * P, base + 2 * D, 3 * D, 0, BC, T);
  cp_async_commit();
  load_tile<DH>(Qs, base, 3 * D, q0, BQ, T, qscale);
  float o[DH / 8][4];
#pragma unroll
  for (int nd = 0; nd < DH / 8; ++nd) o[nd][0] = o[nd][1] = o[nd][2] = o[nd][3] = 0.f;
  float m[2] = {-INFINITY, -INFINITY}, l[2] = {0.f, 0.f};
  const int rq[2] = {q0 + warp * 16 + g, q0 + warp * 16 + g + 8};
  int buf = 0;
  for (int k0 = 0; k0 < T; k0 += BC, buf ^= 1) {
    const uint32_t* Ks = KV + buf * 2 * BC * P;
    const uint32_t* Vs = Ks + BC * P;
    if (k0 + BC < T) {
      uint32_t* nx = KV + (buf ^ 1) * 2 * BC * P;
      load_tile_async<DH>(nx, base + D, 3 * D, k0 + BC, BC, T);
      load_tile_async<DH>(nx + BC * P, base + 2 * D, 3 * D, k0 + BC, BC, T);
      cp_async_commit();
      cp_async_wait<1>();
    } else {
      cp_async_wait<0>();
    }
    __syncthreads();
    float s[4][4];
#pragma unroll
    for (int nt = 0; nt < 4; ++nt) s[nt][0] = s[nt][1] = s[nt][2] = s[nt][3] = 0.f;
    mma_rows<DH>(s, Qs, warp * 16, Ks, g, t);
    float mx[2] = {m[0], m[1]};
#pragma unroll
    for (int nt = 0; nt < 4; ++nt)
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int key = k0 + nt * 8 + 2 * t + (e & 1);
        if (key >= T) s[nt][e] = -INFINITY;
        mx[e >> 1] = fmaxf(mx[e >> 1], s[nt][e]);
      }
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      mx[r] = fmaxf(mx[r], __shfl_xor_sync(0xffffffffu, mx[r], 1));
      mx[r] = fmaxf(mx[r], __shfl_xor_sync(0xffffffffu, mx[r], 2));
    }
    const float alpha[2] = {expf(m[0] - mx[0]), expf(m[1] - mx[1])};      // exp(-inf) = 0 on the first block
    m[0] = mx[0];
    m[1] = mx[1];
    float rs[2] = {0.f, 0.f};
#pragma unroll
    for (int nt = 0; nt < 4; ++nt) {
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        s[nt][e] = expf(s[nt][e] - mx[e >> 1]);
        rs[e >> 1] += s[nt][e];                    // the softmax denominator sums ALL keys; dropout acts on the weights
      }
      if (drop.kind) {
        const int key = k0 + nt * 8 + 2 * t;
        const float2 k0v = keep_scale2(drop, bh, rq[0], key);
        const float2 k1v = keep_scale2(drop, bh, rq[1], key);
        s[nt][0] *= k0v.x; s[nt][1] *= k0v.y; s[nt][2] *= k1v.x; s[nt][3] *= k1v.y;
      }
    }
    l[0] = l[0] * alpha[0] + rs[0];
    l[1] = l[1] * alpha[1] + rs[1];
#pragma unroll
    for (int nd = 0; nd < DH / 8; ++nd) {
      o[nd][0] *= alpha[0]; o[nd][1] *= alpha[0]; o[nd][2] *= alpha[1]; o[nd][3] *= alpha[1];
    }
    mma_cols<DH>(o, s, Vs, g, t);
    __syncthreads();                 // everyone is done with this buffer before the next iteration's prefetch overwrites it
  }
#pragma unroll
  for (int r = 0; r < 2; ++r) {
    l[r] += __shfl_xor_sync(0xffffffffu, l[r], 1);
    l[r] += __shfl_xor_sync(0xffffffffu, l[r], 2);
  }
#pragma unroll
  for (int r = 0; r < 2; ++r) {
    if (rq[r] >= T) continue;
    const float inv = 1.f / l[r];
    float* dst = out + ((long long)b * T + rq[r]) * D + h * DH;
#pragma unroll
    for (int nd = 0; nd < DH / 8; ++nd)
      *reinterpret_cast<float2*>(dst + nd * 8 + 2 * t) = make_float2(o[nd][2 * r] * inv, o[nd][2 * r + 1] * inv);
    if (t == 0) lse[(long long)bh * T + rq[r]] = m[r] + logf(l[r]);
  }
}

// ---------------------------------------------------------------- backward, dq: one CTA per 64 queries, keys streamed
template <int DH>
__global__ void __launch_bounds__(kThreads)
attn_bwd_q_mma_kernel(const float* __restrict__ qkv, const float* __restrict__ dout, const float* __restrict__ lse,
                      const float* __restrict__ delta, float* __restrict__ dqkv, int T, int H, int D, float qscale,
                      DropoutDesc drop) {
  constexpr int P = DH + 4;
  extern __shared__ uint32_t sm[];
  uint32_t* Qs = sm;                 // [BQ][P] scaled queries
  uint32_t* Gs = Qs + BQ * P;        // [BQ][P] dout rows
  uint32_t* KV = Gs + BQ * P;        // [2 buffers][K: BC x P | V: BC x P]
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  const int h = blockIdx.y, b = blockIdx.z, bh = b * H + h;
  const int q0 = blockIdx.x * BQ;
  const float* base = qkv + (long long)b * T * 3 * D + h * DH;
  load_tile_async<DH>(KV, base + D, 3 * D, 0, BC, T);
  load_tile_async<DH>(KV + BC * P, base + 2 * D, 3 * D, 0, BC, T);
  cp_async_commit();
  load_tile<DH>(Qs, base, 3 * D, q0, BQ, T, qscale);
  load_tile<DH>(Gs, dout + (long long)b * T * D + h * DH, D, q0, BQ, T, 1.f);
  float dq[DH / 8][4];
#pragma unroll
  for (int nd = 0; nd < DH / 8; ++nd) dq[nd][0] = dq[nd][1] = dq[nd][2] = dq[nd][3] = 0.f;
  const int rq[2] = {q0 + warp * 16 + g, q0 + warp * 16 + g + 8};
  float L[2], Dl[2];
#pragma unroll
  for (int r = 0; r < 2; ++r) {
    L[r] = rq[r] < T ? lse[(long long)bh * T + rq[r]] : 0.f;
    Dl[r] = rq[r] < T ? delta[(long long)bh * T + rq[r]] : 0.f;
  }
  int buf = 0;
  for (int k0 = 0; k0 < T; k0 += BC, buf ^= 1) {
    const uint32_t* Ks = KV + buf * 2 * BC * P;
    const uint32_t* Vs = Ks + BC * P;
    if (k0 + BC < T) {
      uint32_t* nx = KV + (buf ^ 1) * 2 * BC * P;
      load_tile_async<DH>(nx, base + D, 3 * D, k0 + BC, BC, T);
      load_tile_async<DH>(nx + BC * P, base + 2 * D, 3 * D, k0 + BC, BC, T);
      cp_async_commit();
      cp_async_wait<1>();
    } else {
      cp_async_wait<0>();
    }
    __syncthreads();
    float s[4][4], dp[4][4];
#pragma unroll
    for (int nt = 0; nt < 4; ++nt)
#pragma unroll
      for (int e = 0; e < 4; ++e) s[nt][e] = dp[nt][e] = 0.f;
    mma_rows<DH>(s, Qs, warp * 16, Ks, g, t);
    mma_rows<DH>(dp, Gs, warp * 16, Vs, g, t);
#pragma unroll
    for (int nt = 0; nt < 4; ++nt) {
      const int key = k0 + nt * 8 + 2 * t;
      float2 kv[2] = {make_float2(1.f, 1.f), make_float2(1.f, 1.f)};
      if (drop.kind) {
        kv[0] = keep_scale2(drop, bh, rq[0], key);
        kv[1] = keep_scale2(drop, bh, rq[1], key);
      }
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int r = e >> 1;
        const float ks = (e & 1) ? kv[r].y : kv[r].x;
        const bool valid = key + (e & 1) < T && rq[r] < T;
        const float p = valid ? expf(s[nt][e] - L[r]) : 0.f;
        s[nt][e] = p * (dp[nt][e] * ks - Dl[r]);             // dS
      }
    }
    mma_cols<DH>(dq, s, Ks, g, t);
    __syncthreads();
  }
#pragma unroll
  for (int r = 0; r < 2; ++r) {
    if (rq[r] >= T) continue;
    float* dst = dqkv + ((long long)b * T + rq[r]) * 3 * D + h * DH;
#pragma unroll
    for (int nd = 0; nd < DH / 8; ++nd)
      *reinterpret_cast<float2*>(dst + nd * 8 + 2 * t) = make_float2(dq[nd][2 * r] * qscale, dq[nd][2 * r + 1] * qscale);
  }
}

// ---------------------------------------------------------------- backward, dk / dv: one CTA per 64 keys, queries streamed
template <int DH>
__global__ void __launch_bounds__(kThreads)
attn_bwd_kv_mma_kernel(const float* __restrict__ qkv, const float* __restrict__ dout, const float* __restrict__ lse,
                       const float* __restrict__ delta, float* __restrict__ dqkv, int T, int H, int D, float qscale,
                       DropoutDesc drop) {
  constexpr int P = DH + 4;
  extern __shared__ uint32_t sm[];
  uint32_t* Ks = sm;                 // [BQ][P] this CTA's keys
  uint32_t* Vs = Ks + BQ * P;        // [BQ][P]
  uint32_t* QG = Vs + BQ * P;        // [2 buffers][Q: BC x P (unscaled) | dout: BC x P] of the streamed query block
  float* LD = reinterpret_cast<float*>(QG + 4 * BC * P);   // [2 buffers][lse: BC | delta: BC]
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  const int h = blockIdx.y, b = blockIdx.z, bh = b * H + h;
  const int kbase = blockIdx.x * BQ;
  const float* base = qkv + (long long)b * T * 3 * D + h * DH;
  const float* gbase = dout + (long long)b * T * D + h * DH;
  auto prefetch = [&](int q0, int bf) {
    load_tile_async<DH>(QG + bf * 2 * BC * P, base, 3 * D, q0, BC, T);
    load_tile_async<DH>(QG + bf * 2 * BC * P + BC * P, gbase, D, q0, BC, T);
    cp_async_commit();
    if (threadIdx.x < BC) {
      const int tq = q0 + threadIdx.x;
      LD[bf * 2 * BC + threadIdx.x] = tq < T ? lse[(long long)bh * T + tq] : 0.f;
      LD[bf * 2 * BC + BC + threadIdx.x] = tq < T ? delta[(long long)bh * T + tq] : 0.f;
    }
  };
  prefetch(0, 0);
  load_tile<DH>(Ks, base + D, 3 * D, kbase, BQ, T, 1.f);
  load_tile<DH>(Vs, base + 2 * D, 3 * D, kbase, BQ, T, 1.f);
  float dk[DH / 8][4], dv[DH / 8][4];
#pragma unroll
  for (int nd = 0; nd < DH / 8; ++nd)
#pragma unroll
    for (int e = 0; e < 4; ++e) dk[nd][e] = dv[nd][e] = 0.f;
  const int rk[2] = {kbase + warp * 16 + g, kbase + warp * 16 + g + 8};
  int buf = 0;
  for (int q0 = 0; q0 < T; q0 += BC, buf ^= 1) {
    const uint32_t* Qs = QG + buf * 2 * BC * P;
    const uint32_t* Gs = Qs + BC * P;
    const float* Ls = LD + buf * 2 * BC;
    const float* Ds = Ls + BC;
    if (q0 + BC < T) {
      prefetch(q0 + BC, buf ^ 1);
      cp_async_wait<1>();
    } else {
      cp_async_wait<0>();
    }
    __syncthreads();
    // transposed tiles: rows = this warp's keys, columns = the block's queries
    float st[4][4], dpt[4][4];
#pragma unroll
    for (int nt = 0; nt < 4; ++nt)
#pragma unroll
      for (int e = 0; e < 4; ++e) st[nt][e] = dpt[nt][e] = 0.f;
    mma_rows<DH>(st, Ks, warp * 16, Qs, g, t);
    mma_rows<DH>(dpt, Vs, warp * 16, Gs, g, t);
#pragma unroll
    for (int nt = 0; nt < 4; ++nt)
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int qc = nt * 8 + 2 * t + (e & 1), tq = q0 + qc, key = rk[e >> 1];
        const bool valid = tq < T && key < T;
        const float p = valid ? expf(st[nt][e] * qscale - Ls[qc]) : 0.f;      // the streamed queries are unscaled
        const float ks = (drop.kind && valid) ? keep_scale(drop, bh, tq, key) : 1.f;
        st[nt][e] = p * ks;                                   // dropped weights P~^T
        dpt[nt][e] = p * (dpt[nt][e] * ks - Ds[qc]);          // dS^T
      }
    mma_cols<DH>(dv, st, Gs, g, t);
    mma_cols<DH>(dk, dpt, Qs, g, t);                          // d s / d k = scale * q: the scale is applied to the sum below
    __syncthreads();
  }
#pragma unroll
  for (int r = 0; r < 2; ++r) {
    if (rk[r] >= T) continue;
    float* dst = dqkv + ((long long)b * T + rk[r]) * 3 * D + h * DH;
#pragma unroll
    for (int nd = 0; nd < DH / 8; ++nd) {
      *reinterpret_cast<float2*>(dst + D + nd * 8 + 2 * t) = make_float2(dk[nd][2 * r] * qscale, dk[nd][2 * r + 1] * qscale);
      *reinterpret_cast<float2*>(dst + 2 * D + nd * 8 + 2 * t) = make_float2(dv[nd][2 * r], dv[nd][2 * r + 1]);
    }
  }
}

// ---------------------------------------------------------------- row terms and the mask (256-thread grid-stride kernels)
// delta[bh, t] = sum_d dout[t, h, d] * out[t, h, d]
__global__ void __launch_bounds__(256)
attn_delta_kernel(const float* __restrict__ out, const float* __restrict__ dout, float* __restrict__ delta, int B, int T, int H,
                  int dh) {
  const int lane = threadIdx.x & 31;
  const long long warps = ((long long)gridDim.x * blockDim.x) >> 5;
  const long long total = (long long)B * H * T;
  const int D = H * dh;
  for (long long w = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5; w < total; w += warps) {
    const long long bh = w / T;
    const int t = int(w - bh * T);
    const long long b = bh / H;
    const int h = int(bh - b * H);
    const long long off = (b * T + t) * D + h * dh;
    float s = 0.f;
    for (int d = lane; d < dh; d += 32) s = fmaf(out[off + d], dout[off + d], s);
    s = warp_sum(s);
    if (lane == 0) delta[w] = s;
  }
}

// mask[bh, i, j] = 1 when the attention kernels keep weight (bh, query i, key j) under `drop` (the parity-test surface)
__global__ void __launch_bounds__(256)
dropout_mask_kernel(DropoutDesc drop, long long n, uint8_t* __restrict__ mask) {
  const long long T = drop.T;
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (long long)gridDim.x * blockDim.x) {
    const long long row = e / T;
    mask[e] = keep_scale(drop, int(row / T), int(row % T), int(e % T)) != 0.f;
  }
}

template <typename K>
int set_smem(K kernel, size_t bytes) {
  IEF_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(bytes)));
  return IEFVAD_OK;
}

}  // namespace

bool attn_train_supported(int dh) { return dh == 32 || dh == 64 || dh == 96 || dh == 128; }

int attn_train_fwd(const float* qkv, int B, int T, int H, int dh, DropoutDesc drop, float* out, float* lse,
                   cudaStream_t stream) {
  if (B == 0 || T == 0) return IEFVAD_OK;
  const dim3 grid((T + BQ - 1) / BQ, H, B);
  const float qs = 1.0f / sqrtf(float(dh));
  drop.T = T;
#define IEF_FWD(DH_)                                                                                                  \
  {                                                                                                                    \
    const size_t smem = size_t(BQ + 4 * BC) * (DH_ + 4) * 4;                                                           \
    static bool set = false;                                                                                           \
    if (!set) { IEF_TRY(set_smem(attn_fwd_mma_kernel<DH_>, smem)); set = true; }                                       \
    attn_fwd_mma_kernel<DH_><<<grid, kThreads, smem, stream>>>(qkv, out, lse, T, H, H * dh, qs, drop);         \
  }
  switch (dh) {
    case 32: IEF_FWD(32) break;
    case 64: IEF_FWD(64) break;
    case 96: IEF_FWD(96) break;
    case 128: IEF_FWD(128) break;
    default: set_error("attn_train: head dim %d unsupported (32, 64, 96, 128)", dh); return IEFVAD_ERR_INVALID;
  }
#undef IEF_FWD
  count_launches(1);
  IEF_CUDA(cudaGetLastError());
  return IEFVAD_OK;
}

int attn_train_bwd(const float* qkv, const float* out, const float* dout, const float* lse, int B, int T, int H, int dh,
                   DropoutDesc drop, float* delta_scratch, float* dqkv, int num_sms, cudaStream_t stream) {
  if (B == 0 || T == 0) return IEFVAD_OK;
  const dim3 grid((T + BQ - 1) / BQ, H, B);
  const int delta_grid = blocks_for((long long)B * H * T * 32, num_sms);
  const float qs = 1.0f / sqrtf(float(dh));
  drop.T = T;
#define IEF_BWD(DH_)                                                                                                            \
  {                                                                                                                              \
    const size_t smem = size_t(2 * BQ + 4 * BC) * (DH_ + 4) * 4 + 4 * BC * 4;                                                    \
    static bool set = false;                                                                                                     \
    if (!set) {                                                                                                                  \
      IEF_TRY(set_smem(attn_bwd_q_mma_kernel<DH_>, smem));                                                                       \
      IEF_TRY(set_smem(attn_bwd_kv_mma_kernel<DH_>, smem));                                                                      \
      set = true;                                                                                                                \
    }                                                                                                                            \
    attn_delta_kernel<<<delta_grid, 256, 0, stream>>>(out, dout, delta_scratch, B, T, H, dh);                                    \
    attn_bwd_q_mma_kernel<DH_><<<grid, kThreads, smem, stream>>>(qkv, dout, lse, delta_scratch, dqkv, T, H, H * dh, qs, drop);   \
    attn_bwd_kv_mma_kernel<DH_><<<grid, kThreads, smem, stream>>>(qkv, dout, lse, delta_scratch, dqkv, T, H, H * dh, qs, drop);  \
  }
  switch (dh) {
    case 32: IEF_BWD(32) break;
    case 64: IEF_BWD(64) break;
    case 96: IEF_BWD(96) break;
    case 128: IEF_BWD(128) break;
    default: set_error("attn_train: head dim %d unsupported (32, 64, 96, 128)", dh); return IEFVAD_ERR_INVALID;
  }
#undef IEF_BWD
  count_launches(3);
  IEF_CUDA(cudaGetLastError());
  return IEFVAD_OK;
}

int dropout_mask(DropoutDesc drop, int B, int H, int T, uint8_t* mask, cudaStream_t stream) {
  const long long n = (long long)B * H * T * T;
  if (n == 0) return IEFVAD_OK;
  int sms = 0;
  IEF_TRY(device_sms(&sms));
  drop.T = T;
  dropout_mask_kernel<<<blocks_for(n, sms), 256, 0, stream>>>(drop, n, mask);
  count_launches(1);
  IEF_CUDA(cudaGetLastError());
  return IEFVAD_OK;
}

}  // namespace iefvad
