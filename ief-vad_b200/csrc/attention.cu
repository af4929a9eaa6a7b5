// Self-attention core of nn.MultiheadAttention as the reference uses it (model/imf_vad.py:115,121:
// no mask, keys = all T rows of the batch element including zero pads; q pre-scaled by d_h^-1/2,
// torch/nn/functional.py:6632) - softmax(Q K^T) V without ever materialising the [B,H,T,T] scores.
//
// attn_tc : tcgen05 flash-style kernel.  One CTA = 128 query rows of one (batch, head); key blocks of 64
//           stream through a 2-stage TMA ring; S = Q.K^T lands in one of two 64-column TMEM buffers, the
//           four softmax warps (thread == query row, so row max / sum need no shuffles) turn it into bf16 P in
//           128B-swizzled smem, P.V^T-major accumulates a per-block O in TMEM which the same threads fold into
//           fp32 registers with the online-softmax rescale.  Optional additive mask / key-padding mask serve
//           the model/module.py block (D4).
// attn_simt : fp32 reference plan (one warp per query row), same math in IEEE fp32.
#include "attention.cuh"
#include "common.cuh"
#include "tensormap.cuh"

namespace iefvad {

namespace {

constexpr int QB = 128;   // query rows per CTA
// Keys per block.  64 rather than 128 halves every per-CTA resource (104 KB smem, 256 TMEM columns) so that TWO CTAs
// share an SM and one CTA's softmax overlaps the other's MMAs / loads (T_c = 256 has only two 128-key blocks to
// pipeline within a CTA); two CTAs per SM measured faster at every T (7.75 vs 7.95 ms on config 5).
constexpr int KB = 64;
constexpr float kLog2e = 1.4426950408889634f;

// 2^x on the SFU in one instruction (ex2.approx.ftz: 2 ulp, flushes denormal results - they vanish in the 16-bit P)
__device__ __forceinline__ float fast_exp2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

template <int DH, int DHP>
struct AttnCfg {
  static constexpr uint32_t kQBytes = QB * DHP * 2;
  static constexpr uint32_t kKBytes = KB * DHP * 2;
  static constexpr uint32_t kVSub = DH * 128;            // one [DH x 64 keys] sub-tile
  static constexpr uint32_t kVBytes = (KB / 64) * kVSub;
  static constexpr uint32_t kPBytes = QB * KB * 2;
  static constexpr uint32_t kOffK = kQBytes;
  static constexpr uint32_t kOffV = kOffK + 2 * kKBytes;
  static constexpr uint32_t kOffP = kOffV + 2 * kVBytes;
  static constexpr uint32_t kOffBar = kOffP + kPBytes;
  static constexpr size_t kSmemBytes = 1024 + kOffBar + 256;
  static constexpr uint32_t kOffO = 2 * KB;              // TMEM: S0 [0,KB) S1 [KB,2KB) O [2KB, 2KB+DH)
  static constexpr uint32_t kTmemCols = 256;
  static_assert(kOffO + DH <= kTmemCols, "S0, S1 and O fit the TMEM allocation");
};

template <int DH, int DHP>
__global__ void __launch_bounds__(192, 2)
attn_tc_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmK,
               const __grid_constant__ CUtensorMap tmVt, bf16* __restrict__ out, int ldo, int T, int H,
               const float* __restrict__ attn_mask /* [T,T] additive or null */,
               const uint8_t* __restrict__ key_pad /* [B,T] 1 = ignore, or null */, int fp16,
               const int* __restrict__ row_out) {
  using Cfg = AttnCfg<DH, DHP>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + Cfg::kOffBar);
  uint64_t* q_full = bars + 0;
  uint64_t* k_full = bars + 1;    // [2]
  uint64_t* v_full = bars + 3;    // [2]
  uint64_t* kv_empty = bars + 5;  // [2]
  uint64_t* s_full = bars + 7;    // [2]
  uint64_t* s_empty = bars + 9;   // [2]
  uint64_t* p_full = bars + 11;
  uint64_t* o_full = bars + 12;
  uint64_t* o_empty = bars + 13;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 14);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int qt = blockIdx.x, h = blockIdx.y, b = blockIdx.z;
  const int bh = b * H + h;
  const int nb = (T + KB - 1) / KB;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmQ);
    tma_prefetch_desc(&tmK);
    tma_prefetch_desc(&tmVt);
    mbar_init(q_full, 1);
    for (int s = 0; s < 2; ++s) {
      mbar_init(&k_full[s], 1);
      mbar_init(&v_full[s], 1);
      mbar_init(&kv_empty[s], 1);
      mbar_init(&s_full[s], 1);
      mbar_init(&s_empty[s], 128);
    }
    mbar_init(p_full, 128);
    mbar_init(o_full, 1);
    mbar_init(o_empty, 128);
    fence_barrier_init();
  }
  if (warp == 1) {
    tmem_alloc(tmem_slot, Cfg::kTmemCols);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      mbar_arrive_expect_tx(q_full, Cfg::kQBytes);
#pragma unroll
      for (int c = 0; c < DHP / 64; ++c) tma_load_3d(&tmQ, q_full, smem + c * (QB * 128), c * 64, qt * QB, bh);
      for (int j = 0; j < nb; ++j) {
        const int s = j & 1;
        mbar_wait(&kv_empty[s], ((j >> 1) & 1) ^ 1);
        uint8_t* sk = smem + Cfg::kOffK + s * Cfg::kKBytes;
        uint8_t* sv = smem + Cfg::kOffV + s * Cfg::kVBytes;
        mbar_arrive_expect_tx(&k_full[s], Cfg::kKBytes);
#pragma unroll
        for (int c = 0; c < DHP / 64; ++c) tma_load_3d(&tmK, &k_full[s], sk + c * (KB * 128), c * 64, j * KB, bh);
        mbar_arrive_expect_tx(&v_full[s], Cfg::kVBytes);
#pragma unroll
        for (int c = 0; c < KB / 64; ++c) tma_load_3d(&tmVt, &v_full[s], sv + c * Cfg::kVSub, j * KB + c * 64, 0, bh);
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    if (lane == 0) {
      const uint32_t idesc_s = fp16 ? make_idesc_f16(QB, KB) : make_idesc_bf16(QB, KB);
      const uint32_t idesc_o = fp16 ? make_idesc_f16(QB, DH) : make_idesc_bf16(QB, DH);
      const uint32_t sq = smem_u32(smem);
      auto issue_s = [&](int j) {
        const int s = j & 1;
        const uint32_t par = (j >> 1) & 1;
        mbar_wait(&k_full[s], par);
        mbar_wait(&s_empty[s], par ^ 1);
        tc_fence_after();
        const uint32_t sk = smem_u32(smem + Cfg::kOffK + s * Cfg::kKBytes);
        const uint32_t d = tmem_base + uint32_t(s * KB);
#pragma unroll
        for (int kk = 0; kk < DH / 16; ++kk) {   // only the DH real columns of the DHP-padded rows
          const int c = kk >> 2, k4 = kk & 3;
          umma_bf16(d, make_smem_desc_sw128(sq + c * (QB * 128)) + uint64_t(2 * k4),
                    make_smem_desc_sw128(sk + c * (KB * 128)) + uint64_t(2 * k4), idesc_s, kk != 0 ? 1u : 0u);
        }
        tc_commit(&s_full[s]);
      };
      mbar_wait(q_full, 0);
      issue_s(0);
      for (int j = 0; j < nb; ++j) {
        if (j + 1 < nb) issue_s(j + 1);
        const int s = j & 1;
        mbar_wait(p_full, j & 1);
        mbar_wait(&v_full[s], (j >> 1) & 1);
        mbar_wait(o_empty, (j & 1) ^ 1);
        tc_fence_after();
        const uint32_t sp = smem_u32(smem + Cfg::kOffP);
        const uint32_t sv = smem_u32(smem + Cfg::kOffV + s * Cfg::kVBytes);
        const uint32_t d = tmem_base + Cfg::kOffO;
#pragma unroll
        for (int kk = 0; kk < KB / 16; ++kk) {
          const int c = kk >> 2, k4 = kk & 3;
          umma_bf16(d, make_smem_desc_sw128(sp + c * (QB * 128)) + uint64_t(2 * k4),
                    make_smem_desc_sw128(sv + c * Cfg::kVSub) + uint64_t(2 * k4), idesc_o, kk != 0 ? 1u : 0u);
        }
        tc_commit(o_full);
        tc_commit(&kv_empty[s]);
      }
    }
  } else {
    // ===================== softmax / accumulate / store (warps 2..5) =====================
    const int quarter = warp & 3;
    const int r = quarter * 32 + lane;             // query row inside the tile == TMEM lane
    const int tq = qt * QB + r;
    const uint32_t lane_off = uint32_t(quarter * 32) << 16;
    float m = -INFINITY, l = 0.f;
    float alpha_prev = 0.f;       // rescale factor of the previous block: applied when that block's P.V is folded in
    float o_acc[DH];
#pragma unroll
    for (int d = 0; d < DH; ++d) o_acc[d] = 0.f;
    const bool masked = (attn_mask != nullptr) || (key_pad != nullptr);
    const float* mrow = attn_mask ? attn_mask + (long long)(tq < T ? tq : T - 1) * T : nullptr;
    const uint8_t* prow = key_pad ? key_pad + (long long)b * T : nullptr;

    for (int j = 0; j < nb; ++j) {
      const int s = j & 1;
      mbar_wait(&s_full[s], (j >> 1) & 1);
      tc_fence_after();
      const uint32_t ts = tmem_base + uint32_t(s * KB) + lane_off;
      const int key0 = j * KB;
      const bool tail = masked || (key0 + KB > T);
      // ---- pass 1: running max
      float mx = m;
#pragma unroll 1
      for (int c = 0; c < KB / 32; ++c) {
        float v[32];
        tmem_ld32(ts + uint32_t(c * 32), v);
        tmem_ld_wait();
        if (tail) {
#pragma unroll
          for (int i = 0; i < 32; ++i) {
            const int key = key0 + c * 32 + i;
            float x = v[i];
            if (key >= T) x = -INFINITY;
            else {
              if (mrow) x += mrow[key];
              if (prow && prow[key]) x = -INFINITY;
            }
            mx = fmaxf(mx, x);
          }
        } else {
#pragma unroll
          for (int i = 0; i < 32; ++i) mx = fmaxf(mx, v[i]);
        }
      }
      // ---- fold the previous block's P.V into the register accumulator (also frees P smem).  The accumulator is
      // kept relative to the max BEFORE the previous block; one FFMA per element rescales it and adds the block.
      if (j > 0) {
        mbar_wait(o_full, (j - 1) & 1);
        tc_fence_after();
#pragma unroll
        for (int c = 0; c < DH / 32; ++c) {
          float v[32];
          tmem_ld32(tmem_base + Cfg::kOffO + lane_off + uint32_t(c * 32), v);
          tmem_ld_wait();
#pragma unroll
          for (int i = 0; i < 32; ++i) o_acc[c * 32 + i] = fmaf(o_acc[c * 32 + i], alpha_prev, v[i]);
        }
        tc_fence_before();
        mbar_arrive(o_empty);
      }
      // a fully masked prefix keeps mx == -inf: use 0 as the reference point so exp2 stays finite
      const float mref = (mx == -INFINITY) ? 0.f : mx;
      const float alpha = fast_exp2((m - mref) * kLog2e);   // m == -inf -> 0
      m = mx;
      l *= alpha;
      alpha_prev = alpha;
      // ---- pass 2: P = exp(S - m) -> 16-bit, swizzled K-major smem (A operand of P.V)
      const float mscaled = mref * kLog2e;
      float lsum = 0.f;
#pragma unroll 1
      for (int c = 0; c < KB / 32; ++c) {
        float v[32];
        tmem_ld32(ts + uint32_t(c * 32), v);
        tmem_ld_wait();
#pragma unroll
        for (int i = 0; i < 32; ++i) {
          float x = v[i];
          if (tail) {
            const int key = key0 + c * 32 + i;
            if (key >= T) x = -INFINITY;
            else {
              if (mrow) x += mrow[key];
              if (prow && prow[key]) x = -INFINITY;
            }
          }
          const float p = fast_exp2(fmaf(x, kLog2e, -mscaled));
          lsum += p;
          v[i] = p;
        }
        uint8_t* ptile = smem + Cfg::kOffP + (c >> 1) * (QB * 128) + r * 128;
#pragma unroll
        for (int g = 0; g < 4; ++g) {
          const int chunk = ((c & 1) * 4 + g) ^ (r & 7);
          *reinterpret_cast<uint4*>(ptile + chunk * 16) = pack_16x8(v + g * 8, fp16);
        }
      }
      l += lsum;
      tc_fence_before();
      fence_proxy_async_smem();     // generic-proxy smem writes -> visible to the tensor-core (async) proxy
      mbar_arrive(&s_empty[s]);
      mbar_arrive(p_full);
    }
    // ---- last block's P.V
    mbar_wait(o_full, (nb - 1) & 1);
    tc_fence_after();
#pragma unroll
    for (int c = 0; c < DH / 32; ++c) {
      float v[32];
      tmem_ld32(tmem_base + Cfg::kOffO + lane_off + uint32_t(c * 32), v);
      tmem_ld_wait();
#pragma unroll
      for (int i = 0; i < 32; ++i) o_acc[c * 32 + i] = fmaf(o_acc[c * 32 + i], alpha_prev, v[i]);
    }
    long long ro = (long long)b * T + (tq < T ? tq : 0);
    if (row_out) ro = __ldg(row_out + ro);
    if (tq < T && ro >= 0) {
      const float inv = 1.f / l;
      bf16* dst = out + ro * ldo + h * DH;
#pragma unroll
      for (int d = 0; d < DH; d += 8) *reinterpret_cast<uint4*>(dst + d) = pack_16x8(o_acc + d, fp16, inv);
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, Cfg::kTmemCols);
  }
}

template <int DH, int DHP>
int launch_attn_tc(const AttnTcArgs& a, cudaStream_t stream) {
  using Cfg = AttnCfg<DH, DHP>;
  static bool attr_set = false;
  if (!attr_set) {
    IEF_CUDA(cudaFuncSetAttribute(attn_tc_kernel<DH, DHP>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  static_cast<int>(Cfg::kSmemBytes)));
    attr_set = true;
  }
  const uint64_t BH = uint64_t(a.B) * a.H;
  CUtensorMap tq, tk, tv;
  IEF_TRY(make_tmap_3d(&tq, a.q, DHP, a.T, BH, uint64_t(DHP) * 2, uint64_t(a.T) * DHP * 2, 64, QB, 1));
  IEF_TRY(make_tmap_3d(&tk, a.k, DHP, a.T, BH, uint64_t(DHP) * 2, uint64_t(a.T) * DHP * 2, 64, KB, 1));
  IEF_TRY(make_tmap_3d(&tv, a.vt, a.T, DH, BH, uint64_t(a.Tpad) * 2, uint64_t(DH) * a.Tpad * 2, 64, DH, 1));
  dim3 grid((a.T + QB - 1) / QB, a.H, a.B);
  attn_tc_kernel<DH, DHP><<<grid, 192, Cfg::kSmemBytes, stream>>>(tq, tk, tv, a.out, a.ldo, a.T, a.H, a.attn_mask,
                                                              a.key_pad, a.fp16, a.row_out);
  count_launches(1);
  IEF_CUDA(cudaGetLastError());
  return IEFVAD_OK;
}

// ------------------------------------------------------------------------------------------------
// fp32 SIMT plan: qkv fp32 [M, 3D] (bias already added, q NOT yet scaled), one warp per query row.
// ------------------------------------------------------------------------------------------------
constexpr int SROWS = 16;  // query rows per block (4 warps x 4 rows)

template <int DH>
__global__ void __launch_bounds__(128)
attn_simt_kernel(const float* __restrict__ qkv, float* __restrict__ out, int T, int H, int D, float qscale,
                 const float* __restrict__ attn_mask, const uint8_t* __restrict__ key_pad) {
  constexpr int NPL = DH / 32;  // output dims per lane
  __shared__ float Ks[32][DH + 1];
  __shared__ float Vs[32][DH];
  __shared__ float Qs[SROWS][DH];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int h = blockIdx.y, b = blockIdx.z;
  const int q0 = blockIdx.x * SROWS;
  const long long base = (long long)b * T;
  for (int i = threadIdx.x; i < SROWS * DH; i += 128) {
    const int rr = i / DH, d = i - rr * DH;
    const int t = q0 + rr;
    Qs[rr][d] = (t < T) ? qkv[(base + t) * 3 * D + h * DH + d] * qscale : 0.f;
  }
  float m[4], l[4], o[4][NPL];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    m[i] = -INFINITY;
    l[i] = 0.f;
#pragma unroll
    for (int e = 0; e < NPL; ++e) o[i][e] = 0.f;
  }
  for (int k0 = 0; k0 < T; k0 += 32) {
    __syncthreads();
    for (int i = threadIdx.x; i < 32 * DH; i += 128) {
      const int kr = i / DH, d = i - kr * DH;
      const int t = k0 + kr;
      Ks[kr][d] = (t < T) ? qkv[(base + t) * 3 * D + D + h * DH + d] : 0.f;
      Vs[kr][d] = (t < T) ? qkv[(base + t) * 3 * D + 2 * D + h * DH + d] : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int rr = warp * 4 + i;
      const int tq = q0 + rr;
      float s = 0.f;
#pragma unroll 8
      for (int d = 0; d < DH; ++d) s = fmaf(Qs[rr][d], Ks[lane][d], s);
      const int key = k0 + lane;
      if (key >= T) s = -INFINITY;
      else {
        if (attn_mask && tq < T) s += attn_mask[(long long)tq * T + key];
        if (key_pad && key_pad[base + key]) s = -INFINITY;
      }
      const float mx = fmaxf(m[i], warp_max(s));
      const float mref = (mx == -INFINITY) ? 0.f : mx;
      const float alpha = expf(m[i] - mref);
      const float p = expf(s - mref);
      l[i] = l[i] * alpha + warp_sum(p);
      m[i] = mx;
#pragma unroll
      for (int e = 0; e < NPL; ++e) o[i][e] *= alpha;
      for (int jj = 0; jj < 32; ++jj) {
        const float pj = __shfl_sync(0xffffffffu, p, jj);
#pragma unroll
        for (int e = 0; e < NPL; ++e) o[i][e] = fmaf(pj, Vs[jj][lane + 32 * e], o[i][e]);
      }
    }
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int tq = q0 + warp * 4 + i;
    if (tq < T) {
#pragma unroll
      for (int e = 0; e < NPL; ++e) out[(base + tq) * D + h * DH + lane + 32 * e] = o[i][e] / l[i];
    }
  }
}

}  // namespace

int attn_qk_cols(const AttnTcArgs& a) {
  return (attn_short_supported(a) && a.dh % 32 == 0) ? a.dh : (a.dh + 63) / 64 * 64;
}

int attn_tc(const AttnTcArgs& a, cudaStream_t stream) {
  IEF_CHECK(a.B > 0 && a.T > 0 && a.H > 0, "attn_tc: empty problem");
  IEF_CHECK(a.Tpad % 8 == 0 && a.Tpad >= a.T, "attn_tc: Tpad=%d must be a multiple of 8 and >= T=%d", a.Tpad, a.T);
  IEF_CHECK(a.ldo % 8 == 0, "attn_tc: ldo must be a multiple of 8");
  if (attn_short_supported(a)) return attn_short(a, stream);
  if (attn_long_supported(a)) return attn_long(a, stream);
  IEF_CHECK(a.B <= 65535 && a.H <= 65535, "attn_tc: B=%d / H=%d exceed the grid limits", a.B, a.H);
#define IEF_ATTN(DH_, DHP_) \
  if (a.dh == DH_ && a.dhp == DHP_) return launch_attn_tc<DH_, DHP_>(a, stream);
  IEF_ATTN(96, 128)
  IEF_ATTN(64, 64)
  IEF_ATTN(128, 128)
  IEF_ATTN(32, 64)
#undef IEF_ATTN
  set_error("attn_tc: unsupported head dim %d (padded %d); supported: 32, 64, 96, 128", a.dh, a.dhp);
  return IEFVAD_ERR_INVALID;
}

int attn_simt(const float* qkv, float* out, int B, int T, int H, int dh, const float* attn_mask,
              const uint8_t* key_pad, cudaStream_t stream) {
  IEF_CHECK(B > 0 && T > 0 && H > 0, "attn_simt: empty problem");
  IEF_CHECK(B <= 65535 && H <= 65535, "attn_simt: B/H exceed the grid limits");
  const int D = H * dh;
  const float qscale = 1.0f / sqrtf(static_cast<float>(dh));
  dim3 grid((T + SROWS - 1) / SROWS, H, B);
  switch (dh) {
    case 32: attn_simt_kernel<32><<<grid, 128, 0, stream>>>(qkv, out, T, H, D, qscale, attn_mask, key_pad); break;
    case 64: attn_simt_kernel<64><<<grid, 128, 0, stream>>>(qkv, out, T, H, D, qscale, attn_mask, key_pad); break;
    case 96: attn_simt_kernel<96><<<grid, 128, 0, stream>>>(qkv, out, T, H, D, qscale, attn_mask, key_pad); break;
    case 128: attn_simt_kernel<128><<<grid, 128, 0, stream>>>(qkv, out, T, H, D, qscale, attn_mask, key_pad); break;
    default: set_error("attn_simt: unsupported head dim %d", dh); return IEFVAD_ERR_INVALID;
  }
  count_launches(1);
  IEF_CUDA(cudaGetLastError());
  return IEFVAD_OK;
}

}  // namespace iefvad
