// HBM-bound kernels of the forward: input ingest, LayerNorm (single / double), the uncertainty-weighted
// fusion (model/imf_vad.py:130-144) and the 768->1 classifier (model/imf_vad.py:150).  All fp32 IEEE
// arithmetic (no fast-math), 128-bit global accesses, grids sized in multiples of the SM count.
#include "common.cuh"
#include "elementwise.cuh"

namespace iefvad {

namespace {

constexpr int kThreads = 256;

__host__ int grid_for(long long work_items, int num_sms, int per_sm = 8) {
  long long blocks = (work_items + kThreads - 1) / kThreads;
  long long cap = (long long)num_sms * per_sm;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  return static_cast<int>(blocks);
}

// ---------------------------------------------------------------- ingest: any float dtype -> fp32 (+bf16 hi)
template <typename Tin>
__device__ __forceinline__ void load8(const Tin* p, float* v);
template <>
__device__ __forceinline__ void load8<float>(const float* p, float* v) {
  const float4 a = __ldcs(reinterpret_cast<const float4*>(p));
  const float4 b = __ldcs(reinterpret_cast<const float4*>(p) + 1);
  v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
}
template <>
__device__ __forceinline__ void load8<__half>(const __half* p, float* v) {
  const uint4 u = __ldcs(reinterpret_cast<const uint4*>(p));
  const __half2* h = reinterpret_cast<const __half2*>(&u);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float2 f = __half22float2(h[i]);
    v[2 * i] = f.x; v[2 * i + 1] = f.y;
  }
}
template <>
__device__ __forceinline__ void load8<bf16>(const bf16* p, float* v) {
  const uint4 u = __ldcs(reinterpret_cast<const uint4*>(p));
  const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&u);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float2 f = __bfloat1622float2(h[i]);
    v[2 * i] = f.x; v[2 * i + 1] = f.y;
  }
}

template <typename Tin>
__global__ void __launch_bounds__(kThreads)
ingest_kernel(const Tin* __restrict__ in, long long n8, float* __restrict__ out_f32, bf16* __restrict__ out_hi,
              bf16* __restrict__ out_lo, int hi_fp16) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n8; i += (long long)gridDim.x * blockDim.x) {
    float v[8];
    load8<Tin>(in + i * 8, v);
    if (out_f32) {
      float4* o = reinterpret_cast<float4*>(out_f32 + i * 8);
      o[0] = make_float4(v[0], v[1], v[2], v[3]);
      o[1] = make_float4(v[4], v[5], v[6], v[7]);
    }
    uint32_t hi[4], lo[4];                    // fp16: exact for fp16 inputs, the remainder is zero then
#pragma unroll
    for (int q = 0; q < 4; ++q) split_16x2(v[2 * q], v[2 * q + 1], hi_fp16, hi[q], lo[q]);
    if (out_hi) *reinterpret_cast<uint4*>(out_hi + i * 8) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
    if (out_lo) *reinterpret_cast<uint4*>(out_lo + i * 8) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
  }
}

// ragged ingest: row (c, t) of the zero-padded [n_chunks, T, D] batch comes from packed[chunk_start[c] - base + t] when
// t < chunk_valid[c] and is zero otherwise - process_split (data/tools.py:100-114) folded into the ingest, so the
// pad rows never cross PCIe nor get read from HBM
template <typename Tin>
__global__ void __launch_bounds__(kThreads)
ingest_ragged_kernel(const Tin* __restrict__ packed, const long long* __restrict__ chunk_start, long long start_base,
                     const int* __restrict__ chunk_valid, long long n8, int T, int D8, float* __restrict__ out_f32,
                     bf16* __restrict__ out_hi, int hi_fp16) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n8; i += (long long)gridDim.x * blockDim.x) {
    const long long row = i / D8;
    const int col8 = int(i - row * D8);
    const long long c = row / T;
    const int t = int(row - c * T);
    float v[8];
    if (t < chunk_valid[c]) {
      load8<Tin>(packed + ((chunk_start[c] - start_base + t) * D8 + col8) * 8, v);
    } else {
#pragma unroll
      for (int e = 0; e < 8; ++e) v[e] = 0.f;
    }
    if (out_f32) {
      float4* o = reinterpret_cast<float4*>(out_f32 + i * 8);
      o[0] = make_float4(v[0], v[1], v[2], v[3]);
      o[1] = make_float4(v[4], v[5], v[6], v[7]);
    }
    if (out_hi) *reinterpret_cast<uint4*>(out_hi + i * 8) = pack_16x8(v, hi_fp16);
  }
}

// four consecutive values -> their 16-bit pairs at hi[off, off + 4) and (when lo != null) lo[off, off + 4)
__device__ __forceinline__ void store_split4(const float* v, int f16, bf16* hi, bf16* lo, long long off) {
  uint2 h, l;
  split_16x2(v[0], v[1], f16, h.x, l.x);
  split_16x2(v[2], v[3], f16, h.y, l.y);
  *reinterpret_cast<uint2*>(hi + off) = h;
  if (lo) *reinterpret_cast<uint2*>(lo + off) = l;
}

// ---------------------------------------------------------------- LayerNorm: one warp per row, row in registers
template <int NV>   // D = 128 * NV
__global__ void __launch_bounds__(kThreads)
layernorm_kernel(const float* __restrict__ x, long long M, const float* __restrict__ w1, const float* __restrict__ b1,
                 const float* __restrict__ w2, const float* __restrict__ b2, float eps, float* __restrict__ out_f32,
                 bf16* __restrict__ out_hi, bf16* __restrict__ out_lo, int hi_fp16,
                 const int* __restrict__ f32_row_out) {
  constexpr int D = 128 * NV;
  const int lane = threadIdx.x & 31;
  const long long warps = ((long long)gridDim.x * blockDim.x) >> 5;
  for (long long row = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5; row < M; row += warps) {
    float v[NV * 4];
    const float4* xr = reinterpret_cast<const float4*>(x + row * D);
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const float4 t = xr[lane + 32 * i];
      v[4 * i] = t.x; v[4 * i + 1] = t.y; v[4 * i + 2] = t.z; v[4 * i + 3] = t.w;
    }
#pragma unroll
    for (int pass = 0; pass < 2; ++pass) {
      const float* w = pass ? w2 : w1;
      const float* b = pass ? b2 : b1;
      if (w == nullptr) break;
      float s = 0.f;
#pragma unroll
      for (int i = 0; i < NV * 4; ++i) s += v[i];
      const float mean = warp_sum(s) * (1.f / D);
      float q = 0.f;
#pragma unroll
      for (int i = 0; i < NV * 4; ++i) {
        const float c = v[i] - mean;
        q = fmaf(c, c, q);
      }
      const float rstd = 1.f / sqrtf(warp_sum(q) * (1.f / D) + eps);
#pragma unroll
      for (int i = 0; i < NV; ++i) {
        const float4 wv = __ldg(reinterpret_cast<const float4*>(w) + lane + 32 * i);
        const float4 bv = __ldg(reinterpret_cast<const float4*>(b) + lane + 32 * i);
        v[4 * i + 0] = (v[4 * i + 0] - mean) * rstd * wv.x + bv.x;
        v[4 * i + 1] = (v[4 * i + 1] - mean) * rstd * wv.y + bv.y;
        v[4 * i + 2] = (v[4 * i + 2] - mean) * rstd * wv.z + bv.z;
        v[4 * i + 3] = (v[4 * i + 3] - mean) * rstd * wv.w + bv.w;
      }
    }
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const long long off = row * D + (lane + 32 * i) * 4;
      if (out_f32) {
        // the fp32 copy may go to a compact row (or nowhere): only rows that survive the valid-row cut need it
        const long long ro = f32_row_out ? (long long)__ldg(f32_row_out + row) : row;
        if (ro >= 0)
          *reinterpret_cast<float4*>(out_f32 + ro * D + (lane + 32 * i) * 4) =
              make_float4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
      }
      if (out_hi) store_split4(v + 4 * i, hi_fp16, out_hi, out_lo, off);
    }
  }
}

// ---------------------------------------------------------------- uncertainty-weighted fusion
__global__ void __launch_bounds__(kThreads)
fuse_kernel(const float4* __restrict__ mu_i, const float4* __restrict__ mu_e, const float4* __restrict__ lv_i,
            const float4* __restrict__ lv_e, long long n4, float factor, float eps, float4* __restrict__ w_i,
            float4* __restrict__ w_e, float4* __restrict__ fused, bf16* __restrict__ fused_hi,
            bf16* __restrict__ fused_lo, int hi_fp16) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
    const float4 a = __ldcs(mu_i + i), b = __ldcs(mu_e + i), c = __ldcs(lv_i + i), d = __ldcs(lv_e + i);
    const float mi[4] = {a.x, a.y, a.z, a.w}, me[4] = {b.x, b.y, b.z, b.w};
    const float li[4] = {c.x, c.y, c.z, c.w}, le[4] = {d.x, d.y, d.z, d.w};
    float wi[4], we[4], f[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) f[e] = fuse_one(mi[e], me[e], li[e], le[e], factor, eps, wi[e], we[e]);
    if (w_i) {                                  // the evaluation forward does not return the fusion weights
      __stcs(w_i + i, make_float4(wi[0], wi[1], wi[2], wi[3]));
      __stcs(w_e + i, make_float4(we[0], we[1], we[2], we[3]));
    }
    if (fused) fused[i] = make_float4(f[0], f[1], f[2], f[3]);
    if (fused_hi) store_split4(f, hi_fp16, fused_hi, fused_lo, i * 4);   // operand pair of the refinement chain
  }
}

// The same fusion with one warp per row, which also reduces w_i / w_e over the row: the evaluation loop of the reference
// keeps only w_i.mean(-1) and w_e.mean(-1) per frame (train/ucf_test.py:124-131) - 8 bytes per row instead of 6 KB.
__global__ void __launch_bounds__(kThreads)
fuse_rows_kernel(const float4* __restrict__ mu_i, const float4* __restrict__ mu_e, const float4* __restrict__ lv_i,
                 const float4* __restrict__ lv_e, long long rows, int D4, float factor, float eps, float inv_d,
                 float* __restrict__ wi_mean, float* __restrict__ we_mean, float4* __restrict__ fused,
                 bf16* __restrict__ fused_hi, bf16* __restrict__ fused_lo, int hi_fp16) {
  const int lane = threadIdx.x & 31;
  const long long warps = ((long long)gridDim.x * blockDim.x) >> 5;
  for (long long row = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5; row < rows; row += warps) {
    float si = 0.f, se = 0.f;
    for (int c = lane; c < D4; c += 32) {
      const long long i = row * D4 + c;
      const float4 a = __ldcs(mu_i + i), b = __ldcs(mu_e + i), cc = __ldcs(lv_i + i), d = __ldcs(lv_e + i);
      const float mi[4] = {a.x, a.y, a.z, a.w}, me[4] = {b.x, b.y, b.z, b.w};
      const float li[4] = {cc.x, cc.y, cc.z, cc.w}, le[4] = {d.x, d.y, d.z, d.w};
      float f[4];
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        float wi, we;
        f[e] = fuse_one(mi[e], me[e], li[e], le[e], factor, eps, wi, we);
        si += wi;
        se += we;
      }
      if (fused) fused[i] = make_float4(f[0], f[1], f[2], f[3]);
      if (fused_hi) store_split4(f, hi_fp16, fused_hi, fused_lo, i * 4);
    }
    si = warp_sum(si);
    se = warp_sum(se);
    if (lane == 0) {
      wi_mean[row] = si * inv_d;
      we_mean[row] = se * inv_d;
    }
  }
}

__global__ void __launch_bounds__(kThreads)
inverse_rowmap_kernel(const int* __restrict__ rowmap, long long row_base, long long n_rows, int* __restrict__ inv) {
  for (long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x; j < n_rows; j += (long long)gridDim.x * blockDim.x)
    inv[(long long)rowmap[j] - row_base] = int(j);
}

// one block per chunk item (see ChunkItem / ChunkAux)
__global__ void __launch_bounds__(kThreads)
pack_chunks_kernel(const uint4* __restrict__ src, const ChunkItem* __restrict__ items, const ChunkAux* __restrict__ aux,
                   int D8, uint4* __restrict__ dst) {
  const ChunkItem it = items[blockIdx.x];
  const ChunkAux ax = aux[blockIdx.x];
  const long long n_valid = (long long)it.valid * D8, n_all = (long long)ax.span * D8;
  const uint4* s = src + ax.src * D8;
  uint4* d = dst + (long long)it.start * D8;
  // gridDim.y blocks share a chunk (a chunk is at most 256 rows: one block per chunk leaves most SMs with too little in flight)
  for (long long i = (long long)blockIdx.y * blockDim.x + threadIdx.x; i < n_all; i += (long long)gridDim.y * blockDim.x)
    d[i] = i < n_valid ? __ldcs(s + i) : make_uint4(0, 0, 0, 0);
}

__global__ void __launch_bounds__(kThreads)
inverse_rowmap_items_kernel(const ChunkItem* __restrict__ items, const ChunkAux* __restrict__ aux, int* __restrict__ inv,
                            const int* __restrict__ rowmap, long long row_base, int* __restrict__ status) {
  const ChunkItem it = items[blockIdx.x];
  const ChunkAux ax = aux[blockIdx.x];
  bool bad = false;
  for (int t = threadIdx.x; t < ax.span; t += blockDim.x) {
    inv[it.start + t] = t < it.valid ? ax.out + t : -1;
    // pad de-duplication takes the valid rows of a chunk to be its FIRST rows: the caller's row map must say the same
    if (rowmap && t < it.valid && (long long)rowmap[ax.out + t] - row_base != ax.src + t) bad = true;
  }
  if (bad && status) atomicOr(status, 2);
}

// one warp per output row: 16-byte vectors, D % 8 == 0
__global__ void __launch_bounds__(kThreads)
gather_rows_kernel(const bf16* __restrict__ ctx, const float* __restrict__ x, const int* __restrict__ rowmap,
                   long long row_base, long long n_rows, int D, bf16* __restrict__ ctx_c, float* __restrict__ x_c) {
  const int lane = threadIdx.x & 31;
  const long long warps = ((long long)gridDim.x * blockDim.x) >> 5;
  for (long long j = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5; j < n_rows; j += warps) {
    const long long r = (long long)rowmap[j] - row_base;
    const uint4* cs = reinterpret_cast<const uint4*>(ctx + r * D);
    uint4* cd = reinterpret_cast<uint4*>(ctx_c + j * D);
    for (int i = lane; i < D / 8; i += 32) cd[i] = cs[i];
    const float4* xs = reinterpret_cast<const float4*>(x + r * D);
    float4* xd = reinterpret_cast<float4*>(x_c + j * D);
    for (int i = lane; i < D / 4; i += 32) xd[i] = xs[i];
  }
}

__global__ void __launch_bounds__(kThreads)
to_half_kernel(const float* __restrict__ in, long long n, __half* __restrict__ out) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    out[i] = __float2half_rn(in[i]);
}

// ---------------------------------------------------------------- classifier: warp-per-row fp32 dot product
__global__ void __launch_bounds__(kThreads)
classifier_kernel(const float* __restrict__ x, long long M, int D, const float* __restrict__ w,
                  const float* __restrict__ bias, float* __restrict__ logits, float* __restrict__ scores,
                  int* __restrict__ nonfinite) {
  const int lane = threadIdx.x & 31;
  const long long warps = ((long long)gridDim.x * blockDim.x) >> 5;
  const float b = __ldg(bias);
  for (long long row = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5; row < M; row += warps) {
    const float4* xr = reinterpret_cast<const float4*>(x + row * D);
    float s = 0.f;
    for (int i = lane; i < D / 4; i += 32) {
      const float4 xv = xr[i];
      const float4 wv = __ldg(reinterpret_cast<const float4*>(w) + i);
      s = fmaf(xv.x, wv.x, s);
      s = fmaf(xv.y, wv.y, s);
      s = fmaf(xv.z, wv.z, s);
      s = fmaf(xv.w, wv.w, s);
    }
    s = warp_sum(s) + b;
    if (lane == 0) {
      logits[row] = s;
      if (scores) scores[row] = 1.f / (1.f + expf(-s));
      // range guard of the 16-bit plans: an operand that overflowed fp16 / bf16 anywhere upstream reaches the last
      // activation row as inf / NaN (every stage propagates them), so one test per row here sees all of them
      if (nonfinite && !(fabsf(s) <= 3.0e38f)) atomicOr(nonfinite, 1);
    }
  }
}

// out[i] = alpha * sum_s part[s * n + i], slices added in index order (split-K reduction: run-to-run deterministic)
__global__ void __launch_bounds__(kThreads)
sum_slices_kernel(const float4* __restrict__ part, int S, long long n4, float alpha, float4* __restrict__ out) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
    float4 a = part[i];
    for (int s = 1; s < S; ++s) {
      const float4 b = part[(long long)s * n4 + i];
      a.x += b.x; a.y += b.y; a.z += b.z; a.w += b.w;
    }
    out[i] = make_float4(alpha * a.x, alpha * a.y, alpha * a.z, alpha * a.w);
  }
}

}  // namespace

int ingest(const void* in, int dtype, long long n, float* out_f32, bf16* out_hi, bf16* out_lo, int num_sms,
           cudaStream_t stream, int hi_fp16) {
  IEF_CHECK(n % 8 == 0, "ingest: element count %lld must be a multiple of 8", n);
  if (n == 0) return IEFVAD_OK;
  const long long n8 = n / 8;
  const int grid = grid_for(n8, num_sms);
  switch (dtype) {
    case IEFVAD_DT_F32:
      ingest_kernel<float><<<grid, kThreads, 0, stream>>>(static_cast<const float*>(in), n8, out_f32, out_hi, out_lo, hi_fp16);
      break;
    case IEFVAD_DT_F16:
      ingest_kernel<__half><<<grid, kThreads, 0, stream>>>(static_cast<const __half*>(in), n8, out_f32, out_hi, out_lo, hi_fp16);
      break;
    case IEFVAD_DT_BF16:
      ingest_kernel<bf16><<<grid, kThreads, 0, stream>>>(static_cast<const bf16*>(in), n8, out_f32, out_hi, out_lo, hi_fp16);
      break;
    default:
      set_error("ingest: unsupported dtype code %d (0 = f32, 1 = f16, 2 = bf16)", dtype);
      return IEFVAD_ERR_INVALID;
  }
  count_launches(1);
  IEF_CUDA(cudaGetLastError());
  return IEFVAD_OK;
}

int ingest_ragged(const void* packed, int dtype, const long long* chunk_start, long long start_base, const int* chunk_valid,
                  long long n_chunks, int T, int D, float* out_f32, bf16* out_hi, int hi_fp16, int num_sms,
                  cudaStream_t stream) {
  IEF_CHECK(D % 8 == 0, "ingest_ragged: D=%d must be a multiple of 8", D);
  if (n_chunks == 0 || T == 0) return IEFVAD_OK;
  const long long n8 = n_chunks * T * (D / 8);
  const int grid = grid_for(n8, num_sms);
  switch (dtype) {
    case IEFVAD_DT_F32:
      ingest_ragged_kernel<float><<<grid, kThreads, 0, stream>>>(static_cast<const float*>(packed), chunk_start, start_base,
                                                                  chunk_valid, n8, T, D / 8, out_f32, out_hi, hi_fp16);
      break;
    case IEFVAD_DT_F16:
      ingest_ragged_kernel<__half><<<grid, kThreads, 0, stream>>>(static_cast<const __half*>(packed), chunk_start, start_base,
                                                                   chunk_valid, n8, T, D / 8, out_f32, out_hi, hi_fp16);
      break;
    case IEFVAD_DT_BF16:
      ingest_ragged_kernel<bf16><<<grid, kThreads, 0, stream>>>(static_cast<const bf16*>(packed), chunk_start, start_base,
                                                                 chunk_valid, n8, T, D / 8, out_f32, out_hi, hi_fp16);
      break;
    default:
      set_error("ingest_ragged: unsupported dtype code %d", dtype);
      return IEFVAD_ERR_INVALID;
  }
  count_launches(1);
  IEF_CUDA(cudaGetLastError());
  return IEFVAD_OK;
}

int layernorm(const float* x, long long M, int D, const float* w1, const float* b1, const float* w2, const float* b2,
              float eps, float* out_f32, bf16* out_hi, bf16* out_lo, int num_sms, cudaStream_t stream, int hi_fp16,
              const int* f32_row_out) {
  IEF_CHECK(D % 128 == 0 && D >= 128 && D <= 1024, "layernorm: D=%d must be a multiple of 128 in [128, 1024]", D);
  IEF_CHECK(w1 && b1 && (w2 == nullptr) == (b2 == nullptr), "layernorm: bad affine pointers");
  if (M == 0) return IEFVAD_OK;
  const int grid = grid_for(M * 32, num_sms);
#define IEF_LN(NV)                                                                                              \
  case NV:                                                                                                      \
    layernorm_kernel<NV><<<grid, kThreads, 0, stream>>>(x, M, w1, b1, w2, b2, eps, out_f32, out_hi, out_lo, hi_fp16, f32_row_out);  \
    break;
  switch (D / 128) {
    IEF_LN(1) IEF_LN(2) IEF_LN(3) IEF_LN(4) IEF_LN(5) IEF_LN(6) IEF_LN(7) IEF_LN(8)
  }
#undef IEF_LN
  count_launches(1);
  IEF_CUDA(cudaGetLastError());
  return IEFVAD_OK;
}

int fuse(const float* mu_i, const float* mu_e, const float* lv_i, const float* lv_e, long long n, float factor,
         float eps, float* w_i, float* w_e, float* fused, bf16* fused_hi, bf16* fused_lo, int num_sms,
         cudaStream_t stream, int hi_fp16) {
  IEF_CHECK(n % 4 == 0, "fuse: element count %lld must be a multiple of 4", n);
  if (n == 0) return IEFVAD_OK;
  const long long n4 = n / 4;
  fuse_kernel<<<grid_for(n4, num_sms), kThreads, 0, stream>>>(
      reinterpret_cast<const float4*>(mu_i), reinterpret_cast<const float4*>(mu_e),
      reinterpret_cast<const float4*>(lv_i), reinterpret_cast<const float4*>(lv_e), n4, factor, eps,
      reinterpret_cast<float4*>(w_i), reinterpret_cast<float4*>(w_e), reinterpret_cast<float4*>(fused), fused_hi,
      fused_lo, hi_fp16);
  count_launches(1);
  IEF_CUDA(cudaGetLastError());
  return IEFVAD_OK;
}

int fuse_rows(const float* mu_i, const float* mu_e, const float* lv_i, const float* lv_e, long long rows, int D, float factor,
              float eps, float* wi_mean, float* we_mean, float* fused, bf16* fused_hi, bf16* fused_lo, int num_sms,
              cudaStream_t stream, int hi_fp16) {
  IEF_CHECK(D % 4 == 0 && wi_mean && we_mean, "fuse_rows: D %% 4 == 0 and both mean outputs are required");
  if (rows == 0) return IEFVAD_OK;
  fuse_rows_kernel<<<grid_for(rows * 32, num_sms), kThreads, 0, stream>>>(
      reinterpret_cast<const float4*>(mu_i), reinterpret_cast<const float4*>(mu_e), reinterpret_cast<const float4*>(lv_i),
      reinterpret_cast<const float4*>(lv_e), rows, D / 4, factor, eps, 1.0f / float(D), wi_mean, we_mean,
      reinterpret_cast<float4*>(fused), fused_hi, fused_lo, hi_fp16);
  count_launches(1);
  IEF_CUDA(cudaGetLastError());
  return IEFVAD_OK;
}

int gather_rows(const bf16* ctx, const float* x, const int* rowmap, long long row_base, long long n_rows, int D,
                bf16* ctx_c, float* x_c, int num_sms, cudaStream_t stream) {
  IEF_CHECK(D % 8 == 0, "gather_rows: D=%d must be a multiple of 8", D);
  if (n_rows == 0) return IEFVAD_OK;
  gather_rows_kernel<<<grid_for(n_rows * 32, num_sms), kThreads, 0, stream>>>(ctx, x, rowmap, row_base, n_rows, D, ctx_c, x_c);
  count_launches(1);
  IEF_CUDA(cudaGetLastError());
  return IEFVAD_OK;
}

int pack_chunks(const void* src16, const ChunkItem* items, const ChunkAux* aux, int n_items, int D, void* dst16,
                cudaStream_t stream) {
  IEF_CHECK(D % 8 == 0, "pack_chunks: D=%d must be a multiple of 8", D);
  if (n_items == 0) return IEFVAD_OK;
  pack_chunks_kernel<<<dim3(n_items, 8), kThreads, 0, stream>>>(static_cast<const uint4*>(src16), items, aux, D / 8,
                                                       static_cast<uint4*>(dst16));
  count_launches(1);
  IEF_CUDA(cudaGetLastError());
  return IEFVAD_OK;
}

int inverse_rowmap_items(const ChunkItem* items, const ChunkAux* aux, int n_items, int* inv, cudaStream_t stream,
                         const int* rowmap, long long row_base, int* status) {
  if (n_items == 0) return IEFVAD_OK;
  inverse_rowmap_items_kernel<<<n_items, kThreads, 0, stream>>>(items, aux, inv, rowmap, row_base, status);
  count_launches(1);
  IEF_CUDA(cudaGetLastError());
  return IEFVAD_OK;
}

int inverse_rowmap(const int* rowmap, long long row_base, long long n_rows, long long M, int* inv, int num_sms,
                   cudaStream_t stream) {
  if (M == 0) return IEFVAD_OK;
  IEF_CUDA(cudaMemsetAsync(inv, 0xFF, size_t(M) * sizeof(int), stream));        // -1 = row does not survive
  if (n_rows == 0) return IEFVAD_OK;
  inverse_rowmap_kernel<<<grid_for(n_rows, num_sms), kThreads, 0, stream>>>(rowmap, row_base, n_rows, inv);
  count_launches(1);
  IEF_CUDA(cudaGetLastError());
  return IEFVAD_OK;
}

int to_half(const float* in, long long n, void* out_f16, int num_sms, cudaStream_t stream) {
  if (n == 0) return IEFVAD_OK;
  to_half_kernel<<<grid_for(n, num_sms), kThreads, 0, stream>>>(in, n, static_cast<__half*>(out_f16));
  count_launches(1);
  IEF_CUDA(cudaGetLastError());
  return IEFVAD_OK;
}

int classifier(const float* x, long long M, int D, const float* w, const float* bias, float* logits, float* scores,
               int num_sms, cudaStream_t stream, int* nonfinite) {
  IEF_CHECK(D % 4 == 0, "classifier: D=%d must be a multiple of 4", D);
  if (M == 0) return IEFVAD_OK;
  classifier_kernel<<<grid_for(M * 32, num_sms), kThreads, 0, stream>>>(x, M, D, w, bias, logits, scores, nonfinite);
  count_launches(1);
  IEF_CUDA(cudaGetLastError());
  return IEFVAD_OK;
}

int sum_slices(const float* part, int S, long long n, float alpha, float* out, int num_sms, cudaStream_t stream) {
  IEF_CHECK(n % 4 == 0 && S >= 1, "sum_slices: element count %lld must be a multiple of 4", n);
  if (n == 0) return IEFVAD_OK;
  sum_slices_kernel<<<grid_for(n / 4, num_sms), kThreads, 0, stream>>>(reinterpret_cast<const float4*>(part), S, n / 4, alpha,
                                                                       reinterpret_cast<float4*>(out));
  count_launches(1);
  IEF_CUDA(cudaGetLastError());
  return IEFVAD_OK;
}

}  // namespace iefvad
