#pragma once
#include "common.cuh"

namespace iefvad {

enum : int { IEFVAD_DT_F32 = 0, IEFVAD_DT_F16 = 1, IEFVAD_DT_BF16 = 2 };

// in (f32 / f16 / bf16, n elements, n % 8 == 0) -> optional fp32 copy, optional 16-bit hi, optional 16-bit lo
int ingest(const void* in, int dtype, long long n, float* out_f32, bf16* out_hi, bf16* out_lo, int num_sms,
           cudaStream_t stream, int hi_fp16 = 0 /* out_hi / out_lo receive fp16 instead of bf16 */);

// The same for a ragged batch: `packed` holds only the valid rows of the n_chunks zero-padded [T, D] chunks, chunk c's
// rows starting at packed row chunk_start[c] - start_base (device arrays); pad rows are written as zeros.
int ingest_ragged(const void* packed, int dtype, const long long* chunk_start, long long start_base, const int* chunk_valid,
                  long long n_chunks, int T, int D, float* out_f32, bf16* out_hi, int hi_fp16, int num_sms,
                  cudaStream_t stream);

// out = LN(x; w1, b1) or LN(LN(x; w1, b1); w2, b2) when w2 != null.  x [M, D] fp32.
int layernorm(const float* x, long long M, int D, const float* w1, const float* b1, const float* w2, const float* b2,
              float eps, float* out_f32, bf16* out_hi, bf16* out_lo, int num_sms, cudaStream_t stream,
              int hi_fp16 = 0 /* out_hi / out_lo receive fp16 instead of bf16 */,
              const int* f32_row_out = nullptr /* [M]: row of out_f32 that receives source row r, < 0 = none */);

// Packed ("dedup-pad") row layout of a batch of zero-padded chunks: chunk c owns rows [start, start + span) of which the
// first `valid` hold its real rows, the next one (when the chunk has pads) is ONE zero row standing for all of them,
// the rest is alignment (zero).  ChunkItem is what the attention kernel reads, ChunkAux what the packers read.
struct ChunkItem { int start, rows, valid, mult; };            // rows = valid + (mult > 0); mult = T - valid
struct ChunkAux { long long src; int span; int out; };          // src = first source row, out = first compact row
// dst[start + t] = src16[src + t] (t < valid), 0 elsewhere in the span; 16-bit rows of D elements
int pack_chunks(const void* src16, const ChunkItem* items, const ChunkAux* aux, int n_items, int D, void* dst16,
                cudaStream_t stream);
// inv[start + t] = out + t (t < valid), -1 elsewhere in the span.  rowmap (optional, dense sources): the caller's compact
// row map, checked to be the prefix map the packed layout assumes (rowmap[out + t] - row_base == src + t); bit 1 of
// *status is set otherwise
int inverse_rowmap_items(const ChunkItem* items, const ChunkAux* aux, int n_items, int* inv, cudaStream_t stream,
                         const int* rowmap = nullptr, long long row_base = 0, int* status = nullptr);

// inv[rowmap[j] - row_base] = j for j < n_rows, every other entry of inv[0, M) = -1
int inverse_rowmap(const int* rowmap, long long row_base, long long n_rows, long long M, int* inv, int num_sms,
                   cudaStream_t stream);

// The fusion of one element, model/imf_vad.py:134-144 in its exact op order, every product / sum rounded separately
// like ATen: w_i, w_e and the returned fused value.  fuse, fuse_rows and heads_fuse all compute it here, which keeps
// them bit-identical with one another.
__device__ __forceinline__ float fuse_one(float mu_i, float mu_e, float lv_i, float lv_e, float factor, float eps,
                                          float& w_i, float& w_e) {
  const float ri = __fmul_rn(factor, expf(-lv_i));
  const float re = __fmul_rn(factor, expf(-lv_e));
  const float den = __fadd_rn(__fadd_rn(ri, re), eps);
  w_i = __fdiv_rn(ri, den);
  w_e = __fdiv_rn(re, den);
  return __fadd_rn(__fmul_rn(w_i, mu_i), __fmul_rn(w_e, mu_e));
}

// model/imf_vad.py:130-144.  n elements; fused / fused_hi / fused_lo optional.
int fuse(const float* mu_i, const float* mu_e, const float* lv_i, const float* lv_e, long long n, float factor,
         float eps, float* w_i, float* w_e, float* fused, bf16* fused_hi, bf16* fused_lo, int num_sms,
         cudaStream_t stream, int hi_fp16 = 0 /* fused_hi / fused_lo receive fp16 instead of bf16 */);

// The same with one warp per row, which also writes the row means of w_i / w_e (what the reference's evaluation loop keeps
// of them, train/ucf_test.py:124-131) instead of the [rows, D] weight tensors.
int fuse_rows(const float* mu_i, const float* mu_e, const float* lv_i, const float* lv_e, long long rows, int D, float factor,
              float eps, float* wi_mean, float* we_mean, float* fused, bf16* fused_hi, bf16* fused_lo, int num_sms,
              cudaStream_t stream, int hi_fp16 = 0);

// compact the rows listed in rowmap (minus row_base): ctx_c[j] = ctx[rowmap[j] - base] (16-bit rows), x_c[j] = x[...] (fp32)
int gather_rows(const bf16* ctx, const float* x, const int* rowmap, long long row_base, long long n_rows, int D,
                bf16* ctx_c, float* x_c, int num_sms, cudaStream_t stream);

// out[i] = alpha * sum_s part[s * n + i] (slices in index order): the reduction of a split-K GEMM
int sum_slices(const float* part, int S, long long n, float alpha, float* out, int num_sms, cudaStream_t stream);

// fp32 -> fp16 (weights of the fp16-operand refinement GEMMs)
int to_half(const float* in, long long n, void* out_f16, int num_sms, cudaStream_t stream);

// logits[row] = x[row, :] . w + bias;  scores (optional) = sigmoid(logits)
// nonfinite (optional device int): bit 0 is set when a logit is inf / NaN (the range guard of the 16-bit plans)
int classifier(const float* x, long long M, int D, const float* w, const float* bias, float* logits, float* scores,
               int num_sms, cudaStream_t stream, int* nonfinite = nullptr);

}  // namespace iefvad
