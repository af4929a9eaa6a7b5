// Internal C++ interface of the two GEMM engines (tcgen05 16-bit and fp32 SIMT) and their epilogue parameters.
#pragma once
#include "common.cuh"

namespace iefvad {

enum : int { ACT_NONE = 0, ACT_RELU = 1, ACT_QUICKGELU = 2 };
enum : int { EPI_ROWMAJOR = 0, EPI_QKV = 1, EPI_DISCARD = 2 /* micro-benchmarks: mainloop only */ };

// Both engines read mode EPI_ROWMAJOR, bias, act, the fp32 resid with alpha and the fp32 outputs.  Only the tcgen05
// engine reads EPI_QKV, EPI_DISCARD, out_hi / out_lo / hi_fp16 and resid_h16 / resid_l16.
struct EpiParams {
  int mode = EPI_ROWMAJOR;
  const float* bias = nullptr;   // [N] or null
  int act = ACT_NONE;
  // out = (resid ? resid[row, col] : 0) + alpha * act(acc + bias)
  const float* resid = nullptr;  // fp32 [M, ld_resid] or null
  int ld_resid = 0;
  // the residual as fp16 [M, ld_resid] (exact for fp16 inputs), optionally plus an fp16 remainder (resid = hi + lo,
  // ~22 mantissa bits); replaces `resid`
  const void* resid_h16 = nullptr;
  const void* resid_l16 = nullptr;
  float alpha = 1.f;
  // row-major outputs (any subset)
  float* out_f32 = nullptr;      // columns [0, split_col)
  float* out_f32_b = nullptr;    // columns [split_col, N) land in out_f32_b[row, col - split_col]
  int ld_f32 = 0;
  int split_col = 1 << 30;
  bf16* out_hi = nullptr;        // 16-bit(out)
  bf16* out_lo = nullptr;        // 16-bit(out - hi), optional
  int ld_bf = 0;
  int hi_fp16 = 0;               // out_hi / out_lo receive fp16 instead of bf16
  // EPI_QKV: packed in-projection scattered into the attention kernel's operand layouts
  //   q  [B, H, T, dhp]  (scaled by qscale; columns >= dh are neither written nor read by the attention kernels)
  //   k  [B, H, T, dhp]
  //   vt [B, H, dh, Tpad] (transposed so that P.V is a K-major x K-major UMMA)
  bf16* q = nullptr;
  bf16* k = nullptr;
  bf16* vt = nullptr;
  int T = 0, H = 0, dh = 0, dhp = 0, Tpad = 0, D = 0;
  float qscale = 1.f;
};

__device__ __forceinline__ float apply_act(float v, int act) {
  if (act == ACT_RELU) return fmaxf(v, 0.f);
  if (act == ACT_QUICKGELU) return v / (1.f + __expf(-1.702f * v));
  return v;
}

struct GemmTcArgs {
  const bf16* A_hi = nullptr;  // [M, lda]  activations (K-major)
  const bf16* A_lo = nullptr;  // residual of the bf16 rounding, only for nsplit == 3
  const bf16* W_hi = nullptr;  // [N, ldw]  nn.Linear weight layout (K-major)
  const bf16* W_lo = nullptr;
  int M = 0, N = 0, K = 0;
  int lda = 0, ldw = 0;
  int nsplit = 1;              // 1: plain bf16;  3: hi.hi + hi.lo + lo.hi
  int fp16 = 0;                // A_hi / W_hi hold fp16 (E5M10) instead of bf16: 8x finer operand rounding, same MMA rate
  int force_bn = 0;            // 0 = heuristic, else 64 / 128 / 256 (tests, tuning)
  int force_stages = 0;        // 0 = as many smem stages as fit beside the epilogue buffers (tuning)
  int ksplit = 1;              // split-K (small M x N, long K: the wgrad GEMMs): slice s accumulates into rows [s M, (s + 1) M) of
                               // out_f32, which must hold ksplit x M rows; the caller sums the slices (fixed order)
  int force_cg = 0;            // 0 = heuristic, 1 = one CTA per tile, 2 = CTA pair (cta_group::2, 256-row tiles)
};

// C = epilogue(A . W^T): 16-bit operands through TMA, tcgen05.mma into TMEM, and an epilogue whose global traffic
// (fp32 or fp16-pair residual in; fp32 / 16-bit hi / lo / q / k out) moves through TMA bulk tensor copies as well.
int gemm_tc(const GemmTcArgs& g, const EpiParams& ep, int num_sms, cudaStream_t stream);

// fp32 FFMA GEMM with a per-thread epilogue: the "fp32 plan" (1e-5 class) and the on-device yardstick the tcgen05
// path is debugged against.  A [M, lda] fp32, W [N, ldw] fp32; `ep` as above, without the tcgen05-only fields.
int gemm_simt(const float* A, int lda, const float* W, int ldw, int M, int N, int K, const EpiParams& ep,
              cudaStream_t stream);

}  // namespace iefvad
