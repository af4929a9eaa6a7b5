// GEMM operands of the stand-alone operators in the representation a precision plan needs, and the GEMM calls that
// read them.  Plan codes: -1 fp32 FFMA, 0 bf16, 1 split-bf16 (hi + lo, three MMA passes), 2 fp16 (E5M10).
#pragma once
#include "gemm.cuh"
#include "scratch.cuh"

namespace iefvad {

// grid of the 256-thread grid-stride kernels: one thread per item, at most 8 CTAs per SM
inline int blocks_for(long long n, int num_sms) {
  const long long b = (n + 255) / 256, cap = (long long)num_sms * 8;
  return int(b < 1 ? 1 : (b > cap ? cap : b));
}

int check_plan(const char* who, int plan);

// one operand / result in the representation the plan needs: fp32 (plan < 0), bf16 hi (+ lo when plan == 1) or fp16
// in `hi` (plan == 2)
struct Mat {
  float* f = nullptr;
  bf16* hi = nullptr;
  bf16* lo = nullptr;
  int ld = 0;
};

int alloc_mat(Scratch& sc, Mat* m, size_t rows, int ld, int plan);

// src fp32 [rows, cols] (pitch ld_src) -> operand [rows_p, cols_p], zero outside [rows, cols).  hi = rn(x) and
// lo = rn(x - hi) whichever kernel runs.  An unpadded dense source is converted by the vectorised ingest kernel, or
// under plan -1 read in place (m->f aliases src and must not be written).
int to_mat(Scratch& sc, Mat* m, const float* src, int rows, int cols, long long ld_src, int rows_p, int cols_p, int plan,
           int num_sms, cudaStream_t st);

// GemmTcArgs of C = A . W^T under a 16-bit plan
GemmTcArgs tc_args(int plan, const Mat& A, const Mat& W, int M, int N, int K);

// C = epilogue(A . W^T) in the plan's arithmetic; `ep` carries bias / act / resid / alpha and the fp32 output, `dst`
// (optional) receives the result in operand form for a following contraction.
int gemm_plan(int plan, const Mat& A, const Mat& W, int M, int N, int K, EpiParams ep, const Mat* dst, int num_sms,
              cudaStream_t st);

// gemm_tc for an epilogue out_f32 = alpha * A . W^T (row-major fp32 only, ld_f32 = N, no bias, residual, activation or
// 16-bit output) with the tiling left to the heuristic, split along K where the output is small and the contraction
// long (the wgrad GEMMs of the training step: [768, 768] = dY^T [768, 16 384] . X^T, which without it walk 768
// k-blocks on 72 CTAs).  K slices become extra row tiles of an [S x M, N] partial buffer from `sc` (256-column tiles
// on CTA pairs), summed in slice order afterwards: deterministic, unlike atomics.  Any other GEMM runs as one gemm_tc.
int gemm_tc_split_k(GemmTcArgs g, EpiParams ep, Scratch& sc, int num_sms, cudaStream_t st);

}  // namespace iefvad
