#include "operand.cuh"

#include "elementwise.cuh"

namespace iefvad {

namespace {

// dst[r, c] = (r < rows && c < cols) ? src[r, c] : 0  for r < rows_p, c < cols_p (fp32 and/or bf16 hi / lo copies;
// hi_fp16: dst_hi receives fp16 instead, no lo)
__global__ void __launch_bounds__(256)
pad2d_kernel(const float* __restrict__ src, int rows, int cols, long long ld_src, int rows_p, int cols_p,
             float* __restrict__ dst_f32, bf16* __restrict__ dst_hi, bf16* __restrict__ dst_lo, int hi_fp16) {
  const long long total = (long long)rows_p * cols_p;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int r = int(i / cols_p), c = int(i - (long long)r * cols_p);
    const float v = (r < rows && c < cols) ? src[r * ld_src + c] : 0.f;
    if (dst_f32) dst_f32[i] = v;
    if (dst_hi && hi_fp16) {
      reinterpret_cast<__half*>(dst_hi)[i] = __float2half_rn(v);
    } else if (dst_hi) {
      bf16 h, l;
      split_bf16(v, h, l);
      dst_hi[i] = h;
      if (dst_lo) dst_lo[i] = l;
    }
  }
}

}  // namespace

int check_plan(const char* who, int plan) {
  IEF_CHECK(plan >= -1 && plan <= 2, "%s: plan must be -1 (fp32), 0 (bf16), 1 (split-bf16) or 2 (fp16), got %d", who, plan);
  return IEFVAD_OK;
}

int alloc_mat(Scratch& sc, Mat* m, size_t rows, int ld, int plan) {
  *m = Mat();
  m->ld = ld;
  if (plan < 0) return sc.get(&m->f, rows * ld);
  IEF_TRY(sc.get(&m->hi, rows * ld));
  if (plan == 1) IEF_TRY(sc.get(&m->lo, rows * ld));
  return IEFVAD_OK;
}

int to_mat(Scratch& sc, Mat* m, const float* src, int rows, int cols, long long ld_src, int rows_p, int cols_p, int plan,
           int num_sms, cudaStream_t st) {
  const long long n = (long long)rows * cols;
  // the GEMMs and the ingest kernel read 16-byte vectors
  if (rows_p == rows && cols_p == cols && ld_src == cols && (reinterpret_cast<uintptr_t>(src) & 15) == 0) {
    if (plan < 0) {
      *m = Mat();
      m->f = const_cast<float*>(src);
      m->ld = cols;
      return IEFVAD_OK;
    }
    if (n % 8 == 0) {
      IEF_TRY(alloc_mat(sc, m, size_t(rows), cols, plan));
      return ingest(src, IEFVAD_DT_F32, n, nullptr, m->hi, m->lo, num_sms, st, plan == 2);
    }
  }
  IEF_TRY(alloc_mat(sc, m, size_t(rows_p), cols_p, plan));
  pad2d_kernel<<<blocks_for((long long)rows_p * cols_p, num_sms), 256, 0, st>>>(src, rows, cols, ld_src, rows_p, cols_p,
                                                                                 m->f, m->hi, m->lo, plan == 2);
  count_launches(1);
  IEF_CUDA(cudaGetLastError());
  return IEFVAD_OK;
}

GemmTcArgs tc_args(int plan, const Mat& A, const Mat& W, int M, int N, int K) {
  GemmTcArgs g;
  g.A_hi = A.hi; g.A_lo = A.lo; g.W_hi = W.hi; g.W_lo = W.lo;
  g.M = M; g.N = N; g.K = K; g.lda = A.ld; g.ldw = W.ld; g.nsplit = (plan == 1) ? 3 : 1; g.fp16 = (plan == 2);
  return g;
}

int gemm_plan(int plan, const Mat& A, const Mat& W, int M, int N, int K, EpiParams ep, const Mat* dst, int num_sms,
              cudaStream_t st) {
  if (dst) {
    if (plan < 0) { ep.out_f32 = dst->f; ep.ld_f32 = dst->ld; }
    else { ep.out_hi = dst->hi; ep.out_lo = dst->lo; ep.ld_bf = dst->ld; ep.hi_fp16 = (plan == 2); }
  }
  if (plan < 0) return gemm_simt(A.f, A.ld, W.f, W.ld, M, N, K, ep, st);
  return gemm_tc(tc_args(plan, A, W, M, N, K), ep, num_sms, st);
}

int gemm_tc_split_k(GemmTcArgs g, EpiParams ep, Scratch& sc, int num_sms, cudaStream_t st) {
  const int tiles = (g.M / 256) * (g.N / 256);
  const bool plain = ep.mode == EPI_ROWMAJOR && !ep.bias && !ep.resid && !ep.resid_h16 && ep.act == ACT_NONE &&
                     !ep.out_hi && !ep.out_f32_b && ep.ld_f32 == g.N;
  if (plain && !g.force_bn && !g.force_cg && g.M % 256 == 0 && g.N % 256 == 0 && g.K >= 4096 && tiles * 2 <= num_sms / 2) {
    int S = (num_sms / 2) / tiles;
    while (S > 1 && (g.K / 64) % S != 0) --S;
    if (S > 1) {
      float* out = ep.out_f32;
      const float alpha = ep.alpha;
      float* part = nullptr;
      IEF_TRY(sc.get(&part, size_t(S) * g.M * g.N));
      ep.alpha = 1.f;
      ep.out_f32 = part;
      g.ksplit = S; g.force_bn = 256; g.force_cg = 2;
      IEF_TRY(gemm_tc(g, ep, num_sms, st));
      return sum_slices(part, S, (long long)g.M * g.N, alpha, out, num_sms, st);
    }
  }
  return gemm_tc(g, ep, num_sms, st);
}

}  // namespace iefvad
