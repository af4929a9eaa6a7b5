// fp32 FFMA GEMM: C = epilogue(A[M,K] . W[N,K]^T).  Precision plan "fp32" of the forward (every
// contraction in IEEE fp32 like the reference, model/imf_vad.py:109-150) and the on-device yardstick
// for the tcgen05 path.  Classic 64x64x16 smem tiling, 128 threads, 4x8 register micro-tiles.
#include "common.cuh"
#include "gemm.cuh"

namespace iefvad {

namespace {

constexpr int SBM = 64, SBN = 64, SBK = 16;

// Store NC (multiple of 4, <= 32) consecutive fp32 columns [col0, col0+NC) of one output row.  `v` holds the raw
// accumulators.  Every pointer dereferenced here is 16-byte aligned because col0 % 4 == 0 and all leading dimensions
// are multiples of 8.
template <int NC>
__device__ __forceinline__ void epi_store_row(const EpiParams& p, long long row, int col0, float* v) {
#pragma unroll
  for (int j = 0; j < NC; ++j) {
    float x = v[j];
    if (p.bias) x += __ldg(p.bias + col0 + j);
    v[j] = apply_act(x, p.act);
  }
  if (p.resid) {
    const float* r = p.resid + row * p.ld_resid + col0;
#pragma unroll
    for (int j = 0; j < NC; j += 4) {
      const float4 rv = *reinterpret_cast<const float4*>(r + j);
      v[j + 0] = rv.x + p.alpha * v[j + 0];
      v[j + 1] = rv.y + p.alpha * v[j + 1];
      v[j + 2] = rv.z + p.alpha * v[j + 2];
      v[j + 3] = rv.w + p.alpha * v[j + 3];
    }
  } else if (p.alpha != 1.f) {
#pragma unroll
    for (int j = 0; j < NC; ++j) v[j] *= p.alpha;
  }
  if (p.out_f32) {
    float* o = (col0 < p.split_col) ? p.out_f32 + row * p.ld_f32 + col0
                                    : p.out_f32_b + row * p.ld_f32 + (col0 - p.split_col);
#pragma unroll
    for (int j = 0; j < NC; j += 4) *reinterpret_cast<float4*>(o + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
  }
}

__global__ void __launch_bounds__(128)
gemm_simt_kernel(const float* __restrict__ A, int lda, const float* __restrict__ W, int ldw, int M, int N, int K,
                 EpiParams ep) {
  __shared__ float As[SBK][SBM + 4];
  __shared__ float Ws[SBK][SBN + 4];
  const int tid = threadIdx.x;
  const int tx = tid & 7, ty = tid >> 3;
  const long long m0 = (long long)blockIdx.x * SBM;
  const int n0 = blockIdx.y * SBN;
  float acc[4][8];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;

  const int lr = tid >> 2;         // 0..31
  const int lk = (tid & 3) * 4;    // 0,4,8,12
  for (int k0 = 0; k0 < K; k0 += SBK) {
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int r = lr + 32 * h;
      float4 a = make_float4(0.f, 0.f, 0.f, 0.f), w = a;
      if (m0 + r < M) a = *reinterpret_cast<const float4*>(A + (m0 + r) * lda + k0 + lk);
      if (n0 + r < N) w = *reinterpret_cast<const float4*>(W + (long long)(n0 + r) * ldw + k0 + lk);
      As[lk + 0][r] = a.x; As[lk + 1][r] = a.y; As[lk + 2][r] = a.z; As[lk + 3][r] = a.w;
      Ws[lk + 0][r] = w.x; Ws[lk + 1][r] = w.y; Ws[lk + 2][r] = w.z; Ws[lk + 3][r] = w.w;
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < SBK; ++k) {
      const float4 a = *reinterpret_cast<const float4*>(&As[k][ty * 4]);
      const float4 b0 = *reinterpret_cast<const float4*>(&Ws[k][tx * 8]);
      const float4 b1 = *reinterpret_cast<const float4*>(&Ws[k][tx * 8 + 4]);
      const float av[4] = {a.x, a.y, a.z, a.w};
      const float bv[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
    }
    __syncthreads();
  }
  const int col0 = n0 + tx * 8;
  if (col0 < N) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const long long row = m0 + ty * 4 + i;
      if (row < M) epi_store_row<8>(ep, row, col0, acc[i]);
    }
  }
}

}  // namespace

int gemm_simt(const float* A, int lda, const float* W, int ldw, int M, int N, int K, const EpiParams& ep,
              cudaStream_t stream) {
  IEF_CHECK(M > 0 && N > 0 && K > 0, "gemm_simt: empty problem");
  IEF_CHECK(K % SBK == 0 && N % 8 == 0 && lda % 4 == 0 && ldw % 4 == 0,
            "gemm_simt: need K %% 16 == 0, N %% 8 == 0, lda/ldw %% 4 == 0 (K=%d N=%d)", K, N);
  IEF_CHECK(ep.mode == EPI_ROWMAJOR && !ep.out_hi && !ep.resid_h16, "gemm_simt: the epilogue writes fp32 rows only");
  dim3 grid((M + SBM - 1) / SBM, (N + SBN - 1) / SBN);
  gemm_simt_kernel<<<grid, 128, 0, stream>>>(A, lda, W, ldw, M, N, K, ep);
  count_launches(1);
  IEF_CUDA(cudaGetLastError());
  return IEFVAD_OK;
}

}  // namespace iefvad
