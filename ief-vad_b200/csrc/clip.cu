// CLIP VisionTransformer forward (extracting/clip/model.py:206-241):
//   patches = im2col(x) . conv1^T          one GEMM, K = 3 P^2 zero-padded to a multiple of 64 (588 -> 640 at P = 14)
//   x = ln_pre([cls; patches] + pos)       one warp-per-row kernel writing the fp32 residual [N, T, W] batch-first
//   x = transformer(x)                     transformer_blocks (graph.cu), no layout swap
//   out = ln_post(x[:, 0]) @ proj          one kernel over the N class-token rows, fp32 throughout
// The im2col rows and the conv weight are written in the plan's operand type (fp16, or fp32 for the FFMA plan).
#include "clip.cuh"

#include <cmath>
#include <vector>

#include "elementwise.cuh"
#include "gemm.cuh"
#include "scratch.cuh"

namespace iefvad {

namespace {

int grid_of(long long n, int num_sms) {
  const long long b = (n + 255) / 256, cap = (long long)num_sms * 8;
  return int(b < 1 ? 1 : (b > cap ? cap : b));
}

__device__ __forceinline__ float load_f(const float* p, long long i) { return p[i]; }
__device__ __forceinline__ float load_f(const __half* p, long long i) { return __half2float(p[i]); }
__device__ __forceinline__ float load_f(const bf16* p, long long i) { return __bfloat162float(p[i]); }
__device__ __forceinline__ void store_f(float* p, long long i, float v) { p[i] = v; }
__device__ __forceinline__ void store_f(__half* p, long long i, float v) { p[i] = __float2half_rn(v); }

// dst[n*G*G + gy*G + gx, c*P*P + ky*P + kx] = x[n, c, gy*P + ky, gx*P + kx]; columns [3 P^2, Kp) are zero.
// This is Conv2d(3, W, P, stride P, bias=False) as a product with conv1.weight viewed as [W, 3 P^2].
template <typename Tin, typename Tout>
__global__ void __launch_bounds__(256)
clip_im2col_kernel(const Tin* __restrict__ x, long long rows, int R, int P, int G, int Kp, Tout* __restrict__ dst) {
  const int K = 3 * P * P, GG = G * G;
  const long long total = rows * Kp;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long r = i / Kp;
    const int c = int(i - r * Kp);
    float v = 0.f;
    if (c < K) {
      const long long n = r / GG;
      const int g = int(r - n * GG), gy = g / G, gx = g - gy * G;
      const int ch = c / (P * P), rem = c - ch * P * P, ky = rem / P, kx = rem - ky * P;
      v = load_f(x, ((n * 3 + ch) * R + gy * P + ky) * (long long)R + gx * P + kx);
    }
    store_f(dst, i, v);
  }
}

// conv1.weight [W, K] -> [W, Kp] in the operand type, zero columns [K, Kp)
template <typename Tout>
__global__ void __launch_bounds__(256)
clip_pad_weight_kernel(const float* __restrict__ w, int rows, int K, int Kp, Tout* __restrict__ dst) {
  const long long total = (long long)rows * Kp;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long r = i / Kp;
    const int c = int(i - r * Kp);
    store_f(dst, i, c < K ? w[r * K + c] : 0.f);
  }
}

// One warp per token row (n, t) of the residual [N, T, W], W = 128 NV:
//   v = (t == 0 ? class_embedding : patches[n*(T-1) + t-1]) + positional_embedding[t];  x[n, t] = ln_pre(v)
// (model.py:229-233).  Two-pass mean / variance in registers, as the library's LayerNorm kernel.
template <int NV>
__global__ void __launch_bounds__(256)
clip_tokens_kernel(const float* __restrict__ patches, const float* __restrict__ cls, const float* __restrict__ pos,
                   const float* __restrict__ lnw, const float* __restrict__ lnb, int T, long long rows,
                   float* __restrict__ x) {
  constexpr int W = 128 * NV;
  const int lane = threadIdx.x & 31;
  const long long warps = ((long long)gridDim.x * blockDim.x) >> 5;
  for (long long row = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5; row < rows; row += warps) {
    const long long n = row / T;
    const int t = int(row - n * T);
    const float4* src = reinterpret_cast<const float4*>(t == 0 ? cls : patches + (n * (T - 1) + t - 1) * W);
    const float4* pr = reinterpret_cast<const float4*>(pos + (long long)t * W);
    float v[NV * 4];
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const float4 a = src[lane + 32 * i], b = __ldg(pr + lane + 32 * i);
      v[4 * i] = a.x + b.x; v[4 * i + 1] = a.y + b.y; v[4 * i + 2] = a.z + b.z; v[4 * i + 3] = a.w + b.w;
    }
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < NV * 4; ++i) s += v[i];
    const float mean = warp_sum(s) * (1.f / W);
    float q = 0.f;
#pragma unroll
    for (int i = 0; i < NV * 4; ++i) {
      const float c = v[i] - mean;
      q = fmaf(c, c, q);
    }
    const float rstd = 1.f / sqrtf(warp_sum(q) * (1.f / W) + 1e-5f);
    float4* o = reinterpret_cast<float4*>(x + row * W);
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const float4 wv = __ldg(reinterpret_cast<const float4*>(lnw) + lane + 32 * i);
      const float4 bv = __ldg(reinterpret_cast<const float4*>(lnb) + lane + 32 * i);
      o[lane + 32 * i] = make_float4((v[4 * i + 0] - mean) * rstd * wv.x + bv.x, (v[4 * i + 1] - mean) * rstd * wv.y + bv.y,
                                     (v[4 * i + 2] - mean) * rstd * wv.z + bv.z, (v[4 * i + 3] - mean) * rstd * wv.w + bv.w);
    }
  }
}

// out[n] = ln_post(x[n, 0]) @ proj (model.py:237-241) in fp32.  A CTA takes HEAD_IMGS images and 256 output columns:
// its warps normalise the class-token rows into shared memory, then each thread runs the k-loop of one column for all
// of them (each proj element is read once per CTA).  An image's result does not depend on the others in its CTA.
constexpr int HEAD_IMGS = 8;

__global__ void __launch_bounds__(256)
clip_head_kernel(const float* __restrict__ x, int N, int T, int W, const float* __restrict__ lnw,
                 const float* __restrict__ lnb, const float* __restrict__ proj, int out_dim, float* __restrict__ out) {
  __shared__ float xs[HEAD_IMGS][1024];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n0 = blockIdx.x * HEAD_IMGS;
  const int nimg = (N - n0 < HEAD_IMGS) ? N - n0 : HEAD_IMGS;
  if (warp < nimg) {
    const float* r = x + (long long)(n0 + warp) * T * W;      // token 0 of image n0 + warp
    float s = 0.f;
    for (int k = lane; k < W; k += 32) s += r[k];
    const float mean = warp_sum(s) / float(W);
    float q = 0.f;
    for (int k = lane; k < W; k += 32) {
      const float c = r[k] - mean;
      q = fmaf(c, c, q);
    }
    const float rstd = 1.f / sqrtf(warp_sum(q) / float(W) + 1e-5f);
    for (int k = lane; k < W; k += 32) xs[warp][k] = (r[k] - mean) * rstd * lnw[k] + lnb[k];
  }
  __syncthreads();
  const int j = blockIdx.y * 256 + threadIdx.x;
  if (j >= out_dim) return;
  float acc[HEAD_IMGS];
#pragma unroll
  for (int i = 0; i < HEAD_IMGS; ++i) acc[i] = 0.f;
  for (int k = 0; k < W; ++k) {
    const float p = __ldg(proj + (long long)k * out_dim + j);
#pragma unroll
    for (int i = 0; i < HEAD_IMGS; ++i) acc[i] = fmaf(xs[i][k], p, acc[i]);
  }
  for (int i = 0; i < nimg; ++i) out[(long long)(n0 + i) * out_dim + j] = acc[i];
}

template <typename Tout>
int launch_im2col(const void* x, int dtype, long long rows, int R, int P, int G, int Kp, Tout* dst, int sms,
                  cudaStream_t st) {
  const int grid = grid_of(rows * Kp, sms);
  if (dtype == IEFVAD_DT_F32)
    clip_im2col_kernel<<<grid, 256, 0, st>>>(static_cast<const float*>(x), rows, R, P, G, Kp, dst);
  else if (dtype == IEFVAD_DT_F16)
    clip_im2col_kernel<<<grid, 256, 0, st>>>(static_cast<const __half*>(x), rows, R, P, G, Kp, dst);
  else
    clip_im2col_kernel<<<grid, 256, 0, st>>>(static_cast<const bf16*>(x), rows, R, P, G, Kp, dst);
  count_launches(1);
  IEF_CUDA(cudaGetLastError());
  return IEFVAD_OK;
}

}  // namespace

int clip_visual(const void* x, int dtype, int N, int R, int P, int W, int layers, int heads, int out_dim,
                const ClipVisualParams& p, int plan, float* out, cudaStream_t st) {
  IEF_CHECK(plan == -1 || plan == 2, "clip_visual: plan must be -1 (fp32) or 2 (fp16), got %d", plan);
  IEF_CHECK(dtype == IEFVAD_DT_F32 || dtype == IEFVAD_DT_F16 || dtype == IEFVAD_DT_BF16,
            "clip_visual: unsupported dtype code %d", dtype);
  IEF_CHECK(N >= 0 && N <= 65535, "clip_visual: batch %d outside [0, 65535]", N);
  IEF_CHECK(P > 0 && R > 0 && R % P == 0, "clip_visual: resolution %d must be a positive multiple of patch %d", R, P);
  IEF_CHECK(W >= 128 && W <= 1024 && W % 128 == 0, "clip_visual: width %d must be a multiple of 128 in [128, 1024]", W);
  IEF_CHECK(heads > 0 && W % heads == 0, "clip_visual: width %d is not divisible by heads=%d", W, heads);
  const int dh = W / heads;
  IEF_CHECK(dh == 32 || dh == 64 || dh == 96 || dh == 128, "clip_visual: head dim %d unsupported (32, 64, 96, 128)", dh);
  IEF_CHECK(layers >= 0 && layers <= 64, "clip_visual: layers %d outside [0, 64]", layers);
  IEF_CHECK(out_dim > 0, "clip_visual: output_dim %d must be positive", out_dim);
  IEF_CHECK(p.conv1 && p.cls && p.pos && p.ln_pre_w && p.ln_pre_b && p.ln_post_w && p.ln_post_b && p.proj &&
            (p.blocks || layers == 0), "clip_visual: null parameter");
  for (int i = 0; i < layers; ++i) {
    const ResBlockParams& b = p.blocks[i];
    IEF_CHECK(b.ln1_w && b.ln1_b && b.in_w && b.in_b && b.out_w && b.out_b && b.ln2_w && b.ln2_b && b.fc_w && b.fc_b &&
              b.proj_w && b.proj_b, "clip_visual: block %d has a null parameter", i);
  }
  const int G = R / P, T = G * G + 1;
  const long long M = (long long)N * T, Mp = (long long)N * G * G;
  IEF_CHECK(M < (1LL << 31), "clip_visual: %lld token rows exceed the GEMM row limit", M);
  IEF_CHECK(N == 0 || (x && out), "clip_visual: null input or output");
  if (N == 0) return IEFVAD_OK;
  int dev = 0, sms = 0;
  IEF_CUDA(cudaGetDevice(&dev));
  IEF_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));

  const int K = 3 * P * P, Kp = (K + 63) / 64 * 64;
  Scratch sc(st);
  float *patches, *xr;
  IEF_TRY(sc.get(&patches, size_t(Mp) * W));
  IEF_TRY(sc.get(&xr, size_t(M) * W));
  // patch embedding (model.py:226)
  EpiParams ep;
  ep.out_f32 = patches; ep.ld_f32 = W;
  if (plan < 0) {
    float *col, *wf;
    IEF_TRY(sc.get(&col, size_t(Mp) * Kp));
    IEF_TRY(sc.get(&wf, size_t(W) * Kp));
    IEF_TRY(launch_im2col(x, dtype, Mp, R, P, G, Kp, col, sms, st));
    clip_pad_weight_kernel<<<grid_of((long long)W * Kp, sms), 256, 0, st>>>(p.conv1, W, K, Kp, wf);
    count_launches(1);
    IEF_TRY(gemm_simt(col, Kp, wf, Kp, int(Mp), W, Kp, ep, st));
  } else {
    __half *col, *wh;
    IEF_TRY(sc.get(&col, size_t(Mp) * Kp));
    IEF_TRY(sc.get(&wh, size_t(W) * Kp));
    IEF_TRY(launch_im2col(x, dtype, Mp, R, P, G, Kp, col, sms, st));
    clip_pad_weight_kernel<<<grid_of((long long)W * Kp, sms), 256, 0, st>>>(p.conv1, W, K, Kp, wh);
    count_launches(1);
    GemmTcArgs g;
    g.A_hi = reinterpret_cast<const bf16*>(col); g.W_hi = reinterpret_cast<const bf16*>(wh);
    g.M = int(Mp); g.N = W; g.K = Kp; g.lda = Kp; g.ldw = Kp; g.fp16 = 1;
    IEF_TRY(gemm_tc(g, ep, sms, st));
  }
  // class token, positional embedding and ln_pre -> the fp32 residual [N, T, W] (model.py:227-230)
  {
    const int grid = grid_of(M * 32, sms);
#define IEF_TOK(NV)                                                                                                  \
  case NV:                                                                                                           \
    clip_tokens_kernel<NV><<<grid, 256, 0, st>>>(patches, p.cls, p.pos, p.ln_pre_w, p.ln_pre_b, T, M, xr);          \
    break;
    switch (W / 128) { IEF_TOK(1) IEF_TOK(2) IEF_TOK(3) IEF_TOK(4) IEF_TOK(5) IEF_TOK(6) IEF_TOK(7) IEF_TOK(8) }
#undef IEF_TOK
    count_launches(1);
    IEF_CUDA(cudaGetLastError());
  }
  // the residual attention blocks (model.py:232-234; the permutes there are the seq-first convention, not arithmetic)
  IEF_TRY(transformer_blocks(xr, p.blocks, layers, T, N, W, heads, nullptr, nullptr, plan, sms, st));
  // ln_post on the class token and the projection (model.py:236-241)
  clip_head_kernel<<<dim3((N + HEAD_IMGS - 1) / HEAD_IMGS, (out_dim + 255) / 256), 256, 0, st>>>(
      xr, N, T, W, p.ln_post_w, p.ln_post_b, p.proj, out_dim, out);
  count_launches(1);
  IEF_CUDA(cudaGetLastError());
  return IEFVAD_OK;
}

}  // namespace iefvad
