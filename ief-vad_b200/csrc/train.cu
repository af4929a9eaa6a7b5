// Kernels of the TRAINING step (SURVEY 8f row N3; reference: train/ucf_train.py:60-106 calls loss.backward() through
// model/imf_vad.py:109-161 and train/loss.py:18-30): what the backward pass needs besides the GEMMs, which reuse the
// tcgen05 kernel of the forward (dgrad = dY . W with W^T as the K-major "weight", wgrad = dY^T . X on transposed
// activations) and the attention, which has its own file (train_attn.cu).  Everything here is fp32 IEEE arithmetic;
// reductions over rows are two-stage and fixed-order, so the gradients are run-to-run deterministic.
//
//   layernorm_bwd                           dx, dgamma, dbeta of nn.LayerNorm
//   colsum                                  column sums (bias gradients), optionally row-weighted
//   fuse_bwd                                backward of the uncertainty-weighted fusion (model/imf_vad.py:130-144)
//   relu_bwd, quickgelu, axpy, outer        small elementwise helpers
//   transpose_f32, transpose_split          transposes for the wgrad GEMMs (fp32, or straight into bf16 hi / lo operands)
//   clas2_bwd                               backward of the MIL top-k BCE loss (train/loss.py:18-30)
#include "common.cuh"
#include "train.cuh"

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

// ---------------------------------------------------------------- LayerNorm backward
// one warp per row: dx = rstd * (g - mean(g) - xhat * mean(g * xhat)), g = dy * gamma; stats[row] = (mean, rstd)
__global__ void __launch_bounds__(kThreads)
ln_bwd_rows_kernel(const float* __restrict__ x, const float* __restrict__ gamma, const float* __restrict__ dy, long long rows,
                   int D, float eps, float* __restrict__ dx, float2* __restrict__ stats) {
  const int lane = threadIdx.x & 31;
  const long long warps = ((long long)gridDim.x * blockDim.x) >> 5;
  for (long long row = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5; row < rows; row += warps) {
    const float* xr = x + row * D;
    const float* gr = dy + row * D;
    float s = 0.f;
    for (int c = lane; c < D; c += 32) s += xr[c];
    const float mean = warp_sum(s) / float(D);
    float v = 0.f;
    for (int c = lane; c < D; c += 32) { const float d = xr[c] - mean; v = fmaf(d, d, v); }
    const float rstd = rsqrtf(warp_sum(v) / float(D) + eps);
    float m1 = 0.f, m2 = 0.f;
    for (int c = lane; c < D; c += 32) {
      const float g = gr[c] * __ldg(gamma + c);
      m1 += g;
      m2 = fmaf(g, (xr[c] - mean) * rstd, m2);
    }
    m1 = warp_sum(m1) / float(D);
    m2 = warp_sum(m2) / float(D);
    for (int c = lane; c < D; c += 32) {
      const float xh = (xr[c] - mean) * rstd;
      dx[row * D + c] = rstd * (gr[c] * __ldg(gamma + c) - m1 - xh * m2);
    }
    if (lane == 0) stats[row] = make_float2(mean, rstd);
  }
}

// column sums over a slab of rows, one thread per column: part[blk, 0, c] = sum dy * xhat (or dy * wgt), part[blk, 1, c] = sum dy
// mode 0: plain column sum of a (part[.,0,.] only); 1: LayerNorm (a = dy, b = x, stats); 2: a weighted by wgt[row]
__global__ void __launch_bounds__(kThreads)
colsum_partial_kernel(const float* __restrict__ a, const float* __restrict__ b, const float2* __restrict__ stats,
                      const float* __restrict__ wgt, long long rows, int D, int rows_per_block, int mode,
                      float* __restrict__ part) {
  const long long r0 = (long long)blockIdx.x * rows_per_block;
  long long r1 = r0 + rows_per_block;
  if (r1 > rows) r1 = rows;
  for (int c = threadIdx.x; c < D; c += blockDim.x) {
    float s0 = 0.f, s1 = 0.f;
    for (long long r = r0; r < r1; ++r) {
      const float av = a[r * D + c];
      if (mode == 1) {
        const float2 st = stats[r];
        s0 = fmaf(av, (b[r * D + c] - st.x) * st.y, s0);
        s1 += av;
      } else if (mode == 2) {
        s0 = fmaf(av, wgt[r], s0);
      } else {
        s0 += av;
      }
    }
    part[((long long)blockIdx.x * 2) * D + c] = s0;
    if (mode == 1) part[((long long)blockIdx.x * 2 + 1) * D + c] = s1;
  }
}
__global__ void __launch_bounds__(kThreads)
colsum_final_kernel(const float* __restrict__ part, int nblk, int D, int which, float* __restrict__ out) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= D) return;
  float s = 0.f;
  for (int k = 0; k < nblk; ++k) s += part[((long long)k * 2 + which) * D + c];      // fixed order: deterministic
  out[c] = s;
}

// ---------------------------------------------------------------- fusion backward (model/imf_vad.py:130-144)
__global__ void __launch_bounds__(kThreads)
fuse_bwd_kernel(const float* __restrict__ mu_i, const float* __restrict__ mu_e, const float* __restrict__ lv_i,
                const float* __restrict__ lv_e, const float* __restrict__ g_fused, const float* __restrict__ g_wi,
                const float* __restrict__ g_we, const float* __restrict__ g_mu_i, const float* __restrict__ g_mu_e,
                const float* __restrict__ g_lv_i, const float* __restrict__ g_lv_e, long long n, float factor, float eps,
                float* __restrict__ d_mu_i, float* __restrict__ d_mu_e, float* __restrict__ d_lv_i, float* __restrict__ d_lv_e) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const float ri = factor * expf(-lv_i[i]), re = factor * expf(-lv_e[i]);
    const float den = ri + re + eps;
    const float wi = ri / den, we = re / den;
    const float gf = g_fused ? g_fused[i] : 0.f;
    // total gradient reaching the normalised weights: through fused (= wi mu_i + we mu_e) and through the outputs w_i / w_e
    const float gwi = gf * mu_i[i] + (g_wi ? g_wi[i] : 0.f);
    const float gwe = gf * mu_e[i] + (g_we ? g_we[i] : 0.f);
    // d wi / d lv_i = -wi (1 - wi), d wi / d lv_e = wi we, d we / d lv_e = -we (1 - we), d we / d lv_i = wi we
    d_mu_i[i] = gf * wi + (g_mu_i ? g_mu_i[i] : 0.f);
    d_mu_e[i] = gf * we + (g_mu_e ? g_mu_e[i] : 0.f);
    d_lv_i[i] = -gwi * wi * (1.f - wi) + gwe * wi * we + (g_lv_i ? g_lv_i[i] : 0.f);
    d_lv_e[i] = gwi * wi * we - gwe * we * (1.f - we) + (g_lv_e ? g_lv_e[i] : 0.f);
  }
}

// ---------------------------------------------------------------- small elementwise / layout helpers
__global__ void __launch_bounds__(kThreads)
relu_bwd_kernel(const float* __restrict__ dh, const float* __restrict__ h, long long n, float* __restrict__ out) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    out[i] = h[i] > 0.f ? dh[i] : 0.f;
}
// QuickGELU of model/module.py:15-17: x * sigmoid(1.702 x)
__global__ void __launch_bounds__(kThreads)
quickgelu_kernel(const float* __restrict__ x, long long n, float* __restrict__ out) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const float v = x[i];
    out[i] = v / (1.f + expf(-1.702f * v));
  }
}
__global__ void __launch_bounds__(kThreads)
axpy_kernel(float* __restrict__ y, const float* __restrict__ x, float alpha, long long n) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    y[i] = fmaf(alpha, x[i], y[i]);
}
// out[r, c] = a[r] * w[c]
__global__ void __launch_bounds__(kThreads)
outer_kernel(const float* __restrict__ a, const float* __restrict__ w, long long rows, int D, float* __restrict__ out) {
  const long long n = rows * D;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const long long r = i / D;
    out[i] = a[r] * __ldg(w + (i - r * D));
  }
}
// dst[c, r] = src[r, c]; dst has ld_dst >= rows columns, columns [rows, ld_dst) are zero-filled
__global__ void __launch_bounds__(256)
transpose_kernel(const float* __restrict__ src, long long rows, int cols, float* __restrict__ dst, long long ld_dst) {
  __shared__ float tile[32][33];
  const long long r0 = (long long)blockIdx.x * 32;
  const int c0 = blockIdx.y * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  for (int k = ty; k < 32; k += 8) {
    const long long r = r0 + k;
    const int c = c0 + tx;
    tile[k][tx] = (r < rows && c < cols) ? src[r * cols + c] : 0.f;
  }
  __syncthreads();
  for (int k = ty; k < 32; k += 8) {
    const int c = c0 + k;
    const long long r = r0 + tx;
    if (c < cols && r < ld_dst) dst[(long long)c * ld_dst + r] = tile[tx][k];
  }
}

// the same transposition straight into the GEMM's operand format: bf16 hi = bf16(x), lo = bf16(x - hi), [cols, ld_dst]
__global__ void __launch_bounds__(256)
transpose_split_kernel(const float* __restrict__ src, long long rows, int cols, bf16* __restrict__ dst_hi, bf16* __restrict__ dst_lo,
                       long long ld_dst) {
  __shared__ float tile[32][33];
  const long long r0 = (long long)blockIdx.x * 32;
  const int c0 = blockIdx.y * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  for (int k = ty; k < 32; k += 8) {
    const long long r = r0 + k;
    const int c = c0 + tx;
    tile[k][tx] = (r < rows && c < cols) ? src[r * cols + c] : 0.f;
  }
  __syncthreads();
  for (int k = ty; k < 32; k += 8) {
    const int c = c0 + k;
    const long long r = r0 + tx;
    if (c < cols && r < ld_dst) {
      bf16 h, l;
      split_bf16(tile[tx][k], h, l);
      dst_hi[(long long)c * ld_dst + r] = h;
      dst_lo[(long long)c * ld_dst + r] = l;
    }
  }
}

// ---------------------------------------------------------------- CLAS2 backward (train/loss.py:18-30)
// loss = mean_b BCE(v_b, y_b), v_b = mean of the k_b largest sigmoid(logits[b, :len_b]), k_b = int(len_b / 16 + 1).
// idx [B, kmax]: the chosen positions (-1 padded) from the forward's top-k kernel.
__global__ void __launch_bounds__(kThreads)
clas2_bwd_kernel(const float* __restrict__ logits, const float* __restrict__ means, const float* __restrict__ labels,
                 long long label_stride, const int* __restrict__ idx, int B, int T, int kmax, const float* __restrict__ g_loss,
                 float* __restrict__ dlogits) {
  const int b = blockIdx.x;
  for (int t = threadIdx.x; t < T; t += blockDim.x) dlogits[(long long)b * T + t] = 0.f;
  __syncthreads();
  int k = 0;
  for (int j = 0; j < kmax; ++j) k += idx[(long long)b * kmax + j] >= 0 ? 1 : 0;
  if (k == 0) return;
  const float y = 1.f - labels[(long long)b * label_stride];            // :20 target = 1 - labels[:, 0]
  // ATen's binary_cross_entropy backward: grad * (v - y) / max((1 - v) v, 1e-12), mean reduction over the B rows
  const float v = means[b];
  const float dv = (v - y) / fmaxf((1.f - v) * v, 1e-12f);
  const float g = (g_loss ? g_loss[0] : 1.f) * dv / (float(B) * float(k));
  for (int j = threadIdx.x; j < kmax; j += blockDim.x) {
    const int t = idx[(long long)b * kmax + j];
    if (t >= 0) {
      const float p = 1.f / (1.f + expf(-logits[(long long)b * T + t]));
      dlogits[(long long)b * T + t] = g * p * (1.f - p);
    }
  }
}

}  // namespace

// ================================================================ host wrappers
static int colsum_run(const float* a, const float* b, const float2* stats, const float* wgt, long long rows, int D, int mode,
                      float* part, float* out0, float* out1, int num_sms, cudaStream_t stream) {
  const int nblk = train_colsum_blocks(rows, num_sms);
  const int rpb = int((rows + nblk - 1) / nblk);
  colsum_partial_kernel<<<nblk, kThreads, 0, stream>>>(a, b, stats, wgt, rows, D, rpb, mode, part);
  colsum_final_kernel<<<(D + kThreads - 1) / kThreads, kThreads, 0, stream>>>(part, nblk, D, 0, out0);
  if (mode == 1) colsum_final_kernel<<<(D + kThreads - 1) / kThreads, kThreads, 0, stream>>>(part, nblk, D, 1, out1);
  count_launches(mode == 1 ? 3 : 2);
  IEF_CUDA(cudaGetLastError());
  return IEFVAD_OK;
}

int train_colsum_blocks(long long rows, int num_sms) {
  long long nblk = (rows + 63) / 64;
  if (nblk > 4LL * num_sms) nblk = 4LL * num_sms;
  if (nblk < 1) nblk = 1;
  return int(nblk);
}

int layernorm_bwd(const float* x, const float* gamma, const float* dy, long long rows, int D, float eps, float* dx, float* dgamma,
                  float* dbeta, float* scratch, int num_sms, cudaStream_t stream) {
  if (rows == 0) return IEFVAD_OK;
  float2* stats = reinterpret_cast<float2*>(scratch);
  float* part = scratch + 2 * rows;
  ln_bwd_rows_kernel<<<grid_for(rows * 32, num_sms), kThreads, 0, stream>>>(x, gamma, dy, rows, D, eps, dx, stats);
  count_launches(1);
  return colsum_run(dy, x, stats, nullptr, rows, D, 1, part, dgamma, dbeta, num_sms, stream);
}

int colsum(const float* a, const float* wgt, long long rows, int D, float* out, float* scratch, int num_sms, cudaStream_t stream) {
  if (rows == 0) { IEF_CUDA(cudaMemsetAsync(out, 0, size_t(D) * 4, stream)); return IEFVAD_OK; }
  return colsum_run(a, nullptr, nullptr, wgt, rows, D, wgt ? 2 : 0, scratch, out, nullptr, num_sms, stream);
}

int fuse_bwd(const float* mu_i, const float* mu_e, const float* lv_i, const float* lv_e, const float* g_fused, const float* g_wi,
             const float* g_we, const float* g_mu_i, const float* g_mu_e, const float* g_lv_i, const float* g_lv_e, long long n,
             float factor, float eps, float* d_mu_i, float* d_mu_e, float* d_lv_i, float* d_lv_e, int num_sms, cudaStream_t stream) {
  if (n == 0) return IEFVAD_OK;
  fuse_bwd_kernel<<<grid_for(n, num_sms), kThreads, 0, stream>>>(mu_i, mu_e, lv_i, lv_e, g_fused, g_wi, g_we, g_mu_i, g_mu_e,
                                                                g_lv_i, g_lv_e, n, factor, eps, d_mu_i, d_mu_e, d_lv_i, d_lv_e);
  count_launches(1);
  IEF_CUDA(cudaGetLastError());
  return IEFVAD_OK;
}

int relu_bwd(const float* dh, const float* h, long long n, float* out, int num_sms, cudaStream_t stream) {
  if (n == 0) return IEFVAD_OK;
  relu_bwd_kernel<<<grid_for(n, num_sms), kThreads, 0, stream>>>(dh, h, n, out);
  count_launches(1);
  IEF_CUDA(cudaGetLastError());
  return IEFVAD_OK;
}

int quickgelu(const float* x, long long n, float* out, int num_sms, cudaStream_t stream) {
  if (n == 0) return IEFVAD_OK;
  quickgelu_kernel<<<grid_for(n, num_sms), kThreads, 0, stream>>>(x, n, out);
  count_launches(1);
  IEF_CUDA(cudaGetLastError());
  return IEFVAD_OK;
}

int axpy(float* y, const float* x, float alpha, long long n, int num_sms, cudaStream_t stream) {
  if (n == 0) return IEFVAD_OK;
  axpy_kernel<<<grid_for(n, num_sms), kThreads, 0, stream>>>(y, x, alpha, n);
  count_launches(1);
  IEF_CUDA(cudaGetLastError());
  return IEFVAD_OK;
}

int outer(const float* a, const float* w, long long rows, int D, float* out, int num_sms, cudaStream_t stream) {
  if (rows == 0) return IEFVAD_OK;
  outer_kernel<<<grid_for(rows * D, num_sms), kThreads, 0, stream>>>(a, w, rows, D, out);
  count_launches(1);
  IEF_CUDA(cudaGetLastError());
  return IEFVAD_OK;
}

int transpose_f32(const float* src, long long rows, int cols, float* dst, long long ld_dst, cudaStream_t stream) {
  IEF_CHECK(ld_dst >= rows, "transpose: ld_dst %lld < rows %lld", ld_dst, rows);
  if (rows == 0 || cols == 0) return IEFVAD_OK;
  const dim3 grid(unsigned((ld_dst + 31) / 32), unsigned((cols + 31) / 32));
  transpose_kernel<<<grid, 256, 0, stream>>>(src, rows, cols, dst, ld_dst);
  count_launches(1);
  IEF_CUDA(cudaGetLastError());
  return IEFVAD_OK;
}

int transpose_split(const float* src, long long rows, int cols, bf16* dst_hi, bf16* dst_lo, long long ld_dst, cudaStream_t stream) {
  IEF_CHECK(ld_dst >= rows, "transpose_split: ld_dst %lld < rows %lld", ld_dst, rows);
  if (rows == 0 || cols == 0) return IEFVAD_OK;
  const dim3 grid(unsigned((ld_dst + 31) / 32), unsigned((cols + 31) / 32));
  transpose_split_kernel<<<grid, 256, 0, stream>>>(src, rows, cols, dst_hi, dst_lo, ld_dst);
  count_launches(1);
  IEF_CUDA(cudaGetLastError());
  return IEFVAD_OK;
}

int clas2_bwd(const float* logits, const float* means, const float* labels, long long label_stride, const int* idx, int B, int T,
              int kmax, const float* g_loss, float* dlogits, cudaStream_t stream) {
  if (B == 0) return IEFVAD_OK;
  clas2_bwd_kernel<<<B, kThreads, 0, stream>>>(logits, means, labels, label_stride, idx, B, T, kmax, g_loss, dlogits);
  count_launches(1);
  IEF_CUDA(cudaGetLastError());
  return IEFVAD_OK;
}

}  // namespace iefvad
