// The training objective of the reference's loop (train/ucf_train.py:73-102), which the loop builds after the model from
// its outputs, and its backward (SURVEY 8f row N3):
//
//   loss_cls = CLAS2(logits, labels, lengths)                                   train/loss.py:18-30 (rank.cu, train.cu)
//   cos      = cosine_similarity(normalize(mu_i), normalize(mu_e))              per row of [B*T, D]
//   loss_reg = mean(1 - cos) + mean |norm(mu_i) - norm(mu_e)|
//   loss_kl  = -0.5 mean(1 + eli - mu_i^2 - exp(eli)) - 0.5 mean(1 + ele - mu_e^2 - exp(ele)),  el = lv + log(nu / (nu + 1))
//   total    = loss_cls + reg_weight loss_reg + kl_weight loss_kl
//
// Every row is reduced by one warp: ||mu_i||^2, ||mu_e||^2 and mu_i . mu_e in float64, and the KL row sum in float64 of
// fp32 terms (el and exp(el) in fp32, so exp overflows to +inf exactly where torch's fp32 exp does).  The row sums are
// kept in a [B*T, 4] float64 record for the backward; rows are summed in slabs of kSlabRows in a fixed order and the slab
// sums by one block in a fixed order, so the scalars do not depend on the grid or the SM count and no atomics are used.
// The backward's gradient of a row is a per-row linear combination of mu_i and mu_e (plus the elementwise KL terms), with
// the coefficients computed in float64 from the record.  torch's edge rules are kept: F.normalize divides by
// max(|x|, 1e-12) and its clamp passes no gradient below it; cosine_similarity divides each factor by max(|x|, 1e-8) with
// the clamp outside autograd, so the gradient reaches the norm unclamped; the gradients of |x| at 0 and of a norm at the
// zero vector are 0.  oracle/train_objective.py restates the same arithmetic.
#include <cmath>

#include "common.cuh"
#include "rank.cuh"
#include "train.cuh"

namespace iefvad {

namespace {

constexpr int kSlabRows = 16;                 // rows per block and per slab sum: one warp per row
constexpr int kRowThreads = 32 * kSlabRows;
constexpr int kFinalThreads = 256;

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);    // butterfly: every lane ends with the same bits
  return v;
}

struct RowTerms {
  double na, nb, ca, cb, cu, cv, cos;
};

__device__ __forceinline__ RowTerms row_terms(double sa, double sb, double sab) {
  RowTerms t;
  t.na = sqrt(sa);
  t.nb = sqrt(sb);
  t.ca = fmax(t.na, 1e-12);                   // F.normalize
  t.cb = fmax(t.nb, 1e-12);
  t.cu = fmax(t.na / t.ca, 1e-8);             // cosine_similarity of the normalised rows
  t.cv = fmax(t.nb / t.cb, 1e-8);
  t.cos = sab / (t.ca * t.cb * t.cu * t.cv);
  return t;
}

__device__ __forceinline__ double kl_term(float mu, float lv, float c) {
  const float el = lv + c;
  return (1.0 + double(el)) - double(mu) * double(mu) - double(expf(el));
}

__global__ void __launch_bounds__(kRowThreads)
train_loss_rows_kernel(const float4* __restrict__ mu_i, const float4* __restrict__ mu_e, const float4* __restrict__ lv_i,
                       const float4* __restrict__ lv_e, long long M, int D4, float c, double4* __restrict__ record,
                       double2* __restrict__ slab_sum) {
  __shared__ double s_reg[kSlabRows], s_kl[kSlabRows];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long r = (long long)blockIdx.x * kSlabRows + warp;
  double reg = 0.0, kl = 0.0;
  if (r < M) {
    double sa = 0.0, sb = 0.0, sab = 0.0;
    const long long base = r * D4;
#pragma unroll 2
    for (int k = lane; k < D4; k += 32) {
      const float4 a = __ldg(mu_i + base + k), b = __ldg(mu_e + base + k);
      const float4 la = __ldg(lv_i + base + k), lb = __ldg(lv_e + base + k);
      sa = fma(double(a.x), double(a.x), sa); sa = fma(double(a.y), double(a.y), sa);
      sa = fma(double(a.z), double(a.z), sa); sa = fma(double(a.w), double(a.w), sa);
      sb = fma(double(b.x), double(b.x), sb); sb = fma(double(b.y), double(b.y), sb);
      sb = fma(double(b.z), double(b.z), sb); sb = fma(double(b.w), double(b.w), sb);
      sab = fma(double(a.x), double(b.x), sab); sab = fma(double(a.y), double(b.y), sab);
      sab = fma(double(a.z), double(b.z), sab); sab = fma(double(a.w), double(b.w), sab);
      kl += kl_term(a.x, la.x, c) + kl_term(a.y, la.y, c) + kl_term(a.z, la.z, c) + kl_term(a.w, la.w, c);
      kl += kl_term(b.x, lb.x, c) + kl_term(b.y, lb.y, c) + kl_term(b.z, lb.z, c) + kl_term(b.w, lb.w, c);
    }
    sa = warp_sum(sa);
    sb = warp_sum(sb);
    sab = warp_sum(sab);
    kl = warp_sum(kl);
    const RowTerms t = row_terms(sa, sb, sab);
    reg = (1.0 - t.cos) + fabs(t.na - t.nb);
    if (lane == 0) record[r] = make_double4(sa, sb, sab, kl);
  }
  if (lane == 0) {
    s_reg[warp] = reg;
    s_kl[warp] = kl;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    double sr = 0.0, sk = 0.0;
    for (int j = 0; j < kSlabRows; ++j) {
      sr += s_reg[j];
      sk += s_kl[j];
    }
    slab_sum[blockIdx.x] = make_double2(sr, sk);
  }
}

// one block: the slab sums in a fixed order, then the three losses and the total (CLAS2's scalar read from the device)
__global__ void __launch_bounds__(kFinalThreads)
train_loss_final_kernel(const double2* __restrict__ slab_sum, int nslab, double inv_M, double inv_N, double reg_w, double kl_w,
                        const float* __restrict__ loss_cls, float* __restrict__ total, float* __restrict__ loss_reg,
                        float* __restrict__ loss_kl) {
  __shared__ double sr[kFinalThreads], sk[kFinalThreads];
  double r = 0.0, k = 0.0;
  for (int i = threadIdx.x; i < nslab; i += kFinalThreads) {
    r += slab_sum[i].x;
    k += slab_sum[i].y;
  }
  sr[threadIdx.x] = r;
  sk[threadIdx.x] = k;
  __syncthreads();
  for (int s = kFinalThreads / 2; s > 0; s >>= 1) {
    if (threadIdx.x < s) {
      sr[threadIdx.x] += sr[threadIdx.x + s];
      sk[threadIdx.x] += sk[threadIdx.x + s];
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    const double reg = sr[0] * inv_M, kl = -0.5 * sk[0] * inv_N;
    *loss_reg = float(reg);
    *loss_kl = float(kl);
    *total = float(double(*loss_cls) + reg_w * reg + kl_w * kl);
  }
}

__device__ __forceinline__ double upstream(const float* g) { return g ? double(*g) : 0.0; }

__device__ __forceinline__ float4 lin2(double alpha, float4 y, double beta, float4 x) {
  return make_float4(float(alpha * y.x + beta * x.x), float(alpha * y.y + beta * x.y), float(alpha * y.z + beta * x.z),
                     float(alpha * y.w + beta * x.w));
}

__device__ __forceinline__ float4 kl_grad(float k, float4 lv, float c) {
  return make_float4(k * expm1f(lv.x + c), k * expm1f(lv.y + c), k * expm1f(lv.z + c), k * expm1f(lv.w + c));
}

// one warp per row: d_mu_i = alpha_a mu_e + beta_a mu_i, d_mu_e = alpha_b mu_i + beta_b mu_e,
// d_lv = 0.5 G_kl / N (exp(el) - 1).  Block 0 also writes the CLAS2 backward's coefficient g_total + g_cls.
__global__ void __launch_bounds__(kRowThreads)
train_loss_bwd_kernel(const float4* __restrict__ mu_i, const float4* __restrict__ mu_e, const float4* __restrict__ lv_i,
                      const float4* __restrict__ lv_e, const double4* __restrict__ record, long long M, int D4, float c,
                      double inv_M, double inv_N, double reg_w, double kl_w, const float* __restrict__ g_total,
                      const float* __restrict__ g_cls, const float* __restrict__ g_reg, const float* __restrict__ g_kl,
                      float* __restrict__ g_cls_total, float4* __restrict__ d_mu_i, float4* __restrict__ d_mu_e,
                      float4* __restrict__ d_lv_i, float4* __restrict__ d_lv_e) {
  const double gt = upstream(g_total);
  if (blockIdx.x == 0 && threadIdx.x == 0) *g_cls_total = float(gt + upstream(g_cls));
  const long long r = (long long)blockIdx.x * kSlabRows + (threadIdx.x >> 5);
  if (r >= M) return;
  const int lane = threadIdx.x & 31;
  const double G_reg = gt * reg_w + upstream(g_reg), G_kl = gt * kl_w + upstream(g_kl);
  const double4 rec = record[r];
  const double sa = rec.x, sb = rec.y, sab = rec.z;
  const RowTerms t = row_terms(sa, sb, sab);
  const double gc = -G_reg * inv_M;                       // d loss / d cos of this row
  const double inv_na = t.na > 0.0 ? 1.0 / t.na : 0.0, inv_nb = t.nb > 0.0 ? 1.0 / t.nb : 0.0;
  const double sgn = t.na > t.nb ? 1.0 : (t.na < t.nb ? -1.0 : 0.0);
  const double g_norm = G_reg * inv_M * sgn;              // d loss / d (norm_a - norm_b)
  const double kl_mu = G_kl * inv_N;
  // u = a / ca, w = b / cb: d cos / d u = w / (cu cv) - (cos / cu) a / na; through normalize,
  // d / da = g_u / ca - (g_u . a) / ca^2 [na >= 1e-12] a / na
  const double gw = gc / (t.cu * t.cv);
  const double gxa = -gc * t.cos / t.cu * inv_na, gxb = -gc * t.cos / t.cv * inv_nb;
  const double dota = gw * (sab / t.cb) + gxa * sa, dotb = gw * (sab / t.ca) + gxb * sb;
  const double alpha_a = gw / (t.cb * t.ca), alpha_b = alpha_a;
  const double beta_a = gxa / t.ca - dota / (t.ca * t.ca) * (t.na >= 1e-12 ? inv_na : 0.0) + g_norm * inv_na + kl_mu;
  const double beta_b = gxb / t.cb - dotb / (t.cb * t.cb) * (t.nb >= 1e-12 ? inv_nb : 0.0) - g_norm * inv_nb + kl_mu;
  const float k_lv = float(0.5 * G_kl * inv_N);
  const long long base = r * D4;
  for (int k = lane; k < D4; k += 32) {
    const float4 a = __ldg(mu_i + base + k), b = __ldg(mu_e + base + k);
    const float4 la = __ldg(lv_i + base + k), lb = __ldg(lv_e + base + k);
    d_mu_i[base + k] = lin2(alpha_a, b, beta_a, a);
    d_mu_e[base + k] = lin2(alpha_b, a, beta_b, b);
    d_lv_i[base + k] = kl_grad(k_lv, la, c);
    d_lv_e[base + k] = kl_grad(k_lv, lb, c);
  }
}

}  // namespace

int train_loss_slabs(long long rows) { return int((rows + kSlabRows - 1) / kSlabRows); }

int train_loss_fwd(const float* logits, const float* labels, long long label_stride, const long long* lengths, int B, int T,
                   const float* mu_i, const float* mu_e, const float* lv_i, const float* lv_e, int D, double nu, double reg_w,
                   double kl_w, float* means, int* idx, int kmax, double* record, double* slab_scratch, float* total,
                   float* loss_cls, float* loss_reg, float* loss_kl, cudaStream_t stream) {
  const long long M = (long long)B * T;
  const int nslab = train_loss_slabs(M);
  const float c = float(std::log(nu / (nu + 1.0)));
  IEF_TRY(clas2(logits, labels, label_stride, lengths, B, T, means, loss_cls, stream, idx, kmax));
  train_loss_rows_kernel<<<nslab, kRowThreads, 0, stream>>>(
      reinterpret_cast<const float4*>(mu_i), reinterpret_cast<const float4*>(mu_e), reinterpret_cast<const float4*>(lv_i),
      reinterpret_cast<const float4*>(lv_e), M, D / 4, c, reinterpret_cast<double4*>(record),
      reinterpret_cast<double2*>(slab_scratch));
  train_loss_final_kernel<<<1, kFinalThreads, 0, stream>>>(reinterpret_cast<const double2*>(slab_scratch), nslab, 1.0 / double(M),
                                                           1.0 / (double(M) * D), reg_w, kl_w, loss_cls, total, loss_reg, loss_kl);
  count_launches(2);
  IEF_CUDA(cudaGetLastError());
  return IEFVAD_OK;
}

int train_loss_bwd(const float* logits, const float* means, const float* labels, long long label_stride, const int* idx, int B,
                   int T, int kmax, const float* mu_i, const float* mu_e, const float* lv_i, const float* lv_e, int D,
                   const double* record, double nu, double reg_w, double kl_w, const float* g_total, const float* g_cls,
                   const float* g_reg, const float* g_kl, float* g_cls_scratch, float* d_logits, float* d_mu_i, float* d_mu_e,
                   float* d_lv_i, float* d_lv_e, cudaStream_t stream) {
  const long long M = (long long)B * T;
  const float c = float(std::log(nu / (nu + 1.0)));
  train_loss_bwd_kernel<<<train_loss_slabs(M), kRowThreads, 0, stream>>>(
      reinterpret_cast<const float4*>(mu_i), reinterpret_cast<const float4*>(mu_e), reinterpret_cast<const float4*>(lv_i),
      reinterpret_cast<const float4*>(lv_e), reinterpret_cast<const double4*>(record), M, D / 4, c, 1.0 / double(M),
      1.0 / (double(M) * D), reg_w, kl_w, g_total, g_cls, g_reg, g_kl, g_cls_scratch, reinterpret_cast<float4*>(d_mu_i),
      reinterpret_cast<float4*>(d_mu_e), reinterpret_cast<float4*>(d_lv_i), reinterpret_cast<float4*>(d_lv_e));
  count_launches(1);
  IEF_CUDA(cudaGetLastError());
  return clas2_bwd(logits, means, labels, label_stride, idx, B, T, kmax, g_cls_scratch, d_logits, stream);
}

}  // namespace iefvad
