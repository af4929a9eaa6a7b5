// Rows D1-D4: SimilarityAdj / DistanceAdj / GraphConvolution (model/layers.py) and the CLIP-style Transformer
// (model/module.py).  The dense contractions reuse gemm_tc / gemm_simt / attn_tc; this file adds the HBM-bound
// pieces (adjacency writers, row softmax, the bidirectional distance scan, padding / layout copies) and the host
// orchestration.  Shapes are padded to multiples of 64 rows in scratch so that every GEMM constraint holds for
// ragged T; the valid region is copied out at the end (no-ops when T % 64 == 0).
#include "graph.cuh"

#include <cmath>
#include <vector>

#include "attention.cuh"
#include "elementwise.cuh"
#include "gemm.cuh"

namespace iefvad {

namespace {

inline int round_up(int v, int a) { return (v + a - 1) / a * a; }

// ------------------------------------------------------------------------------------------------ D2
// exp(-d / e) depends on d = |i - j| only: a T-entry table in smem, then pure 128-bit row writes.
__global__ void __launch_bounds__(256)
distance_adj_kernel(float* __restrict__ out, int T, long long rows_total) {
  extern __shared__ float table[];
  const float e = expf(1.0f);                                  // torch.exp(torch.tensor(1.)), layers.py:177
  for (int d = threadIdx.x; d < T; d += blockDim.x) table[d] = expf(-float(d) / e);
  __syncthreads();
  for (long long row = blockIdx.x; row < rows_total; row += gridDim.x) {
    const int i = int(row % T);
    float* o = out + row * T;
    for (int j = threadIdx.x; j < T; j += blockDim.x) o[j] = table[i > j ? i - j : j - i];
  }
}

// ------------------------------------------------------------------------------------------------ D3 scan
// y_t = sum_k r^|t-k| s_k = s_t + f_t + g_t with f_t = r (f_{t-1} + s_{t-1}), g_t = r (g_{t+1} + s_{t+1}).
// The map carry -> carry * r^len + E of a segment is affine, so segments compose associatively:
//   pass 1  (segment, column): exit values E_f = sum_i r^(len-i) s_i and E_b = sum_i r^(i+1) s_i of a 64-row segment
//   pass 2  (column)         : scan of the affine maps over the segments -> carry entering every segment (both ways)
//   pass 3  (segment, column): replay the segment from registers with its carries, write y
// Lanes run along the feature dimension (coalesced 128-byte rows), the 64 rows of a segment sit in registers.
constexpr int SEG = 64;

__global__ void __launch_bounds__(128)
scan_reduce_kernel(const float* __restrict__ s, int T, int D, int nseg, float r, float* __restrict__ Ef,
                   float* __restrict__ Eb) {
  const int col = blockIdx.x * 128 + threadIdx.x;
  const int seg = blockIdx.y;
  const long long b = blockIdx.z;
  if (col >= D) return;
  const int t0 = seg * SEG;
  const int len = (T - t0 < SEG) ? T - t0 : SEG;
  const float* p = s + (b * T + t0) * D + col;
  float ef = 0.f, eb = 0.f, pw = r;
  for (int i = 0; i < len; ++i) {
    const float v = p[(long long)i * D];
    ef = r * (ef + v);
    eb = fmaf(pw, v, eb);
    pw *= r;
  }
  Ef[(b * nseg + seg) * D + col] = ef;
  Eb[(b * nseg + seg) * D + col] = eb;
}

// in place: Ef[seg] <- forward carry entering segment seg, Eb[seg] <- backward carry entering it from the right
__global__ void __launch_bounds__(128)
scan_carry_kernel(float* __restrict__ Ef, float* __restrict__ Eb, int T, int D, int nseg, float r) {
  const int col = blockIdx.x * 128 + threadIdx.x;
  const long long b = blockIdx.y;
  if (col >= D) return;
  float* ef = Ef + b * nseg * D + col;
  float* eb = Eb + b * nseg * D + col;
  const float rseg = powf(r, float(SEG));
  float c = 0.f;
  for (int g = 0; g < nseg; ++g) {                        // carry_{g+1} = r^len_g carry_g + E_g  (len_g = SEG but for the tail,
    const float e = ef[(long long)g * D];                 // whose exit value is never consumed)
    ef[(long long)g * D] = c;
    c = fmaf(rseg, c, e);
  }
  c = 0.f;
  for (int g = nseg - 1; g >= 0; --g) {
    const int len = (T - g * SEG < SEG) ? T - g * SEG : SEG;
    const float e = eb[(long long)g * D];
    eb[(long long)g * D] = c;
    c = fmaf(powf(r, float(len)), c, e);
  }
}

__global__ void __launch_bounds__(128)
scan_apply_kernel(const float* __restrict__ s, int T, int D, int nseg, float r, const float* __restrict__ Cf,
                  const float* __restrict__ Cb, float* __restrict__ y) {
  const int col = blockIdx.x * 128 + threadIdx.x;
  const int seg = blockIdx.y;
  const long long b = blockIdx.z;
  if (col >= D) return;
  const int t0 = seg * SEG;
  const int len = (T - t0 < SEG) ? T - t0 : SEG;
  const float* p = s + (b * T + t0) * D + col;
  float* q = y + (b * T + t0) * D + col;
  float v[SEG], f[SEG];
#pragma unroll
  for (int i = 0; i < SEG; ++i) v[i] = (i < len) ? p[(long long)i * D] : 0.f;
  float c = Cf[(b * nseg + seg) * D + col];                // f at the first row of the segment
#pragma unroll
  for (int i = 0; i < SEG; ++i) {
    f[i] = c;
    c = r * (c + v[i]);
  }
  c = Cb[(b * nseg + seg) * D + col];                      // g at the last row of the segment
#pragma unroll
  for (int i = SEG - 1; i >= 0; --i) {
    if (i < len) {
      q[(long long)i * D] = v[i] + f[i] + c;
      c = r * (c + v[i]);
    }
  }
}

// ------------------------------------------------------------------------------------------------ D1 pieces
__global__ void __launch_bounds__(256)
row_norm_kernel(const float* __restrict__ x, long long rows, int D, int ld, float* __restrict__ nrm) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (long long row = (long long)blockIdx.x * 8 + warp; row < rows; row += (long long)gridDim.x * 8) {
    const float* p = x + row * ld;
    float s = 0.f;
    for (int j = lane; j < D; j += 32) s = fmaf(p[j], p[j], s);
    s = warp_sum(s);
    if (lane == 0) nrm[row] = sqrtf(s);
  }
}

// sim [Tp, Tp] (raw theta.theta^T of one batch element) -> out [T, T]: cosine, threshold(0.7 -> 0), row softmax over
// the first `len` columns; rows / columns >= len stay 0 (layers.py:142-156).  One CTA per row, row staged in smem.
__global__ void __launch_bounds__(256)
simadj_softmax_kernel(const float* __restrict__ sim, int ld, const float* __restrict__ nrm, int T, int len,
                      float* __restrict__ out) {
  extern __shared__ float rowbuf[];
  __shared__ float red[8];
  const int i = blockIdx.x;
  float* o = out + (long long)i * T;
  if (i >= len) {
    for (int j = threadIdx.x; j < T; j += blockDim.x) o[j] = 0.f;
    return;
  }
  const float ni = nrm[i];
  const float* srow = sim + (long long)i * ld;
  float mx = -INFINITY;
  for (int j = threadIdx.x; j < len; j += blockDim.x) {
    float c = srow[j] / (ni * nrm[j] + 1e-20f);
    c = (c > 0.7f) ? c : 0.f;                               // F.threshold(x, 0.7, 0)
    rowbuf[j] = c;
    mx = fmaxf(mx, c);
  }
  mx = warp_max(mx);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = mx;
  __syncthreads();
  mx = red[0];
#pragma unroll
  for (int w = 1; w < 8; ++w) mx = fmaxf(mx, red[w]);
  __syncthreads();
  float sum = 0.f;
  for (int j = threadIdx.x; j < len; j += blockDim.x) {
    const float e = expf(rowbuf[j] - mx);
    rowbuf[j] = e;
    sum += e;
  }
  sum = warp_sum(sum);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = sum;
  __syncthreads();
  sum = 0.f;
#pragma unroll
  for (int w = 0; w < 8; ++w) sum += red[w];
  for (int j = threadIdx.x; j < T; j += blockDim.x) o[j] = (j < len) ? rowbuf[j] / sum : 0.f;
}

// ------------------------------------------------------------------------------------------------ copies
// im2col of Conv1d(k = 5, pad = 2) along T: dst[t, k * Din + c] = x[t + k - 2, c] (0 outside [0, T)), rows t < Tp
__global__ void __launch_bounds__(256)
im2col5_kernel(const float* __restrict__ x, int T, int Din, int Tp, float* __restrict__ dst_f32, bf16* __restrict__ dst_hi,
               bf16* __restrict__ dst_lo) {
  const long long total = (long long)Tp * 5 * Din;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int t = int(i / (5 * Din));
    const int rem = int(i - (long long)t * 5 * Din);
    const int k = rem / Din, c = rem - k * Din;
    const int ts = t + k - 2;
    const float v = (t < T && ts >= 0 && ts < T) ? x[(long long)ts * Din + c] : 0.f;
    if (dst_f32) dst_f32[i] = v;
    if (dst_hi) {
      bf16 h, l;
      split_bf16(v, h, l);
      dst_hi[i] = h;
      if (dst_lo) dst_lo[i] = l;
    }
  }
}

// dst[r, :cols] = src[r, :cols] for r < rows (row pitches differ)
__global__ void __launch_bounds__(256)
crop2d_kernel(const float* __restrict__ src, long long ld_src, int rows, int cols, float* __restrict__ dst, long long ld_dst) {
  const long long total = (long long)rows * cols;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int r = int(i / cols), c = int(i - (long long)r * cols);
    dst[r * ld_dst + c] = src[r * ld_src + c];
  }
}

// [A, B, D] -> [B, A, D] (seq-first <-> batch-first), 128-bit rows
__global__ void __launch_bounds__(256)
swap01_kernel(const float* __restrict__ src, int A, int B, int D4, float* __restrict__ dst) {
  const long long total = (long long)A * B * D4;
  const float4* s4 = reinterpret_cast<const float4*>(src);
  float4* d4 = reinterpret_cast<float4*>(dst);
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int c = int(i % D4);
    const long long rb = i / D4;                 // = b * A + a in the destination
    const int a = int(rb % A), b = int(rb / A);
    d4[i] = s4[((long long)a * B + b) * D4 + c];
  }
}

// o = s + bias[col] + resid (bias / resid optional), 128-bit
__global__ void __launch_bounds__(256)
add_bias_resid_kernel(const float* __restrict__ s, const float* __restrict__ bias, const float* __restrict__ resid,
                      float* __restrict__ o, int D4, long long n4) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
    float4 v = reinterpret_cast<const float4*>(s)[i];
    if (bias) {
      const float4 b = __ldg(reinterpret_cast<const float4*>(bias) + int(i % D4));
      v.x += b.x; v.y += b.y; v.z += b.z; v.w += b.w;
    }
    if (resid) {
      const float4 r = reinterpret_cast<const float4*>(resid)[i];
      v.x += r.x; v.y += r.y; v.z += r.z; v.w += r.w;
    }
    reinterpret_cast<float4*>(o)[i] = v;
  }
}

int check_dims(const char* who, int Din, int Dout, int plan) {
  const int a = plan < 0 ? 16 : 64;
  IEF_CHECK(Din > 0 && Dout > 0 && Din % a == 0 && Dout % a == 0,
            "%s: feature sizes must be multiples of %d for this plan (Din=%d, Dout=%d)", who, a, Din, Dout);
  IEF_CHECK(plan >= -1 && plan <= 1, "%s: plan must be -1 (fp32), 0 (bf16) or 1 (split-bf16)", who);
  return IEFVAD_OK;
}

}  // namespace

int distance_adj(float* out, long long B, int T, cudaStream_t stream) {
  IEF_CHECK(B >= 0 && T >= 0 && T <= 49152 / 4 * 4 && out, "distance_adj: need out, B >= 0, 0 <= T <= 49152");
  if (B == 0 || T == 0) return IEFVAD_OK;
  const long long rows = B * T;
  const size_t smem = size_t(T) * sizeof(float);
  static bool attr_set = false;
  if (!attr_set) {
    IEF_CUDA(cudaFuncSetAttribute(distance_adj_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 49152 * 4));
    attr_set = true;
  }
  const int grid = int(rows < 148 * 8 ? rows : 148 * 8);
  distance_adj_kernel<<<grid, 256, smem, stream>>>(out, T, rows);
  count_launches(1);
  IEF_CUDA(cudaGetLastError());
  return IEFVAD_OK;
}

int distance_scan(const float* s, long long B, int T, int D, float* y, cudaStream_t stream) {
  IEF_CHECK(s && y && B >= 0 && T >= 0 && D > 0, "distance_scan: bad argument");
  IEF_CHECK(B <= 65535, "distance_scan: batch %lld exceeds the grid limit", B);
  if (B == 0 || T == 0) return IEFVAD_OK;
  const int nseg = (T + SEG - 1) / SEG;
  IEF_CHECK(nseg <= 65535, "distance_scan: T too long");
  const float r = expf(-1.0f / expf(1.0f));
  Scratch sc(stream);
  float *Ef, *Eb;
  IEF_TRY(sc.get(&Ef, size_t(B) * nseg * D));
  IEF_TRY(sc.get(&Eb, size_t(B) * nseg * D));
  const int cg = (D + 127) / 128;
  scan_reduce_kernel<<<dim3(cg, nseg, unsigned(B)), 128, 0, stream>>>(s, T, D, nseg, r, Ef, Eb);
  scan_carry_kernel<<<dim3(cg, unsigned(B)), 128, 0, stream>>>(Ef, Eb, T, D, nseg, r);
  scan_apply_kernel<<<dim3(cg, nseg, unsigned(B)), 128, 0, stream>>>(s, T, D, nseg, r, Ef, Eb, y);
  count_launches(3);
  IEF_CUDA(cudaGetLastError());
  return IEFVAD_OK;
}

int similarity_adj(const float* x, const float* w0t, const long long* seq_len_host, long long B, int T, int Din,
                   int Dout, int plan, float* out, int num_sms, cudaStream_t st) {
  IEF_CHECK(x && w0t && out && B >= 0 && T >= 0, "similarity_adj: bad argument");
  IEF_TRY(check_dims("similarity_adj", Din, Dout, plan));
  IEF_CHECK(T <= 49152, "similarity_adj: T=%d exceeds the row buffer (49152)", T);
  if (B == 0 || T == 0) return IEFVAD_OK;
  const int Tp = round_up(T, 64);
  Scratch sc(st);
  Mat w;
  IEF_TRY(to_mat(sc, &w, w0t, Dout, Din, Din, Dout, Din, plan, num_sms, st));
  float *theta32, *nrm, *sim;
  IEF_TRY(sc.get(&theta32, size_t(Tp) * Dout));
  IEF_TRY(sc.get(&nrm, size_t(Tp)));
  IEF_TRY(sc.get(&sim, size_t(Tp) * Tp));
  static bool attr_set = false;
  if (!attr_set) {
    IEF_CUDA(cudaFuncSetAttribute(simadj_softmax_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 49152 * 4));
    attr_set = true;
  }
  for (long long b = 0; b < B; ++b) {
    const int len = seq_len_host ? int(seq_len_host[b] < 0 ? 0 : (seq_len_host[b] > T ? T : seq_len_host[b])) : T;
    Mat xb, theta;
    IEF_TRY(to_mat(sc, &xb, x + b * T * Din, T, Din, Din, Tp, Din, plan, num_sms, st));
    IEF_TRY(alloc_mat(sc, &theta, size_t(Tp), Dout, plan));
    // theta = x W0 (layers.py:132; phi is the same product, :133): fp32 copy for the norms + operand copy for theta theta^T
    EpiParams e1;
    e1.out_f32 = theta32; e1.ld_f32 = Dout;
    if (plan >= 0) { e1.out_hi = theta.hi; e1.out_lo = theta.lo; e1.ld_bf = Dout; }
    else theta.f = theta32;
    IEF_TRY(gemm_plan(plan, xb, w, Tp, Dout, Din, e1, nullptr, num_sms, st));
    row_norm_kernel<<<blocks_for((long long)Tp * 32, num_sms), 256, 0, st>>>(theta32, Tp, Dout, Dout, nrm);
    EpiParams e2;
    e2.out_f32 = sim; e2.ld_f32 = Tp;
    IEF_TRY(gemm_plan(plan, theta, theta, Tp, Tp, Dout, e2, nullptr, num_sms, st));
    simadj_softmax_kernel<<<T, 256, size_t(T) * sizeof(float), st>>>(sim, Tp, nrm, T, len, out + b * T * T);
    count_launches(2);
    IEF_CUDA(cudaGetLastError());
  }
  return IEFVAD_OK;
}

int graph_convolution(const float* x, const float* adj, const float* wt, const float* bias, int residual,
                      const float* conv_w, const float* conv_b, long long B, int T, int Din, int Dout, int plan,
                      float* out, int num_sms, cudaStream_t st) {
  IEF_CHECK(x && wt && out && B >= 0 && T >= 0, "graph_convolution: bad argument");
  IEF_TRY(check_dims("graph_convolution", Din, Dout, plan));
  IEF_CHECK(residual >= 0 && residual <= 2, "graph_convolution: residual mode in {0, 1, 2}");
  IEF_CHECK(residual != 1 || Din == Dout, "graph_convolution: the identity residual needs Din == Dout");
  IEF_CHECK(residual != 2 || (conv_w && conv_b), "graph_convolution: the Conv1d residual needs conv_w and conv_b");
  if (B == 0 || T == 0) return IEFVAD_OK;
  const int Tp = round_up(T, 64);
  Scratch sc(st);
  Mat w, cw;
  IEF_TRY(to_mat(sc, &w, wt, Dout, Din, Din, Dout, Din, plan, num_sms, st));
  if (residual == 2) IEF_TRY(to_mat(sc, &cw, conv_w, Dout, 5 * Din, 5 * Din, Dout, 5 * Din, plan, num_sms, st));
  float *outp, *res32 = nullptr, *sup32 = nullptr;
  IEF_TRY(sc.get(&outp, size_t(Tp) * Dout));
  if (residual == 2) IEF_TRY(sc.get(&res32, size_t(Tp) * Dout));
  for (long long b = 0; b < B; ++b) {
    Scratch sb(st);                               // this batch element's operands, back to the pool at the end of the loop body
    const float* xb32 = x + b * T * Din;
    Mat xb;
    IEF_TRY(to_mat(sb, &xb, xb32, T, Din, Din, Tp, Din, plan, num_sms, st));
    // residual term (layers.py:98-104): identity -> the (zero-padded) input itself; Conv1d -> one GEMM over im2col rows
    const float* resid = nullptr;
    if (residual == 1) {
      Mat xf;                                     // the fp32 form of x_b (xb itself under plan -1)
      if (plan >= 0) IEF_TRY(to_mat(sb, &xf, xb32, T, Din, Din, Tp, Din, -1, num_sms, st));
      resid = plan < 0 ? xb.f : xf.f;
    } else if (residual == 2) {
      Mat col;
      IEF_TRY(alloc_mat(sb, &col, size_t(Tp), 5 * Din, plan));
      im2col5_kernel<<<blocks_for((long long)Tp * 5 * Din, num_sms), 256, 0, st>>>(xb32, T, Din, Tp, col.f, col.hi, col.lo);
      count_launches(1);
      EpiParams ec;
      ec.bias = conv_b; ec.out_f32 = res32; ec.ld_f32 = Dout;
      IEF_TRY(gemm_plan(plan, col, cw, Tp, Dout, 5 * Din, ec, nullptr, num_sms, st));
      resid = res32;
    }
    if (adj == nullptr) {
      // DistanceAdj adjacency: support = x W in fp32, then the bidirectional scan; bias / residual in a last pass
      if (!sup32) IEF_TRY(sc.get(&sup32, size_t(Tp) * Dout));
      EpiParams es;
      es.out_f32 = sup32; es.ld_f32 = Dout;
      IEF_TRY(gemm_plan(plan, xb, w, Tp, Dout, Din, es, nullptr, num_sms, st));
      IEF_TRY(distance_scan(sup32, 1, T, Dout, outp, st));
      // out = scan + bias + residual (rows of the scan output, the padded residual and `out` share the pitch Dout)
      add_bias_resid_kernel<<<blocks_for((long long)T * Dout / 4, num_sms), 256, 0, st>>>(
          outp, bias, resid, out + b * T * Dout, Dout / 4, (long long)T * Dout / 4);
      count_launches(1);
      IEF_CUDA(cudaGetLastError());
      continue;
    }
    // supportT [Dout, Tp] = W^T . x_b^T: C = A . W'^T with A = W^T [Dout, Din], W' = x_b [Tp, Din] -> K-major operand
    Mat supT;
    IEF_TRY(alloc_mat(sb, &supT, size_t(Dout), Tp, plan));
    EpiParams e1;
    IEF_TRY(gemm_plan(plan, w, xb, Dout, Tp, Din, e1, &supT, num_sms, st));
    Mat ab;
    IEF_TRY(to_mat(sb, &ab, adj + b * T * T, T, T, T, Tp, Tp, plan, num_sms, st));
    EpiParams e2;
    e2.bias = bias; e2.resid = resid; e2.ld_resid = Dout; e2.out_f32 = outp; e2.ld_f32 = Dout;
    IEF_TRY(gemm_plan(plan, ab, supT, Tp, Dout, Tp, e2, nullptr, num_sms, st));
    crop2d_kernel<<<blocks_for((long long)T * Dout, num_sms), 256, 0, st>>>(outp, Dout, T, Dout, out + b * T * Dout, Dout);
    count_launches(1);
    IEF_CUDA(cudaGetLastError());
  }
  return IEFVAD_OK;
}

int alloc_attn_work(Scratch& sc, AttnWork* w, int plan, int N, int L, int D, int heads) {
  const size_t M = size_t(N) * L;
  const int dh = D / heads, dhp = (dh + 63) / 64 * 64, Tpad = (L + 7) / 8 * 8;
  IEF_TRY(alloc_mat(sc, &w->ctx, M, D, plan == 1 ? 0 : plan));
  if (plan < 0) return sc.get(&w->qkv32, M * 3 * D);
  IEF_TRY(sc.get(&w->q, M * heads * dhp));
  IEF_TRY(sc.get(&w->k, M * heads * dhp));
  return sc.get(&w->vt, size_t(N) * heads * dh * Tpad);
}

int attention_sublayer(int plan, const Mat& x, const Mat& in_w, const float* in_b, const Mat& out_w, const float* out_b,
                       int N, int L, int D, int heads, const float* attn_mask, const uint8_t* key_pad, const float* resid,
                       float* out, const AttnWork& w, int num_sms, cudaStream_t st) {
  const int M = N * L, dh = D / heads;
  EpiParams e1;
  e1.bias = in_b;
  AttnTcArgs at;
  if (plan < 0) {
    e1.out_f32 = w.qkv32; e1.ld_f32 = 3 * D;
  } else {
    at.q = w.q; at.k = w.k; at.vt = w.vt; at.out = w.ctx.hi; at.ldo = D;
    at.B = N; at.T = L; at.H = heads; at.dh = dh; at.Tpad = (L + 7) / 8 * 8;
    at.attn_mask = attn_mask; at.key_pad = key_pad; at.fp16 = (plan == 2);
    at.dhp = attn_qk_cols(at);
    e1.mode = EPI_QKV; e1.q = w.q; e1.k = w.k; e1.vt = w.vt; e1.hi_fp16 = at.fp16;
    e1.T = L; e1.H = heads; e1.dh = dh; e1.dhp = at.dhp; e1.Tpad = at.Tpad; e1.D = D; e1.qscale = 1.0f / sqrtf(float(dh));
  }
  IEF_TRY(gemm_plan(plan, x, in_w, M, 3 * D, D, e1, nullptr, num_sms, st));
  IEF_TRY(plan < 0 ? attn_simt(w.qkv32, w.ctx.f, N, L, heads, dh, attn_mask, key_pad, st) : attn_tc(at, st));
  EpiParams e2;
  e2.bias = out_b; e2.resid = resid; e2.ld_resid = D; e2.out_f32 = out; e2.ld_f32 = D;
  return gemm_plan(plan == 1 ? 0 : plan, w.ctx, out_w, M, D, D, e2, nullptr, num_sms, st);
}

int transformer_blocks(float* xa, const ResBlockParams* blocks, int layers, int L, int N, int D, int heads,
                       const float* attn_mask, const uint8_t* key_pad, int plan, int num_sms, cudaStream_t st) {
  if (layers == 0 || L == 0 || N == 0) return IEFVAD_OK;
  const long long M = (long long)N * L;
  const int f16 = (plan == 2);
  Scratch sc(st);
  float* xb;                                      // second residual buffer: x alternates xa -> xb -> xa in each block
  IEF_TRY(sc.get(&xb, size_t(M) * D));
  Mat h, u;
  IEF_TRY(alloc_mat(sc, &h, size_t(M), D, plan));
  IEF_TRY(alloc_mat(sc, &u, size_t(M), 4 * D, plan));
  AttnWork aw;
  IEF_TRY(alloc_attn_work(sc, &aw, plan, N, L, D, heads));
  std::vector<Mat> wmats(size_t(layers) * 4);
  for (int i = 0; i < layers; ++i) {
    const ResBlockParams& p = blocks[i];
    IEF_CHECK(p.ln1_w && p.ln1_b && p.in_w && p.in_b && p.out_w && p.out_b && p.ln2_w && p.ln2_b && p.fc_w && p.fc_b &&
              p.proj_w && p.proj_b, "transformer: block %d has a null parameter", i);
    Mat &wi = wmats[4 * i], &wo = wmats[4 * i + 1], &wf = wmats[4 * i + 2], &wp = wmats[4 * i + 3];
    IEF_TRY(to_mat(sc, &wi, p.in_w, 3 * D, D, D, 3 * D, D, plan, num_sms, st));
    IEF_TRY(to_mat(sc, &wo, p.out_w, D, D, D, D, D, plan, num_sms, st));
    IEF_TRY(to_mat(sc, &wf, p.fc_w, 4 * D, D, D, 4 * D, D, plan, num_sms, st));
    IEF_TRY(to_mat(sc, &wp, p.proj_w, D, 4 * D, 4 * D, D, 4 * D, plan, num_sms, st));
    // x = x + attn(ln_1(x))   (module.py:41)
    IEF_TRY(layernorm(xa, M, D, p.ln1_w, p.ln1_b, nullptr, nullptr, 1e-5f, h.f, h.hi, h.lo, num_sms, st, f16));
    IEF_TRY(attention_sublayer(plan, h, wi, p.in_b, wo, p.out_b, N, L, D, heads, attn_mask, key_pad, xa, xb, aw, num_sms, st));
    // x = x + mlp(ln_2(x))   (module.py:42): c_fc + QuickGELU, then c_proj with the residual
    IEF_TRY(layernorm(xb, M, D, p.ln2_w, p.ln2_b, nullptr, nullptr, 1e-5f, h.f, h.hi, h.lo, num_sms, st, f16));
    EpiParams e3;
    e3.bias = p.fc_b; e3.act = ACT_QUICKGELU;
    IEF_TRY(gemm_plan(plan, h, wf, int(M), 4 * D, D, e3, &u, num_sms, st));
    EpiParams e4;
    e4.bias = p.proj_b; e4.resid = xb; e4.ld_resid = D; e4.out_f32 = xa; e4.ld_f32 = D;
    IEF_TRY(gemm_plan(plan, u, wp, int(M), D, 4 * D, e4, nullptr, num_sms, st));
  }
  IEF_CUDA(cudaGetLastError());
  return IEFVAD_OK;
}

int transformer(const float* x, const ResBlockParams* blocks, int layers, int L, int N, int D, int heads,
                const float* attn_mask, const uint8_t* key_pad, int plan, float* out, int num_sms, cudaStream_t st) {
  IEF_CHECK(x && out && blocks && layers >= 0 && L >= 0 && N >= 0, "transformer: bad argument");
  IEF_TRY(check_plan("transformer", plan));
  IEF_CHECK(D > 0 && D % 128 == 0 && heads > 0 && D % heads == 0, "transformer: width %d must be a multiple of 128 and of heads=%d", D, heads);
  const int dh = D / heads;
  IEF_CHECK(dh == 32 || dh == 64 || dh == 96 || dh == 128, "transformer: head dim %d unsupported (32, 64, 96, 128)", dh);
  IEF_CHECK(N <= 65535, "transformer: batch %d exceeds the grid limit", N);
  if (L == 0 || N == 0) return IEFVAD_OK;
  const long long M = (long long)N * L;
  IEF_CHECK(M < (1LL << 31), "transformer: too many rows");
  Scratch sc(st);
  float* xa;                                      // residual stream, batch-first [N, L, D]
  IEF_TRY(sc.get(&xa, size_t(M) * D));
  swap01_kernel<<<blocks_for(M * D / 4, num_sms), 256, 0, st>>>(x, L, N, D / 4, xa);   // [L, N, D] -> [N, L, D]
  count_launches(1);
  IEF_TRY(transformer_blocks(xa, blocks, layers, L, N, D, heads, attn_mask, key_pad, plan, num_sms, st));
  swap01_kernel<<<blocks_for(M * D / 4, num_sms), 256, 0, st>>>(xa, N, L, D / 4, out);   // [N, L, D] -> [L, N, D]
  count_launches(1);
  IEF_CUDA(cudaGetLastError());
  return IEFVAD_OK;
}

}  // namespace iefvad
