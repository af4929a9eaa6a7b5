// Ranking kernels of the hot path's tail:
//   * MIL top-k pooling of train/loss.py:18-30 (CLAS2): per-row sigmoid -> top-k (k = int(len/16 + 1)) -> mean -> BCE,
//     one CTA per row with a shared-memory bitonic sort; k comes from the device `lengths`, no host sync.
//   * frame-level AUC / AP of train/ucf_test.py:151-152 (scikit-learn's roc_auc_score / average_precision_score on
//     16x-repeated segment scores): stable descending LSD radix sort of the fp32 scores (hand-written: per-tile
//     histograms, bin-major offset scan, stable warp-match scatter), one associative scan producing cumulative
//     TP / FP (int64) and the tie-group index, then exact-integer trapezoid sums and a fixed-order float64 AP sum.
#include "common.cuh"
#include "rank.cuh"

namespace iefvad {

namespace {

// order-preserving fp32 -> u32 key, ascending in the float order; -0 and +0 collapse (numpy / torch treat them equal)
__device__ __forceinline__ uint32_t asc_key(float x) {
  if (x == 0.f) x = 0.f;
  const uint32_t u = __float_as_uint(x);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

// =================================================================================================
// MIL top-k mean
// =================================================================================================
__global__ void __launch_bounds__(256)
mil_topk_kernel(const float* __restrict__ x, const long long* __restrict__ lengths, int T, int npow2, int apply_sigmoid,
                float* __restrict__ mean_out, int* __restrict__ idx_out, int kmax) {
  extern __shared__ unsigned long long skeys[];
  __shared__ double red[8];
  const int row = blockIdx.x;
  long long len64 = lengths ? lengths[row] : T;
  const int len = int(len64 < 0 ? 0 : (len64 > T ? T : len64));
  const int k = len / 16 + 1;                                   // int(len / 16 + 1), train/loss.py:25
  const float* xr = x + (long long)row * T;
  for (int i = threadIdx.x; i < npow2; i += blockDim.x) {
    unsigned long long key = 0ull;                              // padding sorts last
    if (i < len) {
      float v = xr[i];
      if (apply_sigmoid) v = 1.f / (1.f + expf(-v));            // train/loss.py:22
      key = (static_cast<unsigned long long>(asc_key(v)) << 32) | (0xFFFFFFFFu - uint32_t(i));
    }
    skeys[i] = key;
  }
  __syncthreads();
  // bitonic sort, descending: larger value first, equal values by ascending index
  for (int size = 2; size <= npow2; size <<= 1) {
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      for (int i = threadIdx.x; i < npow2 / 2; i += blockDim.x) {
        const int lo = 2 * i - (i & (stride - 1));
        const int hi = lo + stride;
        const bool desc = ((lo & size) == 0);
        const unsigned long long a = skeys[lo], b = skeys[hi];
        if ((a < b) == desc) { skeys[lo] = b; skeys[hi] = a; }
      }
      __syncthreads();
    }
  }
  // mean of the first k values (fixed-order double accumulation)
  double s = 0.0;
  if (len > 0) {
    for (int i = threadIdx.x; i < k; i += blockDim.x) {
      const uint32_t a = uint32_t(skeys[i] >> 32);
      const uint32_t u = (a & 0x80000000u) ? (a & 0x7FFFFFFFu) : ~a;   // inverse of asc_key
      s += double(__uint_as_float(u));
      if (idx_out && i < kmax) idx_out[(long long)row * kmax + i] = int(0xFFFFFFFFu - uint32_t(skeys[i]));
    }
  }
  if (idx_out) for (int i = k + threadIdx.x; i < kmax; i += blockDim.x) idx_out[(long long)row * kmax + i] = -1;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int w = 0; w < int(blockDim.x >> 5); ++w) t += red[w];
    mean_out[row] = (len > 0) ? float(t / double(k)) : __int_as_float(0x7fc00000);
  }
}

// binary cross entropy of train/loss.py:20,29 on the per-row means; one block, fixed-order double sum
__global__ void __launch_bounds__(256)
bce_kernel(const float* __restrict__ v, const float* __restrict__ labels, long long label_stride, int B,
           float* __restrict__ loss) {
  __shared__ double red[8];
  double s = 0.0;
  for (int i = threadIdx.x; i < B; i += blockDim.x) {
    const float y = 1.f - labels[(long long)i * label_stride];  // 1 - labels[:, 0]
    const float p = v[i];
    const float lp = fmaxf(logf(p), -100.f);                    // torch clamps each log term at -100
    const float lq = fmaxf(logf(1.f - p), -100.f);
    s += double(-(y * lp + (1.f - y) * lq));
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int w = 0; w < 8; ++w) t += red[w];
    *loss = float(t / double(B));
  }
}

// =================================================================================================
// LSD radix sort: 32-bit keys + 32-bit payload, 8 bits per pass, stable
// =================================================================================================
constexpr int RS_THREADS = 256;
constexpr int RS_MAX_ITEMS = 16;                 // up to 4096 keys per CTA
// keys per thread: as many as keep ~2 CTAs per SM busy (a real split is <= 150 k scores: with 4096-key tiles 19 CTAs did all
// the work, and the scatter - 16 sequential rounds per CTA - took 25 us per pass), 16 for large inputs
static int rs_items(long long n) {
  long long it = n / (long long)(RS_THREADS) / 296;
  return it < 1 ? 1 : (it > RS_MAX_ITEMS ? RS_MAX_ITEMS : int(it));
}
constexpr int RS_BINS = 256;

__global__ void __launch_bounds__(RS_THREADS)
rs_init_kernel(const float* __restrict__ scores, long long n, uint32_t* __restrict__ keys, uint32_t* __restrict__ vals) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    keys[i] = ~asc_key(scores[i]);   // ascending sort of ~asc == descending by score
    vals[i] = uint32_t(i);
  }
}

__global__ void __launch_bounds__(RS_THREADS)
rs_hist_kernel(const uint32_t* __restrict__ keys, long long n, int shift, uint32_t* __restrict__ hist, int nblocks, int items) {
  __shared__ uint32_t h[RS_BINS];
  h[threadIdx.x] = 0;
  __syncthreads();
  const long long base = (long long)blockIdx.x * (RS_THREADS * items);
  for (int r = 0; r < items; ++r) {
    const long long i = base + r * RS_THREADS + threadIdx.x;
    if (i < n) atomicAdd(&h[(keys[i] >> shift) & 0xFF], 1u);
  }
  __syncthreads();
  hist[(long long)threadIdx.x * nblocks + blockIdx.x] = h[threadIdx.x];   // bin-major
}

// one CTA per bin: exclusive scan of that bin's per-tile counts (in place) + bin total
__global__ void __launch_bounds__(RS_THREADS)
rs_scan_bins_kernel(uint32_t* __restrict__ hist, int nblocks, uint32_t* __restrict__ totals) {
  __shared__ uint32_t warp_sums[RS_THREADS / 32];
  __shared__ uint32_t carry;
  uint32_t* row = hist + (long long)blockIdx.x * nblocks;
  if (threadIdx.x == 0) carry = 0;
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int b0 = 0; b0 < nblocks; b0 += RS_THREADS) {
    const int i = b0 + threadIdx.x;
    const uint32_t v = (i < nblocks) ? row[i] : 0u;
    uint32_t inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t t = __shfl_up_sync(0xffffffffu, inc, o);
      if (lane >= o) inc += t;
    }
    if (lane == 31) warp_sums[warp] = inc;
    __syncthreads();
    uint32_t woff = 0;
    for (int w = 0; w < warp; ++w) woff += warp_sums[w];
    const uint32_t c = carry;
    if (i < nblocks) row[i] = c + woff + inc - v;
    __syncthreads();
    if (threadIdx.x == RS_THREADS - 1) carry = c + woff + inc;
    __syncthreads();
  }
  if (threadIdx.x == 0) totals[blockIdx.x] = carry;
}

__global__ void __launch_bounds__(RS_THREADS)
rs_scatter_kernel(const uint32_t* __restrict__ keys_in, const uint32_t* __restrict__ vals_in, long long n, int shift,
                  const uint32_t* __restrict__ hist, int nblocks, const uint32_t* __restrict__ totals,
                  uint32_t* __restrict__ keys_out, uint32_t* __restrict__ vals_out, int items) {
  __shared__ uint32_t bin_base[RS_BINS];                  // global offset of this tile's first key of each bin
  __shared__ uint32_t running[RS_BINS];                   // keys of each bin already placed by earlier rounds
  __shared__ uint32_t warp_cnt[RS_THREADS / 32][RS_BINS];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  {
    // exclusive scan of the 256 bin totals (every CTA redoes it: 256 values, cheaper than another launch)
    __shared__ uint32_t ws[RS_THREADS / 32];
    const uint32_t v = totals[threadIdx.x];
    uint32_t inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t t = __shfl_up_sync(0xffffffffu, inc, o);
      if (lane >= o) inc += t;
    }
    if (lane == 31) ws[warp] = inc;
    __syncthreads();
    uint32_t woff = 0;
    for (int w = 0; w < warp; ++w) woff += ws[w];
    bin_base[threadIdx.x] = woff + inc - v + hist[(long long)threadIdx.x * nblocks + blockIdx.x];
    running[threadIdx.x] = 0;
  }
  for (int w = 0; w < RS_THREADS / 32; ++w) warp_cnt[w][threadIdx.x] = 0;
  __syncthreads();
  const long long base = (long long)blockIdx.x * (RS_THREADS * items);
  for (int r = 0; r < items; ++r) {
    const long long i = base + r * RS_THREADS + threadIdx.x;
    const bool valid = i < n;
    uint32_t key = 0, val = 0, digit = 0;
    if (valid) { key = keys_in[i]; val = vals_in[i]; digit = (key >> shift) & 0xFF; }
    // stable rank inside the warp: lanes with the same digit, ordered by lane
    const uint32_t active = __ballot_sync(0xffffffffu, valid);
    uint32_t peers = 0, rank_in_warp = 0;
    if (valid) {
      peers = __match_any_sync(active, digit);
      rank_in_warp = __popc(peers & ((1u << lane) - 1u));
      if (rank_in_warp == 0) warp_cnt[warp][digit] = __popc(peers);   // one writer per (warp, digit)
    }
    __syncthreads();
    uint32_t dst = 0;
    if (valid) {
      uint32_t before = running[digit];
      for (int w = 0; w < warp; ++w) before += warp_cnt[w][digit];
      dst = bin_base[digit] + before + rank_in_warp;
    }
    __syncthreads();
    {
      uint32_t tot = 0;
      for (int w = 0; w < RS_THREADS / 32; ++w) { tot += warp_cnt[w][threadIdx.x]; warp_cnt[w][threadIdx.x] = 0; }
      running[threadIdx.x] += tot;
    }
    __syncthreads();
    if (valid) { keys_out[dst] = key; vals_out[dst] = val; }
  }
}

// =================================================================================================
// Associative scan over the sorted segments: (cumulative positives, cumulative negatives, tie-group index)
// =================================================================================================
struct Tri { long long p, n, g; };
__device__ __forceinline__ Tri tri_add(const Tri& a, const Tri& b) { return {a.p + b.p, a.n + b.n, a.g + b.g}; }

constexpr int SC_THREADS = 256;
constexpr int SC_ITEMS = 8;
constexpr int SC_TILE = SC_THREADS * SC_ITEMS;

// `member` (optional): bit s of member[j] says whether segment j belongs to subset s.  Subsets share the GLOBAL
// ranking and the global tie groups: a segment outside the subset weighs (0, 0), and a tie group without members
// adds nothing to either sum, so the filtered result equals ranking the subset on its own (the stable sort keeps
// the relative order of its members) - class-wise and Ano-AUC cost one sort instead of one per class.
__device__ __forceinline__ Tri load_item(const uint32_t* keys, const uint32_t* order, const int* pos,
                                         const uint32_t* member, int subset, int repeat, long long i, long long n) {
  Tri t = {0, 0, 0};
  if (i < n) {
    const uint32_t j = order[i];
    if (member == nullptr || ((member[j] >> subset) & 1u)) {
      const int p = pos[j];
      t.p = p;
      t.n = repeat - p;
    }
    t.g = (i > 0 && keys[i] != keys[i - 1]) ? 1 : 0;       // a new (global) tie group starts here
  }
  return t;
}

__device__ __forceinline__ Tri block_exclusive_scan(Tri v, Tri* total_out) {
  __shared__ Tri ws[SC_THREADS / 32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  Tri inc = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    Tri t;
    t.p = __shfl_up_sync(0xffffffffu, inc.p, o);
    t.n = __shfl_up_sync(0xffffffffu, inc.n, o);
    t.g = __shfl_up_sync(0xffffffffu, inc.g, o);
    if (lane >= o) inc = tri_add(t, inc);
  }
  if (lane == 31) ws[warp] = inc;
  __syncthreads();
  Tri off = {0, 0, 0};
  for (int w = 0; w < warp; ++w) off = tri_add(off, ws[w]);
  if (total_out && threadIdx.x == SC_THREADS - 1) *total_out = tri_add(off, inc);
  Tri ex = tri_add(off, inc);
  ex.p -= v.p; ex.n -= v.n; ex.g -= v.g;
  __syncthreads();
  return ex;
}

// pass 1: per-tile totals
__global__ void __launch_bounds__(SC_THREADS)
sc_reduce_kernel(const uint32_t* __restrict__ keys, const uint32_t* __restrict__ order, const int* __restrict__ pos,
                 const uint32_t* __restrict__ member, int repeat, long long n, Tri* __restrict__ tile_sums) {
  __shared__ Tri total;
  const int subset = blockIdx.y;
  const long long base = (long long)blockIdx.x * SC_TILE + (long long)threadIdx.x * SC_ITEMS;
  Tri s = {0, 0, 0};
#pragma unroll
  for (int j = 0; j < SC_ITEMS; ++j) s = tri_add(s, load_item(keys, order, pos, member, subset, repeat, base + j, n));
  block_exclusive_scan(s, &total);
  __syncthreads();
  if (threadIdx.x == 0) tile_sums[(long long)subset * gridDim.x + blockIdx.x] = total;
}

// pass 2: exclusive scan of the tile totals (single CTA, sequential over chunks of 256 tiles)
__global__ void __launch_bounds__(SC_THREADS)
sc_scan_tiles_kernel(Tri* __restrict__ tile_sums, int ntiles, Tri* __restrict__ grand_total) {
  __shared__ Tri carry, total;
  tile_sums += (long long)blockIdx.x * ntiles;              // one CTA per subset
  grand_total += blockIdx.x;
  if (threadIdx.x == 0) carry = {0, 0, 0};
  __syncthreads();
  for (int b0 = 0; b0 < ntiles; b0 += SC_THREADS) {
    const int i = b0 + threadIdx.x;
    Tri v = {0, 0, 0};
    if (i < ntiles) v = tile_sums[i];
    Tri ex = block_exclusive_scan(v, &total);
    const Tri c = carry;
    if (i < ntiles) tile_sums[i] = tri_add(c, ex);
    __syncthreads();
    if (threadIdx.x == 0) carry = tri_add(c, total);
    __syncthreads();
  }
  if (threadIdx.x == 0) *grand_total = carry;
}

// pass 3: full scan; at every tie-group end write the cumulative (TP, FP) into the compacted group arrays
__global__ void __launch_bounds__(SC_THREADS)
sc_apply_kernel(const uint32_t* __restrict__ keys, const uint32_t* __restrict__ order, const int* __restrict__ pos,
                const uint32_t* __restrict__ member, int repeat, long long n, const Tri* __restrict__ tile_sums,
                long long* __restrict__ gtp, long long* __restrict__ gfp) {
  const int subset = blockIdx.y;
  gtp += (long long)subset * n;
  gfp += (long long)subset * n;
  const long long base = (long long)blockIdx.x * SC_TILE + (long long)threadIdx.x * SC_ITEMS;
  Tri items[SC_ITEMS];
  Tri s = {0, 0, 0};
#pragma unroll
  for (int j = 0; j < SC_ITEMS; ++j) {
    items[j] = load_item(keys, order, pos, member, subset, repeat, base + j, n);
    s = tri_add(s, items[j]);
  }
  Tri run = tri_add(tile_sums[(long long)subset * gridDim.x + blockIdx.x], block_exclusive_scan(s, nullptr));
#pragma unroll
  for (int j = 0; j < SC_ITEMS; ++j) {
    const long long i = base + j;
    run = tri_add(run, items[j]);                          // inclusive at i
    if (i < n) {
      const bool is_end = (i == n - 1) || (keys[i + 1] != keys[i]);
      if (is_end) { gtp[run.g] = run.p; gfp[run.g] = run.n; }
    }
  }
}

// per tie group: 2 x trapezoid area (exact int64) and the AP term (float64); fixed-order block partials
__global__ void __launch_bounds__(SC_THREADS)
auc_terms_kernel(const long long* __restrict__ gtp, const long long* __restrict__ gfp, long long n,
                 const Tri* __restrict__ grand, unsigned long long* __restrict__ area2_partial,
                 double* __restrict__ ap_partial) {
  __shared__ unsigned long long ra[SC_THREADS / 32];
  __shared__ double rp[SC_THREADS / 32];
  const int subset = blockIdx.y;
  gtp += (long long)subset * n;
  gfp += (long long)subset * n;
  grand += subset;
  area2_partial += (long long)subset * gridDim.x;
  ap_partial += (long long)subset * gridDim.x;
  const long long G = grand->g + 1;
  const double P = double(grand->p);
  unsigned long long a = 0;
  double ap = 0.0;
  for (long long g = (long long)blockIdx.x * SC_THREADS + threadIdx.x; g < G; g += (long long)gridDim.x * SC_THREADS) {
    const long long tp = gtp[g], fp = gfp[g];
    const long long tp0 = g ? gtp[g - 1] : 0, fp0 = g ? gfp[g - 1] : 0;
    a += static_cast<unsigned long long>((fp - fp0) * (tp + tp0));
    if (tp > tp0) ap += (double(tp - tp0) / P) * (double(tp) / double(tp + fp));
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    a += __shfl_xor_sync(0xffffffffu, a, o);
    ap += __shfl_xor_sync(0xffffffffu, ap, o);
  }
  if ((threadIdx.x & 31) == 0) { ra[threadIdx.x >> 5] = a; rp[threadIdx.x >> 5] = ap; }
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned long long ta = 0;
    double tp_ = 0.0;
    for (int w = 0; w < SC_THREADS / 32; ++w) { ta += ra[w]; tp_ += rp[w]; }
    area2_partial[blockIdx.x] = ta;
    ap_partial[blockIdx.x] = tp_;
  }
}

__global__ void auc_final_kernel(const unsigned long long* __restrict__ area2_partial,
                                 const double* __restrict__ ap_partial, int nparts, const Tri* __restrict__ grand,
                                 double* __restrict__ out) {
  area2_partial += (long long)blockIdx.x * nparts;          // one CTA (of one thread) per subset
  ap_partial += (long long)blockIdx.x * nparts;
  grand += blockIdx.x;
  out += 4 * blockIdx.x;
  unsigned long long a = 0;
  double ap = 0.0;
  for (int i = 0; i < nparts; ++i) { a += area2_partial[i]; ap += ap_partial[i]; }
  const double P = double(grand->p), N = double(grand->n);
  const double nan = __longlong_as_double(0x7ff8000000000000LL);
  out[0] = (grand->p > 0 && grand->n > 0) ? double(a) / (2.0 * P * N) : nan;   // roc_auc_score (NaN: one class only)
  out[1] = (grand->p > 0) ? ap : 0.0;                                          // average_precision_score
  out[2] = P;
  out[3] = N;
}

// dst[dst_off[s] + i] = src[src_off[s] + i], i < len[s]: drops the zero-pad rows of chunked videos
// (train/ucf_test.py:113 `logits1[0:len_cur]`) and re-orders gathered per-rank score vectors into list order.
__global__ void __launch_bounds__(256)
segment_copy_kernel(const float* __restrict__ src, const long long* __restrict__ src_off, float* __restrict__ dst,
                    const long long* __restrict__ dst_off, const long long* __restrict__ len, int nseg) {
  for (int s = blockIdx.x; s < nseg; s += gridDim.x) {
    const float* a = src + src_off[s];
    float* b = dst + dst_off[s];
    const long long n = len[s];
    for (long long i = threadIdx.x; i < n; i += blockDim.x) b[i] = a[i];
  }
}

struct Tmp {
  cudaStream_t s;
  void* ptrs[16];
  int n = 0;
  explicit Tmp(cudaStream_t st) : s(st) {}
  ~Tmp() { for (int i = 0; i < n; ++i) cudaFreeAsync(ptrs[i], s); }
  template <typename T> int get(T** out, size_t count) {
    void* p = nullptr;
    IEF_CUDA(cudaMallocAsync(&p, (count ? count : 1) * sizeof(T), s));
    ptrs[n++] = p;
    *out = static_cast<T*>(p);
    return IEFVAD_OK;
  }
};

// sorts (keys, vals) ascending by key, stable; result ends in (keys_a, vals_a)
int radix_sort_pairs(uint32_t* keys_a, uint32_t* vals_a, uint32_t* keys_b, uint32_t* vals_b, long long n,
                     uint32_t* hist, uint32_t* totals, cudaStream_t st) {
  const int items = rs_items(n);
  const int nblocks = int((n + RS_THREADS * items - 1) / (RS_THREADS * items));
  uint32_t *ki = keys_a, *vi = vals_a, *ko = keys_b, *vo = vals_b;
  for (int pass = 0; pass < 4; ++pass) {
    const int shift = pass * 8;
    rs_hist_kernel<<<nblocks, RS_THREADS, 0, st>>>(ki, n, shift, hist, nblocks, items);
    rs_scan_bins_kernel<<<RS_BINS, RS_THREADS, 0, st>>>(hist, nblocks, totals);
    rs_scatter_kernel<<<nblocks, RS_THREADS, 0, st>>>(ki, vi, n, shift, hist, nblocks, totals, ko, vo, items);
    count_launches(3);
    uint32_t* t = ki; ki = ko; ko = t;
    t = vi; vi = vo; vo = t;
  }
  IEF_CUDA(cudaGetLastError());
  return IEFVAD_OK;   // 4 passes: data is back in (keys_a, vals_a)
}

}  // namespace

int mil_topk_mean(const float* x, const long long* lengths, long long B, long long T, int apply_sigmoid, float* mean,
                  int* idx, int kmax, cudaStream_t stream) {
  IEF_CHECK(B >= 0 && T >= 1 && T <= 16384, "mil_topk_mean: T=%lld must be in [1, 16384]", T);
  IEF_CHECK(x && mean, "mil_topk_mean: null argument");
  if (B == 0) return IEFVAD_OK;
  int npow2 = 32;
  while (npow2 < T) npow2 <<= 1;
  const size_t smem = size_t(npow2) * sizeof(unsigned long long);
  static bool attr_set = false;
  if (!attr_set) {
    IEF_CUDA(cudaFuncSetAttribute(mil_topk_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 16384 * 8));
    attr_set = true;
  }
  mil_topk_kernel<<<unsigned(B), 256, smem, stream>>>(x, lengths, int(T), npow2, apply_sigmoid, mean, idx, kmax);
  count_launches(1);
  IEF_CUDA(cudaGetLastError());
  return IEFVAD_OK;
}

int clas2(const float* logits, const float* labels, long long label_stride, const long long* lengths, long long B,
          long long T, float* means, float* loss, cudaStream_t stream, int* idx, int kmax) {
  IEF_CHECK(logits && labels && lengths && means && loss, "clas2: null argument");
  IEF_CHECK(B >= 1, "clas2: empty batch");
  IEF_TRY(mil_topk_mean(logits, lengths, B, T, 1, means, idx, kmax, stream));
  bce_kernel<<<1, 256, 0, stream>>>(means, labels, label_stride, int(B), loss);
  count_launches(1);
  IEF_CUDA(cudaGetLastError());
  return IEFVAD_OK;
}

int segment_copy(const float* src, const long long* src_off, float* dst, const long long* dst_off,
                 const long long* len, long long nseg, cudaStream_t st) {
  IEF_CHECK(nseg >= 0 && nseg < (1LL << 31), "segment_copy: bad segment count");
  if (nseg == 0) return IEFVAD_OK;
  IEF_CHECK(src && src_off && dst && dst_off && len, "segment_copy: null argument");
  segment_copy_kernel<<<unsigned(nseg < 4736 ? nseg : 4736), 256, 0, st>>>(src, src_off, dst, dst_off, len, int(nseg));
  count_launches(1);
  IEF_CUDA(cudaGetLastError());
  return IEFVAD_OK;
}

int sort_scores(const float* scores, long long n, int* order, uint32_t* keys_sorted, cudaStream_t st) {
  IEF_CHECK(n >= 0 && n < (1LL << 31), "sort_scores: bad n");
  IEF_CHECK(scores && order, "sort_scores: null argument");
  if (n == 0) return IEFVAD_OK;
  Tmp tmp(st);
  const int nblocks = int((n + RS_THREADS * rs_items(n) - 1) / (RS_THREADS * rs_items(n)));
  uint32_t *ka, *kb, *vb, *hist, *totals;
  IEF_TRY(tmp.get(&ka, n));
  IEF_TRY(tmp.get(&kb, n));
  IEF_TRY(tmp.get(&vb, n));
  IEF_TRY(tmp.get(&hist, size_t(RS_BINS) * nblocks));
  IEF_TRY(tmp.get(&totals, RS_BINS));
  uint32_t* va = reinterpret_cast<uint32_t*>(order);
  rs_init_kernel<<<(nblocks < 1184 ? nblocks : 1184), RS_THREADS, 0, st>>>(scores, n, ka, va);
  count_launches(1);
  IEF_TRY(radix_sort_pairs(ka, va, kb, vb, n, hist, totals, st));
  if (keys_sorted) IEF_CUDA(cudaMemcpyAsync(keys_sorted, ka, size_t(n) * 4, cudaMemcpyDeviceToDevice, st));
  return IEFVAD_OK;
}

int auc_ap_multi(const float* scores, const int* pos, const uint32_t* member, long long n, int repeat, int nsub,
                 double* out, int* order_out, cudaStream_t st) {
  IEF_CHECK(n >= 0 && n < (1LL << 31), "auc_ap: bad n");
  IEF_CHECK(out && (n == 0 || (scores && pos)), "auc_ap: null argument");
  IEF_CHECK(repeat >= 1, "auc_ap: repeat must be >= 1");
  IEF_CHECK(nsub >= 1 && nsub <= 32 && (member != nullptr || nsub == 1), "auc_ap: 1..32 subsets, a member mask when > 1");
  Tmp tmp(st);
  if (n == 0) {
    const double nan = __builtin_nan("");
    double h[4 * 32];
    for (int s = 0; s < nsub; ++s) { h[4 * s] = nan; h[4 * s + 1] = nan; h[4 * s + 2] = 0.0; h[4 * s + 3] = 0.0; }
    IEF_CUDA(cudaMemcpyAsync(out, h, sizeof(double) * 4 * nsub, cudaMemcpyHostToDevice, st));
    IEF_CUDA(cudaStreamSynchronize(st));
    return IEFVAD_OK;
  }
  const int nblocks = int((n + RS_THREADS * rs_items(n) - 1) / (RS_THREADS * rs_items(n)));
  const int ntiles = int((n + SC_TILE - 1) / SC_TILE);
  uint32_t *ka, *kb, *va, *vb, *hist, *totals;
  Tri *tile_sums, *grand;
  long long *gtp, *gfp;
  unsigned long long* area_part;
  double* ap_part;
  IEF_TRY(tmp.get(&ka, n));
  IEF_TRY(tmp.get(&kb, n));
  IEF_TRY(tmp.get(&va, n));
  IEF_TRY(tmp.get(&vb, n));
  IEF_TRY(tmp.get(&hist, size_t(RS_BINS) * nblocks));
  IEF_TRY(tmp.get(&totals, RS_BINS));
  IEF_TRY(tmp.get(&tile_sums, size_t(ntiles) * nsub));
  IEF_TRY(tmp.get(&grand, nsub));
  IEF_TRY(tmp.get(&gtp, size_t(n) * nsub));
  IEF_TRY(tmp.get(&gfp, size_t(n) * nsub));
  const int term_blocks = ntiles < 256 ? ntiles : 256;
  IEF_TRY(tmp.get(&area_part, size_t(term_blocks) * nsub));
  IEF_TRY(tmp.get(&ap_part, size_t(term_blocks) * nsub));
  rs_init_kernel<<<(nblocks < 1184 ? nblocks : 1184), RS_THREADS, 0, st>>>(scores, n, ka, va);
  count_launches(1);
  IEF_TRY(radix_sort_pairs(ka, va, kb, vb, n, hist, totals, st));
  sc_reduce_kernel<<<dim3(ntiles, nsub), SC_THREADS, 0, st>>>(ka, va, pos, member, repeat, n, tile_sums);
  sc_scan_tiles_kernel<<<nsub, SC_THREADS, 0, st>>>(tile_sums, ntiles, grand);
  sc_apply_kernel<<<dim3(ntiles, nsub), SC_THREADS, 0, st>>>(ka, va, pos, member, repeat, n, tile_sums, gtp, gfp);
  auc_terms_kernel<<<dim3(term_blocks, nsub), SC_THREADS, 0, st>>>(gtp, gfp, n, grand, area_part, ap_part);
  auc_final_kernel<<<nsub, 1, 0, st>>>(area_part, ap_part, term_blocks, grand, out);
  count_launches(5);
  if (order_out) IEF_CUDA(cudaMemcpyAsync(order_out, va, size_t(n) * 4, cudaMemcpyDeviceToDevice, st));
  IEF_CUDA(cudaGetLastError());
  return IEFVAD_OK;
}

int auc_ap(const float* scores, const int* pos, long long n, int repeat, double* out, int* order_out, cudaStream_t st) {
  return auc_ap_multi(scores, pos, nullptr, n, repeat, 1, out, order_out, st);
}

}  // namespace iefvad
