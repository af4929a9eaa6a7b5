// tcgen05 / TMEM / TMA GEMM for sm_100a:  C[M,N] = epilogue( A[M,K] . W[N,K]^T ), bf16 operands, fp32 accumulate.
//
// Covers every dense layer of the IEF-VAD forward (model/imf_vad.py:115,121 in/out projections,
// :125-128 heads, :148 refinement MLPs) - K-major A (activations) and K-major W (nn.Linear stores
// [out, in]) are exactly the layouts UMMA wants, so no transposes anywhere.
//
// Structure (one CTA per SM, persistent over output tiles, 320 threads):
//   warp 0     TMA producer   : cp.async.bulk.tensor 128x64 (A) and BNx64 (W) bf16 boxes, 128B swizzle,
//                               into a smem ring guarded by full/empty mbarriers
//   warp 1     MMA issuer     : one thread issues 4 x tcgen05.mma (128 x BN x 16) per k-block into one of two
//                               TMEM accumulator buffers; tcgen05.commit releases smem slots / publishes tiles
//   warps 2-9  epilogue       : each warp owns 32 accumulator rows (its TMEM lane quarter; two warps per quarter take
//                               the even / odd chunks so that every scheduler has two warps to interleave) and
//                               walks them in 32-column chunks: tcgen05.ld (thread == row) -> bias / activation / residual /
//                               bf16 hi+lo split in registers -> swizzled per-warp smem boxes -> TMA bulk tensor
//                               stores.  The fp32 residual arrives the same way (TMA loads into a per-warp ring,
//                               prefetched several chunks - and across tile boundaries - ahead), so no epilogue
//                               thread ever waits on a global load and every byte of epilogue traffic is issued as
//                               full 32x32 boxes by the copy engine.  Rows past M are clipped by the tensor maps.
// The two TMEM buffers let the epilogue of tile i overlap the MMAs of tile i+1.  The smem that is left after the
// per-warp epilogue boxes decides the depth of the operand ring (3 stages beside a residual ring, 4 otherwise).
//
// "split-bf16" (nsplit == 3): A ~= A_hi + A_lo, W ~= W_hi + W_lo and the product is accumulated as
// A_hi.W_hi + A_hi.W_lo + A_lo.W_hi in the same fp32 accumulator - implemented as a 3x longer K loop whose
// k-blocks pick the (A, W) tensor-map pair, so the pipeline is unchanged.
#include <cstring>

#include "common.cuh"
#include "gemm.cuh"
#include "tensormap.cuh"

namespace iefvad {

namespace {

constexpr int BM = 128;
constexpr int BK = 64;
constexpr int CW = 32;                        // epilogue chunk width (columns)
constexpr int kMaxStages = 8;
constexpr int kMaxResidSlots = 4;
constexpr uint32_t kF32Box = 32 * CW * 4;     // one 32-row x 32-col fp32 box (128-byte rows, SWIZZLE_128B)
constexpr uint32_t kBfBox = 32 * CW * 2;      // the same box in bf16 (64-byte rows, SWIZZLE_64B)
constexpr uint32_t kBarBytes = 768;
constexpr int kEpiWarps = 8;                  // two per TMEM lane quarter: one takes the even, one the odd column chunks
constexpr int kThreads = 64 + 32 * kEpiWarps;
constexpr uint32_t kSmemLimit = 232448;       // 227 KB opt-in maximum per CTA on sm_100

// everything the device epilogue needs besides the tensor maps
struct TcEpi {
  int mode = EPI_ROWMAJOR;
  const float* bias = nullptr;
  int act = ACT_NONE;
  float alpha = 1.f;
  int has_resid = 0, has_f32 = 0, has_hi = 0, has_lo = 0;
  int split_col = 1 << 30;
  int nr = 0;              // residual ring depth (per warp)
  int inplace = 0;         // the fp32 output is written over the residual box it was computed from (ring slot)
  uint32_t warp_bytes = 0; // per-warp epilogue smem
  int stages = 4;
  uint32_t idesc = 0;      // tcgen05 instruction descriptor (operand format bf16 / fp16, tile shape)
  int hi_fp16 = 0;         // the 16-bit output is fp16 instead of bf16
  uint32_t rslot = kF32Box; // bytes per residual ring slot
  int resid_lo = 0;        // R16 instances: the fp16 residual has a remainder part (second box of the ring slot)
  // EPI_QKV
  bf16* q = nullptr;
  bf16* k = nullptr;
  bf16* vt = nullptr;
  int T = 0, H = 0, dh = 0, dhp = 0, Tpad = 0, D = 0;
  float qscale = 1.f;
  int qk_tma = 0;          // q / k leave through 4-D TMA stores (T % 32 == 0), else per-thread 16-byte stores
  int ksplit = 1;          // split-K: slice s of the K range accumulates into rows [s * M, (s + 1) * M) of the output
};

struct TcMaps {
  CUtensorMap a0, a1, b0, b1;   // operands (hi / lo)
  CUtensorMap r;                // fp32 residual [M, N] (R16 instances: its fp16 form, r2 = fp16 remainder)
  CUtensorMap r2;
  CUtensorMap o0, o1;           // fp32 outputs (columns below / from split_col)
  CUtensorMap h, l;             // bf16 hi / lo outputs; in EPI_QKV: q / k as 4-D {d, t, head, batch}
  CUtensorMap v;                // EPI_QKV: V^T as 3-D {t, head * dh + d, batch}
};

template <int BN, int CG = 1>
struct TcCfg {
  static constexpr uint32_t kABytes = BM * BK * 2;
  static constexpr uint32_t kBBytes = (BN / CG) * BK * 2;    // a CTA pair splits the W tile: each CTA loads BN/2 rows
  static constexpr uint32_t kStageBytes = kABytes + kBBytes;
  static constexpr uint32_t kTmemCols = (2 * BN <= 32) ? 32 : (2 * BN <= 64) ? 64 : (2 * BN <= 128) ? 128
                                        : (2 * BN <= 256) ? 256 : 512;
};

// swizzled 16-byte slot of (row, 16-byte group g) inside a TMA box whose rows are 128 B (fp32) or 64 B (bf16)
__device__ __forceinline__ uint32_t sw128(int row, int g) { return uint32_t(row) * 128u + (uint32_t(g ^ (row & 7)) << 4); }
__device__ __forceinline__ uint32_t sw64(int row, int g) { return uint32_t(row) * 64u + (uint32_t(g ^ ((row >> 1) & 3)) << 4); }

// MODE (EPI_ROWMAJOR / EPI_QKV) and ACT are compile-time so that each instance carries only the epilogue code it
// runs: the epilogue warps execute long straight-line chunk bodies and a kernel with every variant inlined
// spent most of its epilogue time in instruction-cache misses (ncu: stall_no_inst).
//
// CG == 2 runs the same roles on a CTA pair (cluster of 2, tcgen05 cta_group::2): one 256 x BN tile per pair, each
// CTA owning 128 rows of A / of the accumulator and HALF of the W tile, which the tensor cores of both SMs share.
// That cuts the smem fill + operand-read traffic per flop by a third - the resource the 1-CTA kernel saturates
// (mainloop ~80 % of the tensor rate, and every epilogue byte staged through smem slows it further).  Only the
// leader CTA issues MMAs; its commits multicast to the mbarriers of both CTAs; both producers signal the leader's
// `full` barrier; both epilogues arrive on the leader's `tempty`.
// R16: the residual arrives as fp16 (+ optional fp16 remainder) boxes instead of fp32 ones.
template <int BN, int MODE, int ACT, int CG, int R16>
__global__ void __launch_bounds__(kThreads, 1)
gemm_tc_kernel(const __grid_constant__ TcMaps tm, int M, int N, int K, int nsplit, const TcEpi ep) {
  using Cfg = TcCfg<BN, CG>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int STAGES = ep.stages;
  uint8_t* epi_base = smem + size_t(STAGES) * Cfg::kStageBytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(epi_base + kEpiWarps * ep.warp_bytes);
  uint64_t* full = bars;
  uint64_t* empty = full + kMaxStages;
  uint64_t* tfull = empty + kMaxStages;
  uint64_t* tempty = tfull + 2;
  uint64_t* rfull_all = tempty + 2;                                  // [4 warps][kMaxResidSlots]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(rfull_all + kEpiWarps * kMaxResidSlots);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t rank = (CG == 2) ? cluster_ctarank() : 0u;     // rank in the CTA pair; 0 = leader
  const int num_m = (M + BM * CG - 1) / (BM * CG);               // tiles of BM * CG rows (one per CTA / pair)
  const int num_n = (N + BN - 1) / BN;
  const int num_tiles = num_m * num_n * ep.ksplit;               // split-K: the output has ksplit row slices of M rows each
  const int tile0 = blockIdx.x / CG, tile_step = gridDim.x / CG;
  const int kb_per_seg = K / BK / ep.ksplit;                      // k-blocks a tile walks per operand pair
  const int total_kb = kb_per_seg * nsplit;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tm.a0);
    tma_prefetch_desc(&tm.b0);
    if (nsplit > 1) {
      tma_prefetch_desc(&tm.a1);
      tma_prefetch_desc(&tm.b1);
    }
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(&tfull[s], 1);
      mbar_init(&tempty[s], kEpiWarps * CG);      // the epilogue warps of every CTA of the pair arrive on the leader's
    }
    for (int s = 0; s < kEpiWarps * kMaxResidSlots; ++s) mbar_init(&rfull_all[s], 1);
    fence_barrier_init();
  }
  if (warp == 1) {
    if (CG == 2) {
      tmem_alloc_cg2(tmem_slot, Cfg::kTmemCols);
      tmem_relinquish_cg2();
    } else {
      tmem_alloc(tmem_slot, Cfg::kTmemCols);
      tmem_relinquish();
    }
  }
  tc_fence_before();
  if (CG == 2) cluster_sync_all(); else __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      int s = 0;
      uint32_t ph = 0;
      for (int tile = tile0; tile < num_tiles; tile += tile_step) {
        const int m_out = (tile / num_n) * CG + int(rank), n_blk = tile % num_n;
        const int m_blk = m_out % (num_m * CG);                    // operand row block; m_out / (num_m * CG) = the K slice
        const int k_first = (m_out / (num_m * CG)) * kb_per_seg;
        for (int kb = 0; kb < total_kb; ++kb) {
          const int seg = kb / kb_per_seg, kk = k_first + kb - seg * kb_per_seg;
          const CUtensorMap* ma = (seg == 2) ? &tm.a1 : &tm.a0;   // hi.hi, hi.lo, lo.hi
          const CUtensorMap* mb = (seg == 1) ? &tm.b1 : &tm.b0;
          mbar_wait(&empty[s], ph ^ 1);
          uint8_t* sa = smem + size_t(s) * Cfg::kStageBytes;
          if (CG == 2) {
            // both CTAs' boxes complete on the LEADER's full barrier, which expects the bytes of the whole pair
            const uint32_t lead_full = mapa_shared(smem_u32(&full[s]), 0);
            if (rank == 0) mbar_arrive_expect_tx(&full[s], 2 * Cfg::kStageBytes);
            tma_load_2d_cg2(ma, lead_full, sa, kk * BK, m_blk * BM);
            tma_load_2d_cg2(mb, lead_full, sa + Cfg::kABytes, kk * BK, n_blk * BN + int(rank) * (BN / 2));
          } else {
            mbar_arrive_expect_tx(&full[s], Cfg::kStageBytes);
            tma_load_2d(ma, &full[s], sa, kk * BK, m_blk * BM);
            tma_load_2d(mb, &full[s], sa + Cfg::kABytes, kk * BK, n_blk * BN);
          }
          if (++s == STAGES) { s = 0; ph ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    if (lane == 0 && rank == 0) {
      const uint32_t idesc = ep.idesc;
      int s = 0;
      uint32_t ph = 0;
      int it = 0;
      for (int tile = tile0; tile < num_tiles; tile += tile_step, ++it) {
        const int as = it & 1;
        const uint32_t aph = (it >> 1) & 1;
        mbar_wait(&tempty[as], aph ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + uint32_t(as * BN);
        for (int kb = 0; kb < total_kb; ++kb) {
          mbar_wait(&full[s], ph);
          tc_fence_after();
          const uint32_t sa = smem_u32(smem + size_t(s) * Cfg::kStageBytes);
          const uint64_t da = make_smem_desc_sw128(sa);
          const uint64_t db = make_smem_desc_sw128(sa + Cfg::kABytes);
#pragma unroll
          for (int k4 = 0; k4 < BK / 16; ++k4) {
            if (CG == 2) umma_bf16_cg2(d_tmem, da + uint64_t(2 * k4), db + uint64_t(2 * k4), idesc, (kb | k4) != 0 ? 1u : 0u);
            else umma_bf16(d_tmem, da + uint64_t(2 * k4), db + uint64_t(2 * k4), idesc, (kb | k4) != 0 ? 1u : 0u);
          }
          if (CG == 2) tc_commit_cg2(&empty[s], 3); else tc_commit(&empty[s]);   // smem slot reusable once these MMAs retire
          if (++s == STAGES) { s = 0; ph ^= 1; }
        }
        if (CG == 2) tc_commit_cg2(&tfull[as], 3); else tc_commit(&tfull[as]);   // accumulator complete (both CTAs)
      }
    }
  } else {
    // ===================== epilogue (warps 2..5) =====================
    const int quarter = warp & 3;         // TMEM lanes [32*quarter, 32*quarter+32) belong to this warp
    const int par = (warp - 2) >> 2;      // the two warps of a quarter split the column chunks: c = par, par + 2, ...
    uint8_t* wb = epi_base + size_t(warp - 2) * ep.warp_bytes;
    uint8_t* Rb = wb;                                                      // [nr] fp32 residual (/ in-place output) boxes
    uint8_t* Ob = Rb + size_t(ep.nr) * ep.rslot;                            // [2] fp32 output boxes (no residual ring)
    uint8_t* Hb = Ob + ((ep.has_f32 && !ep.inplace) ? 2 * kF32Box : 0);    // [2] bf16 hi (or q / k) boxes
    uint8_t* Lb = Hb + (ep.has_hi ? 2 * kBfBox : 0);                       // [2] bf16 lo boxes
    uint64_t* rfull = rfull_all + (warp - 2) * kMaxResidSlots;
    const bool discard = ep.mode == EPI_DISCARD;

    // residual prefetch cursor (lane 0): walks the same (tile, chunk) sequence as the consumer, ahead of it
    int pf_tile = tile0, pf_c = par;
    uint32_t pf_n = 0;
    auto chunks_of = [&](int tile) {
      const int n_blk = tile % num_n;
      const int w = N - n_blk * BN;
      return (w < BN ? w : BN) / CW;
    };
    auto prefetch_resid = [&]() {
      if (pf_tile >= num_tiles) return;
      const int m_blk = (pf_tile / num_n) * CG + int(rank), n_blk = pf_tile % num_n;
      const int slot = int(pf_n % uint32_t(ep.nr));
      if (R16) {
        mbar_arrive_expect_tx(&rfull[slot], ep.resid_lo ? 2 * kBfBox : kBfBox);
        tma_load_2d(&tm.r, &rfull[slot], Rb + size_t(slot) * ep.rslot, n_blk * BN + pf_c * CW, m_blk * BM + quarter * 32);
        if (ep.resid_lo)
          tma_load_2d(&tm.r2, &rfull[slot], Rb + size_t(slot) * ep.rslot + kBfBox, n_blk * BN + pf_c * CW,
                      m_blk * BM + quarter * 32);
      } else {
        mbar_arrive_expect_tx(&rfull[slot], kF32Box);
        tma_load_2d(&tm.r, &rfull[slot], Rb + size_t(slot) * ep.rslot, n_blk * BN + pf_c * CW, m_blk * BM + quarter * 32);
      }
      ++pf_n;
      pf_c += 2;
      while (pf_tile < num_tiles && pf_c >= chunks_of(pf_tile)) { pf_c = par; pf_tile += tile_step; }
    };
    while (pf_tile < num_tiles && pf_c >= chunks_of(pf_tile)) pf_tile += tile_step;   // tiles too narrow for this parity
    if (ep.has_resid && lane == 0) {
      tma_prefetch_desc(&tm.r);
      if (R16 && ep.resid_lo) tma_prefetch_desc(&tm.r2);
      for (int i = 0; i < ep.nr; ++i) prefetch_resid();
    }
    uint32_t n_cons = 0;       // residual chunks consumed
    uint32_t n_out = 0;        // output chunks handed to TMA (one bulk group each)

    // bias of the next chunk, fetched one chunk ahead (8 x 16-byte broadcast loads per thread)
    float4 bnext[8];
    auto fetch_bias = [&](int col0) {
      if (ep.bias == nullptr) return;
#pragma unroll
      for (int g = 0; g < 8; ++g) bnext[g] = __ldg(reinterpret_cast<const float4*>(ep.bias + col0) + g);
    };

    // Output discipline: chunk n writes boxes [n & 1] (or its in-place residual slot).  After committing the
    // stores of chunk n lane 0 waits until every group but the newest has finished READING smem, so when the warp
    // meets again at the top of the next store phase the boxes of chunk n - 1 are free.
    auto finish_chunk = [&]() {      // lane 0, after issuing the stores of one chunk
      bulk_commit();
      bulk_wait_read<1>();
      if (ep.inplace && n_out > 0) prefetch_resid();     // the slot of the previous chunk is free again
    };

    int tile = tile0;
    int it = 0;
    int m_blk = 0, n_blk = 0, row0 = 0, nchunks = 0;

    auto process = [&](float (&v)[32], int c) {
      const int col0 = n_blk * BN + c * CW;
      if (ep.bias) {
#pragma unroll
        for (int g = 0; g < 8; ++g) {
          v[g * 4 + 0] += bnext[g].x; v[g * 4 + 1] += bnext[g].y; v[g * 4 + 2] += bnext[g].z; v[g * 4 + 3] += bnext[g].w;
        }
        if (c + 2 < nchunks) fetch_bias(col0 + 2 * CW);
      }
      if (ACT != ACT_NONE) {
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] = apply_act(v[j], ACT);
      }

      if (MODE == EPI_QKV) {
        const int which = col0 / ep.D;                 // 0 = q, 1 = k, 2 = v (a chunk never straddles: D % 32 == 0)
        const int cc = col0 - which * ep.D;
        const int h = cc / ep.dh;                      // dh % 32 == 0 -> a chunk stays inside one head
        const int d0 = cc - h * ep.dh;
        const long long row = (long long)row0 + lane;
        const long long b = row / ep.T;
        const int t = int(row - b * ep.T);
        if (which == 2 && ep.qk_tma) {
          // V^T [B, H, dh, Tpad] through a transposed box: lane = t writes its 32 d values down a column (each instruction
          // fills one 64-byte box row, conflict-free), then ONE TMA store instead of 32 scattered 2-byte stores per thread
          uint8_t* hb = Hb + size_t(n_out & 1) * kBfBox;
          __syncwarp();                                  // lane 0 is back from bulk_wait_read: box [n_out & 1] is free
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            if (ep.hi_fp16) *reinterpret_cast<__half*>(hb + j * 64 + lane * 2) = __float2half_rn(v[j]);
            else *reinterpret_cast<bf16*>(hb + j * 64 + lane * 2) = __float2bfloat16_rn(v[j]);
          }
          fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0) {
            const long long b0 = (long long)row0 / ep.T;   // T % 32 == 0: all 32 rows share the batch element
            tma_store_3d(&tm.v, hb, int(row0 - b0 * ep.T), h * ep.dh + d0, int(b0));
            finish_chunk();
          }
          ++n_out;
          return;
        }
        if (which == 2) {
          // V^T [B, H, dh, Tpad]: consecutive lanes = consecutive t, so each of the 32 stores is one 64-byte run
          if (row < M) {
            bf16* dst = ep.vt + ((b * ep.H + h) * ep.dh + d0) * (long long)ep.Tpad + t;
#pragma unroll
            for (int j = 0; j < 32; ++j) {
              if (ep.hi_fp16) reinterpret_cast<__half*>(dst)[(long long)j * ep.Tpad] = __float2half_rn(v[j]);
              else dst[(long long)j * ep.Tpad] = __float2bfloat16_rn(v[j]);
            }
          }
          return;
        }
        const float s = (which == 0) ? ep.qscale : 1.f;
        uint4 u[4];
#pragma unroll
        for (int g = 0; g < 4; ++g) u[g] = pack_16x8(v + g * 8, ep.hi_fp16, s);
        if (!ep.qk_tma) {
          if (row < M) {
            bf16* dst = (which == 0 ? ep.q : ep.k) + ((b * ep.H + h) * ep.T + t) * (long long)ep.dhp + d0;
#pragma unroll
            for (int g = 0; g < 4; ++g) *reinterpret_cast<uint4*>(dst + g * 8) = u[g];
          }
          return;
        }
        uint8_t* hb = Hb + size_t(n_out & 1) * kBfBox;
        __syncwarp();                                  // lane 0 is back from bulk_wait_read: box [n_out & 1] is free
#pragma unroll
        for (int g = 0; g < 4; ++g) *reinterpret_cast<uint4*>(hb + sw64(lane, g)) = u[g];
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) {
          const long long b0 = (long long)row0 / ep.T;   // T % 32 == 0: all 32 rows share the batch element
          tma_store_4d(which == 0 ? &tm.h : &tm.l, hb, d0, int(row0 - b0 * ep.T), h, int(b0));
          finish_chunk();
        }
        ++n_out;
        return;
      }

      // ---- row-major outputs: out = resid + alpha * x
      uint8_t* fb = Ob + size_t(n_out & 1) * kF32Box;
      if (ep.has_resid) {
        const int slot = int(n_cons % uint32_t(ep.nr));
        mbar_wait(&rfull[slot], (n_cons / uint32_t(ep.nr)) & 1);
        uint8_t* rb = Rb + size_t(slot) * ep.rslot;
        if (R16) {
#pragma unroll
          for (int g = 0; g < 4; ++g) {
            float r[8];
            unpack_f16x8(*reinterpret_cast<const uint4*>(rb + sw64(lane, g)),
                         ep.resid_lo ? reinterpret_cast<const uint4*>(rb + kBfBox + sw64(lane, g)) : nullptr, r);
#pragma unroll
            for (int j = 0; j < 8; ++j) v[g * 8 + j] = fmaf(ep.alpha, v[g * 8 + j], r[j]);
          }
        } else {
#pragma unroll
          for (int g = 0; g < 8; ++g) {
            const float4 r4 = *reinterpret_cast<const float4*>(rb + sw128(lane, g));
            v[g * 4 + 0] = fmaf(ep.alpha, v[g * 4 + 0], r4.x);
            v[g * 4 + 1] = fmaf(ep.alpha, v[g * 4 + 1], r4.y);
            v[g * 4 + 2] = fmaf(ep.alpha, v[g * 4 + 2], r4.z);
            v[g * 4 + 3] = fmaf(ep.alpha, v[g * 4 + 3], r4.w);
          }
        }
        ++n_cons;
        if (ep.inplace) {
          fb = rb;                                     // every lane overwrites exactly the 128 bytes it just read
        } else {
          __syncwarp();                                // every lane has its residual values: refill the slot
          if (lane == 0) prefetch_resid();
        }
      } else if (ep.alpha != 1.f) {
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] *= ep.alpha;
      }
      if (!(ep.has_f32 || ep.has_hi)) return;
      uint8_t* hb = Hb + size_t(n_out & 1) * kBfBox;
      uint8_t* lb = Lb + size_t(n_out & 1) * kBfBox;
      __syncwarp();                                    // lane 0 is back from bulk_wait_read: boxes [n_out & 1] are free
      if (ep.has_f32) {
#pragma unroll
        for (int g = 0; g < 8; ++g)
          *reinterpret_cast<float4*>(fb + sw128(lane, g)) = make_float4(v[g * 4], v[g * 4 + 1], v[g * 4 + 2], v[g * 4 + 3]);
      }
      if (ep.has_hi) {
#pragma unroll
        for (int g = 0; g < 4; ++g) {
          uint32_t hi[4], lo[4];
#pragma unroll
          for (int q = 0; q < 4; ++q) split_16x2(v[g * 8 + 2 * q], v[g * 8 + 2 * q + 1], ep.hi_fp16, hi[q], lo[q]);
          *reinterpret_cast<uint4*>(hb + sw64(lane, g)) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
          if (ep.has_lo) *reinterpret_cast<uint4*>(lb + sw64(lane, g)) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
        }
      }
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) {
        if (ep.has_f32) {
          if (col0 < ep.split_col) tma_store_2d(&tm.o0, fb, col0, row0);
          else tma_store_2d(&tm.o1, fb, col0 - ep.split_col, row0);
        }
        if (ep.has_hi) tma_store_2d(&tm.h, hb, col0, row0);
        if (ep.has_lo) tma_store_2d(&tm.l, lb, col0, row0);
        finish_chunk();
      }
      ++n_out;
    };

    for (; tile < num_tiles; tile += tile_step, ++it) {
      m_blk = (tile / num_n) * CG + int(rank);
      n_blk = tile % num_n;
      const int as = it & 1;
      const uint32_t aph = (it >> 1) & 1;
      nchunks = chunks_of(tile);
      row0 = m_blk * BM + quarter * 32;               // first row of this warp; this thread owns row0 + lane
      if (!discard && par < nchunks) fetch_bias(n_blk * BN + par * CW);   // in flight while the accumulator is produced
      mbar_wait(&tfull[as], aph);
      tc_fence_after();
      const uint32_t t0 = tmem_base + uint32_t(as * BN) + (uint32_t(quarter * 32) << 16);
      auto release_tmem = [&]() {                     // accumulator fully in registers: hand the buffer back
        tc_fence_before();
        __syncwarp();
        if (lane == 0) {
          if (CG == 2) mbar_arrive_cluster(mapa_shared(smem_u32(&tempty[as]), 0));
          else mbar_arrive(&tempty[as]);
        }
      };
      // the tcgen05.ld of this warp's next chunk is in flight (into vn) while the current one is processed (in v)
      float v[32], vn[32];
      if (par >= nchunks) { release_tmem(); continue; }
      tmem_ld32(t0 + uint32_t(par * CW), vn);
#pragma unroll 1
      for (int c = par; c < nchunks; c += 2) {
        tmem_ld_wait_for(vn);
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] = vn[j];
        if (c + 2 < nchunks) tmem_ld32(t0 + uint32_t((c + 2) * CW), vn);
        else release_tmem();
        if (!discard) process(v, c);
      }
    }
    if (lane == 0) bulk_wait_all<0>();     // smem boxes must outlive their stores
  }

  tc_fence_before();
  if (CG == 2) cluster_sync_all(); else __syncthreads();   // the peer may still signal barriers / read TMEM of this CTA
  if (warp == 1) {
    tc_fence_after();
    if (CG == 2) tmem_dealloc_cg2(tmem_base, Cfg::kTmemCols);
    else tmem_dealloc(tmem_base, Cfg::kTmemCols);
  }
}

template <int BN, int MODE, int ACT, int CG, int R16 = 0>
int launch_inst(const TcMaps& tm, const GemmTcArgs& g, const TcEpi& e, int grid, size_t smem_bytes, cudaStream_t stream) {
  static bool attr_set = false;
  if (!attr_set) {
    IEF_CUDA(cudaFuncSetAttribute(gemm_tc_kernel<BN, MODE, ACT, CG, R16>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  int(kSmemLimit)));
    attr_set = true;
  }
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(kThreads);
  cfg.dynamicSmemBytes = smem_bytes;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = CG;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  IEF_CUDA(cudaLaunchKernelEx(&cfg, gemm_tc_kernel<BN, MODE, ACT, CG, R16>, tm, g.M, g.N, g.K, g.nsplit, e));
  count_launches(1);
  return IEFVAD_OK;
}

template <int BN, int CG>
int launch_bn(const GemmTcArgs& g, const EpiParams& ep, int num_sms, cudaStream_t stream) {
  using Cfg = TcCfg<BN, CG>;
  TcEpi e;
  e.mode = ep.mode; e.bias = ep.bias; e.act = ep.act; e.alpha = ep.alpha; e.split_col = ep.split_col;
  e.idesc = g.fp16 ? make_idesc_f16(BM * CG, BN) : make_idesc_bf16(BM * CG, BN);
  e.hi_fp16 = ep.hi_fp16;
  e.ksplit = g.ksplit > 1 ? g.ksplit : 1;
  if (e.ksplit > 1) {
    IEF_CHECK(ep.mode == EPI_ROWMAJOR && !ep.bias && !ep.resid && !ep.resid_h16 && ep.act == ACT_NONE && ep.out_f32 && !ep.out_hi &&
              ep.split_col >= g.N, "gemm_tc: split-K writes plain fp32 partial sums (no bias / residual / activation)");
    IEF_CHECK(g.M % (BM * CG) == 0 && (g.K / BK) % e.ksplit == 0, "gemm_tc: split-K needs M %% %d == 0 and K / %d divisible by %d",
              BM * CG, BK, e.ksplit);
  }
  IEF_CHECK(!g.fp16 || g.nsplit == 1, "gemm_tc: fp16 operands are single-pass (nsplit == 1)");
  const bool r16 = ep.resid_h16 != nullptr;
  IEF_CHECK(!r16 || (ep.resid == nullptr && ep.mode == EPI_ROWMAJOR && ep.act == ACT_NONE),
            "gemm_tc: the fp16 residual replaces the fp32 one (row-major epilogue, no activation)");
  IEF_CHECK(r16 || ep.resid_l16 == nullptr, "gemm_tc: resid_l16 without resid_h16");
  TcMaps tm;
  memset(&tm, 0, sizeof(tm));
  if (ep.mode == EPI_ROWMAJOR) {
    e.has_resid = ep.resid != nullptr || r16;
    e.resid_lo = ep.resid_l16 != nullptr;
    e.has_f32 = ep.out_f32 != nullptr;
    e.has_hi = ep.out_hi != nullptr;
    e.has_lo = ep.out_hi != nullptr && ep.out_lo != nullptr;
    IEF_CHECK(ep.split_col % CW == 0 || ep.split_col >= g.N, "gemm_tc: split_col must be a multiple of %d", CW);
    IEF_CHECK(!e.has_f32 || (ep.ld_f32 % 4 == 0), "gemm_tc: ld_f32 must be a multiple of 4");
    IEF_CHECK(!e.has_hi || (ep.ld_bf % 8 == 0), "gemm_tc: ld_bf must be a multiple of 8");
    IEF_CHECK(!e.has_resid || (ep.ld_resid % (r16 ? 8 : 4) == 0), "gemm_tc: ld_resid must be a multiple of 4 (fp16: 8)");
  } else if (ep.mode == EPI_QKV) {
    IEF_CHECK(ep.q && ep.k && ep.vt, "gemm_tc: QKV epilogue needs q, k and vt");
    IEF_CHECK(ep.D % CW == 0 && ep.dh % CW == 0 && g.N == 3 * ep.D && ep.T > 0,
              "gemm_tc: QKV epilogue needs D %% 32 == 0, dh %% 32 == 0, N == 3D");
    e.q = ep.q; e.k = ep.k; e.vt = ep.vt; e.T = ep.T; e.H = ep.H; e.dh = ep.dh; e.dhp = ep.dhp; e.Tpad = ep.Tpad;
    e.D = ep.D; e.qscale = ep.qscale;
    e.qk_tma = (ep.T % 32 == 0) ? 1 : 0;
    e.has_hi = e.qk_tma;
  }
  // per-warp epilogue smem: a residual ring whose slots double as the fp32 output boxes (in place), else two fp32
  // output boxes; bf16 boxes always ping-pong
  e.inplace = (e.has_resid && e.has_f32 && !r16) ? 1 : 0;
  e.nr = e.has_resid ? ((e.has_lo || r16) ? 2 : 3) : 0;   // the widest epilogues trade ring depth for an operand stage
  e.rslot = r16 ? (e.resid_lo ? 2 * kBfBox : kBfBox) : kF32Box;
  e.warp_bytes = e.nr * e.rslot + ((e.has_f32 && !e.inplace) ? 2 * kF32Box : 0) + (e.has_hi ? 2 * kBfBox : 0) +
                 (e.has_lo ? 2 * kBfBox : 0);
  const uint32_t fixed = 1024 + kEpiWarps * e.warp_bytes + kBarBytes;
  int stages = int((kSmemLimit - fixed) / Cfg::kStageBytes);
  if (stages > kMaxStages) stages = kMaxStages;
  if (g.force_stages > 0 && g.force_stages < stages) stages = g.force_stages;
  IEF_CHECK(stages >= 2, "gemm_tc: no room for a 2-stage operand ring (BN=%d)", BN);
  e.stages = stages;
  const size_t smem_bytes = fixed + size_t(stages) * Cfg::kStageBytes;

  IEF_TRY(make_tmap_2d(&tm.a0, g.A_hi, g.K, g.M, uint64_t(g.lda) * 2, BK, BM));
  IEF_TRY(make_tmap_2d(&tm.b0, g.W_hi, g.K, g.N, uint64_t(g.ldw) * 2, BK, BN / CG));
  if (g.nsplit == 3) {
    IEF_TRY(make_tmap_2d(&tm.a1, g.A_lo, g.K, g.M, uint64_t(g.lda) * 2, BK, BM));
    IEF_TRY(make_tmap_2d(&tm.b1, g.W_lo, g.K, g.N, uint64_t(g.ldw) * 2, BK, BN / CG));
  } else {
    tm.a1 = tm.a0;
    tm.b1 = tm.b0;
  }
  if (r16) {
    IEF_TRY(make_tmap_2d(&tm.r, ep.resid_h16, g.N, g.M, uint64_t(ep.ld_resid) * 2, CW, 32, TM_BF16, TM_SWIZZLE_64B));
    if (e.resid_lo)
      IEF_TRY(make_tmap_2d(&tm.r2, ep.resid_l16, g.N, g.M, uint64_t(ep.ld_resid) * 2, CW, 32, TM_BF16, TM_SWIZZLE_64B));
  } else if (e.has_resid)
    IEF_TRY(make_tmap_2d(&tm.r, ep.resid, g.N, g.M, uint64_t(ep.ld_resid) * 4, CW, 32, TM_F32, TM_SWIZZLE_128B));
  if (e.has_f32) {
    const uint64_t w0 = ep.split_col < g.N ? ep.split_col : g.N;
    IEF_TRY(make_tmap_2d(&tm.o0, ep.out_f32, w0, uint64_t(g.M) * e.ksplit, uint64_t(ep.ld_f32) * 4, CW, 32, TM_F32, TM_SWIZZLE_128B));
    if (ep.split_col < g.N) {
      IEF_CHECK(ep.out_f32_b != nullptr, "gemm_tc: split_col set without out_f32_b");
      IEF_TRY(make_tmap_2d(&tm.o1, ep.out_f32_b, g.N - ep.split_col, g.M, uint64_t(ep.ld_f32) * 4, CW, 32, TM_F32,
                           TM_SWIZZLE_128B));
    }
  }
  if (ep.mode == EPI_ROWMAJOR && e.has_hi) {
    IEF_TRY(make_tmap_2d(&tm.h, ep.out_hi, g.N, g.M, uint64_t(ep.ld_bf) * 2, CW, 32, TM_BF16, TM_SWIZZLE_64B));
    if (e.has_lo)
      IEF_TRY(make_tmap_2d(&tm.l, ep.out_lo, g.N, g.M, uint64_t(ep.ld_bf) * 2, CW, 32, TM_BF16, TM_SWIZZLE_64B));
  }
  if (ep.mode == EPI_QKV && e.qk_tma) {
    const uint64_t Bn = (uint64_t(g.M) + ep.T - 1) / ep.T;
    const uint64_t dims[4] = {uint64_t(ep.dhp), uint64_t(ep.T), uint64_t(ep.H), Bn};
    const uint64_t strides[3] = {uint64_t(ep.dhp) * 2, uint64_t(ep.T) * ep.dhp * 2, uint64_t(ep.H) * ep.T * ep.dhp * 2};
    const uint32_t box[4] = {CW, 32, 1, 1};
    IEF_TRY(make_tmap_4d(&tm.h, ep.q, dims, strides, box, TM_BF16, TM_SWIZZLE_64B));
    IEF_TRY(make_tmap_4d(&tm.l, ep.k, dims, strides, box, TM_BF16, TM_SWIZZLE_64B));
    IEF_TRY(make_tmap_3d(&tm.v, ep.vt, uint64_t(ep.Tpad), uint64_t(ep.H) * ep.dh, Bn, uint64_t(ep.Tpad) * 2,
                         uint64_t(ep.H) * ep.dh * ep.Tpad * 2, CW, 32, 1, TM_SWIZZLE_NONE));
  }
  const int num_m = (g.M + BM * CG - 1) / (BM * CG), num_n = (g.N + BN - 1) / BN;
  const int tiles = num_m * num_n * e.ksplit;            // one per CTA (CG == 1) or per CTA pair (CG == 2)
  const int max_groups = num_sms / CG;
  const int grid = (tiles < max_groups ? tiles : max_groups) * CG;
  if (ep.mode == EPI_QKV) {
    IEF_CHECK(ep.act == ACT_NONE, "gemm_tc: the QKV epilogue has no activation");
    return launch_inst<BN, EPI_QKV, ACT_NONE, CG>(tm, g, e, grid, smem_bytes, stream);
  }
  if (r16) return launch_inst<BN, EPI_ROWMAJOR, ACT_NONE, CG, 1>(tm, g, e, grid, smem_bytes, stream);
  switch (ep.act) {       // EPI_DISCARD runs the row-major instance and drops the accumulator
    case ACT_NONE: return launch_inst<BN, EPI_ROWMAJOR, ACT_NONE, CG>(tm, g, e, grid, smem_bytes, stream);
    case ACT_RELU: return launch_inst<BN, EPI_ROWMAJOR, ACT_RELU, CG>(tm, g, e, grid, smem_bytes, stream);
    case ACT_QUICKGELU: return launch_inst<BN, EPI_ROWMAJOR, ACT_QUICKGELU, CG>(tm, g, e, grid, smem_bytes, stream);
    default: set_error("gemm_tc: unknown activation %d", ep.act); return IEFVAD_ERR_INVALID;
  }
}

}  // namespace

int gemm_tc(const GemmTcArgs& g, const EpiParams& ep, int num_sms, cudaStream_t stream) {
  IEF_CHECK(g.M > 0 && g.N > 0 && g.K > 0, "gemm_tc: empty problem M=%d N=%d K=%d", g.M, g.N, g.K);
  IEF_CHECK(g.K % BK == 0, "gemm_tc: K=%d must be a multiple of %d", g.K, BK);
  IEF_CHECK(g.N % 32 == 0, "gemm_tc: N=%d must be a multiple of 32", g.N);
  IEF_CHECK(g.lda % 8 == 0 && g.ldw % 8 == 0, "gemm_tc: leading dimensions must be multiples of 8 elements");
  IEF_CHECK(g.nsplit == 1 || g.nsplit == 3, "gemm_tc: nsplit must be 1 or 3");
  IEF_CHECK(g.A_hi && g.W_hi && (g.nsplit == 1 || (g.A_lo && g.W_lo)), "gemm_tc: null operand");
  const int num_m = (g.M + BM - 1) / BM;
  int bn = g.force_bn;
  if (bn == 0) {
    // largest tile that still gives every SM work; small problems trade tile efficiency for parallelism
    if (g.N % 256 == 0 && num_m * (g.N / 256) >= num_sms) bn = 256;
    else if (g.N % 128 == 0 && num_m * (g.N / 128) >= num_sms) bn = 128;
    else bn = 64;
  }
  // CTA pairs (256-row x 256-column tiles) whenever the shape allows and there is a tile for every pair
  int cg = g.force_cg;
  if (cg == 0) cg = (bn == 256 && ((g.M + 255) / 256) * (g.N / 256) >= num_sms / 2) ? 2 : 1;
  IEF_CHECK(cg == 1 || (cg == 2 && bn == 256 && g.N % 256 == 0), "gemm_tc: CTA pairs need BN == 256 and N %% 256 == 0");
  if (cg == 2) return launch_bn<256, 2>(g, ep, num_sms, stream);
  switch (bn) {
    case 256: return launch_bn<256, 1>(g, ep, num_sms, stream);
    case 128: return launch_bn<128, 1>(g, ep, num_sms, stream);
    case 64: return launch_bn<64, 1>(g, ep, num_sms, stream);
    default: set_error("gemm_tc: unsupported BN=%d", bn); return IEFVAD_ERR_INVALID;
  }
}

}  // namespace iefvad
