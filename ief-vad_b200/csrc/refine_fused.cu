// Fused refinement chain for sm_100a (model/imf_vad.py:146-149):
//     for s in 0..R-1:  x <- x - lambda * (W2_s . relu(W1_s . x + b1_s) + b2_s)          x: [M, 768]
// ONE persistent launch for all R steps.  A work unit is (step s, 256-row tile t); CTA pairs (cluster of 2, tcgen05
// cta_group::2, 128 rows per CTA) take units round-robin in (s, t) order, so the R * tiles units spread evenly over the 74
// pairs whatever the row count (no partial last wave per step), and unit (s, t) only waits for unit (s - 1, t) - finished
// about `tiles` units earlier by some other pair - through a per-tile step counter in global memory.
//
// Inside a unit the hidden activation h = relu(W1 x + b1) NEVER leaves the SM:
//   GEMM1  h chunk c (256 hidden units) = fp16(x) . W1[256 c .., :]^T   operands streamed by TMA (A 128 x 64 + the CTA's
//          half of the W tile per 32 KB stage, 6-stage ring), fp32 accumulator of 256 TMEM columns;
//          the epilogue warps turn it IN PLACE into packed fp16 pairs (128 columns) - the A operand of GEMM2;
//   GEMM2  x chunk n (128 columns) = h . W2[128 n .., :]^T with A read from TENSOR MEMORY (tcgen05.mma [d], [a], b-desc),
//          W2 streamed through the same ring; the epilogue adds the residual and writes the new fp16 (hi, lo) pair of x
//          in place in global memory (fp32 on the last step).
// Per row and step the kernel moves 6 KB of activations through HBM (the two-launch form: 10.5 KB) and h not at all.
// The arithmetic is the two-launch form's instruction for instruction (fp16 operands, fp32 accumulation in k order, h
// rounded to fp16 once, x = fp16 hi + lo pair, out = fma(-lambda, acc + b2, hi + lo)), so both forms agree bit for bit.
//
// (A first version kept fp16(x) of a tile resident in shared memory across all steps - 192 KB, which left a 32 KB weight
// ring: 4 stages of 8 KB cannot cover the ~1 700-cycle empty -> TMA -> full round trip, the kernel ran at 40 % of the
// two-launch form's speed (profiles/r2_refine_notes.md).  Streaming x with the weights costs L2 bandwidth, not latency.)
//
// TMEM columns (512 per CTA, lane = row):
//   GEMM1 accumulator of chunk c: [128 c, 128 c + 256)   ->   h chunk c packed in place: [128 c, 128 c + 128)
//   (the upper half of chunk c's accumulator is chunk c + 1's lower half: the epilogue reads it out first and releases it)
//   GEMM2 accumulator: [384, 512)  (= upper half of chunk 2, free once read out); h occupies [0, 384)
// Warp roles (320 threads): warp 0 = TMA producer, warp 1 = MMA issuer (leader CTA only), warps 2..9 = epilogue, two warps
// per TMEM lane quarter, each taking half of the columns.
#include <cstring>

#include "common.cuh"
#include "refine.cuh"
#include "tensormap.cuh"

namespace iefvad {

namespace {

constexpr int D = kRefineDim;
constexpr int BM = 128;                        // rows per CTA
constexpr int BK = 64;
constexpr int NKB = D / BK;                    // 12 k-blocks
constexpr int NCH1 = D / 256;                  // 3 h chunks of 256 hidden units
constexpr int NCH2 = D / 128;                  // 6 x chunks of 128 columns
constexpr int kThreads = 320;
constexpr int kEpiWarps = 8;
constexpr int STAGES = 5;
constexpr uint32_t kABox = BM * BK * 2;        // 16 KB: 128 rows x 64 k of fp16(x)
constexpr uint32_t kW1Box = 128 * BK * 2;      // 16 KB: this CTA's 128 of the 256 W1 rows x 64 k
constexpr uint32_t kW2Box = 64 * BK * 2;       //  8 KB: this CTA's 64 of the 128 W2 rows x 64 k (4 per stage)
constexpr uint32_t kStage = kABox + kW1Box;    // 32 KB
// epilogue staging: three 4 KB tiles (32 rows x 128 B, 16-byte chunks XOR-swizzled by the row) per epilogue warp, through
// which the warp's share of x moves between "one thread = one row" (the TMEM view) and "one instruction = four whole
// 128-byte rows" (the only global access pattern the LSU serves at full rate)
constexpr uint32_t kOffStageBuf = STAGES * kStage;
constexpr uint32_t kWarpStage = 8192;      // Hb, Lb: the (hi, lo) chunk coming in, then the new pair going out
constexpr uint32_t kOffBar = kOffStageBuf + kEpiWarps * kWarpStage;
constexpr uint32_t kSmemBytes = 1024 + kOffBar + 256;
static_assert(kSmemBytes <= 232448, "shared memory budget");
static_assert(4 * kW2Box == kStage, "a GEMM2 stage holds four 64-k boxes of W2");

__device__ __forceinline__ void tma_load_3d_cg2(const CUtensorMap* m, uint32_t bar_cluster_addr, void* smem_dst, int c0, int c1,
                                                int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      :
      : "r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(bar_cluster_addr), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}

// D[tmem] (+)= A[tmem] . B[smem]^T on a CTA pair: each CTA's tensor core reads its own 128 lanes of A
__device__ __forceinline__ void umma_f16_ts_cg2(uint32_t tmem_d, uint32_t tmem_a, uint64_t desc_b, uint32_t idesc,
                                                uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
      :
      : "r"(tmem_d), "r"(tmem_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}

// Arrival on a barrier of the leader CTA that hands TENSOR-MEMORY state over (accumulator read out / h written): the
// tcgen05 fences order those accesses, so the arrive itself is relaxed - a release here would make the warp wait for
// every global store and cp.async it has in flight (ncu: MEMBAR.ALL.CTA + ERRBAR, 15 % of the kernel's stall samples)
__device__ __forceinline__ void mbar_arrive_tmem(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.relaxed.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
// explicit shared-space accesses (the staging pointers are derived from the aligned dynamic-smem base, which the compiler
// only knows as a generic address: LD.E / ST.E to shared memory take the slow generic path)
__device__ __forceinline__ uint4 lds128(uint32_t addr) {
  uint4 v;
  asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr) : "memory");
  return v;
}
__device__ __forceinline__ int ld_relaxed_gpu(const int* p) {
  int v;
  asm volatile("ld.relaxed.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
// smem (shared-space address) -> global tensor store; rows past the tensor bound are clipped
__device__ __forceinline__ void tma_store_2d_s(const CUtensorMap* m, uint32_t smem_src, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
               :
               : "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_src), "r"(c0), "r"(c1)
               : "memory");
}
__device__ __forceinline__ void sts128(uint32_t addr, const uint4& v) {
  asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
__device__ __forceinline__ int ld_acquire_gpu(const int* p) {
  int v;
  asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void fence_proxy_async_all() { asm volatile("fence.proxy.async;" ::: "memory"); }
// 16-byte global -> shared copy that bypasses L1 (L2 is the coherence point); src_bytes = 0 writes zeros
__device__ __forceinline__ void cp_async16(uint32_t smem_dst, const void* gsrc, uint32_t src_bytes) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(smem_dst), "l"(gsrc), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }
__device__ __forceinline__ uint32_t sw128(int row, int c) { return uint32_t(row) * 128u + (uint32_t(c ^ (row & 7)) << 4); }

struct RefineParams {
  const float* b1[kRefineMaxSteps];
  const float* b2[kRefineMaxSteps];
  __half* x_hi;            // [M, 768] fp16(x), rewritten in place every step
  __half* x_lo;            // [M, 768] fp16(x - hi), rewritten in place every step
  float* out;              // fp32 [M, 768]: x after the last step
  int* done;               // [tiles] += 16 whenever a step of the tile is complete (8 epilogue warps x 2 CTAs)
  long long M;
  int steps;
  float lambda;
  int num_tiles;           // tiles of 256 rows
};

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kThreads, 1)
refine_chain_kernel(const __grid_constant__ CUtensorMap tmX, const __grid_constant__ CUtensorMap tmW1,
                    const __grid_constant__ CUtensorMap tmW2, const __grid_constant__ CUtensorMap tmSH,
                    const __grid_constant__ CUtensorMap tmSL, const __grid_constant__ CUtensorMap tmSO, const RefineParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + kOffBar);
  uint64_t* full = bars;                  // [STAGES] leader: stage landed (both CTAs' parts)
  uint64_t* empty = bars + 6;             // [STAGES] each CTA: stage consumed (multicast commit)
  uint64_t* accfull = bars + 12;          // each CTA: a GEMM1 chunk's accumulator is complete (multicast commit)
  uint64_t* upfree = bars + 13;           // leader: the upper half of that accumulator has been read out by the whole pair
  uint64_t* hrdy = bars + 14;             // [3] leader: h chunk c is in TMEM (every epilogue warp of the pair)
  uint64_t* a2full = bars + 17;           // each CTA: a GEMM2 chunk's accumulator is complete
  uint64_t* a2free = bars + 18;           // leader: it has been read out by the whole pair
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 20);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const int pair = blockIdx.x >> 1, npairs = gridDim.x >> 1;
  const int R = p.steps, T = p.num_tiles;
  const int units = R * T;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmX);
    tma_prefetch_desc(&tmW1);
    tma_prefetch_desc(&tmW2);
    tma_prefetch_desc(&tmSH);
    tma_prefetch_desc(&tmSL);
    tma_prefetch_desc(&tmSO);
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], 1);
    }
    mbar_init(accfull, 1);
    mbar_init(upfree, kEpiWarps * 2);
    for (int c = 0; c < NCH1; ++c) mbar_init(&hrdy[c], kEpiWarps * 2);
    mbar_init(a2full, 1);
    mbar_init(a2free, kEpiWarps * 2);
    fence_barrier_init();
  }
  if (warp == 1) {
    tmem_alloc_cg2(tmem_slot, 512);
    tmem_relinquish_cg2();
  }
  tc_fence_before();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  auto lead = [&](uint64_t* bar) { return mapa_shared(smem_u32(bar), 0); };      // the leader CTA's copy of a barrier

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      int st = 0;
      uint32_t ph = 0;
      for (int u = pair; u < units; u += npairs) {
        const int s = u / T, t = u - s * T;
        const int row0 = (t * 2 + int(rank)) * BM;
        if (s > 0) {
          // unit (s - 1, t) - some pair's work ~T units ago - has written this tile's fp16(x): wait for all its 16 warps
          uint32_t spins = 0;
          while (ld_acquire_gpu(p.done + t) < 16 * s) {
            __nanosleep(64);
            if (++spins > (1u << 24)) __trap();
          }
          fence_proxy_async_all();       // the rows were written by generic stores; the TMA reads below are async-proxy
        }
        for (int c = 0; c < NCH1; ++c)
          for (int kb = 0; kb < NKB; ++kb) {
            mbar_wait(&empty[st], ph ^ 1);
            if (rank == 0) mbar_arrive_expect_tx(&full[st], 2 * kStage);
            uint8_t* dst = smem + size_t(st) * kStage;
            tma_load_2d_cg2(&tmX, lead(&full[st]), dst, kb * BK, row0);
            tma_load_3d_cg2(&tmW1, lead(&full[st]), dst + kABox, kb * BK, c * 256 + int(rank) * 128, 2 * s);
            if (++st == STAGES) { st = 0; ph ^= 1; }
          }
        for (int n = 0; n < NCH2; ++n)
          for (int kq = 0; kq < 3; ++kq) {
            mbar_wait(&empty[st], ph ^ 1);
            if (rank == 0) mbar_arrive_expect_tx(&full[st], 2 * kStage);
            uint8_t* dst = smem + size_t(st) * kStage;
#pragma unroll
            for (int j = 0; j < 4; ++j)
              tma_load_3d_cg2(&tmW2, lead(&full[st]), dst + j * kW2Box, kq * 256 + j * BK, n * 128 + int(rank) * 64, 2 * s + 1);
            if (++st == STAGES) { st = 0; ph ^= 1; }
          }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (leader CTA) =====================
    if (lane == 0 && rank == 0) {
      const uint32_t idesc1 = make_idesc_f16(256, 256);
      const uint32_t idesc2 = make_idesc_f16(256, 128);
      int st = 0;
      uint32_t ph = 0, n_up = 0, n_a2 = 0;
      int it = 0;
      for (int u = pair; u < units; u += npairs, ++it) {
        // ---- GEMM1: accumulator of chunk c at columns [128 c, 128 c + 256)
        for (int c = 0; c < NCH1; ++c) {
          if (c > 0) { mbar_wait(upfree, n_up & 1u); ++n_up; }     // chunk c - 1's upper half is in registers
          if (c == 2 && it > 0) { mbar_wait(a2free, n_a2 & 1u); ++n_a2; }   // previous unit's last GEMM2 chunk too
          tc_fence_after();
          const uint32_t d_tmem = tmem_base + uint32_t(128 * c);
          for (int kb = 0; kb < NKB; ++kb) {
            mbar_wait(&full[st], ph);
            tc_fence_after();
            const uint32_t sa = smem_u32(smem + size_t(st) * kStage);
            const uint64_t da = make_smem_desc_sw128(sa), db = make_smem_desc_sw128(sa + kABox);
#pragma unroll
            for (int k4 = 0; k4 < BK / 16; ++k4)
              umma_bf16_cg2(d_tmem, da + uint64_t(2 * k4), db + uint64_t(2 * k4), idesc1, (kb | k4) != 0 ? 1u : 0u);
            tc_commit_cg2(&empty[st], 3);
            if (++st == STAGES) { st = 0; ph ^= 1; }
          }
          tc_commit_cg2(accfull, 3);
        }
        // ---- GEMM2: accumulator at [384, 512) (chunk 2's upper half), A = h chunk kq at columns [128 kq, 128 kq + 128)
        mbar_wait(upfree, n_up & 1u);
        ++n_up;
        const uint32_t d2 = tmem_base + 384u;
        for (int n = 0; n < NCH2; ++n) {
          if (n > 0) { mbar_wait(a2free, n_a2 & 1u); ++n_a2; }
          tc_fence_after();
          for (int kq = 0; kq < 3; ++kq) {
            mbar_wait(&full[st], ph);
            if (n == 0) mbar_wait(&hrdy[kq], uint32_t(it) & 1u);
            tc_fence_after();
            const uint32_t sb = smem_u32(smem + size_t(st) * kStage);
#pragma unroll
            for (int i = 0; i < 16; ++i) {
              const uint32_t a = tmem_base + uint32_t(128 * kq + 8 * i);
              const uint64_t db = make_smem_desc_sw128(sb + uint32_t(i >> 2) * kW2Box) + uint64_t(2 * (i & 3));
              umma_f16_ts_cg2(d2, a, db, idesc2, (kq | i) != 0 ? 1u : 0u);
            }
            tc_commit_cg2(&empty[st], 3);
            if (++st == STAGES) { st = 0; ph ^= 1; }
          }
          tc_commit_cg2(a2full, 3);
        }
      }
    }
  } else {
    // ===================== epilogue (warps 2..9) =====================
    const int q = warp & 3;                       // TMEM lane quarter of this warp
    const int hf = (warp - 2) >> 2;               // which half of the columns
    const int r = q * 32 + lane;                  // row inside the CTA's 128-row tile == TMEM lane
    const uint32_t tlane = tmem_base + (uint32_t(q * 32) << 16);
    const float nlam = -p.lambda;
    const uint32_t Hb = smem_u32(smem + kOffStageBuf + size_t(warp - 2) * kWarpStage);      // shared-space addresses
    const uint32_t Lb = Hb + 4096;
    uint32_t n_acc = 0, n_a2 = 0;
    int publish_t = -1;                           // tile whose step this warp has finished but not yet published
    auto publish = [&]() {                        // this warp's share of a step of tile publish_t is in global memory
      if (publish_t >= 0 && lane == 0) {
        bulk_wait_all<0>();                       // the tensor stores have been performed, not just read out of Ob
        fence_proxy_async_all();
        __threadfence();
        atomicAdd(p.done + publish_t, 1);
      }
      publish_t = -1;
    };
    for (int u = pair; u < units; u += npairs) {
      const int s = u / T, t = u - s * T;
      const bool last = s == R - 1;
      const float* b2 = p.b2[s];
      if (s > 0) {      // unit (s - 1, t) must have written this tile's (hi, lo) before the copies below read them.  Its writer
        // fenced before bumping the counter and the copies read L2 (cp.async.cg) behind a branch on the counter, so a
        // relaxed poll is enough (an acquire costs a MEMBAR + L1 invalidation per warp and unit: 13 % of the stall samples)
        if (lane == 0)
          while (ld_relaxed_gpu(p.done + t) < 16 * s) __nanosleep(32);
        __syncwarp();
      }
      // global side of the staging tiles: instruction j moves rows 4 j + (lane >> 3), 16-byte chunk lane & 7 of this warp's
      // 32 rows x 64 columns - four whole 128-byte rows per instruction
      const long long wrow0 = (long long)(t * 2 + int(rank)) * BM + q * 32;
      const int crow = lane >> 3, cchk = lane & 7;
      auto fetch = [&](int n) {                  // hi / lo of chunk n -> Hb / Lb (asynchronous)
        const int col0 = n * 128 + 64 * hf;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const long long rr = wrow0 + 4 * j + crow;
          const bool ok = rr < p.M;
          const size_t off = size_t(ok ? rr : 0) * D + col0 + 8 * cchk;
          cp_async16(Hb + sw128(4 * j + crow, cchk), p.x_hi + off, ok ? 16u : 0u);
          cp_async16(Lb + sw128(4 * j + crow, cchk), p.x_lo + off, ok ? 16u : 0u);
        }
      };
      fetch(0);                                   // lands while GEMM1 and its epilogue run
      // ---- h = relu(acc + b1) -> packed fp16, in place over the lower half of the chunk's accumulator
      const float* b1 = p.b1[s];
#pragma unroll 1
      for (int c = 0; c < NCH1; ++c) {
        mbar_wait(accfull, n_acc & 1u);
        ++n_acc;
        tc_fence_after();
        float v[64];
        uint32_t pk[64];
        auto pack = [&](const float* bias, uint32_t* dst) {
          const float4* bp = reinterpret_cast<const float4*>(bias);
#pragma unroll
          for (int g = 0; g < 16; ++g) {
            const float4 b = __ldg(bp + g);
            const __half2 h01 = __floats2half2_rn(fmaxf(v[4 * g] + b.x, 0.f), fmaxf(v[4 * g + 1] + b.y, 0.f));
            const __half2 h23 = __floats2half2_rn(fmaxf(v[4 * g + 2] + b.z, 0.f), fmaxf(v[4 * g + 3] + b.w, 0.f));
            dst[2 * g] = *reinterpret_cast<const uint32_t*>(&h01);
            dst[2 * g + 1] = *reinterpret_cast<const uint32_t*>(&h23);
          }
        };
        // upper half first: it is the next chunk's (or GEMM2's) accumulator
        const uint32_t tu = tlane + uint32_t(128 * c + 128 + 64 * hf);
        tmem_ld32(tu, v);
        tmem_ld32(tu + 32, v + 32);
        tmem_ld_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_tmem(lead(upfree));
        if (c == 0) publish();                    // the previous unit's results (nothing waits on this warp meanwhile)
        pack(b1 + c * 256 + 128 + 64 * hf, pk + 32);
        const uint32_t tl = tlane + uint32_t(128 * c + 64 * hf);
        tmem_ld32(tl, v);
        tmem_ld32(tl + 32, v + 32);
        tmem_ld_wait();
        tc_fence_before();
        named_bar_sync(1 + q, 64);                // both warps of the quarter hold their lower-half columns
        pack(b1 + c * 256 + 64 * hf, pk);
        tc_fence_after();
        const uint32_t th = tlane + uint32_t(128 * c + 32 * hf);
        tmem_st16(th, pk);                        // hidden units [64 hf, 64 hf + 64) of the chunk
        tmem_st16(th + 16, pk + 16);
        tmem_st16(th + 64, pk + 32);              // hidden units [128 + 64 hf, ...)
        tmem_st16(th + 80, pk + 48);
        tmem_st_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_tmem(lead(&hrdy[c]));
      }
      // ---- x <- fma(-lambda, acc + b2, hi + lo); new fp16 pair in place (fp32 on the last step)
#pragma unroll 1
      for (int n = 0; n < NCH2; ++n) {
        const int col0 = n * 128 + 64 * hf;
        // the accumulator first: the tensor pipe idles until every warp of the pair has read it out
        mbar_wait(a2full, n_a2 & 1u);
        ++n_a2;
        tc_fence_after();
        float v[64];
        const uint32_t ta = tlane + 384u + uint32_t(64 * hf);
        tmem_ld32(ta, v);
        tmem_ld32(ta + 32, v + 32);
        tmem_ld_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_tmem(lead(a2free));
        cp_async_wait_all();
        __syncwarp();
        uint4 h4[8], l4[8];
#pragma unroll
        for (int c = 0; c < 8; ++c) {            // my row's 64 columns of hi and lo
          h4[c] = lds128(Hb + sw128(lane, c));
          l4[c] = lds128(Lb + sw128(lane, c));
        }
        const float4* bp = reinterpret_cast<const float4*>(b2 + col0);
#pragma unroll
        for (int g = 0; g < 8; ++g) {
          const float4 ba = __ldg(bp + 2 * g), bb = __ldg(bp + 2 * g + 1);
          const float bias[8] = {ba.x, ba.y, ba.z, ba.w, bb.x, bb.y, bb.z, bb.w};
          float x[8];
          unpack_f16x8(h4[g], &l4[g], x);
          // the same operation order as the two-launch epilogue: (acc + bias), then fma(-lambda, ., hi + lo)
#pragma unroll
          for (int e = 0; e < 8; ++e) v[8 * g + e] = fmaf(nlam, v[8 * g + e] + bias[e], x[e]);
          if (!last) {                            // the new pair, kept in the registers the old one came in
            split_16x2(v[8 * g], v[8 * g + 1], 1, h4[g].x, l4[g].x);
            split_16x2(v[8 * g + 2], v[8 * g + 3], 1, h4[g].y, l4[g].y);
            split_16x2(v[8 * g + 4], v[8 * g + 5], 1, h4[g].z, l4[g].z);
            split_16x2(v[8 * g + 6], v[8 * g + 7], 1, h4[g].w, l4[g].w);
          }
        }
        // out through the tiles the chunk came in (every lane rewrites exactly the slots it read): two bulk tensor stores;
        // the next chunk's copies start as soon as the stores have read the tiles
#pragma unroll
        for (int c = 0; c < 8; ++c) {
          if (!last) {
            sts128(Hb + sw128(lane, c), h4[c]);
            sts128(Lb + sw128(lane, c), l4[c]);
          } else {                                // fp32 result: columns [0, 32) of this warp's 64 in Hb, [32, 64) in Lb
            sts128(Hb + sw128(lane, c), make_uint4(__float_as_uint(v[4 * c]), __float_as_uint(v[4 * c + 1]),
                                                   __float_as_uint(v[4 * c + 2]), __float_as_uint(v[4 * c + 3])));
            sts128(Lb + sw128(lane, c), make_uint4(__float_as_uint(v[32 + 4 * c]), __float_as_uint(v[32 + 4 * c + 1]),
                                                   __float_as_uint(v[32 + 4 * c + 2]), __float_as_uint(v[32 + 4 * c + 3])));
          }
        }
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) {
          if (!last) {
            tma_store_2d_s(&tmSH, Hb, col0, int(wrow0));
            tma_store_2d_s(&tmSL, Lb, col0, int(wrow0));
          } else {
            tma_store_2d_s(&tmSO, Hb, col0, int(wrow0));
            tma_store_2d_s(&tmSO, Lb, col0 + 32, int(wrow0));
          }
          bulk_commit();
          bulk_wait_read<0>();                    // the stores have read Hb / Lb
        }
        __syncwarp();
        if (n + 1 < NCH2) fetch(n + 1);
      }
      // Published after the next unit's first accumulator read-out (waiting for the stores here would delay it) - but only
      // when that next unit cannot depend on this one: with more tiles than pairs its predecessor (s, t') lies before this
      // unit in the global order; with T <= npairs it may BE this unit, and deferring would deadlock the pair on itself.
      if (!last) {
        publish_t = t;
        if (T <= npairs) publish();
      }
    }
    publish();
    if (lane == 0) bulk_wait_all<0>();            // Ob must outlive the last stores
  }

  tc_fence_before();
  cluster_sync_all();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc_cg2(tmem_base, 512);
  }
}

}  // namespace

size_t refine_chain_scratch_bytes(long long M) { return size_t((M + 255) / 256) * sizeof(int) + 16; }

bool refine_chain_preferred(long long M, int num_sms) {
  // a unit (256 rows, one step) keeps one CTA pair busy: enough tiles to give every pair work within a step
  return (M + 255) / 256 >= num_sms / 2;
}

int refine_chain(const RefineChainArgs& a, int num_sms, cudaStream_t stream) {
  IEF_CHECK(a.x_hi && a.x_lo && a.w16 && a.out_f32 && a.lo_scratch, "refine_chain: null argument");
  IEF_CHECK(a.steps >= 1 && a.steps <= kRefineMaxSteps, "refine_chain: 1 <= steps <= %d", kRefineMaxSteps);
  IEF_CHECK(a.M > 0 && a.M < (1LL << 31), "refine_chain: bad row count %lld", a.M);
  CUtensorMap tx, tw1, tw2, tsh, tsl, tso;
  IEF_TRY(make_tmap_2d(&tx, a.x_hi, D, uint64_t(a.M), uint64_t(D) * 2, BK, BM));
  // epilogue stores: 32 rows x 128 bytes per warp and box
  IEF_TRY(make_tmap_2d(&tsh, a.x_hi, D, uint64_t(a.M), uint64_t(D) * 2, 64, 32));
  IEF_TRY(make_tmap_2d(&tsl, a.x_lo, D, uint64_t(a.M), uint64_t(D) * 2, 64, 32));
  IEF_TRY(make_tmap_2d(&tso, a.out_f32, D, uint64_t(a.M), uint64_t(D) * 4, 32, 32, TM_F32, TM_SWIZZLE_128B));
  IEF_TRY(make_tmap_3d(&tw1, a.w16, D, D, uint64_t(2 * a.steps), uint64_t(D) * 2, uint64_t(D) * D * 2, BK, 128, 1));
  IEF_TRY(make_tmap_3d(&tw2, a.w16, D, D, uint64_t(2 * a.steps), uint64_t(D) * 2, uint64_t(D) * D * 2, BK, 64, 1));
  RefineParams p;
  memset(&p, 0, sizeof(p));
  for (int s = 0; s < a.steps; ++s) {
    IEF_CHECK(a.b1[s] && a.b2[s], "refine_chain: null bias of step %d", s);
    p.b1[s] = a.b1[s];
    p.b2[s] = a.b2[s];
  }
  p.x_hi = static_cast<__half*>(a.x_hi);
  p.x_lo = static_cast<__half*>(a.x_lo);
  p.out = a.out_f32;
  p.done = static_cast<int*>(a.lo_scratch);
  p.M = a.M;
  p.steps = a.steps;
  p.lambda = a.lambda;
  p.num_tiles = int((a.M + 255) / 256);
  IEF_CUDA(cudaMemsetAsync(p.done, 0, size_t(p.num_tiles) * sizeof(int), stream));
  const int pairs = num_sms / 2;
  const long long units = (long long)p.num_tiles * a.steps;
  const int grid = int(units < pairs ? units : pairs) * 2;
  static bool attr_set = false;
  if (!attr_set) {
    IEF_CUDA(cudaFuncSetAttribute(refine_chain_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(kSmemBytes)));
    attr_set = true;
  }
  refine_chain_kernel<<<grid, kThreads, kSmemBytes, stream>>>(tx, tw1, tw2, tsh, tsl, tso, p);
  IEF_CUDA(cudaGetLastError());
  count_launches(1);
  return IEFVAD_OK;
}

}  // namespace iefvad
