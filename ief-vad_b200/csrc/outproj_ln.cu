// Out-projection + residual + LayerNorm (+ whitening LayerNorm) of one temporal-encoder layer in ONE tcgen05 kernel:
//     y = x + ctx . Wo^T + bo ;  z = LN_i(y) ;  [ out = LN_whiten(z) ]        (model/imf_vad.py:115-117 / :121-123)
// The two-launch form (GEMM writes fp32 y, the LayerNorm kernel reads it back) moves 16-18 bytes per element through HBM
// and both launches are HBM-bound; here y never leaves tensor memory: 8 bytes per element (context and residual in,
// the 16-bit result (pair) out).
//
// * The residual is added BY THE TENSOR CORE: after the 12 k-blocks of ctx . Wo^T the accumulator takes 4 (8 with a
//   remainder part) more blocks  x[:, 64 tile columns] . I_64^T  into the 64 accumulator columns they belong to (N = 64
//   MMAs with a 64 x 64 fp16 identity as the W operand, resident in shared memory; two x boxes share one ring stage) -
//   exact (every product is x * 1 or x * 0, fp32 accumulation) and the tensor pipe has the time, while the CUDA cores,
//   which bound the first version of this kernel, lose a shared-memory ring, two conversions and two additions per element.
// * A LayerNorm row spans all 768 output columns but an accumulator tile is 256 columns wide (a CTA pair owns 256 rows x
//   256 columns, cta_group::2, fp32 accumulators = half of TMEM, double-buffered).  So THREE pairs - a "group" - work on
//   the three column tiles of the same 256-row block at the same time: they are ONE CLUSTER of 6 CTAs and exchange
//   per-row partial sums through distributed shared memory.  Per tile an epilogue warp (32 rows x 128 columns, thread ==
//   row) runs
//     pass 1  tcgen05.ld accumulator chunk -> + bias -> y back into TMEM (tcgen05.st), accumulating the shifted sums of
//             its part; the record goes into the three CTAs that own these rows with st.async ... complete_tx on THEIR
//             mbarrier (no fence on the sending side)
//     merge   wait on the local mbarrier (one expect_tx of 6 records x 32 lanes: 3 column tiles x 2 warps per row quarter),
//             merge the parts in part order
//     pass 2  tcgen05.ld y -> normalise -> fp16 (hi [, lo]) boxes -> TMA stores (or row-mapped stores)
// * The sixteen epilogue warps form TWO TEAMS of eight; team t owns accumulator buffer t and the tiles of its parity, so
//   while one team waits for the exchange (or for its accumulator) the other one computes, and every scheduler holds
//   four epilogue warps to interleave.
// * Both LayerNorms need only ONE exchange: with u_c = w1_c (y_c - mu), z_c = r u_c + b1_c the second LayerNorm's
//   statistics are  mean(z) = r mean(u) + mean(b1),  var(z) = r^2 var(u) + 2 r cov(u, b1) + var(b1), and mean(u),
//   mean(u^2), mean(u b1) follow from the sums of w d, w^2 d, w^2 d^2, w b1 d (d = y - shift) gathered in pass 1 once mu
//   is known.
// Per-row results do not depend on the tile position or the batch size.
#include <cstring>

#include "outproj_ln.cuh"
#include "tensormap.cuh"

namespace iefvad {

namespace {

constexpr int D = kOutprojLnDim;
constexpr int BM = 128;
constexpr int BN = 256;
constexpr int BK = 64;
constexpr int CW = 32;
constexpr int kNT = D / BN;                      // column tiles of a row block = CTA pairs per group
constexpr int kEpiWarps = 16;                    // two teams of 8 (two warps per TMEM lane quarter)
constexpr int kThreads = 64 + 32 * kEpiWarps;
constexpr int kParts = 2 * kNT;                  // partial statistics per row
constexpr int kPartCols = D / kParts;            // 128 columns per part
constexpr int kMaxStages = 6;
constexpr uint32_t kABytes = BM * BK * 2;
constexpr uint32_t kBBytes = (BN / 2) * BK * 2;
constexpr uint32_t kStageBytes = kABytes + kBBytes;
constexpr uint32_t kBox16 = 32 * CW * 2;         // 32 rows x 32 columns of fp16 (64-byte rows, SWIZZLE_64B)
constexpr uint32_t kBarBytes = 384;
constexpr uint32_t kParamBytes = 5 * BN * 4;     // bias, w1, b1, w2, b2 of this CTA's 256 columns
constexpr uint32_t kConstBytes = 128;            // per-part sums of the LayerNorm parameters (see PartConsts)
constexpr uint32_t kSmemLimit = 232448;
constexpr int kClusterCtas = 2 * kNT;             // three CTA pairs
constexpr int kKBMain = D / BK;                  // k-blocks of ctx . Wo^T
constexpr int kKBRes = BN / BK;                  // k-blocks of x[:, 64 tile columns] . I_64^T
constexpr uint32_t kIBytes = (BK / 2) * BK * 2;  // this CTA's half (32 rows) of the 64 x 64 identity

struct LnParams {
  const float* bias;
  const float* w1;
  const float* b1;
  const float* w2;
  const float* b2;
  float eps;
  int M;
  int num_mp;          // 256-row blocks
  int groups;          // blocks in flight (grid = groups * kNT pairs)
  int stages;
  uint32_t warp_bytes;
  const int* row_map;
  __half* out_hi;      // row-mapped stores only
};

// sums over the 128 columns of each part of w1, w1^2 and w1 * b1 (exact inputs of the second LayerNorm's statistics),
// plus mean and variance of b1 over all 768 columns
struct PartConsts {
  float c0[kParts], c1[kParts], c2[kParts];
  float b_mean, b_var;
};

__device__ __forceinline__ uint32_t sw64(int row, int g) { return uint32_t(row) * 64u + (uint32_t(g ^ ((row >> 1) & 3)) << 4); }

// DSMEM exchange: 16-byte asynchronous store into another CTA of the cluster that completes on an mbarrier of that CTA
// (complete_tx, like a TMA copy) - no fence on the sending side (a release at cluster scope compiles to MEMBAR.ALL.GPU,
// which waits for every output store of the previous tile: 16 % of the kernel in the first DSMEM version)
__device__ __forceinline__ void st_async_v4(uint32_t addr, float4 v, uint32_t mbar) {
  asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v4.f32 [%0], {%1, %2, %3, %4}, [%5];" ::"r"(addr),
               "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w), "r"(mbar)
               : "memory");
}

__global__ void outproj_ln_identity_kernel(__half* ident) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < BK * BK) ident[i] = __float2half_rn((i / BK) == (i % BK) ? 1.f : 0.f);
}

// TWO: a second (whitening) LayerNorm follows; RES_LO: the residual has a remainder part; OUT_LO: so has the result
template <int TWO, int RES_LO, int OUT_LO>
__global__ void __launch_bounds__(kThreads, 1)
outproj_ln_kernel(const __grid_constant__ CUtensorMap ta, const __grid_constant__ CUtensorMap tw,
                  const __grid_constant__ CUtensorMap trh, const __grid_constant__ CUtensorMap trl,
                  const __grid_constant__ CUtensorMap tid, const __grid_constant__ CUtensorMap toh,
                  const __grid_constant__ CUtensorMap tol, const LnParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int STAGES = p.stages;
  uint8_t* ident = smem + size_t(STAGES) * kStageBytes;              // this CTA's half (32 rows) of the 64 x 64 identity
  uint8_t* epi_base = ident + kIBytes;
  float* prm = reinterpret_cast<float*>(epi_base + kEpiWarps * p.warp_bytes);      // [5][BN]
  PartConsts* pc = reinterpret_cast<PartConsts*>(reinterpret_cast<uint8_t*>(prm) + kParamBytes);
  constexpr int kRec = TWO ? 8 : 4;                                  // floats per (row, part) record: shift, S1, S2, A1 [, A2, A3, A4, -]
  float* xch = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(pc) + kConstBytes);     // [2 teams][BM rows][kParts][kRec]
  uint64_t* bars = reinterpret_cast<uint64_t*>(xch + 2 * BM * kParts * kRec);
  uint64_t* full = bars;
  uint64_t* empty = full + kMaxStages;
  uint64_t* tfull = empty + kMaxStages;
  uint64_t* tempty = tfull + 2;
  uint64_t* xbar = tempty + 2;                                       // [2 teams][4 quarters]
  uint64_t* ibar = xbar + 8;                                         // the identity halves of both CTAs have landed
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(ibar + 1);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t crank = cluster_ctarank();                          // 0 .. 5: pair = crank / 2, position in the pair = crank % 2
  const uint32_t rank = crank & 1u;
  const uint32_t lead = crank & ~1u;                                 // the pair's leader CTA
  const int grp = blockIdx.x / kClusterCtas;
  const int n_blk = int(crank >> 1);
  constexpr int kResStages = kKBRes * (1 + RES_LO) / 2;              // two 64-column residual boxes per ring stage
  constexpr int kKB = kKBMain + kResStages;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&ta);
    tma_prefetch_desc(&tw);
    tma_prefetch_desc(&trh);
    tma_prefetch_desc(&tid);
    if (RES_LO) tma_prefetch_desc(&trl);
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(&tfull[s], 1);
      mbar_init(&tempty[s], kEpiWarps);          // the 8 warps of the owning team in each CTA of the pair
    }
    for (int s = 0; s < 8; ++s) mbar_init(&xbar[s], 1);        // one local arrive.expect_tx per tile; the records arrive as tx bytes
    mbar_init(ibar, 1);
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

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      {   // the identity, once: both CTAs' halves complete on the leader's barrier
        const uint32_t lead_ibar = mapa_shared(smem_u32(ibar), lead);
        if (rank == 0) mbar_arrive_expect_tx(ibar, 2 * kIBytes);
        tma_load_2d_cg2(&tid, lead_ibar, ident, 0, int(rank) * (BK / 2));
      }
      int s = 0;
      uint32_t ph = 0;
      for (int mp = grp; mp < p.num_mp; mp += p.groups) {
        const int m_blk = mp * 2 + int(rank);
        for (int kb = 0; kb < kKB; ++kb) {
          mbar_wait(&empty[s], ph ^ 1);
          uint8_t* sa = smem + size_t(s) * kStageBytes;
          const uint32_t lead_full = mapa_shared(smem_u32(&full[s]), lead);
          if (rank == 0) mbar_arrive_expect_tx(&full[s], 2 * kStageBytes);
          if (kb < kKBMain) {
            tma_load_2d_cg2(&ta, lead_full, sa, kb * BK, m_blk * BM);
            tma_load_2d_cg2(&tw, lead_full, sa + kABytes, kb * BK, n_blk * BN + int(rank) * (BN / 2));
          } else {
            // residual stage: two A boxes x[rows, tile columns kk * 64 ..] (the W operand is the resident identity)
#pragma unroll
            for (int b = 0; b < 2; ++b) {
              const int kr = 2 * (kb - kKBMain) + b;
              const int kk = kr & (kKBRes - 1);
              const CUtensorMap* tr = (RES_LO && kr >= kKBRes) ? &trl : &trh;
              tma_load_2d_cg2(tr, lead_full, sa + b * kABytes, n_blk * BN + kk * BK, m_blk * BM);
            }
          }
          if (++s == STAGES) { s = 0; ph ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (leader CTA) =====================
    if (lane == 0 && rank == 0) {
      constexpr uint32_t idesc = make_idesc_f16(2 * BM, BN);
      constexpr uint32_t idesc_res = make_idesc_f16(2 * BM, BK);
      const uint16_t pair_mask = uint16_t(3u << lead);
      bool ident_ready = false;
      int s = 0;
      uint32_t ph = 0;
      int it = 0;
      for (int mp = grp; mp < p.num_mp; mp += p.groups, ++it) {
        const int as = it & 1;
        const uint32_t aph = (it >> 1) & 1;
        mbar_wait(&tempty[as], aph ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + uint32_t(as * BN);
        for (int kb = 0; kb < kKB; ++kb) {
          mbar_wait(&full[s], ph);
          tc_fence_after();
          const uint32_t sa = smem_u32(smem + size_t(s) * kStageBytes);
          const uint64_t da = make_smem_desc_sw128(sa);
          const uint64_t db = make_smem_desc_sw128(sa + kABytes);
          if (kb < kKBMain) {
#pragma unroll
            for (int k4 = 0; k4 < BK / 16; ++k4)
              umma_bf16_cg2(d_tmem, da + uint64_t(2 * k4), db + uint64_t(2 * k4), idesc, (kb | k4) != 0 ? 1u : 0u);
          } else {
            if (!ident_ready) {
              mbar_wait(ibar, 0);
              tc_fence_after();
              ident_ready = true;
            }
            const uint64_t di = make_smem_desc_sw128(smem_u32(ident));
#pragma unroll
            for (int b = 0; b < 2; ++b) {
              const int kr = 2 * (kb - kKBMain) + b;
              const uint32_t d_res = d_tmem + uint32_t((kr & (kKBRes - 1)) * BK);     // the 64 columns this box adds to
              const uint64_t dab = make_smem_desc_sw128(sa + uint32_t(b) * kABytes);
#pragma unroll
              for (int k4 = 0; k4 < BK / 16; ++k4)
                umma_bf16_cg2(d_res, dab + uint64_t(2 * k4), di + uint64_t(2 * k4), idesc_res, 1u);
            }
          }
          tc_commit_cg2(&empty[s], pair_mask);
          if (++s == STAGES) { s = 0; ph ^= 1; }
        }
        tc_commit_cg2(&tfull[as], pair_mask);
      }
    }
  } else {
    // ===================== epilogue: two teams of 8 warps, thread == accumulator row =====================
    const int ew = warp - 2;
    const int quarter = warp & 3;          // TMEM lanes [32 * quarter, +32)
    const int team = ew >> 3;              // owns accumulator buffer `team` and the tiles of that parity
    const int par = (ew >> 2) & 1;         // chunks par, par + 2, par + 4, par + 6 of the tile's 8 32-column chunks
    const int part = n_blk * 2 + par;
    uint8_t* Hb = epi_base + size_t(ew) * p.warp_bytes;
    uint8_t* Lb = Hb + kBox16;
    if (lane == 0 && !p.row_map) {
      tma_prefetch_desc(&toh);
      if (OUT_LO) tma_prefetch_desc(&tol);
    }

    // ---- parameters of this CTA's 256 columns -> smem (broadcast reads in the passes); per-part parameter sums
    {
      const int t = int(threadIdx.x) - 64;            // 0 .. 511
      if (t < BN) {
        const int col = n_blk * BN + t;
        prm[0 * BN + t] = __ldg(p.bias + col);
        prm[1 * BN + t] = __ldg(p.w1 + col);
        prm[2 * BN + t] = __ldg(p.b1 + col);
        prm[3 * BN + t] = TWO ? __ldg(p.w2 + col) : 1.f;
        prm[4 * BN + t] = TWO ? __ldg(p.b2 + col) : 0.f;
      }
      if (ew == kEpiWarps - 1 && TWO) {
        float bs = 0.f;
        for (int c = lane; c < D; c += 32) bs += __ldg(p.b1 + c);
        const float bm = warp_sum(bs) * (1.f / D);
        float bq = 0.f;
        for (int c = lane; c < D; c += 32) { const float d = __ldg(p.b1 + c) - bm; bq = fmaf(d, d, bq); }
        const float bv = warp_sum(bq) * (1.f / D);
        for (int pp = 0; pp < kParts; ++pp) {
          float c0 = 0.f, c1 = 0.f, c2 = 0.f;
          for (int j = 0; j < 4; ++j) {
            const int c = (pp >> 1) * BN + ((pp & 1) + 2 * j) * CW + lane;
            const float w = __ldg(p.w1 + c), b = __ldg(p.b1 + c);
            c0 += w; c1 = fmaf(w, w, c1); c2 = fmaf(w, b, c2);
          }
          c0 = warp_sum(c0); c1 = warp_sum(c1); c2 = warp_sum(c2);
          if (lane == 0) { pc->c0[pp] = c0; pc->c1[pp] = c1; pc->c2[pp] = c2; }
        }
        if (lane == 0) { pc->b_mean = bm; pc->b_var = bv; }
      }
      named_bar_sync(1, kEpiWarps * 32);
    }

    const float inv_part = 1.f / float(kPartCols);
    const uint32_t t0 = tmem_base + uint32_t(team * BN) + (uint32_t(quarter * 32) << 16);

    int it = team;
    for (int mp = grp + team * p.groups; mp < p.num_mp; mp += 2 * p.groups, it += 2) {
      const int m_blk = mp * 2 + int(rank);
      const uint32_t aph = (it >> 1) & 1;
      const int row0 = m_blk * BM + quarter * 32;
      const long long row = (long long)row0 + lane;
      int dst_row = -1;
      if (p.row_map && row < p.M) dst_row = __ldg(p.row_map + row);
      float* xrow = xch + ((size_t(team) * BM + size_t(quarter * 32 + lane)) * kParts) * kRec;   // this row's records

      mbar_wait(&tfull[team], aph);
      tc_fence_after();
      float v[32];

      // ---- pass 1: y = acc (= ctx . Wo^T + x) + bias, back into TMEM; shifted sums of this thread's 128 columns
      float shift = 0.f, S1 = 0.f, S2 = 0.f, A1 = 0.f, A2 = 0.f, A3 = 0.f, A4 = 0.f;
#pragma unroll 1
      for (int j = 0; j < 4; ++j) {
        const int c = par + 2 * j;
        const float4* pb = reinterpret_cast<const float4*>(prm + c * CW);
        tmem_ld32(t0 + uint32_t(c * CW), v);
        tmem_ld_wait_for(v);
#pragma unroll
        for (int g = 0; g < 8; ++g) {
          const float4 b4 = pb[g];
          v[g * 4 + 0] += b4.x; v[g * 4 + 1] += b4.y; v[g * 4 + 2] += b4.z; v[g * 4 + 3] += b4.w;
        }
        tmem_st32(t0 + uint32_t(c * CW), v);
        if (j == 0) shift = v[0];
        if (TWO) {
#pragma unroll
          for (int g = 0; g < 8; ++g) {
            const float4 w4 = pb[BN / 4 + g], c4 = pb[2 * BN / 4 + g];
            const float ws[4] = {w4.x, w4.y, w4.z, w4.w}, bs[4] = {c4.x, c4.y, c4.z, c4.w};
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const float d = v[g * 4 + e] - shift;
              const float wd = ws[e] * d;
              S1 += d;
              S2 = fmaf(d, d, S2);
              A1 += wd;
              A2 = fmaf(ws[e], wd, A2);
              A3 = fmaf(wd, wd, A3);
              A4 = fmaf(wd, bs[e], A4);
            }
          }
        } else {
#pragma unroll
          for (int e = 0; e < 32; ++e) {
            const float d = v[e] - shift;
            S1 += d;
            S2 = fmaf(d, d, S2);
          }
        }
      }
      tmem_st_wait();

      // ---- publish this part's sums to the three CTAs that work on these rows (same position in their pair), then wait
      // for all six parts of the rows of this quarter
      {
        uint64_t* xb = &xbar[team * 4 + quarter];
        if (par == 0 && lane == 0) mbar_arrive_expect_tx(xb, uint32_t(kParts * 32 * kRec * 4));
        const uint32_t rec = smem_u32(xrow + part * kRec);
#pragma unroll
        for (int j = 0; j < kNT; ++j) {
          const uint32_t cta = uint32_t(2 * j) + rank;
          const uint32_t dst = mapa_shared(rec, cta), bar = mapa_shared(smem_u32(xb), cta);
          st_async_v4(dst, make_float4(shift, S1, S2, A1), bar);
          if (TWO) st_async_v4(dst + 16, make_float4(A2, A3, A4, 0.f), bar);
        }
        mbar_wait(xb, uint32_t(it >> 1) & 1u);
      }
      float mean, rstd, zbar = 0.f, rstd2 = 1.f;
      {
        float sh[kParts], a1[kParts], ml[kParts];
        float sm = 0.f, m2 = 0.f;
#pragma unroll
        for (int i = 0; i < kParts; ++i) {
          const float4 a = *reinterpret_cast<const float4*>(xrow + i * kRec);
          sh[i] = a.x; a1[i] = a.w;
          ml[i] = fmaf(a.y, inv_part, a.x);
          sm += ml[i];
          m2 += fmaxf(fmaf(-a.y * inv_part, a.y, a.z), 0.f);
        }
        mean = sm * (1.f / kParts);
        float dev = 0.f;
#pragma unroll
        for (int i = 0; i < kParts; ++i) { const float d = ml[i] - mean; dev = fmaf(d, d, dev); }
        const float var = fmaf(dev, float(kPartCols), m2) * (1.f / D);
        rstd = 1.f / sqrtf(var + p.eps);
        if (TWO) {
          // u_c = w1_c (y_c - mean):  sum u, sum u^2, sum u b1 from the shifted sums (delta = mean - shift of the part)
          float su = 0.f, suu = 0.f, sub = 0.f;
#pragma unroll
          for (int i = 0; i < kParts; ++i) {
            const float4 b = *reinterpret_cast<const float4*>(xrow + i * kRec + 4);
            const float dl = mean - sh[i];
            su += fmaf(-dl, pc->c0[i], a1[i]);
            suu += fmaf(dl, fmaf(dl, pc->c1[i], -2.f * b.x), b.y);
            sub += fmaf(-dl, pc->c2[i], b.z);
          }
          const float ubar = su * (1.f / D);
          const float var_u = fmaxf(fmaf(-ubar, ubar, suu * (1.f / D)), 0.f);
          const float cov = fmaf(-ubar, pc->b_mean, sub * (1.f / D));
          const float var_z = fmaxf(fmaf(rstd * rstd, var_u, fmaf(2.f * rstd, cov, pc->b_var)), 0.f);
          rstd2 = 1.f / sqrtf(var_z + p.eps);
          zbar = fmaf(rstd, ubar, pc->b_mean);
        }
      }

      // ---- pass 2: normalise and store
#pragma unroll 1
      for (int j = 0; j < 4; ++j) {
        const int c = par + 2 * j;
        const int col0 = n_blk * BN + c * CW;
        const float4* pb = reinterpret_cast<const float4*>(prm + c * CW);
        tmem_ld32(t0 + uint32_t(c * CW), v);
        tmem_ld_wait_for(v);
        if (j == 3) {                                    // accumulator fully read: hand the buffer back to the MMA warp
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive_cluster(mapa_shared(smem_u32(&tempty[team]), lead));
        }
#pragma unroll
        for (int g = 0; g < 8; ++g) {
          const float4 w4 = pb[BN / 4 + g], c4 = pb[2 * BN / 4 + g];
          v[g * 4 + 0] = (v[g * 4 + 0] - mean) * rstd * w4.x + c4.x;
          v[g * 4 + 1] = (v[g * 4 + 1] - mean) * rstd * w4.y + c4.y;
          v[g * 4 + 2] = (v[g * 4 + 2] - mean) * rstd * w4.z + c4.z;
          v[g * 4 + 3] = (v[g * 4 + 3] - mean) * rstd * w4.w + c4.w;
        }
        if (TWO) {
#pragma unroll
          for (int g = 0; g < 8; ++g) {
            const float4 w4 = pb[3 * BN / 4 + g], c4 = pb[4 * BN / 4 + g];
            v[g * 4 + 0] = (v[g * 4 + 0] - zbar) * rstd2 * w4.x + c4.x;
            v[g * 4 + 1] = (v[g * 4 + 1] - zbar) * rstd2 * w4.y + c4.y;
            v[g * 4 + 2] = (v[g * 4 + 2] - zbar) * rstd2 * w4.z + c4.z;
            v[g * 4 + 3] = (v[g * 4 + 3] - zbar) * rstd2 * w4.w + c4.w;
          }
        }
        // the finished 32 x 32 chunk -> fp16 (hi [, lo]) boxes -> global
        if (!p.row_map && lane == 0) bulk_wait_read<0>();  // the previous chunk's stores have read the boxes
        __syncwarp();
#pragma unroll
        for (int g = 0; g < 4; ++g) {
          uint32_t hi[4], lo[4];
#pragma unroll
          for (int q = 0; q < 4; ++q) split_16x2(v[g * 8 + 2 * q], v[g * 8 + 2 * q + 1], 1, hi[q], lo[q]);
          *reinterpret_cast<uint4*>(Hb + sw64(lane, g)) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
          if (OUT_LO) *reinterpret_cast<uint4*>(Lb + sw64(lane, g)) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
        }
        if (p.row_map) {
          // 64-byte row pieces to mapped rows: 4 lanes per row, 8 rows per instruction
          __syncwarp();
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const int r = i * 8 + (lane >> 2), g = lane & 3;
            const int dr = __shfl_sync(0xffffffffu, dst_row, r);
            const uint4 u = *reinterpret_cast<const uint4*>(Hb + sw64(r, g));
            if (dr >= 0) *reinterpret_cast<uint4*>(p.out_hi + (size_t(dr) * D + col0 + g * 8)) = u;
          }
        } else {
          fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0) {
            tma_store_2d(&toh, Hb, col0, row0);
            if (OUT_LO) tma_store_2d(&tol, Lb, col0, row0);
            bulk_commit();
          }
        }
      }
    }
    if (lane == 0) bulk_wait_all<0>();     // smem boxes must outlive their stores
  }

  tc_fence_before();
  cluster_sync_all();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc_cg2(tmem_base, 512);
  }
}

long long padded_rows(long long M) { return (M + 255) / 256 * 256; }

}  // namespace

size_t outproj_ln_scratch_bytes(long long) { return 16; }   // the exchange lives in distributed shared memory now

size_t outproj_ln_identity_bytes() { return size_t(BK) * BK * sizeof(__half); }

int outproj_ln_identity(void* ident, cudaStream_t stream) {
  IEF_CHECK(ident, "outproj_ln_identity: null buffer");
  outproj_ln_identity_kernel<<<(BK * BK + 255) / 256, 256, 0, stream>>>(static_cast<__half*>(ident));
  IEF_CUDA(cudaGetLastError());
  count_launches(1);
  return IEFVAD_OK;
}

int outproj_ln(const OutprojLnArgs& a, int num_sms, cudaStream_t stream) {
  IEF_CHECK(a.ctx && a.w16 && a.bias && a.res_hi && a.ln_w && a.ln_b && a.out_hi && a.scratch && a.identity,
            "outproj_ln: null argument");
  IEF_CHECK((a.ln2_w == nullptr) == (a.ln2_b == nullptr), "outproj_ln: ln2_w and ln2_b go together");
  IEF_CHECK(!(a.row_map && a.out_lo), "outproj_ln: row-mapped output has no remainder part");
  IEF_CHECK(a.M > 0 && a.M < (1LL << 31) - 256, "outproj_ln: bad row count %lld", a.M);
  IEF_CHECK(num_sms >= 2 * kNT, "outproj_ln: needs at least %d SMs", 2 * kNT);
  const long long Mp = padded_rows(a.M);
  LnParams p;
  memset(&p, 0, sizeof(p));
  p.bias = a.bias; p.w1 = a.ln_w; p.b1 = a.ln_b; p.w2 = a.ln2_w; p.b2 = a.ln2_b; p.eps = a.eps;
  p.M = int(a.M);
  p.num_mp = int(Mp / 256);
  const int res_lo = a.res_lo ? 1 : 0, out_lo = a.out_lo ? 1 : 0, two = a.ln2_w ? 1 : 0;
  p.warp_bytes = kBox16 + (out_lo ? kBox16 : 0);
  const uint32_t xch_bytes = 2 * BM * kParts * (two ? 8 : 4) * 4;
  const uint32_t fixed = 1024 + kIBytes + kEpiWarps * p.warp_bytes + kParamBytes + kConstBytes + xch_bytes + kBarBytes;
  p.stages = int((kSmemLimit - fixed) / kStageBytes);
  if (p.stages > kMaxStages) p.stages = kMaxStages;
  IEF_CHECK(p.stages >= 2, "outproj_ln: no room for the operand ring");
  const size_t smem_bytes = fixed + size_t(p.stages) * kStageBytes;
  p.row_map = a.row_map;
  p.out_hi = static_cast<__half*>(a.out_hi);

  CUtensorMap ta, tw, trh, trl, tid, toh, tol;
  IEF_TRY(make_tmap_2d(&ta, a.ctx, D, uint64_t(a.M), uint64_t(D) * 2, BK, BM));
  IEF_TRY(make_tmap_2d(&tw, a.w16, D, D, uint64_t(D) * 2, BK, BN / 2));
  IEF_TRY(make_tmap_2d(&trh, a.res_hi, D, uint64_t(a.M), uint64_t(D) * 2, BK, BM));
  if (a.res_lo) IEF_TRY(make_tmap_2d(&trl, a.res_lo, D, uint64_t(a.M), uint64_t(D) * 2, BK, BM));
  else trl = trh;
  IEF_TRY(make_tmap_2d(&tid, a.identity, BK, BK, uint64_t(BK) * 2, BK, BK / 2));
  if (!a.row_map) IEF_TRY(make_tmap_2d(&toh, a.out_hi, D, uint64_t(a.M), uint64_t(D) * 2, CW, 32, TM_BF16, TM_SWIZZLE_64B));
  else toh = trh;
  if (a.out_lo) IEF_TRY(make_tmap_2d(&tol, a.out_lo, D, uint64_t(a.M), uint64_t(D) * 2, CW, 32, TM_BF16, TM_SWIZZLE_64B));
  else tol = toh;

  const int variant = two * 4 + res_lo * 2 + out_lo;
  using KernelFn = void (*)(CUtensorMap, CUtensorMap, CUtensorMap, CUtensorMap, CUtensorMap, CUtensorMap, CUtensorMap, LnParams);
  static const KernelFn kernels[8] = {outproj_ln_kernel<0, 0, 0>, outproj_ln_kernel<0, 0, 1>, outproj_ln_kernel<0, 1, 0>,
                                      outproj_ln_kernel<0, 1, 1>, outproj_ln_kernel<1, 0, 0>, outproj_ln_kernel<1, 0, 1>,
                                      outproj_ln_kernel<1, 1, 0>, outproj_ln_kernel<1, 1, 1>};
  static bool attr_set[8] = {};
  if (!attr_set[variant]) {
    IEF_CUDA(cudaFuncSetAttribute(kernels[variant], cudaFuncAttributeMaxDynamicSharedMemorySize, int(kSmemLimit)));
    attr_set[variant] = true;
  }
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.blockDim = dim3(kThreads);
  cfg.dynamicSmemBytes = smem_bytes;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = kClusterCtas;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  // as many clusters as can be resident at once (one CTA per SM, six SMs of one GPC per cluster)
  static int max_clusters[8] = {};
  if (max_clusters[variant] == 0) {
    cfg.gridDim = dim3(unsigned(kClusterCtas * (num_sms / kClusterCtas)));
    int n = 0;
    IEF_CUDA(cudaOccupancyMaxActiveClusters(&n, kernels[variant], &cfg));
    IEF_CHECK(n >= 1, "outproj_ln: no cluster of %d CTAs fits on this device", kClusterCtas);
    max_clusters[variant] = n;
  }
  p.groups = p.num_mp < max_clusters[variant] ? p.num_mp : max_clusters[variant];
  cfg.gridDim = dim3(unsigned(p.groups * kClusterCtas));
  IEF_CUDA(cudaLaunchKernelEx(&cfg, kernels[variant], ta, tw, trh, trl, tid, toh, tol, p));
  count_launches(1);
  return IEFVAD_OK;
}

}  // namespace iefvad
