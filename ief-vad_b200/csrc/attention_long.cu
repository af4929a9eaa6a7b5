// Self-attention core for LONG sequences (T > 256, no masks): direct module calls such as the T = 16 384 stress case
// (SURVEY config 5).  softmax(Q K^T) V without materialising the [B, H, T, T] scores (the reference does materialise
// them: need_weights=True, model/imf_vad.py:115,121 -> 8 GiB per layer at T = 16 384).
//
// Persistent, one CTA per SM, 18 warps.  Work item = 256 query rows (two 128-row tiles a, b) of one (batch, head);
// K / V^T stream through a 2-stage TMA ring in blocks of 128 keys, shared by both tiles.  Per tile and block:
//   S = Q_t.K_blk^T (128 x 128 fp32) -> TMEM columns [0, 128) of the tile
//   16 softmax warps (two threads per query row, 64 keys each) read S ONCE: every thread exponentiates against the
//   maximum of its OWN 64 keys, rounded up to an integer in the log2 domain, so that aligning the two halves of a row
//   and, later, the blocks of a row with each other only ever multiplies by exact powers of two (packed fp16 P by
//   HMUL2, the fp32 accumulators by FMUL) - nothing waits for a row maximum before the SFU work, and no rounding is
//   added by the online-softmax rescaling;
//   P (packed 16-bit pairs) goes back into TMEM columns [0, 64) over the consumed S;
//   O += P.V_blk accumulates in TMEM columns [128, 128 + DH) over all key blocks (A operand = P read from TMEM).  P is
//   always written in units of 2^(running maximum); when a row's running maximum grows (rare after the first blocks,
//   rarer still for integer maxima) the threads of that warp rescale their O columns in TMEM by the exact power of
//   two before releasing P - otherwise O is not touched until the item ends.
// The MMA warp alternates the tiles (P.V_a(j), S_a(j+1), P.V_b(j), S_b(j+1)), so one tile's softmax overlaps the other
// tile's tensor work; MMAs of one tile are ordered by the in-order tensor pipe (P.V(j) reads P before S(j+1) overwrites it).
#include "attention.cuh"
#include "common.cuh"
#include "tensormap.cuh"

namespace iefvad {

namespace {

constexpr float kLog2e = 1.4426950408889634f;
constexpr int kSoftmaxWarps = 16;
constexpr int kThreads = (kSoftmaxWarps + 2) * 32;
constexpr float kNone = -30000.f;        // "no key yet" in the integer log2 domain: 2^(kNone - anything sane) == 0

template <int DH, int DHP>
struct LongCfg {
  static constexpr int KB = 128;                                   // keys per block
  static constexpr uint32_t kQChunk = 128 * 128;                   // [128 rows x 64 columns] 128B-swizzled
  static constexpr uint32_t kQTile = (DHP / 64) * kQChunk;
  static constexpr uint32_t kKBytes = (DHP / 64) * kQChunk;        // one 128-key block of K
  static constexpr uint32_t kVSub = DH * 128;                      // [DH rows x 64 keys]
  static constexpr uint32_t kVBytes = (KB / 64) * kVSub;
  static constexpr uint32_t kOffK = 2 * kQTile;
  static constexpr uint32_t kOffV = kOffK + 2 * kKBytes;
  static constexpr uint32_t kOffX = kOffV + 2 * kVBytes;           // per-row exchange between the two key halves
  static constexpr uint32_t kXBytes = 2 * 2 * 2 * 128 * 4;         // parity x tile x half x row
  static constexpr uint32_t kOffBar = kOffX + kXBytes;
  static constexpr size_t kSmemBytes = 1024 + kOffBar + 256;
  static constexpr uint32_t kColO = 128;                           // TMEM columns of a tile: S / P [0, 128), O [128, 128 + DH)
  static_assert(kColO + DH <= 256, "O does not fit behind S");
  static_assert(DH % 32 == 0, "each thread owns DH / 2 columns in 16-column pieces");
};

template <int DH, int DHP>
__global__ void __launch_bounds__(kThreads, 1)
attn_long_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmK,
                 const __grid_constant__ CUtensorMap tmVt, bf16* __restrict__ out, int ldo, int T, int H, int n_items,
                 int fp16, const int* __restrict__ row_out) {
  using Cfg = LongCfg<DH, DHP>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + Cfg::kOffBar);
  uint64_t* q_full = bars + 0;
  uint64_t* q_empty = bars + 1;
  uint64_t* k_full = bars + 2;     // [2]
  uint64_t* v_full = bars + 4;     // [2]
  uint64_t* kv_empty = bars + 6;   // [2]
  uint64_t* s_full = bars + 8;     // [2 tiles]
  uint64_t* p_full = bars + 10;    // [2]
  uint64_t* o_full = bars + 12;    // [2]
  uint64_t* o_empty = bars + 14;   // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 16);
  float* xch = reinterpret_cast<float*>(smem + Cfg::kOffX);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int q_pairs = (T + 255) / 256;          // items per (batch, head)
  const int nb = (T + Cfg::KB - 1) / Cfg::KB;   // key blocks

  if (warp == kSoftmaxWarps && lane == 0) {
    tma_prefetch_desc(&tmQ);
    tma_prefetch_desc(&tmK);
    tma_prefetch_desc(&tmVt);
    mbar_init(q_full, 1);
    mbar_init(q_empty, 1);
    for (int s = 0; s < 2; ++s) {
      mbar_init(&k_full[s], 1);
      mbar_init(&v_full[s], 1);
      mbar_init(&kv_empty[s], 1);
      mbar_init(&s_full[s], 1);
      mbar_init(&p_full[s], 256);
      mbar_init(&o_full[s], 1);
      mbar_init(&o_empty[s], 256);
    }
    fence_barrier_init();
  }
  if (warp == kSoftmaxWarps + 1) {
    tmem_alloc(tmem_slot, 512);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == kSoftmaxWarps) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      int it = 0;
      uint32_t n = 0;                                   // key blocks loaded so far (all items)
      for (int item = blockIdx.x; item < n_items; item += gridDim.x, ++it) {
        const int bh = item / q_pairs, qp = item - bh * q_pairs;
        mbar_wait(q_empty, (it & 1) ^ 1);
        mbar_arrive_expect_tx(q_full, 2 * Cfg::kQTile);
#pragma unroll
        for (int t = 0; t < 2; ++t)
#pragma unroll
          for (int c = 0; c < DHP / 64; ++c)
            tma_load_3d(&tmQ, q_full, smem + t * Cfg::kQTile + c * Cfg::kQChunk, c * 64, qp * 256 + t * 128, bh);
        for (int j = 0; j < nb; ++j, ++n) {
          const int s = int(n & 1);
          mbar_wait(&kv_empty[s], ((n >> 1) & 1) ^ 1);
          uint8_t* sk = smem + Cfg::kOffK + s * Cfg::kKBytes;
          uint8_t* sv = smem + Cfg::kOffV + s * Cfg::kVBytes;
          mbar_arrive_expect_tx(&k_full[s], Cfg::kKBytes);
#pragma unroll
          for (int c = 0; c < DHP / 64; ++c) tma_load_3d(&tmK, &k_full[s], sk + c * Cfg::kQChunk, c * 64, j * Cfg::KB, bh);
          mbar_arrive_expect_tx(&v_full[s], Cfg::kVBytes);
#pragma unroll
          for (int c = 0; c < Cfg::KB / 64; ++c)
            tma_load_3d(&tmVt, &v_full[s], sv + c * Cfg::kVSub, j * Cfg::KB + c * 64, 0, bh);
        }
      }
    }
  } else if (warp == kSoftmaxWarps + 1) {
    // ===================== MMA issuer =====================
    if (lane == 0) {
      const uint32_t idesc_s = fp16 ? make_idesc_f16(128, Cfg::KB) : make_idesc_bf16(128, Cfg::KB);
      const uint32_t idesc_o = fp16 ? make_idesc_f16(128, DH) : make_idesc_bf16(128, DH);
      const uint32_t sq = smem_u32(smem);
      auto issue_s = [&](int t, int s) {
        const uint32_t sk = smem_u32(smem + Cfg::kOffK + s * Cfg::kKBytes);
        const uint32_t d = tmem_base + uint32_t(t * 256);
#pragma unroll
        for (int kk = 0; kk < DH / 16; ++kk) {   // only the DH real columns of the DHP-padded rows
          const int c = kk >> 2, k4 = kk & 3;
          umma_bf16(d, make_smem_desc_sw128(sq + t * Cfg::kQTile + c * Cfg::kQChunk) + uint64_t(2 * k4),
                    make_smem_desc_sw128(sk + c * Cfg::kQChunk) + uint64_t(2 * k4), idesc_s, kk != 0 ? 1u : 0u);
        }
        tc_commit(&s_full[t]);
      };
      auto issue_pv = [&](int t, int s, bool first) {
        const uint32_t sv = smem_u32(smem + Cfg::kOffV + s * Cfg::kVBytes);
        const uint32_t tb = tmem_base + uint32_t(t * 256);
#pragma unroll
        for (int kk = 0; kk < Cfg::KB / 16; ++kk) {
          const int c = kk >> 2, k4 = kk & 3;
          umma_f16_ts(tb + Cfg::kColO, tb + uint32_t(kk * 8), make_smem_desc_sw128(sv + c * Cfg::kVSub) + uint64_t(2 * k4),
                      idesc_o, (first && kk == 0) ? 0u : 1u);
        }
        tc_commit(&o_full[t]);
      };
      int it = 0;
      uint32_t n = 0;                                   // key blocks consumed so far (all items)
      for (int item = blockIdx.x; item < n_items; item += gridDim.x, ++it) {
        mbar_wait(q_full, it & 1);
        mbar_wait(&k_full[n & 1], (n >> 1) & 1);
        tc_fence_after();
        issue_s(0, int(n & 1));
        issue_s(1, int(n & 1));
        for (int j = 0; j < nb; ++j, ++n) {
          const int s = int(n & 1);
          const uint32_t par = n & 1;                   // every per-block barrier flips once per block
          const bool more = j + 1 < nb;
          if (more) mbar_wait(&k_full[s ^ 1], ((n + 1) >> 1) & 1);
          mbar_wait(&v_full[s], (n >> 1) & 1);
#pragma unroll
          for (int t = 0; t < 2; ++t) {
            mbar_wait(&p_full[t], par);                 // P written (and O rescaled if the row maximum moved)
            if (j == 0) mbar_wait(&o_empty[t], (it & 1) ^ 1);   // the previous item's O has been read out
            tc_fence_after();
            issue_pv(t, s, j == 0);
            if (t == 1) tc_commit(&kv_empty[s]);        // K / V stage free once both tiles' P.V retire
            if (more) issue_s(t, s ^ 1);                // in order behind P.V: it reads P before this overwrites S
            else if (t == 1) tc_commit(q_empty);
          }
        }
      }
    }
  } else {
    // ===================== softmax / fold / store (warps 0..15) =====================
    const int t = warp >> 3;                        // query tile
    const int hf = (warp >> 2) & 1;                 // key half of a block: keys [64 hf, 64 hf + 64)
    const int quarter = warp & 3;                   // TMEM lane quarter this warp may access
    const int r = quarter * 32 + lane;              // query row inside the tile == TMEM lane
    const uint32_t tbase = tmem_base + uint32_t(t * 256) + (uint32_t(quarter * 32) << 16);
    auto slot = [&](uint32_t par, int half) { return xch + ((((int(par) * 2 + t) * 2 + half)) << 7) + r; };

    uint32_t n = 0;
    for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
      const int bh = item / q_pairs, qp = item - bh * q_pairs;
      const int b = bh / H, h = bh - b * H;
      const int tq = qp * 256 + t * 128 + r;
      float run = kNone;          // running row maximum (integer, log2 domain), the same in both halves of the row
      float l = 0.f;              // this half's share of the row sum, in units of 2^run

      for (int j = 0; j < nb; ++j, ++n) {
        const uint32_t par = n & 1;
        const int k_lo = j * Cfg::KB + hf * 64;
        mbar_wait(&s_full[t], par);
        tc_fence_after();
        float v[64];
        tmem_ld32(tbase + uint32_t(hf * 64), v);
        tmem_ld32(tbase + uint32_t(hf * 64 + 32), v + 32);
        tmem_ld_wait();
        // ---- this half's own maximum, rounded up to an integer in the log2 domain
        float mx = -INFINITY;
        const bool full = k_lo + 64 <= T;
        if (full) {
#pragma unroll
          for (int i = 0; i < 64; ++i) mx = fmaxf(mx, v[i]);
        } else {
#pragma unroll
          for (int i = 0; i < 64; ++i)
            if (k_lo + i < T) mx = fmaxf(mx, v[i]);
        }
        const float mloc = (mx == -INFINITY) ? kNone : ceilf(mx * kLog2e);
        *slot(par, hf) = mloc;
        // ---- P = 2^(S log2e - mloc) in (0, 1], packed; nothing here depends on the other half or on earlier blocks
        uint32_t pk[32];
        float lsum = 0.f;
#pragma unroll
        for (int i = 0; i < 64; i += 2) {
          float p0 = fast_exp2(fmaf(v[i], kLog2e, -mloc));
          float p1 = fast_exp2(fmaf(v[i + 1], kLog2e, -mloc));
          if (!full) {
            if (k_lo + i >= T) p0 = 0.f;
            if (k_lo + i + 1 >= T) p1 = 0.f;
          }
          lsum += p0 + p1;
          pk[i >> 1] = pack_16x2(p0, p1, fp16);
        }
        // ---- align with the other half of the row and with the running maximum: exact powers of two
        named_bar_sync(1 + t, 256);                                   // also: both halves have read their S
        const float run_new = fmaxf(run, fmaxf(mloc, *slot(par, hf ^ 1)));
        const float sc = fast_exp2(mloc - run_new);                   // 2^-k, k >= 0 (0 for an empty half)
        const float a_old = fast_exp2(run - run_new);                 // rescale of everything accumulated so far
        if (fp16) {
          const __half2 s2 = __float2half2_rn(sc);
#pragma unroll
          for (int i = 0; i < 32; ++i) {
            const __half2 x = __hmul2(*reinterpret_cast<const __half2*>(&pk[i]), s2);
            pk[i] = *reinterpret_cast<const uint32_t*>(&x);
          }
        } else {
          const __nv_bfloat162 s2 = __float2bfloat162_rn(sc);
#pragma unroll
          for (int i = 0; i < 32; ++i) {
            const __nv_bfloat162 x = __hmul2(*reinterpret_cast<const __nv_bfloat162*>(&pk[i]), s2);
            pk[i] = *reinterpret_cast<const uint32_t*>(&x);
          }
        }
        tmem_st16(tbase + uint32_t(hf * 32), pk);
        tmem_st16(tbase + uint32_t(hf * 32 + 16), pk + 16);
        l = fmaf(l, a_old, lsum * sc);
        // ---- the running maximum of some row of this warp moved: bring the accumulated O of the warp's rows to the new
        // unit before P.V of this block adds to it (P.V of the previous block must have retired first)
        const bool moved = (j > 0) && (run_new != run);
        run = run_new;
        if (__any_sync(0xffffffffu, moved)) {
          mbar_wait(&o_full[t], par ^ 1);
          tc_fence_after();
          float o[DH / 2];
#pragma unroll
          for (int c = 0; c < DH / 32; ++c) tmem_ld16(tbase + Cfg::kColO + uint32_t(hf * (DH / 2) + c * 16), o + c * 16);
          tmem_ld_wait();
          const float f = moved ? a_old : 1.f;
#pragma unroll
          for (int d = 0; d < DH / 2; ++d) o[d] *= f;
#pragma unroll
          for (int c = 0; c < DH / 32; ++c)
            tmem_st16(tbase + Cfg::kColO + uint32_t(hf * (DH / 2) + c * 16), reinterpret_cast<const uint32_t*>(o + c * 16));
        }
        tmem_st_wait();
        tc_fence_before();
        mbar_arrive(&p_full[t]);
      }
      // ---- the item's last P.V: read O, add the two halves' row-sum shares (same unit), normalise, store
      mbar_wait(&o_full[t], (n - 1) & 1);
      tc_fence_after();
      float o[DH / 2];
#pragma unroll
      for (int c = 0; c < DH / 32; ++c) tmem_ld16(tbase + Cfg::kColO + uint32_t(hf * (DH / 2) + c * 16), o + c * 16);
      tmem_ld_wait();
      tc_fence_before();
      mbar_arrive(&o_empty[t]);
      const uint32_t parx = n & 1;       // the slot pair the next block (of the next item) will use: idle now
      *slot(parx, hf) = l;
      named_bar_sync(1 + t, 256);
      const float inv = 1.f / (l + *slot(parx, hf ^ 1));
      long long ro = (long long)b * T + (tq < T ? tq : 0);
      if (row_out) ro = __ldg(row_out + ro);              // compact layouts: < 0 = this row is dropped
      if (tq < T && ro >= 0) {
        bf16* dst = out + ro * ldo + h * DH + hf * (DH / 2);
#pragma unroll
        for (int d = 0; d < DH / 2; d += 8) *reinterpret_cast<uint4*>(dst + d) = pack_16x8(o + d, fp16, inv);
      }
      named_bar_sync(1 + t, 256);        // the slots are written again by the next item's first block
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == kSoftmaxWarps + 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

template <int DH, int DHP>
int launch_attn_long(const AttnTcArgs& a, int num_sms, cudaStream_t stream) {
  using Cfg = LongCfg<DH, DHP>;
  static bool attr_set = false;
  if (!attr_set) {
    IEF_CUDA(cudaFuncSetAttribute(attn_long_kernel<DH, DHP>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  static_cast<int>(Cfg::kSmemBytes)));
    attr_set = true;
  }
  const uint64_t BH = uint64_t(a.B) * a.H;
  CUtensorMap tq, tk, tv;
  IEF_TRY(make_tmap_3d(&tq, a.q, DHP, a.T, BH, uint64_t(DHP) * 2, uint64_t(a.T) * DHP * 2, 64, 128, 1));
  IEF_TRY(make_tmap_3d(&tk, a.k, DHP, a.T, BH, uint64_t(DHP) * 2, uint64_t(a.T) * DHP * 2, 64, 128, 1));
  IEF_TRY(make_tmap_3d(&tv, a.vt, a.T, DH, BH, uint64_t(a.Tpad) * 2, uint64_t(DH) * a.Tpad * 2, 64, DH, 1));
  const long long items = (long long)BH * ((a.T + 255) / 256);
  IEF_CHECK(items < (1LL << 31), "attn_long: too many work items");
  const int grid = items < num_sms ? int(items) : num_sms;
  attn_long_kernel<DH, DHP><<<grid, kThreads, Cfg::kSmemBytes, stream>>>(tq, tk, tv, a.out, a.ldo, a.T, a.H, int(items),
                                                                        a.fp16, a.row_out);
  count_launches(1);
  IEF_CUDA(cudaGetLastError());
  return IEFVAD_OK;
}

}  // namespace

bool attn_long_supported(const AttnTcArgs& a) {
  return a.T > 256 && !a.attn_mask && !a.key_pad && !a.items;
}

int attn_long(const AttnTcArgs& a, cudaStream_t stream) {
  static int num_sms = 0;
  if (!num_sms) {
    int dev = 0;
    IEF_CUDA(cudaGetDevice(&dev));
    IEF_CUDA(cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, dev));
  }
#define IEF_ATTN_LONG(DH_, DHP_) \
  if (a.dh == DH_ && a.dhp == DHP_) return launch_attn_long<DH_, DHP_>(a, num_sms, stream);
  IEF_ATTN_LONG(96, 128)
  IEF_ATTN_LONG(64, 64)
  IEF_ATTN_LONG(128, 128)
  IEF_ATTN_LONG(32, 64)
#undef IEF_ATTN_LONG
  set_error("attn_long: unsupported head dim %d (padded %d); supported: 32, 64, 96, 128", a.dh, a.dhp);
  return IEFVAD_ERR_INVALID;
}

}  // namespace iefvad
