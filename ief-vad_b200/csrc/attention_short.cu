// Self-attention core for SHORT sequences (T <= 256, no masks) - the shape every reference caller produces: test-time
// videos are cut into 256-row chunks (data/tools.py:100-114), training clips are pooled / padded to 256
// (data/tools.py:89-97), and nn.MultiheadAttention attends over all rows of the chunk (model/imf_vad.py:115,121).
//
// Persistent kernel, one CTA per SM, work item = one (batch element, head): both 128-row query tiles share one copy of
// K and V^T in shared memory.  The whole key range fits one MMA (N = 256), so there is no online softmax:
//   S_t = Q_t.K^T (128 x 256 fp32) lands in the 256 TMEM columns of tile t,
//   16 softmax warps (two threads per query row, 128 keys each) take the exact row max, write P = exp(S - max) as
//   packed 16-bit pairs back INTO TMEM over the S columns they have already consumed,
//   O_t = P_t.V runs with the A operand read from TMEM (tcgen05.mma [d], [a], b-desc) into free columns of the tile,
//   the same threads normalise and store their half row.
// Nothing of P ever touches shared memory; Q / K / V^T buffers are released by tcgen05.commit as soon as their last
// MMA retires, so the next item's TMA loads overlap this item's softmax.  TMEM columns of tile t (base 256 t):
//   [0, 64) P keys 0..127 | [64, 64 + DH) O | [192, 256) P keys 128..255    (all inside the dead S columns).
#include "attention.cuh"
#include "common.cuh"
#include "tensormap.cuh"

namespace iefvad {

namespace {

constexpr float kLog2e = 1.4426950408889634f;
constexpr int kSoftmaxWarps = 16;
constexpr int kThreads = (kSoftmaxWarps + 2) * 32;

template <int DH, int DHP>
struct ShortCfg {
  static constexpr int TK = 256;                                   // keys covered by one S MMA
  // q / k rows of DHP elements are cut into column chunks of CW elements: 64 (128-byte swizzle) when DHP is a multiple
  // of 64, else 32 (64-byte swizzle) - d_h = 96 then needs no padding to 128 (a quarter less q / k traffic)
  static constexpr int CW = (DHP % 64 == 0) ? 64 : 32;
  static constexpr int NCH = DHP / CW;
  static constexpr uint32_t kRowB = CW * 2;                        // bytes per chunk row
  static constexpr uint32_t kQChunk = 128 * kRowB;                 // [128 rows x CW columns], swizzled
  static constexpr uint32_t kQTile = NCH * kQChunk;
  static constexpr uint32_t kKChunk = TK * kRowB;
  static constexpr uint32_t kKBytes = NCH * kKChunk;
  static_assert(DHP % 32 == 0 && DHP >= DH, "q / k row length");
  static constexpr uint32_t kVSub = DH * 128;                      // [DH rows x 64 keys]
  static constexpr uint32_t kVBytes = (TK / 64) * kVSub;
  static constexpr uint32_t kOffK = 2 * kQTile;
  static constexpr uint32_t kOffV = kOffK + kKBytes;
  static constexpr uint32_t kOffX = kOffV + kVBytes;               // row max / row sum exchange between the two halves
  static constexpr uint32_t kXBytes = 2 * 2 * 2 * 2 * 128 * 4;     // {max, sum} x parity x tile x half x row
  static constexpr uint32_t kOffBar = kOffX + kXBytes;
  static constexpr size_t kSmemBytes = 1024 + kOffBar + 256;
  static constexpr uint32_t kColP0 = 0, kColO = 64, kColP1 = 192;
  static_assert(kColO + DH <= kColP1, "O does not fit between the two P halves");
  static_assert(DH % 32 == 0, "each thread stores DH / 2 columns in 16-column pieces");
};

template <int DH, int DHP>
__global__ void __launch_bounds__(kThreads, 1)
attn_short_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmK,
                  const __grid_constant__ CUtensorMap tmVt, bf16* __restrict__ out, int ldo, int T, int H, int n_items,
                  int fp16, const int* __restrict__ row_out, const int4* __restrict__ items) {
  using Cfg = ShortCfg<DH, DHP>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + Cfg::kOffBar);
  uint64_t* qk_full = bars + 0;
  uint64_t* qk_empty = bars + 1;
  uint64_t* v_full = bars + 2;
  uint64_t* v_empty = bars + 3;
  uint64_t* s_full = bars + 4;    // [2]
  uint64_t* s_empty = bars + 6;   // [2]
  uint64_t* p_full = bars + 8;    // [2]
  uint64_t* o_full = bars + 10;   // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 12);
  float* xch = reinterpret_cast<float*>(smem + Cfg::kOffX);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // Work item -> (first row, rows, valid rows, multiplicity of the last row as a key, tensor-map z coordinate).
  // Dense batches: item = b * H + h over [B*H, T, dhp]; ragged ("items"): item = chunk * H + h over [H, Mtot, dhp],
  // chunk c owning rows [start, start + rows) of which the last one, when mult > 0, stands for `mult` identical
  // zero-pad rows (it enters the softmax with log(mult) added to its score).
  struct Item { int row0, rows, valid, mult, z, orow0; };
  auto get_item = [&](int item) {
    Item d;
    if (items) {
      const int c = item / H;
      const int4 v = __ldg(items + c);
      d.row0 = v.x; d.rows = v.y; d.valid = v.z; d.mult = v.w; d.z = item - c * H; d.orow0 = v.x;
    } else {
      const int b = item / H;
      d.row0 = 0; d.rows = T; d.valid = T; d.mult = 0; d.z = item; d.orow0 = b * T;
    }
    return d;
  };
  // stale K / V rows of earlier items stay in shared memory when a short item loads fewer boxes: they only ever meet
  // P == 0, but must be finite - so the operand buffers start out as zeros
  for (uint32_t i = threadIdx.x * 16u; i < Cfg::kOffX; i += kThreads * 16u) *reinterpret_cast<uint4*>(smem + i) = make_uint4(0, 0, 0, 0);
  fence_proxy_async_smem();

  if (warp == kSoftmaxWarps && lane == 0) {
    tma_prefetch_desc(&tmQ);
    tma_prefetch_desc(&tmK);
    tma_prefetch_desc(&tmVt);
    mbar_init(qk_full, 1);
    mbar_init(qk_empty, 1);
    mbar_init(v_full, 1);
    mbar_init(v_empty, 1);
    for (int t = 0; t < 2; ++t) {
      mbar_init(&s_full[t], 1);
      mbar_init(&s_empty[t], 256);
      mbar_init(&p_full[t], 256);
      mbar_init(&o_full[t], 1);
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
      auto nq = [](const Item& d) { return d.rows > 128 ? 2 : 1; };                    // 128-row Q / K boxes
      auto nv = [](const Item& d) { return (d.rows + 63) >> 6; };                      // 64-key V^T boxes
      auto load_qk = [&](const Item& d) {
        mbar_arrive_expect_tx(qk_full, uint32_t(nq(d)) * (Cfg::kQTile + Cfg::kKBytes / 2));
        for (int t = 0; t < nq(d); ++t)
#pragma unroll
          for (int c = 0; c < Cfg::NCH; ++c) {
            tma_load_3d(&tmQ, qk_full, smem + t * Cfg::kQTile + c * Cfg::kQChunk, c * Cfg::CW, d.row0 + t * 128, d.z);
            tma_load_3d(&tmK, qk_full, smem + Cfg::kOffK + c * Cfg::kKChunk + t * Cfg::kQChunk, c * Cfg::CW, d.row0 + t * 128, d.z);
          }
      };
      auto prefetch = [&](const Item& nx) {
        for (int t = 0; t < nq(nx); ++t)
#pragma unroll
          for (int c = 0; c < Cfg::NCH; ++c) {
            tma_prefetch_3d(&tmQ, c * Cfg::CW, nx.row0 + t * 128, nx.z);
            tma_prefetch_3d(&tmK, c * Cfg::CW, nx.row0 + t * 128, nx.z);
          }
        for (int c = 0; c < nv(nx); ++c) tma_prefetch_3d(&tmVt, nx.row0 + c * 64, 0, nx.z);
      };
      // The S MMAs read Q and K from shared memory at three quarters of its bandwidth: a TMA load landing at the same
      // time slows them down (measured: S issue -> S visible 1.1 k cycles alone, 2.6 k beside the V load).  So V(i)
      // starts when S_a(i) has retired (it is needed after the softmax), Q / K (i+1) when all S MMAs of item i have.
      const int step = int(gridDim.x);
      if (int(blockIdx.x) < n_items) {
        load_qk(get_item(blockIdx.x));
        if (int(blockIdx.x) + step < n_items) prefetch(get_item(blockIdx.x + step));
      }
      int it = 0;
      for (int item = blockIdx.x; item < n_items; item += step, ++it) {
        const uint32_t ph = it & 1;
        const Item d = get_item(item);
        mbar_wait(&s_full[0], ph);                // S_a(i) retired
        mbar_wait(v_empty, ph ^ 1);               // P.V of item i-1 retired
        mbar_arrive_expect_tx(v_full, uint32_t(nv(d)) * Cfg::kVSub);
        for (int c = 0; c < nv(d); ++c)
          tma_load_3d(&tmVt, v_full, smem + Cfg::kOffV + c * Cfg::kVSub, d.row0 + c * 64, 0, d.z);
        if (item + step < n_items) {
          mbar_wait(qk_empty, ph);                // every S MMA of item i retired: Q / K buffers are free
          load_qk(get_item(item + step));
          if (item + 2 * step < n_items) prefetch(get_item(item + 2 * step));
        }
      }
    }
  } else if (warp == kSoftmaxWarps + 1) {
    // ===================== MMA issuer =====================
    if (lane == 0) {
      const uint32_t idesc_s = fp16 ? make_idesc_f16(128, Cfg::TK) : make_idesc_bf16(128, Cfg::TK);
      const uint32_t idesc_o = fp16 ? make_idesc_f16(128, DH) : make_idesc_bf16(128, DH);
      const uint32_t sq = smem_u32(smem), sk = smem_u32(smem + Cfg::kOffK), sv = smem_u32(smem + Cfg::kOffV);
      auto issue_s = [&](int t) {
        const uint32_t d = tmem_base + uint32_t(t * 256);
#pragma unroll
        for (int kk = 0; kk < DH / 16; ++kk) {   // only the DH real columns of DHP-padded rows
          constexpr int KPC = Cfg::CW / 16;      // 16-element K steps per column chunk
          const int c = kk / KPC, ks = kk % KPC;
          const uint32_t qa = sq + t * Cfg::kQTile + c * Cfg::kQChunk, ka = sk + c * Cfg::kKChunk;
          const uint64_t dq = Cfg::CW == 64 ? make_smem_desc_sw128(qa) : make_smem_desc_sw64(qa);
          const uint64_t dk = Cfg::CW == 64 ? make_smem_desc_sw128(ka) : make_smem_desc_sw64(ka);
          umma_bf16(d, dq + uint64_t(2 * ks), dk + uint64_t(2 * ks), idesc_s, kk != 0 ? 1u : 0u);
        }
        tc_commit(&s_full[t]);
      };
      auto issue_pv = [&](int t) {
        const uint32_t tb = tmem_base + uint32_t(t * 256);
#pragma unroll
        for (int kk = 0; kk < Cfg::TK / 16; ++kk) {
          const int c = kk >> 2, k4 = kk & 3;
          const uint32_t a = tb + (kk < 8 ? Cfg::kColP0 + uint32_t(kk * 8) : Cfg::kColP1 + uint32_t((kk - 8) * 8));
          umma_f16_ts(tb + Cfg::kColO, a, make_smem_desc_sw128(sv + c * Cfg::kVSub) + uint64_t(2 * k4), idesc_o,
                      kk != 0 ? 1u : 0u);
        }
        tc_commit(&o_full[t]);
      };
      // The two query tiles run half an item apart: S_a(i), P.V_b(i-1), S_b(i), P.V_a(i).  While tile a's softmax
      // owns the SFU, the tensor pipe serves tile b, and vice versa (in lock-step both would wait at the same time).
      // Items of <= 128 rows have no tile b; tile b's barriers count only the items that use it.
      int it = 0;
      uint32_t nb_s = 0, nb_pv = 0;           // S_b / P.V_b issued so far
      bool pend_b = false;                    // the previous item still owes its P.V_b
      for (int item = blockIdx.x; item < n_items; item += gridDim.x, ++it) {
        const uint32_t ph = it & 1;
        const bool act_b = get_item(item).rows > 128;
        mbar_wait(qk_full, ph);
        mbar_wait(&s_empty[0], ph ^ 1);         // tile 0's columns (P and O of the previous item) have been read out
        tc_fence_after();
        issue_s(0);
        if (pend_b) {
          mbar_wait(&p_full[1], nb_pv & 1);
          tc_fence_after();
          issue_pv(1);                          // previous item, still on the previous V
          tc_commit(v_empty);
          ++nb_pv;
        }
        if (act_b) {
          mbar_wait(&s_empty[1], (nb_s & 1) ^ 1);
          tc_fence_after();
          issue_s(1);
          ++nb_s;
        }
        tc_commit(qk_empty);                    // Q and K may be overwritten once the S MMAs have retired
        mbar_wait(v_full, ph);
        mbar_wait(&p_full[0], ph);
        tc_fence_after();
        issue_pv(0);
        if (!act_b) tc_commit(v_empty);
        pend_b = act_b;
      }
      if (pend_b) {
        mbar_wait(&p_full[1], nb_pv & 1);
        tc_fence_after();
        issue_pv(1);
      }
    }
  } else {
    // ===================== softmax / normalise / store (warps 0..15) =====================
    const int t = warp >> 3;                        // query tile
    const int hf = (warp >> 2) & 1;                 // key half: keys [128 hf, 128 hf + 128)
    const int quarter = warp & 3;                   // TMEM lane quarter this warp may access
    const int r = quarter * 32 + lane;              // query row inside the tile == TMEM lane
    const int tq = t * 128 + r;
    const uint32_t tbase = tmem_base + uint32_t(t * 256) + (uint32_t(quarter * 32) << 16);
    const uint32_t ts = tbase + uint32_t(hf * 128);
    const uint32_t tp = tbase + (hf ? Cfg::kColP1 : Cfg::kColP0);
    const int key0 = hf * 128;
    // exchange slots: xch[((kind * 2 + parity) * 2 + tile) * 2 + half][row]
    auto slot = [&](int kind, uint32_t ph, int half) { return xch + ((((kind * 2 + int(ph)) * 2 + t) * 2 + half) << 7) + r; };

    uint32_t n_mine = 0;                            // items this tile has processed (tile 1 skips the short ones)
    for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
      const Item d = get_item(item);
      if (t == 1 && d.rows <= 128) continue;
      const uint32_t ph = n_mine & 1;
      ++n_mine;
      const int h = items ? d.z : item % H;
      const int Tk = d.rows;                        // keys of this item
      const int padkey = d.mult > 0 ? d.valid : -1; // the key that stands for `mult` identical zero-pad rows
      const float lnm = d.mult > 0 ? __logf(float(d.mult)) : 0.f;
      const int plain_end = padkey >= 0 ? padkey : Tk;   // 32-key chunks that end at or before this key need no masking
      mbar_wait(&s_full[t], ph);
      tc_fence_after();
      // ---- pass 1: row max over this thread's 128 keys.  Only the 32-key chunk that holds the last key needs per-key
      // masking (keys >= Tk are not there; the last key may carry a multiplicity); chunks before it are plain, chunks
      // after it are skipped.  All of this is warp-uniform.
      float mx = -INFINITY;
      auto chunk_max = [&](const float (&v)[32], int k_lo) {
        if (k_lo + 32 <= plain_end) {
#pragma unroll
          for (int i = 0; i < 32; ++i) mx = fmaxf(mx, v[i]);
        } else if (k_lo < Tk) {
#pragma unroll
          for (int i = 0; i < 32; ++i)
            if (k_lo + i < Tk) mx = fmaxf(mx, k_lo + i == padkey ? v[i] + lnm : v[i]);
        }
      };
#pragma unroll
      for (int c2 = 0; c2 < 2; ++c2) {
        if (key0 + c2 * 64 >= Tk) break;
        float v0[32], v1[32];
        tmem_ld32(ts + uint32_t(c2 * 64), v0);
        tmem_ld32(ts + uint32_t(c2 * 64 + 32), v1);
        tmem_ld_wait();
        chunk_max(v0, key0 + c2 * 64);
        chunk_max(v1, key0 + c2 * 64 + 32);
      }
      *slot(0, ph, hf) = mx;
      named_bar_sync(1 + t, 256);
      mx = fmaxf(mx, *slot(0, ph, hf ^ 1));          // key 0 is always valid, so the row max is finite
      const float mscaled = mx * kLog2e;
      // ---- pass 2: P = exp(S - max) -> packed 16-bit pairs over the S columns already consumed.  Half 0 walks its
      // chunks upwards and packs downwards into [0, 64); half 1 walks downwards and packs into [192, 256).
      float lsum = 0.f;
#pragma unroll
      for (int ci = 0; ci < 4; ++ci) {
        const int c = hf ? 3 - ci : ci;
        const int k_lo = key0 + c * 32;
        uint32_t pk[16];
        if (k_lo >= Tk) {                            // no key here: P = 0 (the MMA still reads these columns)
#pragma unroll
          for (int i = 0; i < 16; ++i) pk[i] = 0u;
        } else {
          float v[32];
          tmem_ld32(ts + uint32_t(c * 32), v);
          tmem_ld_wait();
          if (k_lo + 32 <= plain_end) {
#pragma unroll
            for (int i = 0; i < 32; i += 2) {
              const float p0 = fast_exp2(fmaf(v[i], kLog2e, -mscaled));
              const float p1 = fast_exp2(fmaf(v[i + 1], kLog2e, -mscaled));
              lsum += p0 + p1;
              pk[i >> 1] = pack_16x2(p0, p1, fp16);
            }
          } else {                                   // the chunk with the last key
#pragma unroll
            for (int i = 0; i < 32; i += 2) {
              const float x0 = (k_lo + i == padkey) ? v[i] + lnm : v[i];
              const float x1 = (k_lo + i + 1 == padkey) ? v[i + 1] + lnm : v[i + 1];
              float p0 = fast_exp2(fmaf(x0, kLog2e, -mscaled));
              float p1 = fast_exp2(fmaf(x1, kLog2e, -mscaled));
              if (k_lo + i >= Tk) p0 = 0.f;
              if (k_lo + i + 1 >= Tk) p1 = 0.f;
              lsum += p0 + p1;
              pk[i >> 1] = pack_16x2(p0, p1, fp16);
            }
          }
        }
        tmem_st16(tp + uint32_t(c * 16), pk);
      }
      *slot(1, ph, hf) = lsum;
      tmem_st_wait();
      tc_fence_before();
      mbar_arrive(&p_full[t]);
      // ---- O = P.V: this thread normalises and stores columns [hf DH/2, hf DH/2 + DH/2) of its row
      mbar_wait(&o_full[t], ph);
      tc_fence_after();
      named_bar_sync(1 + t, 256);
      const float inv = 1.f / (lsum + *slot(1, ph, hf ^ 1));
      float o[DH / 2];
#pragma unroll
      for (int c = 0; c < DH / 32; ++c) tmem_ld16(tbase + Cfg::kColO + uint32_t(hf * (DH / 2) + c * 16), o + c * 16);
      tmem_ld_wait();
      tc_fence_before();
      mbar_arrive(&s_empty[t]);
      long long ro = (long long)d.orow0 + tq;
      if (tq < Tk && row_out) ro = __ldg(row_out + ro);
      if (tq < Tk && ro >= 0) {
        bf16* dst = out + ro * ldo + h * DH + hf * (DH / 2);
#pragma unroll
        for (int d = 0; d < DH / 2; d += 8) *reinterpret_cast<uint4*>(dst + d) = pack_16x8(o + d, fp16, inv);
      }
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
int launch_attn_short(const AttnTcArgs& a, int num_sms, cudaStream_t stream) {
  using Cfg = ShortCfg<DH, DHP>;
  static bool attr_set = false;
  if (!attr_set) {
    IEF_CUDA(cudaFuncSetAttribute(attn_short_kernel<DH, DHP>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  static_cast<int>(Cfg::kSmemBytes)));
    attr_set = true;
  }
  // dense: [B*H, T, dhp]; ragged items: [H, T = all packed rows, dhp] with `n_chunks` row ranges (AttnTcArgs.items)
  const uint64_t BH = a.items ? uint64_t(a.H) : uint64_t(a.B) * a.H;
  CUtensorMap tq, tk, tv;
  const int qk_sw = Cfg::CW == 64 ? TM_SWIZZLE_128B : TM_SWIZZLE_64B;
  IEF_TRY(make_tmap_3d(&tq, a.q, DHP, a.T, BH, uint64_t(DHP) * 2, uint64_t(a.T) * DHP * 2, Cfg::CW, 128, 1, qk_sw));
  IEF_TRY(make_tmap_3d(&tk, a.k, DHP, a.T, BH, uint64_t(DHP) * 2, uint64_t(a.T) * DHP * 2, Cfg::CW, 128, 1, qk_sw));
  IEF_TRY(make_tmap_3d(&tv, a.vt, a.T, DH, BH, uint64_t(a.Tpad) * 2, uint64_t(DH) * a.Tpad * 2, 64, DH, 1));
  const int n_items = a.items ? a.n_chunks * a.H : int(BH);
  const int grid = n_items < num_sms ? n_items : num_sms;
  attn_short_kernel<DH, DHP><<<grid, kThreads, Cfg::kSmemBytes, stream>>>(tq, tk, tv, a.out, a.ldo, a.T, a.H, n_items,
                                                                         a.fp16, a.row_out, reinterpret_cast<const int4*>(a.items));
  count_launches(1);
  IEF_CUDA(cudaGetLastError());
  return IEFVAD_OK;
}

}  // namespace

bool attn_short_supported(const AttnTcArgs& a) {
  if (a.items) return !a.attn_mask && !a.key_pad;      // ragged items exist only here (every item <= 256 rows)
  return a.T <= 256 && !a.attn_mask && !a.key_pad && uint64_t(a.B) * a.H < (1ull << 31);
}

int attn_short(const AttnTcArgs& a, cudaStream_t stream) {
  static int num_sms = 0;
  if (!num_sms) {
    int dev = 0;
    IEF_CUDA(cudaGetDevice(&dev));
    IEF_CUDA(cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, dev));
  }
#define IEF_ATTN_SHORT(DH_, DHP_) \
  if (a.dh == DH_ && a.dhp == DHP_) return launch_attn_short<DH_, DHP_>(a, num_sms, stream);
  IEF_ATTN_SHORT(96, 96)      // unpadded q / k rows (32-column chunks, 64-byte swizzle)
  IEF_ATTN_SHORT(96, 128)
  IEF_ATTN_SHORT(64, 64)
  IEF_ATTN_SHORT(128, 128)
  IEF_ATTN_SHORT(32, 64)
  IEF_ATTN_SHORT(32, 32)
#undef IEF_ATTN_SHORT
  set_error("attn_short: unsupported head dim %d (padded %d); supported: 32, 64, 96, 128", a.dh, a.dhp);
  return IEFVAD_ERR_INVALID;
}

}  // namespace iefvad
