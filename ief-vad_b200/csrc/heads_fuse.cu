// mu / logvar heads of BOTH modalities + the uncertainty-weighted fusion as ONE tcgen05 kernel (evaluation path):
//     mu_m = x_m . Wmu_m^T + bmu_m,  logvar_m = x_m . Wlv_m^T + blv_m            (model/imf_vad.py:125-128)
//     r_m = factor * exp(-logvar_m);  w_m = r_m / (r_i + r_e + eps);  fused = w_i mu_i + w_e mu_e       (:130-144)
// The two-launch heads GEMMs write 12 KB per row of fp32 mu / logvar that only the fusion kernel reads back (27 KB per row of
// HBM traffic in all); here a CTA pair computes, for 256 rows x 128 features, the image modality's [mu | logvar] into one
// half of tensor memory (N = 256 accumulator) and the event modality's into the other half, and the epilogue fuses them from
// TMEM: 3 KB of x in, the 16-bit (hi, lo) pair of `fused` out - 4.5 KB per row.
// Same arithmetic, instruction for instruction, as gemm_tc (fp16 operands, fp32 accumulation in k order, + bias) followed
// by fuse_kernel (the same fuse_one): the pair is bit-identical to the three-launch form.
// TMEM is full (2 x 256 columns), so the epilogue of a tile does not overlap the MMAs of the next one - but the operand ring
// (6 stages) refills meanwhile, and the kernel still moves a sixth of the bytes.  Sixteen epilogue warps (four per scheduler,
// one 32-feature chunk each, 8 features at a time to stay inside 96 registers) keep that exposed epilogue short: it is bound
// by the CUDA cores (expf and IEEE division per element).
#include <cstring>

#include "elementwise.cuh"
#include "heads_fuse.cuh"
#include "tensormap.cuh"

namespace iefvad {

namespace {

constexpr int D = kHeadsFuseDim;
constexpr int BM = 128;
constexpr int BN = 256;                          // [mu (128 features) | logvar (128 features)] of one modality
constexpr int BF = 128;                          // features per tile
constexpr int BK = 64;
constexpr int CW = 32;
constexpr int kFB = D / BF;                      // feature blocks
constexpr int kEpiWarps = 16;
constexpr int kThreads = 64 + 32 * kEpiWarps;
constexpr int kMaxStages = 6;
constexpr uint32_t kABytes = BM * BK * 2;
constexpr uint32_t kBBytes = (BN / 2) * BK * 2;
constexpr uint32_t kStageBytes = kABytes + kBBytes;
constexpr uint32_t kBox16 = 32 * CW * 2;
constexpr uint32_t kWarpBytes = kBox16;          // one box per warp: the hi part leaves, then the lo part
constexpr uint32_t kBarBytes = 256;
constexpr uint32_t kSmemLimit = 232448;
constexpr int kKB = D / BK;                      // k-blocks per modality

struct HfParams {
  const float* b_i;
  const float* b_e;
  float factor, eps;
  int num_tiles;
  int stages;
};

__device__ __forceinline__ uint32_t sw64(int row, int g) { return uint32_t(row) * 64u + (uint32_t(g ^ ((row >> 1) & 3)) << 4); }

__global__ void __launch_bounds__(kThreads, 1)
heads_fuse_kernel(const __grid_constant__ CUtensorMap txi, const __grid_constant__ CUtensorMap txe,
                  const __grid_constant__ CUtensorMap twi, const __grid_constant__ CUtensorMap twe,
                  const __grid_constant__ CUtensorMap toh, const __grid_constant__ CUtensorMap tol, const HfParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int STAGES = p.stages;
  uint8_t* epi_base = smem + size_t(STAGES) * kStageBytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(epi_base + kEpiWarps * kWarpBytes);
  uint64_t* full = bars;
  uint64_t* empty = full + kMaxStages;
  uint64_t* tfull = empty + kMaxStages;
  uint64_t* tempty = tfull + 1;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 1);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const int tile0 = blockIdx.x >> 1, tile_step = gridDim.x >> 1;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&txi);
    tma_prefetch_desc(&txe);
    tma_prefetch_desc(&twi);
    tma_prefetch_desc(&twe);
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], 1);
    }
    mbar_init(tfull, 1);
    mbar_init(tempty, kEpiWarps * 2);
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
      int s = 0;
      uint32_t ph = 0;
      for (int tile = tile0; tile < p.num_tiles; tile += tile_step) {
        const int m_blk = (tile / kFB) * 2 + int(rank), fb = tile % kFB;
        const int wrow = (rank ? D : 0) + fb * BF;           // rank 0 loads the mu rows of the tile, rank 1 the logvar rows
        for (int kb = 0; kb < 2 * kKB; ++kb) {
          const bool ev = kb >= kKB;
          const int kk = ev ? kb - kKB : kb;
          mbar_wait(&empty[s], ph ^ 1);
          uint8_t* sa = smem + size_t(s) * kStageBytes;
          const uint32_t lead_full = mapa_shared(smem_u32(&full[s]), 0);
          if (rank == 0) mbar_arrive_expect_tx(&full[s], 2 * kStageBytes);
          tma_load_2d_cg2(ev ? &txe : &txi, lead_full, sa, kk * BK, m_blk * BM);
          tma_load_2d_cg2(ev ? &twe : &twi, lead_full, sa + kABytes, kk * BK, wrow);
          if (++s == STAGES) { s = 0; ph ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (leader CTA) =====================
    if (lane == 0 && rank == 0) {
      constexpr uint32_t idesc = make_idesc_f16(2 * BM, BN);
      int s = 0;
      uint32_t ph = 0;
      int it = 0;
      for (int tile = tile0; tile < p.num_tiles; tile += tile_step, ++it) {
        mbar_wait(tempty, uint32_t(it & 1) ^ 1);
        tc_fence_after();
        for (int kb = 0; kb < 2 * kKB; ++kb) {
          const bool ev = kb >= kKB;
          const int kk = ev ? kb - kKB : kb;
          const uint32_t d_tmem = tmem_base + (ev ? uint32_t(BN) : 0u);
          mbar_wait(&full[s], ph);
          tc_fence_after();
          const uint32_t sa = smem_u32(smem + size_t(s) * kStageBytes);
          const uint64_t da = make_smem_desc_sw128(sa);
          const uint64_t db = make_smem_desc_sw128(sa + kABytes);
#pragma unroll
          for (int k4 = 0; k4 < BK / 16; ++k4)
            umma_bf16_cg2(d_tmem, da + uint64_t(2 * k4), db + uint64_t(2 * k4), idesc, (kk | k4) != 0 ? 1u : 0u);
          tc_commit_cg2(&empty[s], 3);
          if (++s == STAGES) { s = 0; ph ^= 1; }
        }
        tc_commit_cg2(tfull, 3);
      }
    }
  } else {
    // ===================== epilogue: 16 warps, thread == row =====================
    const int ew = warp - 2;
    const int quarter = warp & 3;
    const int c32 = ew >> 2;               // this warp's 32-feature chunk of the tile
    uint8_t* Bx = epi_base + size_t(ew) * kWarpBytes;
    if (lane == 0) {
      tma_prefetch_desc(&toh);
      tma_prefetch_desc(&tol);
    }
    const uint32_t t0 = tmem_base + (uint32_t(quarter * 32) << 16);
    int it = 0;
    for (int tile = tile0; tile < p.num_tiles; tile += tile_step, ++it) {
      const int m_blk = (tile / kFB) * 2 + int(rank), fb = tile % kFB;
      const int row0 = m_blk * BM + quarter * 32;
      mbar_wait(tfull, uint32_t(it & 1));
      tc_fence_after();
      uint32_t lo_keep[16];                                  // the remainder halves wait in registers for the box
      if (lane == 0) bulk_wait_read<0>();                    // the previous tile's lo store has read the box
      __syncwarp();
#pragma unroll
      for (int step = 0; step < 4; ++step) {
        const int fo = c32 * CW + step * 8;                  // feature offset inside the tile
        float mi[8], li[8], me[8], le[8];
        tmem_ld8(t0 + uint32_t(fo), mi);
        tmem_ld8(t0 + uint32_t(BF + fo), li);
        tmem_ld8(t0 + uint32_t(BN + fo), me);
        tmem_ld8(t0 + uint32_t(BN + BF + fo), le);
        const int f0 = fb * BF + fo;
        float4 bmi[2], bli[2], bme[2], ble[2];
#pragma unroll
        for (int g = 0; g < 2; ++g) {
          bmi[g] = __ldg(reinterpret_cast<const float4*>(p.b_i + f0) + g);
          bli[g] = __ldg(reinterpret_cast<const float4*>(p.b_i + D + f0) + g);
          bme[g] = __ldg(reinterpret_cast<const float4*>(p.b_e + f0) + g);
          ble[g] = __ldg(reinterpret_cast<const float4*>(p.b_e + D + f0) + g);
        }
        tmem_ld_wait();
        if (step == 3) {                                     // both accumulators fully read: the next tile's MMAs may start
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive_cluster(mapa_shared(smem_u32(tempty), 0));
        }
        float f[8];
#pragma unroll
        for (int g = 0; g < 2; ++g) {
          const float b0[4] = {bmi[g].x, bmi[g].y, bmi[g].z, bmi[g].w}, b1[4] = {bli[g].x, bli[g].y, bli[g].z, bli[g].w};
          const float b2[4] = {bme[g].x, bme[g].y, bme[g].z, bme[g].w}, b3[4] = {ble[g].x, ble[g].y, ble[g].z, ble[g].w};
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const int i = g * 4 + e;
            float wi, we;
            f[i] = fuse_one(__fadd_rn(mi[i], b0[e]), __fadd_rn(me[i], b2[e]), __fadd_rn(li[i], b1[e]),
                            __fadd_rn(le[i], b3[e]), p.factor, p.eps, wi, we);
          }
        }
        uint32_t hi[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) split_16x2(f[2 * q], f[2 * q + 1], 1, hi[q], lo_keep[step * 4 + q]);
        *reinterpret_cast<uint4*>(Bx + sw64(lane, step)) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
      }
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) {
        tma_store_2d(&toh, Bx, fb * BF + c32 * CW, row0);
        bulk_commit();
        bulk_wait_read<0>();
      }
      __syncwarp();
#pragma unroll
      for (int g = 0; g < 4; ++g)
        *reinterpret_cast<uint4*>(Bx + sw64(lane, g)) = make_uint4(lo_keep[g * 4], lo_keep[g * 4 + 1], lo_keep[g * 4 + 2], lo_keep[g * 4 + 3]);
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) {
        tma_store_2d(&tol, Bx, fb * BF + c32 * CW, row0);
        bulk_commit();
      }
    }
    if (lane == 0) bulk_wait_all<0>();
  }

  tc_fence_before();
  cluster_sync_all();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc_cg2(tmem_base, 512);
  }
}

}  // namespace

int heads_fuse(const HeadsFuseArgs& a, int num_sms, cudaStream_t stream) {
  IEF_CHECK(a.x_i && a.x_e && a.w_i16 && a.w_e16 && a.b_i && a.b_e && a.out_hi && a.out_lo, "heads_fuse: null argument");
  IEF_CHECK(a.M > 0 && a.M < (1LL << 31) - 256, "heads_fuse: bad row count %lld", a.M);
  HfParams p;
  memset(&p, 0, sizeof(p));
  p.b_i = a.b_i; p.b_e = a.b_e; p.factor = a.factor; p.eps = a.eps;
  const int num_mp = int((a.M + 255) / 256);
  p.num_tiles = num_mp * kFB;
  const uint32_t fixed = 1024 + kEpiWarps * kWarpBytes + kBarBytes;
  p.stages = int((kSmemLimit - fixed) / kStageBytes);
  if (p.stages > kMaxStages) p.stages = kMaxStages;
  const size_t smem_bytes = fixed + size_t(p.stages) * kStageBytes;

  CUtensorMap txi, txe, twi, twe, toh, tol;
  IEF_TRY(make_tmap_2d(&txi, a.x_i, D, uint64_t(a.M), uint64_t(D) * 2, BK, BM));
  IEF_TRY(make_tmap_2d(&txe, a.x_e, D, uint64_t(a.M), uint64_t(D) * 2, BK, BM));
  IEF_TRY(make_tmap_2d(&twi, a.w_i16, D, 2 * D, uint64_t(D) * 2, BK, BN / 2));
  IEF_TRY(make_tmap_2d(&twe, a.w_e16, D, 2 * D, uint64_t(D) * 2, BK, BN / 2));
  IEF_TRY(make_tmap_2d(&toh, a.out_hi, D, uint64_t(a.M), uint64_t(D) * 2, CW, 32, TM_BF16, TM_SWIZZLE_64B));
  IEF_TRY(make_tmap_2d(&tol, a.out_lo, D, uint64_t(a.M), uint64_t(D) * 2, CW, 32, TM_BF16, TM_SWIZZLE_64B));

  static bool attr_set = false;
  if (!attr_set) {
    IEF_CUDA(cudaFuncSetAttribute(heads_fuse_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(kSmemLimit)));
    attr_set = true;
  }
  const int pairs = num_sms / 2;
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3(unsigned((p.num_tiles < pairs ? p.num_tiles : pairs) * 2));
  cfg.blockDim = dim3(kThreads);
  cfg.dynamicSmemBytes = smem_bytes;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  IEF_CUDA(cudaLaunchKernelEx(&cfg, heads_fuse_kernel, txi, txe, twi, twe, toh, tol, p));
  count_launches(1);
  return IEFVAD_OK;
}

}  // namespace iefvad
