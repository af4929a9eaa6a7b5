// Shared device helpers for the IEF-VAD sm_100a kernels: error plumbing, 16-bit (fp16 / bf16) hi/lo splitting,
// and thin inline-PTX wrappers for mbarrier, TMA (cp.async.bulk.tensor) and tcgen05 / TMEM.
#pragma once

#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace iefvad {

// ----------------------------------------------------------------------------------------------
// host-side error plumbing (C ABI returns int codes; message kept per thread)
// ----------------------------------------------------------------------------------------------
enum : int { IEFVAD_OK = 0, IEFVAD_ERR_INVALID = 1, IEFVAD_ERR_CUDA = 2, IEFVAD_ERR_STATE = 3 };

void set_error(const char* fmt, ...);
void keep_async_pool();              // once per device: the stream-ordered allocator keeps freed blocks (no OS round trips)
void count_launches(int n);          // kernels launched by this library (bench.py's gpu_launches)
unsigned long long launch_count();
int cuda_fail(cudaError_t e, const char* what, const char* file, int line);
int device_sms(int* out);            // SM count of the current device

#define IEF_CUDA(call)                                                                    \
  do {                                                                                    \
    cudaError_t _e = (call);                                                              \
    if (_e != cudaSuccess) return ::iefvad::cuda_fail(_e, #call, __FILE__, __LINE__);     \
  } while (0)

#define IEF_CHECK(cond, ...)                                                              \
  do {                                                                                    \
    if (!(cond)) {                                                                        \
      ::iefvad::set_error(__VA_ARGS__);                                                   \
      return ::iefvad::IEFVAD_ERR_INVALID;                                                \
    }                                                                                     \
  } while (0)

#define IEF_TRY(expr)                                                                     \
  do {                                                                                    \
    int _rc = (expr);                                                                     \
    if (_rc != 0) return _rc;                                                             \
  } while (0)

// ----------------------------------------------------------------------------------------------
// small device utilities
// ----------------------------------------------------------------------------------------------
typedef __nv_bfloat16 bf16;

__device__ __forceinline__ uint32_t pack_bf16x2(float a, float b) {
  __nv_bfloat162 v = __floats2bfloat162_rn(a, b);  // .x = a (low 16 bits), .y = b
  return *reinterpret_cast<uint32_t*>(&v);
}

// two floats -> packed 16-bit pair in either operand format (fp16 when `f16` != 0, else bf16); .x = a in the low half
__device__ __forceinline__ uint32_t pack_16x2(float a, float b, int f16) {
  if (f16) {
    const __half2 h = __floats2half2_rn(a, b);
    return *reinterpret_cast<const uint32_t*>(&h);
  }
  return pack_bf16x2(a, b);
}

// hi = bf16(x), lo = bf16(x - hi): x ~= hi + lo to ~16 mantissa bits
__device__ __forceinline__ void split_bf16(float x, bf16& hi, bf16& lo) {
  hi = __float2bfloat16_rn(x);
  lo = __float2bfloat16_rn(x - __bfloat162float(hi));
}

// The 16-bit operand pair of two floats, packed like pack_16x2: hi = round16(x), lo = round16(x - float(hi)).
// hi + lo carries x to ~16 mantissa bits in bf16 and ~22 in fp16 (E5M10) - the fp16 plans' residual stream.
__device__ __forceinline__ void split_16x2(float a, float b, int f16, uint32_t& hi, uint32_t& lo) {
  if (f16) {
    const __half2 h = __floats2half2_rn(a, b);
    const float2 hf = __half22float2(h);
    const __half2 l = __floats2half2_rn(a - hf.x, b - hf.y);
    hi = *reinterpret_cast<const uint32_t*>(&h);
    lo = *reinterpret_cast<const uint32_t*>(&l);
  } else {
    const __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
    const float2 hf = __bfloat1622float2(h);
    hi = *reinterpret_cast<const uint32_t*>(&h);
    lo = pack_bf16x2(a - hf.x, b - hf.y);
  }
}

// eight floats, each times `s`, -> one 16-byte vector of 16-bit values in element order
__device__ __forceinline__ uint4 pack_16x8(const float* v, int f16, float s = 1.f) {
  return make_uint4(pack_16x2(v[0] * s, v[1] * s, f16), pack_16x2(v[2] * s, v[3] * s, f16),
                    pack_16x2(v[4] * s, v[5] * s, f16), pack_16x2(v[6] * s, v[7] * s, f16));
}

// eight fp16 values -> floats; with `lo`, eight split_16x2 fp16 pairs -> float(hi) + float(lo)
__device__ __forceinline__ void unpack_f16x8(const uint4& hi, const uint4* lo, float* r) {
  const __half2* h = reinterpret_cast<const __half2*>(&hi);
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const float2 f = __half22float2(h[q]);
    r[2 * q] = f.x; r[2 * q + 1] = f.y;
  }
  if (lo) {
    const __half2* l = reinterpret_cast<const __half2*>(lo);
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const float2 f = __half22float2(l[q]);
      r[2 * q] += f.x; r[2 * q + 1] += f.y;
    }
  }
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ bool elect_one() {
  uint32_t pred = 0;
  asm volatile(
      "{\n\t.reg .pred P;\n\t"
      "elect.sync _|P, 0xffffffff;\n\t"
      "selp.b32 %0, 1, 0, P;\n\t}"
      : "=r"(pred));
  return pred != 0;
}

// ----------------------------------------------------------------------------------------------
// mbarrier
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred P;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P, [%1], %2;\n\t"
      "selp.b32 %0, 1, 0, P;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// Bounded wait: a protocol bug traps (-> CUDA error on the host) instead of hanging the GPU box.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if (++spins > (1u << 26)) __trap();
  }
}

// ----------------------------------------------------------------------------------------------
// TMA
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
__device__ __forceinline__ void tma_load_2d(const CUtensorMap* m, uint64_t* bar, void* smem_dst, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      :
      : "r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d(const CUtensorMap* m, uint64_t* bar, void* smem_dst, int c0, int c1,
                                            int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      :
      : "r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}

// L2 prefetch of a tensor box: the data starts moving from HBM long before a shared-memory buffer is free to take it
__device__ __forceinline__ void tma_prefetch_3d(const CUtensorMap* m, int c0, int c1, int c2) {
  asm volatile("cp.async.bulk.prefetch.tensor.3d.L2.global.tile [%0, {%1, %2, %3}];"
               :
               : "l"(reinterpret_cast<uint64_t>(m)), "r"(c0), "r"(c1), "r"(c2)
               : "memory");
}

// smem -> global tensor store (bulk async group); the box is clipped at the tensor bounds
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* m, const void* smem_src, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
               :
               : "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(smem_src)), "r"(c0), "r"(c1)
               : "memory");
}
__device__ __forceinline__ void tma_store_3d(const CUtensorMap* m, const void* smem_src, int c0, int c1, int c2) {
  asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];"
               :
               : "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(smem_src)), "r"(c0), "r"(c1), "r"(c2)
               : "memory");
}
__device__ __forceinline__ void tma_store_4d(const CUtensorMap* m, const void* smem_src, int c0, int c1, int c2,
                                             int c3) {
  asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];"
               :
               : "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(smem_src)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
               : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
// wait until at most N of this thread's bulk groups still have to READ their smem source
template <int N>
__device__ __forceinline__ void bulk_wait_read() {
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
// wait until at most N bulk groups are still in flight at all (writes performed)
template <int N>
__device__ __forceinline__ void bulk_wait_all() {
  asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory");
}
// named barrier among `nthreads` threads of the CTA (id 1..15; 0 is __syncthreads)
__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// ----------------------------------------------------------------------------------------------
// tcgen05 / TMEM
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_dst, uint32_t ncols) {  // one full warp
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)),
               "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {  // same warp as alloc
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// tcgen05.commit: mbarrier arrives once all previously issued tcgen05.mma of this thread complete
__device__ __forceinline__ void tc_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}

// D[tmem] (+)= A[smem] * B[smem]^T, bf16 x bf16 -> fp32, single CTA
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      :
      : "r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}

// Instruction descriptor, kind::f16, A/B = bf16 K-major, D = fp32 (bit layout: cute::UMMA::InstrDescriptor)
__host__ __device__ constexpr uint32_t make_idesc_bf16(int M, int N) {
  return (1u << 4)                          // c_format  = F32
         | (1u << 7)                        // a_format  = BF16
         | (1u << 10)                       // b_format  = BF16
         | (0u << 15) | (0u << 16)          // a_major = b_major = K
         | (static_cast<uint32_t>(N >> 3) << 17) | (static_cast<uint32_t>(M >> 4) << 24);
}

// Same with fp16 (E5M10) operands: a_format = b_format = 0; the tensor pipe runs kind::f16 at the same rate
__host__ __device__ constexpr uint32_t make_idesc_f16(int M, int N) {
  return (1u << 4) | (static_cast<uint32_t>(N >> 3) << 17) | (static_cast<uint32_t>(M >> 4) << 24);
}

// Shared-memory matrix descriptor for a K-major tile stored as rows of 128 bytes (64 bf16) with the
// 128-byte swizzle TMA writes (CU_TENSOR_MAP_SWIZZLE_128B): 8-row groups are 1024 B apart (SBO),
// LBO is unused for swizzled K-major layouts, version = 1 (Blackwell), layout_type = 2 (SWIZZLE_128B).
__device__ __forceinline__ uint64_t make_smem_desc_sw128(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3FFFFu) >> 4);        // start address  [0,14)
  d |= static_cast<uint64_t>(1) << 16;                            // LBO (ignored)  [16,30)
  d |= static_cast<uint64_t>(1024 >> 4) << 32;                    // SBO = 1024 B   [32,46)
  d |= static_cast<uint64_t>(1) << 46;                            // version = 1    [46,48)
  d |= static_cast<uint64_t>(2) << 61;                            // SWIZZLE_128B   [61,64)
  return d;
}

// K-major tile stored as rows of 64 bytes (32 16-bit elements) with the 64-byte swizzle (CU_TENSOR_MAP_SWIZZLE_64B):
// 8-row groups are 512 B apart, layout_type = 4 (cute::UMMA::LayoutType::SWIZZLE_64B).
__device__ __forceinline__ uint64_t make_smem_desc_sw64(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3FFFFu) >> 4);
  d |= static_cast<uint64_t>(1) << 16;
  d |= static_cast<uint64_t>(512 >> 4) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(4) << 61;
  return d;
}

// Same, with the B operand MN-major (N contiguous in smem): used for P.V where V is stored [keys, d] row-major.
__host__ __device__ constexpr uint32_t make_idesc_bf16_bmn(int M, int N) {
  return make_idesc_bf16(M, N) | (1u << 16);
}

// MN-major 128B-swizzled operand: 64 contiguous MN elements (128 B) per K row, 8 K rows per 1024-byte swizzle
// atom; groups of 8 K rows are `sbo` bytes apart, 64-element MN groups `lbo` bytes apart
// (canonical layout ((8,n),(8,k)):((1,LBO),(8,SBO)) in 16-byte units, cute::UMMA::make_umma_desc<Major::MN>).
__device__ __forceinline__ uint64_t make_smem_desc_sw128_mn(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3FFFFu) >> 4);
  d |= static_cast<uint64_t>((lbo_bytes >> 4) & 0x3FFFu) << 16;
  d |= static_cast<uint64_t>((sbo_bytes >> 4) & 0x3FFFu) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(2) << 61;
  return d;
}

// ----------------------------------------------------------------------------------------------
// CTA pair (cta_group::2): two CTAs of a cluster drive both SMs' tensor cores with one instruction stream
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {   // every thread of every CTA of the cluster
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cta address -> shared::cluster address of the same offset in CTA `rank`
__device__ __forceinline__ uint32_t mapa_shared(uint32_t cta_addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(cta_addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
// TMA load whose completion is signalled on an mbarrier that may live in the peer CTA of the pair
__device__ __forceinline__ void tma_load_2d_cg2(const CUtensorMap* m, uint32_t bar_cluster_addr, void* smem_dst, int c0,
                                                int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], "
      "[%2];"
      :
      : "r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(bar_cluster_addr), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tmem_alloc_cg2(uint32_t* smem_dst, uint32_t ncols) {  // one warp in EACH CTA of the pair
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)),
               "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish_cg2() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_cg2(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// D[tmem of both CTAs] (+)= A . B^T with M = 256 split over the pair (128 rows each), B halves from both CTAs
__device__ __forceinline__ void umma_bf16_cg2(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                              uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      :
      : "r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// commit of the pair's MMAs: arrives on the mbarrier at the same smem offset in every CTA of `cta_mask`
__device__ __forceinline__ void tc_commit_cg2(uint64_t* bar, uint16_t cta_mask) {
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
          smem_u32(bar)),
      "h"(cta_mask)
      : "memory");
}

// 32 lanes x 32 consecutive fp32 columns: thread i of the warp receives TMEM lane (base_lane + i)
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float* v) {
  uint32_t* r = reinterpret_cast<uint32_t*>(v);
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
// Same wait, but the 32 destination registers of an earlier tmem_ld32 are threaded through the statement as
// read-write operands: when other work sits between the load and its wait, the compiler must not move a use of
// those registers above the wait (as far as it knows the asm produced them).
__device__ __forceinline__ void tmem_ld_wait_for(float* v) {
  uint32_t* r = reinterpret_cast<uint32_t*>(v);
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]),
                 "+r"(r[8]), "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15]),
                 "+r"(r[16]), "+r"(r[17]), "+r"(r[18]), "+r"(r[19]), "+r"(r[20]), "+r"(r[21]), "+r"(r[22]), "+r"(r[23]),
                 "+r"(r[24]), "+r"(r[25]), "+r"(r[26]), "+r"(r[27]), "+r"(r[28]), "+r"(r[29]), "+r"(r[30]), "+r"(r[31])
               :
               : "memory");
}

// ----------------------------------------------------------------------------------------------
// attention kernels: SFU exp2, MMA with the A operand in TMEM, 16-column TMEM loads / stores
// ----------------------------------------------------------------------------------------------
// 2^x on the SFU in one instruction (ex2.approx.ftz: 2 ulp, flushes denormal results - they vanish in the 16-bit P)
__device__ __forceinline__ float fast_exp2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// D[tmem] (+)= A[tmem] * B[smem]^T : A = 128 lanes x K 16-bit elements, two per 32-bit column
__device__ __forceinline__ void umma_f16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t desc_b, uint32_t idesc,
                                            uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
      :
      : "r"(tmem_d), "r"(tmem_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}

// 32 lanes x 16 consecutive 32-bit columns
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float* v) {
  uint32_t* r = reinterpret_cast<uint32_t*>(v);
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
// 32 lanes x 8 consecutive 32-bit columns
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, float* v) {
  uint32_t* r = reinterpret_cast<uint32_t*>(v);
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr)
               : "memory");
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t* r) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
      :
      : "r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]),
        "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
// 32 lanes x 32 consecutive 32-bit columns back into TMEM (thread i writes lane base_lane + i)
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const float* v) {
  const uint32_t* r = reinterpret_cast<const uint32_t*>(v);
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
      :
      : "r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]),
        "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]),
        "r"(r[18]), "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]),
        "r"(r[27]), "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
      : "memory");
}

}  // namespace iefvad
