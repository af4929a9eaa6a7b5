// Error plumbing + tensor-map encoding shared by all translation units of libiefvad.so.
#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <mutex>
#include <unordered_map>

#include "common.cuh"
#include "tensormap.cuh"

#include <cudaTypedefs.h>

namespace iefvad {

// cudaMallocAsync's default pool hands memory back to the OS at every synchronisation point (release threshold 0):
// an operator that takes gigabytes of scratch (a T = 16384 adjacency) then spends tens of ms per call in the driver.
void keep_async_pool() {
  static bool done[64] = {};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64 || done[dev]) return;
  cudaMemPool_t pool;
  if (cudaDeviceGetDefaultMemPool(&pool, dev) == cudaSuccess) {
    unsigned long long keep = ~0ull;
    cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
  }
  done[dev] = true;
}

static thread_local char g_err[1024] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

const char* last_error() { return g_err; }

static std::atomic<unsigned long long> g_launches{0};
void count_launches(int n) { g_launches.fetch_add(static_cast<unsigned long long>(n), std::memory_order_relaxed); }
unsigned long long launch_count() { return g_launches.load(std::memory_order_relaxed); }

int cuda_fail(cudaError_t e, const char* what, const char* file, int line) {
  set_error("CUDA error %d (%s) at %s:%d in `%s`", static_cast<int>(e), cudaGetErrorString(e), file, line, what);
  return IEFVAD_ERR_CUDA;
}

int device_sms(int* out) {
  int dev = 0;
  IEF_CUDA(cudaGetDevice(&dev));
  IEF_CUDA(cudaDeviceGetAttribute(out, cudaDevAttrMultiProcessorCount, dev));
  return IEFVAD_OK;
}

static PFN_cuTensorMapEncodeTiled_v12000 get_encode() {
  static PFN_cuTensorMapEncodeTiled_v12000 fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(p);
  });
  return fn;
}

// cuTensorMapEncodeTiled costs ~1 us on the host and a forward issues ~270 of them, always for the same few dozen
// (pointer, shape) combinations (the workspace is stable across calls): memoise the 128-byte descriptors.
namespace {
struct TmKey {
  uint64_t v[12];
  bool operator==(const TmKey& o) const { return memcmp(v, o.v, sizeof(v)) == 0; }
};
struct TmHash {
  size_t operator()(const TmKey& k) const {
    uint64_t h = 1469598103934665603ull;
    for (uint64_t x : k.v) { h ^= x; h *= 1099511628211ull; }
    return size_t(h);
  }
};
std::mutex g_tm_mutex;
std::unordered_map<TmKey, CUtensorMap, TmHash> g_tm_cache;
}  // namespace

static int encode_uncached(CUtensorMap* out, const void* base, uint32_t rank, const cuuint64_t* dims,
                           const cuuint64_t* strides, const cuuint32_t* box, int dtype, int swizzle);

static int encode(CUtensorMap* out, const void* base, uint32_t rank, const cuuint64_t* dims, const cuuint64_t* strides,
                  const cuuint32_t* box, int dtype, int swizzle) {
  TmKey key;
  memset(&key, 0, sizeof(key));
  key.v[0] = reinterpret_cast<uint64_t>(base);
  key.v[1] = (uint64_t(rank) << 32) | (uint64_t(uint32_t(dtype)) << 8) | uint64_t(uint32_t(swizzle));
  for (uint32_t i = 0; i < rank; ++i) {
    key.v[2 + i] = dims[i];
    key.v[6 + i] = (i + 1 < rank) ? strides[i] : 0;
    key.v[10 + i / 2] |= uint64_t(box[i]) << (32 * (i & 1));
  }
  {
    std::lock_guard<std::mutex> lock(g_tm_mutex);
    auto it = g_tm_cache.find(key);
    if (it != g_tm_cache.end()) {
      *out = it->second;
      return IEFVAD_OK;
    }
  }
  IEF_TRY(encode_uncached(out, base, rank, dims, strides, box, dtype, swizzle));
  std::lock_guard<std::mutex> lock(g_tm_mutex);
  if (g_tm_cache.size() > 65536) g_tm_cache.clear();      // pointers of short-lived tensors: bound the table
  g_tm_cache.emplace(key, *out);
  return IEFVAD_OK;
}

static int encode_uncached(CUtensorMap* out, const void* base, uint32_t rank, const cuuint64_t* dims,
                           const cuuint64_t* strides, const cuuint32_t* box, int dtype, int swizzle) {
  auto fn = get_encode();
  if (!fn) {
    set_error("cuTensorMapEncodeTiled not available from the CUDA driver");
    return IEFVAD_ERR_CUDA;
  }
  cuuint32_t estr[4] = {1, 1, 1, 1};
  const CUtensorMapDataType dt = (dtype == TM_F32) ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
  const CUtensorMapSwizzle sw = (swizzle == TM_SWIZZLE_NONE) ? CU_TENSOR_MAP_SWIZZLE_NONE
                                : (swizzle == TM_SWIZZLE_64B) ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B;
  CUresult r = fn(out, dt, rank, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, sw,
                  CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed (CUresult %d): rank %u dims {%llu,%llu,%llu} box {%u,%u,%u} base %p "
              "stride0 %llu", static_cast<int>(r), rank, (unsigned long long)dims[0], (unsigned long long)dims[1],
              (unsigned long long)(rank > 2 ? dims[2] : 0), box[0], box[1], rank > 2 ? box[2] : 0, base,
              (unsigned long long)strides[0]);
    return IEFVAD_ERR_CUDA;
  }
  return IEFVAD_OK;
}

int make_tmap_2d(CUtensorMap* out, const void* base, uint64_t inner, uint64_t outer, uint64_t row_stride_bytes,
                 uint32_t box_inner, uint32_t box_outer, int dtype, int swizzle) {
  cuuint64_t dims[2] = {inner, outer};
  cuuint64_t strides[1] = {row_stride_bytes};
  cuuint32_t box[2] = {box_inner, box_outer};
  return encode(out, base, 2, dims, strides, box, dtype, swizzle);
}

int make_tmap_3d(CUtensorMap* out, const void* base, uint64_t d0, uint64_t d1, uint64_t d2, uint64_t stride1_bytes,
                 uint64_t stride2_bytes, uint32_t box0, uint32_t box1, uint32_t box2, int swizzle) {
  cuuint64_t dims[3] = {d0, d1, d2};
  cuuint64_t strides[2] = {stride1_bytes, stride2_bytes};
  cuuint32_t box[3] = {box0, box1, box2};
  return encode(out, base, 3, dims, strides, box, TM_BF16, swizzle);
}

int make_tmap_4d(CUtensorMap* out, const void* base, const uint64_t dims[4], const uint64_t strides_bytes[3],
                 const uint32_t box[4], int dtype, int swizzle) {
  cuuint64_t d[4] = {dims[0], dims[1], dims[2], dims[3]};
  cuuint64_t s[3] = {strides_bytes[0], strides_bytes[1], strides_bytes[2]};
  cuuint32_t b[4] = {box[0], box[1], box[2], box[3]};
  return encode(out, base, 4, d, s, b, dtype, swizzle);
}

}  // namespace iefvad
