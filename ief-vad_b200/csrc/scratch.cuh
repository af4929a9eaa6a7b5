// Per-call device temporaries from the stream-ordered pool, released (stream-ordered) when the object goes out of scope.
// Used by the stateless entry points (capi.cu, graph.cu, clip.cu).
#pragma once
#include <vector>

#include "common.cuh"

namespace iefvad {

struct Scratch {   // stream-ordered temporaries
  cudaStream_t s;
  std::vector<void*> ptrs;
  explicit Scratch(cudaStream_t st) : s(st) { keep_async_pool(); }
  ~Scratch() {
    for (void* p : ptrs) cudaFreeAsync(p, s);
  }
  template <typename T>
  int get(T** out, size_t count) {
    void* p = nullptr;
    const size_t bytes = (count ? count : 1) * sizeof(T);
    IEF_CUDA(cudaMallocAsync(&p, bytes, s));
    ptrs.push_back(p);
    *out = static_cast<T*>(p);
    return IEFVAD_OK;
  }
};

}  // namespace iefvad
