// Counter-based dropout mask of the training attention (documented in include/iefvad.h: iefvad_dropout).
#pragma once
#include "common.cuh"

namespace iefvad {

// Philox4x32-10 (Salmon et al., SC'11)
__device__ __forceinline__ uint4 philox4x32_10(uint4 ctr, uint2 key) {
  constexpr uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(M0, ctr.x), lo0 = M0 * ctr.x;
    const uint32_t hi1 = __umulhi(M1, ctr.z), lo1 = M1 * ctr.z;
    ctr = make_uint4(hi1 ^ ctr.y ^ key.x, lo1, hi0 ^ ctr.w ^ key.y, lo0);
    key.x += W0;
    key.y += W1;
  }
  return ctr;
}

// The dropout mode of one attention call, passed to the kernels by value.
//   kDropOff:    no dropout (p = 0)
//   kDropPhilox: the library's own mask - counter (key >> 2, query, b * H + h, 0), dropped when the word < thresh
//   kDropTorch:  torch.native_dropout's mask of the [B*H, T, T] weights - element e = (bh * T + query) * T + key lies in
//                group v = e / 4, drawn by thread v % threads in iteration v / threads: counter
//                (lo64 = offset / 4 + v / threads, hi64 = v % threads), word e % 4, kept when the curand uniform < keep
enum DropKind : int { kDropOff = 0, kDropPhilox = 1, kDropTorch = 2 };
struct DropoutDesc {
  int kind;
  int T;                             // keys per row (torch: the row pitch of the element index)
  uint32_t thresh;                   // philox: drop threshold (p * 2^32)
  float keep;                        // torch: float32(1 - p)
  float scale;                       // multiplier of a kept weight
  unsigned long long seed;
  unsigned long long offset;         // torch: the generator's offset (a multiple of 4)
  unsigned int threads;              // torch: G = grid * 256 threads of torch's launch
};

__device__ __forceinline__ uint4 torch_group(const DropoutDesc& d, unsigned long long v) {
  unsigned long long it, th;
  if ((v >> 32) == 0) {              // 32-bit division whenever the group index allows it
    const uint32_t v32 = uint32_t(v), i32 = v32 / d.threads;
    it = i32;
    th = v32 - i32 * d.threads;
  } else {
    it = v / d.threads;
    th = v - it * d.threads;
  }
  const unsigned long long c = (d.offset >> 2) + it;
  return philox4x32_10(make_uint4(uint32_t(c), uint32_t(c >> 32), uint32_t(th), uint32_t(th >> 32)),
                       make_uint2(uint32_t(d.seed), uint32_t(d.seed >> 32)));
}
// curand_uniform: float32(word) * 2^-32 + 2^-33 (the product is exact, so a fused multiply-add rounds the same way)
__device__ __forceinline__ float torch_keep(const DropoutDesc& d, uint32_t w) {
  return fmaf(__uint2float_rn(w), 2.3283064365386963e-10f, 1.1641532182693481e-10f) < d.keep ? d.scale : 0.f;
}
__device__ __forceinline__ uint32_t word_of(const uint4& r, unsigned int k) {
  return k == 0 ? r.x : k == 1 ? r.y : k == 2 ? r.z : r.w;
}

// keep (scale) / drop (0) decision of attention weight (bh, query i, key j); philox: one call serves 4 consecutive keys
__device__ __forceinline__ float keep_scale(const DropoutDesc& d, int bh, int i, int j) {
  if (d.kind == kDropTorch) {
    const unsigned long long e = ((unsigned long long)bh * d.T + i) * d.T + j;
    return torch_keep(d, word_of(torch_group(d, e >> 2), unsigned(e & 3)));
  }
  const uint4 r = philox4x32_10(make_uint4(uint32_t(j >> 2), uint32_t(i), uint32_t(bh), 0u),
                                make_uint2(uint32_t(d.seed), uint32_t(d.seed >> 32)));
  const uint32_t v = (j & 3) == 0 ? r.x : (j & 3) == 1 ? r.y : (j & 3) == 2 ? r.z : r.w;
  return v >= d.thresh ? d.scale : 0.f;          // P(drop) = thresh / 2^32
}

// the same decision for the two consecutive keys j, j + 1 (j even).  philox: both lie in one word group.  torch: with an
// odd T the element index e of key j may be odd, and e = 3 mod 4 puts key j + 1 in the next group
__device__ __forceinline__ float2 keep_scale2(const DropoutDesc& d, int bh, int i, int j) {
  if (d.kind == kDropTorch) {
    const unsigned long long e = ((unsigned long long)bh * d.T + i) * d.T + j;
    const unsigned int k = unsigned(e & 3);
    const uint4 r = torch_group(d, e >> 2);
    const uint32_t w1 = k == 3 ? torch_group(d, (e >> 2) + 1).x : word_of(r, k + 1);
    return make_float2(torch_keep(d, word_of(r, k)), torch_keep(d, w1));
  }
  const uint4 r = philox4x32_10(make_uint4(uint32_t(j >> 2), uint32_t(i), uint32_t(bh), 0u),
                                make_uint2(uint32_t(d.seed), uint32_t(d.seed >> 32)));
  const uint32_t v0 = (j & 2) ? r.z : r.x, v1 = (j & 2) ? r.w : r.y;
  return make_float2(v0 >= d.thresh ? d.scale : 0.f, v1 >= d.thresh ? d.scale : 0.f);
}

// host: the descriptor of each mode (p_drop = 0 in philox mode gives kDropOff, the eval-mode arithmetic)
inline DropoutDesc dropout_philox(float p_drop, unsigned long long seed, int T) {
  DropoutDesc d{};
  d.thresh = p_drop > 0.f ? uint32_t(double(p_drop) * 4294967296.0) : 0u;
  d.kind = d.thresh ? kDropPhilox : kDropOff;
  d.T = T;
  d.scale = 1.f / (1.f - p_drop);
  d.seed = seed;
  return d;
}
inline DropoutDesc dropout_torch(double p_drop, unsigned long long seed, unsigned long long offset, unsigned int threads, int T) {
  DropoutDesc d{};
  d.kind = kDropTorch;
  d.T = T;
  d.keep = float(1.0 - p_drop);
  d.scale = float(1.0 / double(d.keep));
  d.seed = seed;
  d.offset = offset;
  d.threads = threads;
  return d;
}

}  // namespace iefvad
