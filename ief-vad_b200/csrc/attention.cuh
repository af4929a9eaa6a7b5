#pragma once
#include "common.cuh"

namespace iefvad {

struct AttnTcArgs {
  const bf16* q = nullptr;   // [B, H, T, dhp]  pre-scaled by dh^-1/2
  const bf16* k = nullptr;   // [B, H, T, dhp]
  const bf16* vt = nullptr;  // [B, H, dh, Tpad]
  bf16* out = nullptr;       // [B*T, ldo], head h writes columns [h*dh, (h+1)*dh)
  int ldo = 0;
  int B = 0, T = 0, H = 0, dh = 0, dhp = 0, Tpad = 0;
  const float* attn_mask = nullptr;    // optional additive [T, T]
  const uint8_t* key_pad = nullptr;    // optional [B, T], non-zero = ignore key
  int fp16 = 0;                        // q / k / vt / out hold fp16 and P is rounded to fp16 (11-bit mantissa), else bf16
  const int* row_out = nullptr;        // optional [B*T]: output row of query row b*T+t (compact layouts), < 0 = drop
  // ragged items (short kernel only): q / k are [H, T, dhp], vt [H, dh, Tpad] over ALL packed rows and items[c] =
  // {first row, rows (<= 256), valid rows, multiplicity of the last row as a key (0 = none)} for n_chunks row ranges
  const int* items = nullptr;          // device, int4 per chunk
  int n_chunks = 0;
};

int attn_tc(const AttnTcArgs& a, cudaStream_t stream);

// T <= 256 without masks (every chunk the reference's callers produce): persistent kernel, P kept in TMEM
// (attention_short.cu).  attn_tc dispatches here when attn_short_supported(a).
// T > 256 without masks: persistent two-tile kernel, single-pass softmax with integer (power-of-two) maxima, O
// accumulated in TMEM (attention_long.cu).  Masked attention, and any other shape neither kernel takes, runs the
// flash-style attn_tc_kernel.
bool attn_long_supported(const AttnTcArgs& a);
int attn_long(const AttnTcArgs& a, cudaStream_t stream);
bool attn_short_supported(const AttnTcArgs& a);
int attn_short(const AttnTcArgs& a, cudaStream_t stream);

// Row width (dhp) of q / k that attn_tc reads for these arguments (dhp itself is not consulted): d_h where the
// short-sequence kernel runs, which takes 32-column chunks under the 64-byte swizzle, else d_h padded to a multiple of
// 64 for the 128-byte-swizzled kernels.
int attn_qk_cols(const AttnTcArgs& a);

// fp32 plan: qkv fp32 [B*T, 3*H*dh] (bias added, q unscaled) -> out fp32 [B*T, H*dh]
int attn_simt(const float* qkv, float* out, int B, int T, int H, int dh, const float* attn_mask,
              const uint8_t* key_pad, cudaStream_t stream);

}  // namespace iefvad
