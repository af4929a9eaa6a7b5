// Device-resident IEF-VAD model: fp32 master parameters (state_dict layout of model/imf_vad.py:69-107),
// packed 16-bit copies for the tensor-core plans, and a grow-only activation workspace.
#pragma once
#include <string>
#include <unordered_map>
#include <vector>

#include "attention.cuh"
#include "common.cuh"
#include "elementwise.cuh"
#include "gemm.cuh"
#include "heads_fuse.cuh"
#include "outproj_ln.cuh"
#include "refine.cuh"

namespace iefvad {

// precision plans (the values of IEFVAD_PLAN_* in include/iefvad.h):
// PLAN_HH: fp16 (E5M10) operands in one MMA pass for every GEMM and the attention core.  fp16 inputs are then exact, and
// one fp16 pass matches the 3-term bf16 split at a third of the MMA work (DESIGN.md section 4)
// PLAN_B: bf16 operands; the heads and the refinement Linears use the 3-term split (A_hi.W_hi + A_hi.W_lo + A_lo.W_hi).
// fp32's exponent range: the fall-back when an fp16 operand overflows
// PLAN_FP32: every contraction in fp32 FFMA
enum : int { PLAN_FP32 = -1, PLAN_B = 6, PLAN_HH = 56 };

struct DevBuf {
  void* p = nullptr;
  size_t bytes = 0;
  int reserve(size_t need);   // grow-only; contents are NOT preserved
  void release();
  template <typename T> T* as() const { return static_cast<T*>(p); }
};

struct Linear {          // y = x W^T + b, W [out, in]
  float* w = nullptr;    // fp32 master
  float* b = nullptr;
  bf16* w_hi = nullptr;
  bf16* w_lo = nullptr;   // bf16(w - hi) for plan B's 3-term split: heads and refinement Linears only
  bf16* w_h16 = nullptr;  // fp16 copy (16-bit storage)
  int out = 0, in = 0;
};

struct ParamSlot {
  float* dst = nullptr;
  long long numel = 0;
  bf16* hi = nullptr;    // packed copies refreshed on upload (weights only)
  bf16* lo = nullptr;    // heads and refinement weights only
  bf16* h16 = nullptr;   // fp16 copy
  bool loaded = false;
};

// Optional "valid rows only" mode of the forward.  Callers that feed zero-padded chunks (data/tools.py:100-114) consume
// only the first len rows of every batch element (train/ucf_test.py:112-114 `logits1[0:len_cur]`), but the pad rows
// still act as attention KEYS.  With this descriptor the encoder runs on all rows up to and including the last
// attention core; everything after it (out-projection, LayerNorms, heads, fusion, refinement, classifier - 65 % of
// the FLOPs) runs on the valid rows only, gathered into a compact matrix.  Every output is then COMPACT
// ([sum len, ...], valid row j of the whole call at index j) and bit-identical to the valid rows of the full forward.
unsigned long long alloc_generation();   // bumped whenever a library workspace is (re)allocated

struct ValidRows {
  const long long* len_host = nullptr;  // HOST [B]: valid rows (a prefix) of each batch element, 0 <= len <= T
  const int* rowmap = nullptr;          // DEVICE [sum len]: row index (b * T + t, relative to this call's first row,
                                        // after subtracting row_base) of every valid row, ascending
  long long row_base = 0;               // subtracted from rowmap entries (lets a caller pass a slice of a global map)
  // ragged inputs (optional, both non-null): img / ev then point at PACKED device buffers that hold only the valid rows
  // (chunk b's rows start at packed row chunk_start[b] - start_base); the pad rows are synthesised as zeros on ingest
  const long long* chunk_start = nullptr;   // DEVICE [B]
  const int* chunk_valid = nullptr;         // DEVICE [B] (== len_host)
  long long start_base = 0;
};

struct Model {
  int D = 0, H = 0, L = 0, R = 0, dh = 0, dhp = 0;
  float lambda_ref = 0.5f, factor = 1.f, eps = 1e-8f;
  int plan = PLAN_HH;
  bool pad_dedup = true;         // valid-rows mode: one representative per chunk for its identical zero-pad rows
  int refine_fused = -1;         // refinement chain as ONE persistent kernel (refine_fused.cu): -1 = when it pays (enough
                                 // rows to fill the CTA pairs), 0 = never (per-step GEMMs), 1 = always
  int heads_fuse_mode = 1;       // heads of both modalities + fusion as one kernel (heads_fuse.cu) when mu / logvar are not kept
  bool heads_outputs_unused = false;   // set per call by the C ABI: the mu / logvar / w pointers of forward() are scratch
  int outproj_ln_mode = 1;       // out-projection + residual + LayerNorm(s) as one kernel (outproj_ln.cu) where the plan allows
  bool refine_contig = false;    // the fp16 refinement weights lie back to back (W1_0, W2_0, W1_1, ...) in params_h16
  // evaluation extras (set per call by the C ABI): per-row means of the fusion weights, written at the call's compact offset
  float* eval_wi_mean = nullptr;
  float* eval_we_mean = nullptr;
  long long max_rows = 262144;   // rows per internal slab (whole batch elements); ~18 KB of workspace per row
  int num_sms = 148;
  int device = 0;

  // parameters, index 0 = image, 1 = event
  std::vector<Linear> in_proj[2], out_proj[2];
  std::vector<float*> ln_w[2], ln_b[2];
  float* whiten_w[2] = {nullptr, nullptr};
  float* whiten_b[2] = {nullptr, nullptr};
  Linear heads[2];               // rows [0, D) = mu, [D, 2D) = logvar
  std::vector<Linear> ref1, ref2;
  float* cls_w = nullptr;
  float* cls_b = nullptr;

  std::unordered_map<std::string, ParamSlot> slots;
  DevBuf params_f32, params_hi, params_lo, params_h16;

  // workspace (one slab)
  DevBuf x32, y32, a_hi, a_lo, h_hi, h_lo, qb, kb, vtb, qkv32, attn32, h32, inv_map, items_dev, aux_dev, ln_scratch, ln_ident;
  DevBuf status;                         // int[4]: [0] bit 0 = a non-finite logit was produced since the last check
  std::vector<ChunkItem> items_host;     // packed-row layout of the current slab (valid-rows mode, see forward)
  std::vector<ChunkAux> aux_host;

  int init(int embed_dim, int heads, int layers, int refine_steps, float lambda, int noise_model, float nu, float epsilon);
  int set_param(const char* key, const float* dptr, long long numel, cudaStream_t stream);
  int check_loaded() const;
  int reserve_workspace(long long rows, int B, int T, bool fp32_plan);
  int forward(const void* img, const void* ev, int in_dtype, long long B, long long T, float* fused, float* logits,
              float* image_mu, float* event_mu, float* image_logvar, float* event_logvar, float* w_i, float* w_e,
              float* scores, cudaStream_t stream, const ValidRows* vr = nullptr);
  void destroy();
};

// Per-kernel-class device timing (CUDA events on the launching stream) for bench.py's roofline block.
enum : int { KC_GEMM_QKV = 0, KC_ATTN_TC, KC_LAYERNORM, KC_FUSE, KC_CLASSIFIER, KC_INGEST, KC_GEMM_SIMT, KC_ATTN_SIMT,
             KC_GEMM_OUT, KC_GEMM_HEADS, KC_GEMM_REF1, KC_GEMM_REF2, KC_GATHER, KC_REFINE_FUSED, KC_HEADS_FUSE, KC_OUTPROJ_LN, KC_COUNT };
struct Profiler {
  bool on = false;
  struct Rec { int cls; double work; cudaEvent_t a, b; };   // work = algorithmic flops (GEMM/attn) or bytes (others)
  std::vector<Rec> recs;
  void begin(int cls, double work, cudaStream_t st);
  void end(cudaStream_t st);
  int read(double* ms, double* work, long long* launches);     // synchronises, sums per class, clears
};
Profiler& profiler();

}  // namespace iefvad
