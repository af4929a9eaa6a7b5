/* libiefvad - C ABI of the B200-native IEF-VAD inference hot path.
 *
 * The reference (EavnJeong/IEF-VAD) has no FFI / plugin boundary: its hot path is the Python nn.Module
 * surface `model.imf_vad.MMFMIL` plus `train.loss.CLAS2` and scikit-learn's AUC / AP.  This header is the
 * boundary a binding for that path would target; every entry point cites the reference interface it
 * replaces.  The Python host side in `ief-vad_b200/` (ctypes) mirrors the reference's module API on top of it.
 *
 * Conventions
 *   - plain C: pointers + sizes only.  Unless a parameter says "host", every data pointer is a DEVICE
 *     pointer on the current CUDA device; `stream` is a cudaStream_t passed as void* (NULL = legacy default).
 *   - every function returns 0 on success; otherwise a non-zero code (1 invalid argument, 2 CUDA error,
 *     3 bad state) and `iefvad_last_error()` holds a message (thread-local).
 *   - nothing synchronises the host unless stated; inputs are never modified.
 *   - there is NO CPU implementation behind this ABI: without an sm_100a device every compute call fails.
 */
#ifndef IEFVAD_H_
#define IEFVAD_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define IEFVAD_ABI_VERSION 1

/* input element types (`in_dtype`) */
#define IEFVAD_F32 0
#define IEFVAD_F16 1
#define IEFVAD_BF16 2

/* noise models, model/imf_vad.py:130-138 */
#define IEFVAD_NOISE_GAUSSIAN 0
#define IEFVAD_NOISE_STUDENT_T 1

/* precision plans of the model (iefvad_model_set_plan), fp32 accumulation throughout; LayerNorm, softmax statistics,
 * fusion and the classifier are fp32 under every plan.  Any other value is rejected (IEFVAD_ERR_INVALID).
 *   IEFVAD_PLAN_HH (default): every GEMM and the attention core take fp16 (E5M10) operands in one tcgen05 pass - the
 *     11-bit mantissa at bf16's MMA rate; the fp16 range (65 504) is guarded, see iefvad_model_check_finite.
 *   IEFVAD_PLAN_B: bf16 operands (fp32's exponent range); the mu / logvar heads and the refinement Linears use the
 *     3-term bf16 split A_hi.W_hi + A_hi.W_lo + A_lo.W_hi.  The fall-back when plan HH overflows.
 *   IEFVAD_PLAN_FP32: every contraction in fp32 FFMA (1e-5 class), the accuracy yardstick. */
#define IEFVAD_PLAN_FP32 (-1)
#define IEFVAD_PLAN_B 6
#define IEFVAD_PLAN_HH 56

int iefvad_abi_version(void);
const char* iefvad_last_error(void);

/* ------------------------------------------------------------------------------------------------
 * Model object - replaces MMFMIL / MultiModal_Fusion_Attn_Iter construction, model/imf_vad.py:6-38, :48-107
 * ---------------------------------------------------------------------------------------------- */
typedef struct iefvad_model iefvad_model;

/* embed_dim: multiple of 128 in [128, 1024]; embed_dim / num_heads in {32, 64, 96, 128}.
 * noise_model other than the two constants fails with the reference's message (model/imf_vad.py:138). */
int iefvad_model_create(iefvad_model** out, int embed_dim, int num_heads, int num_layers, int num_refinement_steps,
                        float lambda_ref, int noise_model, float nu, float epsilon);
void iefvad_model_destroy(iefvad_model* m);

/* Upload one parameter by its reference state_dict key (e.g. "temporal.image_attn_layers.0.in_proj_weight",
 * "temporal.refinement_blocks.3.2.bias"; the 78 tensors of model/imf_vad.py:69-107).  `data`: device fp32,
 * contiguous, `numel` elements.  The 16-bit operand copies of a weight are refreshed on the given stream. */
int iefvad_model_set_param(iefvad_model* m, const char* key, const float* data, int64_t numel, void* stream);

int iefvad_model_set_plan(iefvad_model* m, int plan);
int iefvad_model_get_plan(const iefvad_model* m);
/* Tuning / test knobs by name.  "refine_fused": the refinement chain (model/imf_vad.py:146-149) as ONE persistent kernel
 * whose hidden activations never leave the SM: -1 = when the batch fills the CTA pairs (default), 0 = never (two tcgen05
 * GEMM launches per step), 1 = always.  Both forms give identical bits.
 * "outproj_ln" (default 1): an encoder layer's tail LN(x + out_proj(ctx)) [+ the whitening LayerNorm] (model/imf_vad.py:115-117)
 * as ONE kernel under the all-fp16 plan; 0 = GEMM + LayerNorm launches (results agree to fp32 statistics rounding).
 * "heads_fuse" (default 1): mu / logvar heads of both modalities + fusion (model/imf_vad.py:125-144) as ONE kernel on the
 * evaluation path, used when the call keeps neither mu / logvar nor the fusion weights; 0 = heads GEMMs + fusion kernel
 * (identical bits). */
int iefvad_model_set_option(iefvad_model* m, const char* name, int64_t value);
/* Range guard of the 16-bit operand plans (fp16 saturates at 65 504; the reference computes in fp32): every forward
 * ORs bit 0 of a device flag when it produced a non-finite logit - an operand that overflowed anywhere upstream reaches
 * the classifier as inf / NaN.  Bit 1: a valid-rows call with pad de-duplication was given a row map that is not the prefix
 * map (the valid rows of a chunk must be its first rows; results of that call are undefined).  This call copies the flags
 * to *nonfinite_host, clears them and SYNCHRONISES the stream.
 * Callers re-run with a bf16 plan (IEFVAD_PLAN_B, fp32's exponent range) or IEFVAD_PLAN_FP32 when it is set. */
int iefvad_model_check_finite(iefvad_model* m, int* nonfinite_host, void* stream);
/* rows per internal slab (bounds the activation workspace, ~18 KB per row); default 262144 */
int iefvad_model_set_max_rows(iefvad_model* m, int64_t max_rows);

/* Replaces MMFMIL.forward(img_visual, ev_visual, padding_mask, text, lengths), model/imf_vad.py:40-44 ->
 * :109-161.  padding_mask / text / lengths are ignored by the reference and have no parameter here.
 * img, ev: [B, T, embed_dim] contiguous, element type `in_dtype`.  Outputs (fp32, contiguous):
 * fused, image_mu, event_mu, image_logvar, event_logvar, w_i, w_e: [B, T, embed_dim]; logits: [B, T, 1];
 * scores (optional, may be NULL): sigmoid(logits) [B, T] (train/ucf_test.py:114). */
int iefvad_model_forward(iefvad_model* m, const void* img, const void* ev, int in_dtype, int64_t B, int64_t T,
                         float* fused, float* logits, float* image_mu, float* event_mu, float* image_logvar,
                         float* event_logvar, float* w_i, float* w_e, float* scores, void* stream);

/* Same path with HOST buffers: copies img / ev host->device, runs the forward, copies logits (and, when
 * non-NULL, scores) device->host and synchronises the stream.  The seven wide outputs stay in library-owned device
 * scratch (the evaluation loop only consumes the scores).  Host pointers should be pinned for full copy bandwidth;
 * batches larger than the slab size are streamed slab by slab. */
int iefvad_model_forward_host(iefvad_model* m, const void* img_host, const void* ev_host, int in_dtype, int64_t B,
                              int64_t T, float* logits_host, float* scores_host, void* stream);

/* The same host-input path with DEVICE results and no host synchronisation: logits [B*T] (and scores, optional)
 * are written to device memory on `stream` - the form the batched evaluator uses (scores feed the on-device
 * compaction and AUC).  Both host-input calls pipeline the transfer: the batch is cut into parts of whole batch
 * elements whose sizes grow geometrically (x 1.4) from `host_part_rows` / 4 rows (default 32768 / 4), and part
 * p+1 is copied on an internal copy stream while part p computes, so only the small first part's copy is exposed.  The host buffers must stay valid and unchanged
 * until `stream` has finished the call. */
int iefvad_model_forward_host_to_device(iefvad_model* m, const void* img_host, const void* ev_host, int in_dtype,
                                        int64_t B, int64_t T, float* logits, float* scores, void* stream);
int iefvad_model_set_host_part_rows(iefvad_model* m, int64_t rows);
/* Valid-rows mode: compute the identical zero-pad rows of a chunk once (1, default) or row by row (0). */
int iefvad_model_set_pad_dedup(iefvad_model* m, int on);

/* Evaluation forward: only logits / scores are returned (the seven wide tensors stay in library scratch), from
 * device inputs (inputs_on_host == 0) or through the pipelined host-input path (!= 0).
 * Optional "valid rows" mode (both pointers non-NULL): callers that feed zero-padded chunks consume only the first
 * len rows of each batch element (train/ucf_test.py:112-114 `logits1[0:len_cur]`) while the pad rows still act as
 * attention keys.  valid_len_host: HOST int64 [B]; rowmap: DEVICE int32 [sum len] = b * T + t of every valid row,
 * ascending.  The encoder then runs on all rows up to and including the last attention core; out-projection,
 * LayerNorms, heads, fusion, refinement and classifier (65 %% of the FLOPs) run on the valid rows only, and
 * logits / scores are COMPACT ([sum len]).
 * Pad de-duplication (default on, iefvad_model_set_pad_dedup; fp16 inputs, plan HH, T <= 256, >= 2
 * layers): the rows past len are taken to be the all-zero pads process_split writes (data/tools.py:100-114) and are
 * not read - identical rows stay identical through the encoder, so ONE representative per chunk is computed and
 * enters every softmax with multiplicity T - len (+ log(T - len) on its score).  Same arithmetic as the dense
 * forward up to the rounding of that key's probability; with de-duplication off the compact results are
 * bit-identical to the valid rows of the full forward. */
int iefvad_model_forward_scores(iefvad_model* m, const void* img, const void* ev, int in_dtype, int inputs_on_host,
                                int64_t B, int64_t T, const int64_t* valid_len_host, const int32_t* rowmap,
                                float* logits, float* scores, void* stream);

/* The evaluation forward from RAGGED pinned host features: img_packed_host / ev_packed_host hold only the valid rows
 * of the B zero-padded [T, D] chunks, chunk after chunk (i.e. the videos' [T_v, D] arrays back to back, as the .npy
 * files hold them) - process_split (data/tools.py:100-114) happens on the device inside the ingest kernel, so the
 * pad rows neither cross PCIe nor are read from HBM.  valid_len_host / rowmap as for iefvad_model_forward_scores;
 * chunk_start: DEVICE int64 [B] = exclusive prefix sums of the valid lengths; chunk_valid: DEVICE int32 [B].
 * Pipelined like the other host-input calls; logits / scores are compact DEVICE vectors [sum len]. */
int iefvad_model_forward_scores_ragged(iefvad_model* m, const void* img_packed_host, const void* ev_packed_host,
                                       int in_dtype, int64_t B, int64_t T, const int64_t* valid_len_host,
                                       const int32_t* rowmap, const int64_t* chunk_start, const int32_t* chunk_valid,
                                       float* logits, float* scores, void* stream);

/* What the reference's evaluation loop derives from the forward besides the scores (train/ucf_test.py:124-144):
 * `w_i.mean(dim=-1)`, `w_e.mean(dim=-1)` per frame and the frames' `fused`, `image_mu`, `event_mu` rows.  Registers
 * optional DEVICE output buffers for the following iefvad_model_forward_scores[_ragged] calls (sticky; NULL = not
 * wanted; all-NULL restores the default): wi_mean / we_mean [rows] (both or neither; the row reduction is fused into the
 * fusion kernel - 8 bytes per frame instead of the two [rows, embed_dim] weight tensors), fused / image_mu / event_mu
 * [rows, embed_dim], where rows = sum of the valid lengths in valid-rows mode (compact, like logits / scores), else B * T. */
int iefvad_model_set_eval_outputs(iefvad_model* m, float* wi_mean, float* we_mean, float* fused, float* image_mu,
                                  float* event_mu);

/* ------------------------------------------------------------------------------------------------
 * Stand-alone operators (device pointers) - the same kernels the forward uses, exposed for parity tests
 * ---------------------------------------------------------------------------------------------- */

/* Uncertainty-weighted fusion, model/imf_vad.py:130-144.  n = number of elements (multiple of 4).
 * factor = 1 (Gaussian) or (nu+1)/nu (StudentT).  fused may be NULL. */
int iefvad_fuse(const float* mu_i, const float* mu_e, const float* logvar_i, const float* logvar_e, int64_t n,
                float factor, float epsilon, float* w_i, float* w_e, float* fused, void* stream);

/* nn.LayerNorm (eps 1e-5) applied once, or twice when w2/b2 are non-NULL (model/imf_vad.py:116-117). */
int iefvad_layernorm(const float* x, int64_t rows, int dim, const float* w1, const float* b1, const float* w2,
                     const float* b2, float eps, float* out, void* stream);

/* nn.Linear with fused epilogue: out = (resid ? resid : 0) + alpha * act(x W^T + bias); act: 0 none, 1 ReLU,
 * 2 QuickGELU (model/module.py:15-17).  x [rows, in_f] fp32, w [out_f, in_f] fp32, out [rows, out_f] fp32.
 * plan: -1 fp32 FFMA, 0 bf16 tcgen05, 1 split-bf16 tcgen05, 2 fp16 (E5M10) tcgen05 - the default model plan's GEMM.  tile_n: 0 = heuristic, or 64 / 128 / 256 (one CTA per
 * 128-row tile), or 512 = 256-column tiles on CTA pairs (tcgen05 cta_group::2, 256-row tiles; out_f %% 256 == 0). */
int iefvad_linear(const float* x, const float* w, const float* bias, const float* resid, float alpha, int act,
                  int64_t rows, int in_f, int out_f, int plan, int tile_n, float* out, void* stream);

/* The tail of one temporal-encoder layer as ONE launch (model/imf_vad.py:115-117 / :121-123):
 *   LN(resid + ctx . w^T + bias; ln_w, ln_b), then LN(.; ln2_w, ln2_b) when ln2_w / ln2_b are non-NULL (the whitening
 * LayerNorm after the last layer).  Plan HH's arithmetic: ctx and w rounded to fp16, fp32 accumulation, resid carried as an
 * fp16 hi + lo pair, LayerNorm statistics in fp32.  ctx, resid [rows, 768], w [768, 768] ([out, in]) fp32 device tensors.
 * out_hi_f16 receives fp16(result); out_lo_f16 (optional) fp16(result - hi).  row_map (optional, device, [rows]): result
 * row r goes to row row_map[r] of out_hi_f16 (negative: dropped); out_lo_f16 must be NULL then. */
int iefvad_outproj_ln(const float* ctx, const float* w, const float* bias, const float* resid, const float* ln_w,
                      const float* ln_b, const float* ln2_w, const float* ln2_b, float eps, int64_t rows,
                      const int32_t* row_map, void* out_hi_f16, void* out_lo_f16, void* stream);

/* nn.MultiheadAttention(batch_first=True)(x, x, x)[0] in eval mode (model/imf_vad.py:115; torch/nn/functional.py:6244).
 * x [B, T, D] fp32; in_w [3D, D], in_b [3D], out_w [D, D], out_b [D].  attn_mask: optional additive [T, T] fp32;
 * key_padding_mask: optional [B, T] uint8 (non-zero = ignore).  plan as for iefvad_linear. */
int iefvad_mha(const float* x, const float* in_w, const float* in_b, const float* out_w, const float* out_b,
               int64_t B, int64_t T, int D, int num_heads, const float* attn_mask, const uint8_t* key_padding_mask,
               int plan, float* out, void* stream);

/* Linear(embed_dim -> 1), model/imf_vad.py:150 (+ optional sigmoid). */
int iefvad_classifier(const float* x, int64_t rows, int dim, const float* w, const float* bias, float* logits,
                      float* scores, void* stream);

/* ------------------------------------------------------------------------------------------------
 * MIL top-k pooling and frame-level AUC / AP
 * ---------------------------------------------------------------------------------------------- */

/* Per-row top-k mean of train/loss.py:24-27: k = int(len/16 + 1) largest of x[row, :len] (after sigmoid when
 * apply_sigmoid != 0), averaged.  x [B, T] fp32 (T <= 16384); lengths [B] int64 (device; NULL = every row full).
 * mean [B] fp32.  idx (optional) [B, kmax] int32: the selected positions in descending-value order, ties by
 * ascending position, padded with -1. */
int iefvad_mil_topk_mean(const float* x, const int64_t* lengths, int64_t B, int64_t T, int apply_sigmoid, float* mean,
                         int32_t* idx, int kmax, void* stream);

/* CLAS2 of train/loss.py:18-30: logits [B, T] (the [B, T, 1] logits tensor), labels [B, *] fp32 with row stride
 * `label_stride` elements (column 0 = normal), lengths [B] int64.  means [B] and the scalar loss are written. */
int iefvad_clas2(const float* logits, const float* labels, int64_t label_stride, const int64_t* lengths, int64_t B,
                 int64_t T, float* means, float* loss, void* stream);

/* Stable descending argsort of fp32 scores: order[i] = index of the i-th largest score, ties by ascending index
 * (== numpy.argsort(-scores, kind="stable"), the ranking sklearn/metrics/_ranking.py builds). */
int iefvad_sort_scores(const float* scores, int64_t n, int32_t* order, void* stream);

/* roc_auc_score / average_precision_score (train/ucf_test.py:151-152) of np.repeat(scores, repeat) against labels
 * in which segment j has pos[j] positive frames out of `repeat`.  scores [n] fp32, pos [n] int32,
 * out: DEVICE double[4] = {AUC (NaN if one class only), AP, #positive frames, #negative frames};
 * order (optional) [n] int32 receives the rank permutation. */
int iefvad_auc_ap(const float* scores, const int32_t* pos, int64_t n, int repeat, double* out, int32_t* order,
                  void* stream);

/* The same for `num_subsets` (1..32) subsets of the segments in ONE ranking pass - the class-wise AUC / AP loop of
 * train/ucf_test.py:164-178 and compute_ano_auc (:336-353), which re-run sklearn per class on concatenated slices.
 * member [n] uint32: bit s set = segment belongs to subset s (NULL allowed when num_subsets == 1).  A subset's
 * AUC / AP equals ranking its members alone: the stable sort keeps their relative order and tie groups without
 * members contribute nothing.  out: DEVICE double[num_subsets][4] laid out as for iefvad_auc_ap. */
int iefvad_auc_ap_multi(const float* scores, const int32_t* pos, const uint32_t* member, int64_t n, int repeat,
                        int num_subsets, double* out, int32_t* order, void* stream);

/* Segmented copy: dst[dst_off[s] + i] = src[src_off[s] + i] for i < len[s] (all arrays on the device, int64).
 * Drops the zero-pad rows of chunked videos (train/ucf_test.py:113 `logits1[0:len_cur]`), and re-orders the
 * per-rank score vectors into list order after the multi-GPU gather. */
int iefvad_segment_copy(const float* src, const int64_t* src_off, float* dst, const int64_t* dst_off,
                        const int64_t* len, int64_t nseg, void* stream);

/* ------------------------------------------------------------------------------------------------
 * The VadCLIP-style graph / transformer classes named by the north star (model/layers.py, model/module.py; not
 * wired into the live reference graph).  plan: -1 fp32 FFMA (feature sizes %% 16), 0 bf16 / 1 split-bf16 tcgen05
 * (feature sizes %% 64).  Weights are passed TRANSPOSED ([out_f, in_f] contiguous; the reference stores [in_f, out_f]).
 * ---------------------------------------------------------------------------------------------- */

/* DistanceAdj.forward(batch_size, max_seqlen), model/layers.py:172-179: out[b, i, j] = exp(-|i-j| / e). */
int iefvad_distance_adj(int64_t batch_size, int max_seqlen, float* out, void* stream);

/* SimilarityAdj.forward(input, seq_len), model/layers.py:130-158.  x [B, T, in_f]; weight0_t = weight0^T
 * [out_f, in_f]; seq_len_host: HOST int64[B] or NULL; out [B, T, T] (cosine of theta = x W0 with itself,
 * threshold 0.7, row softmax on the top-left len x len block, zeros elsewhere). */
int iefvad_similarity_adj(const float* x, const float* weight0_t, const int64_t* seq_len_host, int64_t B, int T, int in_f,
                          int out_f, int plan, float* out, void* stream);

/* GraphConvolution.forward(input, adj), model/layers.py:91-106: out = adj @ (x @ W) (+ bias) + residual.
 * residual: 0 none, 1 identity (in_f == out_f), 2 Conv1d(in_f -> out_f, k = 5, pad = 2) with conv_w [out_f, 5, in_f]
 * (= the reference's [out_f, in_f, 5] with the last two axes swapped) and conv_b [out_f].
 * adj [B, T, T], or NULL = the DistanceAdj adjacency evaluated as a bidirectional first-order scan over T. */
int iefvad_graph_convolution(const float* x, const float* adj, const float* weight_t, const float* bias, int residual,
                             const float* conv_w, const float* conv_b, int64_t B, int T, int in_f, int out_f, int plan,
                             float* out, void* stream);

/* y[b, t, :] = sum_k exp(-|t-k| / e) s[b, k, :]  ==  DistanceAdj(B, T) @ s, as forward + backward linear
 * recurrences (segment reduce, carry scan, apply).  s, y [B, T, D] fp32. */
int iefvad_distance_scan(const float* s, int64_t B, int T, int D, float* y, void* stream);

/* Transformer.forward((x, padding_mask)), model/module.py:20-54, x SEQ-FIRST [L, N, D]; params: HOST array of
 * layers * 12 device pointers per block in the order ln_1.weight, ln_1.bias, attn.in_proj_weight, attn.in_proj_bias,
 * attn.out_proj.weight, attn.out_proj.bias, ln_2.weight, ln_2.bias, mlp.c_fc.weight, mlp.c_fc.bias,
 * mlp.c_proj.weight, mlp.c_proj.bias.  attn_mask: optional additive [L, L]; key_padding_mask: optional [N, L] uint8.
 * plan: as above, or 2 = fp16 operands (fp32 accumulation, LayerNorm and residual stream). */
int iefvad_transformer(const float* x, const float* const* params, int layers, int L, int N, int D, int heads,
                       const float* attn_mask, const uint8_t* key_padding_mask, int plan, float* out, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Input shaping of the reference's data layer (data/tools.py:65-114) for a packed list of V videos:
 * src [sum T_v, D] (element type `dtype`), row_off DEVICE int64 [V + 1] = prefix sums of T_v.
 * ---------------------------------------------------------------------------------------------- */

/* process_split (data/tools.py:100-114): video v -> int(T_v / length) + 1 zero-padded chunks of `length` rows (one chunk
 * when T_v < length; an extra all-zero chunk when T_v %% length == 0).  chunk_off DEVICE int64 [V + 1] = prefix sums of
 * the chunk counts, total_chunks = chunk_off[V]; dst [total_chunks, length, D] in the input's element type.
 * nan_to_num != 0 applies torch.nan_to_num (train/ucf_test.py:83-88). */
int iefvad_process_split(const void* src, int dtype, const int64_t* row_off, int64_t V, int D, int length,
                         const int64_t* chunk_off, int64_t total_chunks, void* dst, int nan_to_num, void* stream);

/* process_feat (data/tools.py:89-97, is_random=False) -> dst [V, length, D] fp32, out_len DEVICE int64 [V]:
 * T_v > length: uniform_extract (:65-73), the mean over np.linspace(0, T_v, length + 1, dtype=int32) bins; else zero-pad. */
int iefvad_process_feat(const void* src, int dtype, const int64_t* row_off, int64_t V, int D, int length, float* dst,
                        int64_t* out_len, int nan_to_num, void* stream);

/* Synthetic event frames (row N4), extracting/ucf_gen_event.py: generate_event_image (:21-37) and the clamp / normalise /
 * stack lines of its caller (:91-95).  frames: DEVICE uint8 [B, C, H, W, 3] (C decoded frames per stack, 16 in the
 * reference).  sum_out (DEVICE fp32 [B, H, W], may be NULL) = number of the C - 1 frame-to-frame differences of the
 * gray image 0.2989 R + 0.5870 G + 0.1140 B whose magnitude exceeds `threshold` (what generate_event_image returns);
 * event_out (DEVICE fp32 [B, 3, H, W], may be NULL) = clamp(sum, 0, clamp_max) / max over the whole batch, the same
 * plane in all three channels (an event-free batch gives 0 / 0 = NaN, as in the reference). */
int iefvad_event_image(const uint8_t* frames, int64_t B, int C, int H, int W, float threshold, float clamp_max,
                       float* sum_out, float* event_out, void* stream);

/* CLIP image encoder of the extraction step (row N4): VisionTransformer.forward(x), extracting/clip/model.py:206-241
 * (ViT-L/14 in the reference's feature extraction).  x: DEVICE [N, 3, resolution, resolution] normalised pixels,
 * dtype 0 fp32 / 1 fp16 / 2 bf16; out: DEVICE fp32 [N, output_dim].  Grid G = resolution / patch, T = G*G + 1 tokens.
 * params: HOST array of 8 + 12 * layers DEVICE fp32 pointers in the order
 *   conv1.weight [width, 3, patch, patch], class_embedding [width], positional_embedding [T, width],
 *   ln_pre.weight, ln_pre.bias,
 *   per block the 12 pointers of iefvad_transformer's table (transformer.resblocks.{i}.*),
 *   ln_post.weight, ln_post.bias, proj [width, output_dim].
 * plan: -1 fp32 FFMA, 2 fp16 operands with fp32 accumulation; LayerNorms, the residual stream and the projection are
 * fp32 under both.  Constraints: resolution % patch == 0, width % 128 == 0 and <= 1024, width / heads in {32, 64, 96,
 * 128}, 0 <= N <= 65535, layers <= 64; a malformed argument fails before the device is touched.
 * Stateless like iefvad_transformer: the weights are converted on every call.  Device scratch (stream-ordered pool,
 * released at the end of the call) under plan 2 is about 26 * width bytes per token (26 KB at ViT-L/14's width 1024,
 * 6.7 MB per 224 px image) plus the fp16 weights (2 bytes per parameter, 0.6 GB for ViT-L/14); plan -1 needs about
 * 44 * width bytes per token and 4 bytes per parameter. */
int iefvad_clip_visual(const void* x, int dtype, int N, int resolution, int patch, int width, int layers, int heads,
                       int output_dim, const float* const* params, int plan, float* out, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Instrumentation used by bench.py
 * ---------------------------------------------------------------------------------------------- */

/* Micro-benchmark of the tcgen05 GEMM on library-allocated buffers (synchronises; default stream): M x N x K,
 * nsplit 1 | 3, tile_n 0 | 64 | 128 | 256 | 512 (as for iefvad_linear), stages 0 (= as many as fit) or a cap on the operand ring depth, epi_kind 0 = mainloop only (discard), 1 = fp32 out, 2 = refinement
 * epilogue (fp32 residual in, fp32 + bf16 hi/lo out), 3 = ReLU -> bf16 hi/lo, 4 = QKV scatter, 5 = fp16 operands,
 * ReLU -> fp16, 6 = fp16 operands, fp32 residual in, fp32 + fp16 out, 7 = fp16 operands, fp16 hi + lo pair residual in, fp16 pair out in
 * place (5 and 7 = the two refinement Linears of the default plan).  Writes the mean
 * device time of `iters` back-to-back launches (CUDA events). */
int iefvad_bench_gemm(int64_t M, int N, int K, int nsplit, int tile_n, int stages, int epi_kind, int iters,
                      float* ms_per_iter);

/* ------------------------------------------------------------------------------------------------
 * Training step (SURVEY 8f row N3): the pieces `loss.backward()` of train/ucf_train.py:105 needs besides the GEMMs
 * (which go through iefvad_linear: dgrad = linear(dY, W^T), wgrad = linear(dY^T, X^T)).  All tensors fp32, device.
 * ---------------------------------------------------------------------------------------------- */

/* nn.MultiheadAttention's core in TRAIN mode (model/imf_vad.py:53,70: dropout 0.1 on the attention weights,
 * torch/nn/functional.py:6643-6647): out = dropout(softmax(q k^T / sqrt(head_dim))) v per (batch element, head).
 * qkv [B*T, 3*heads*head_dim] (in-projection output, bias added, q unscaled); out [B*T, heads*head_dim]; lse [B, heads, T]
 * = log-sum-exp of the scores (saved for the backward).  The dropout mask is a pure function of (seed, head, query, key):
 * Philox4x32-10 with key = (seed & 0xffffffff, seed >> 32) and counter = (key >> 2, query, b * heads + h, 0), word (key & 3),
 * dropped when the word < uint32(double(p_drop) * 2^32), kept weights scaled by 1.f / (1.f - p_drop) (restated in
 * oracle/iefvad_oracle.py: attention_keep) - NOT PyTorch's generator stream (no kernel can reproduce that),
 * so train-mode parity with the reference is statistical; p_drop = 0 gives the eval-mode arithmetic. */
int iefvad_attention_train_fwd(const float* qkv, int64_t B, int64_t T, int heads, int head_dim, float p_drop, uint64_t seed,
                               float* out, float* lse, void* stream);
/* dqkv [B*T, 3*heads*head_dim] <- dout [B*T, heads*head_dim], recomputing the weights (and the same mask) from qkv / lse */
int iefvad_attention_train_bwd(const float* qkv, const float* out, const float* dout, const float* lse, int64_t B, int64_t T,
                               int heads, int head_dim, float p_drop, uint64_t seed, float* dqkv, void* stream);
/* nn.LayerNorm backward: x [rows, dim] = the layer's input, dy = gradient of its output -> dx, dweight [dim], dbias [dim] */
int iefvad_layernorm_bwd(const float* x, const float* weight, const float* dy, int64_t rows, int dim, float eps, float* dx,
                         float* dweight, float* dbias, void* stream);
/* out[c] = sum_r a[r, c] (bias gradients), optionally weighted by row_weight[r] (classifier weight gradient); fixed order */
int iefvad_colsum(const float* a, const float* row_weight, int64_t rows, int dim, float* out, void* stream);
/* Backward of the uncertainty-weighted fusion (model/imf_vad.py:130-144).  g_* = upstream gradients of fused, w_i, w_e and of
 * the returned image_mu / event_mu / image_logvar / event_logvar (any may be NULL = 0); d_* = total gradients of the four
 * head outputs (fusion path + their own upstream gradient). */
int iefvad_fuse_bwd(const float* mu_i, const float* mu_e, const float* logvar_i, const float* logvar_e, const float* g_fused,
                    const float* g_wi, const float* g_we, const float* g_mu_i, const float* g_mu_e, const float* g_logvar_i,
                    const float* g_logvar_e, int64_t n, float factor, float epsilon, float* d_mu_i, float* d_mu_e,
                    float* d_logvar_i, float* d_logvar_e, void* stream);
/* Weight gradient of a Linear: dw [out_f, in_f] = alpha * dy^T . x for dy [rows, out_f], x [rows, in_f] (row-major fp32), with
 * the 3-term bf16 split of the forward GEMMs (fp32's exponent range, ~16 mantissa bits) and split-K over the rows. */
int iefvad_wgrad(const float* dy, const float* x, int64_t rows, int out_f, int in_f, float alpha, float* dw, void* stream);
int iefvad_quickgelu(const float* x, int64_t n, float* out, void* stream);   /* model/module.py:15-17: x * sigmoid(1.702 x) */
int iefvad_relu_bwd(const float* dh, const float* h, int64_t n, float* out, void* stream);      /* out = h > 0 ? dh : 0 */
int iefvad_axpy(float* y, const float* x, float alpha, int64_t n, void* stream);                /* y += alpha x */
int iefvad_outer(const float* a, const float* w, int64_t rows, int dim, float* out, void* stream); /* out[r, c] = a[r] w[c] */
/* dst[c, r] = src[r, c]; dst rows are ld_dst >= rows long, the tail [rows, ld_dst) is zero-filled (GEMM K padding) */
int iefvad_transpose(const float* src, int64_t rows, int cols, float* dst, int64_t ld_dst, void* stream);
/* Backward of CLAS2 (train/loss.py:18-30): dlogits [B, T] from the chosen top-k positions idx [B, kmax] (-1 padded) and the
 * per-row means of iefvad_mil_topk_mean(apply_sigmoid = 1); g_loss: device scalar (NULL = 1). */
int iefvad_clas2_bwd(const float* logits, const float* means, const float* labels, int64_t label_stride, const int32_t* idx,
                     int64_t B, int64_t T, int kmax, const float* g_loss, float* dlogits, void* stream);
/* Training objective of the reference's loop (train/ucf_train.py:73-102, the loss it builds from the module's outputs), with
 * mu_i, mu_e, lv_i, lv_e the [B, T, D] fp32 outputs image_mu, event_mu, image_logvar, event_logvar:
 *   loss_cls = CLAS2(logits, labels, lengths)                               (train/loss.py:18-30, as iefvad_clas2)
 *   cos      = cosine_similarity(normalize(mu_i), normalize(mu_e)) per row  (:75-82)
 *   loss_reg = mean(1 - cos) + mean |norm(mu_i) - norm(mu_e)|               (:75-82)
 *   c = log(nu / (nu + 1)), eli = lv_i + c, ele = lv_e + c                  (:93-98)
 *   loss_kl  = -0.5 mean(1 + eli - mu_i^2 - exp(eli)) - 0.5 mean(1 + ele - mu_e^2 - exp(ele))
 *   total    = loss_cls + reg_weight loss_reg + kl_weight loss_kl
 * The means run over all B*T rows (B*T*D elements for the KL term), pad rows beyond `lengths` included, as in the loop.
 * torch's edge rules hold: normalize divides by max(|x|, 1e-12), cosine_similarity by max(|x|, 1e-8) per factor; the
 * gradients of |x| at 0 and of a norm at the zero vector are 0; exp overflows to +inf as fp32 does.  Reductions are in
 * float64 in a fixed order (run-to-run identical, independent of the device's SM count).  D % 4 == 0, the wide tensors
 * 16-byte aligned, kmax = T / 16 + 1.
 * Forward: means [B], idx [B, kmax] (top-k positions, as iefvad_mil_topk_mean) and record [B*T, 4] (float64, 32-byte
 * aligned) are kept for the backward; total, loss_cls, loss_reg, loss_kl are device scalars.  4 kernel launches. */
int iefvad_train_loss_fwd(const float* logits, const float* labels, int64_t label_stride, const int64_t* lengths, int64_t B,
                          int64_t T, const float* mu_i, const float* mu_e, const float* logvar_i, const float* logvar_e, int D,
                          double nu, double reg_weight, double kl_weight, float* means, int32_t* idx, int kmax, double* record,
                          float* total, float* loss_cls, float* loss_reg, float* loss_kl, void* stream);
/* Backward: d_logits [B, T] and d_mu_i, d_mu_e, d_logvar_i, d_logvar_e [B*T, D] (fp32) of
 * g_total total + g_cls loss_cls + g_reg loss_reg + g_kl loss_kl; each g_* is a device scalar, NULL = 0.  2 launches. */
int iefvad_train_loss_bwd(const float* logits, const float* means, const float* labels, int64_t label_stride, const int32_t* idx,
                          int64_t B, int64_t T, int kmax, const float* mu_i, const float* mu_e, const float* logvar_i,
                          const float* logvar_e, int D, const double* record, double nu, double reg_weight, double kl_weight,
                          const float* g_total, const float* g_cls, const float* g_reg, const float* g_kl, float* d_logits,
                          float* d_mu_i, float* d_mu_e, float* d_logvar_i, float* d_logvar_e, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Temporal-localisation mAP (SURVEY 8f row N5) - replaces getDetectionMAP / getLocMAP / nms, train/metrics.py:19-136
 * (imported by train/ucf_test.py:13 as dmAP, never called by the reference).
 * ---------------------------------------------------------------------------------------------- */

/* Per (video, class): class score = mean of the top int(T/16) values of the column (:60-64); for classes with a positive
 * score, runs of >= 2 frames above max - 0.6 (max - min) become proposals scored max + 0.7 class score (:75-83), sorted by
 * score, greedy NMS at IoU 0.6 (:19-41).  pred: the videos' [T_v, num_classes] fp32 predictions back to back (video v at
 * row vid_off[v], vid_len[v] <= 4096 rows); prop_count [V, C] (-1: more than 512 proposals, unsupported), prop_se
 * [V, C, 512, 2] (start, end), prop_score [V, C, 512], class_score [V, C]. */
int iefvad_locmap_proposals(const float* pred, const int64_t* vid_off, const int32_t* vid_len, int64_t num_videos,
                            int num_classes, int max_len, int32_t* prop_count, int32_t* prop_se, float* prop_score,
                            float* class_score, void* stream);
/* Per class: proposals of all videos sorted by score (:96), greedy matching against that class's ground-truth segments with
 * deletion of the matched one (:104-122, IoU of the integer frame sets >= iou_threshold), ap[c] = sum(precision * tp) / #gt
 * (:123-128; 0 without a true positive).  gt [num_gt, 3] = (video, start, end) GROUPED BY CLASS in the reference's order,
 * class c owning rows [gt_off[c], gt_off[c + 1]); n_pred[c] = proposals of class c (the reference returns 0 for the whole
 * call as soon as one class has none, :92-93 - the host side reproduces that). */
int iefvad_locmap_match(const int32_t* prop_count, const int32_t* prop_se, const float* prop_score, int64_t num_videos,
                        int num_classes, const int32_t* gt, const int32_t* gt_off, int64_t num_gt, double iou_threshold,
                        double* ap, int32_t* n_pred, void* stream);

/* number of CUDA kernels this library has launched since load (process-wide) */
uint64_t iefvad_launch_count(void);
/* bumped whenever a library workspace is (re)allocated: a CUDA graph captured around a forward call holds workspace
 * addresses and must be re-captured once this value has changed (the Python module does that for its small-batch graphs) */
uint64_t iefvad_alloc_generation(void);
/* a caller that replays a CUDA graph captured around library calls reports the kernels of one replay here, so that
 * iefvad_launch_count keeps counting launches rather than host calls */
void iefvad_add_launches(uint64_t n);

/* Per-kernel-class device timing of the model forward with CUDA events on the launching stream.
 * classes (IEFVAD_PROFILE_CLASSES = 15): 0 gemm_tc QKV in-projection, 1 attn_tc, 2 layernorm, 3 fuse, 4 classifier,
 * 5 ingest, 6 gemm_simt, 7 attn_simt, 8 gemm_tc out-projection, 9 gemm_tc heads, 10 gemm_tc refinement Linear 1
 * (ReLU), 11 gemm_tc refinement Linear 2 (residual), 12 valid-row gather, 13 fused refinement chain, 14 heads + fusion.
 * iefvad_profile_read synchronises, fills ms / work (executed
 * FLOPs for the GEMM and attention classes, bytes moved otherwise) / launches (arrays of IEFVAD_PROFILE_CLASSES) for everything
 * recorded since the last read, and clears the record. */
#define IEFVAD_PROFILE_CLASSES 15
int iefvad_profile_enable(int on);
int iefvad_profile_read(double* ms, double* work, int64_t* launches);

#ifdef __cplusplus
}
#endif
#endif /* IEFVAD_H_ */
