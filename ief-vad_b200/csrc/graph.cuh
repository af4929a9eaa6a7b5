// Rows D1-D4 of the scope table: the VadCLIP-style graph / transformer classes of model/layers.py and
// model/module.py (dead code in the live reference graph, named by the north star), built from the same tcgen05
// GEMM / attention / LayerNorm kernels as the live forward plus the kernels of graph.cu.
#pragma once
#include "common.cuh"

namespace iefvad {

// DistanceAdj.forward, model/layers.py:172-179: out[b, i, j] = exp(-|i - j| / e), [B, T, T] fp32.
int distance_adj(float* out, long long B, int T, cudaStream_t stream);

// SimilarityAdj.forward, model/layers.py:130-158.  x [B, T, Din]; w0t = weight0^T [Dout, Din]; seq_len: HOST int64[B]
// or null; out [B, T, T].  plan: -1 fp32 FFMA, 0 bf16, 1 split-bf16.
int similarity_adj(const float* x, const float* w0t, const long long* seq_len_host, long long B, int T, int Din,
                   int Dout, int plan, float* out, int num_sms, cudaStream_t stream);

// GraphConvolution.forward, model/layers.py:91-106: out = adj @ (x @ W) (+ bias) + residual.
// wt = weight^T [Dout, Din]; residual: 0 none, 1 identity (Din == Dout), 2 Conv1d(k = 5, pad = 2) with
// conv_w [Dout, 5, Din] (tap-major rearrangement of the reference's [Dout, Din, 5]) and conv_b [Dout].
// adj [B, T, T] or null = the DistanceAdj adjacency, evaluated as a bidirectional first-order scan over T
// (O(T.D) instead of O(T^2.D); SURVEY.md F3).
int graph_convolution(const float* x, const float* adj, const float* wt, const float* bias, int residual,
                      const float* conv_w, const float* conv_b, long long B, int T, int Din, int Dout, int plan,
                      float* out, int num_sms, cudaStream_t stream);

// y[b, t, :] = sum_k r^|t - k| s[b, k, :], r = exp(-1 / e): the DistanceAdj product as forward + backward scans.
int distance_scan(const float* s, long long B, int T, int D, float* y, cudaStream_t stream);

struct ResBlockParams {   // one ResidualAttentionBlock, model/module.py:20-43 (fp32 device pointers)
  const float *ln1_w, *ln1_b, *in_w, *in_b, *out_w, *out_b, *ln2_w, *ln2_b, *fc_w, *fc_b, *proj_w, *proj_b;
};

// Transformer.forward, model/module.py:46-54, on SEQ-FIRST x [L, N, D] like the reference: `layers` pre-LN blocks
// x += MHA(LN1 x); x += c_proj(QuickGELU(c_fc(LN2 x))).  attn_mask: optional additive [L, L]; key_pad: optional
// [N, L] uint8 (non-zero = ignore).  out [L, N, D].  plan: -1 fp32 FFMA, 0 bf16, 1 split-bf16, 2 fp16 operands.
int transformer(const float* x, const ResBlockParams* blocks, int layers, int L, int N, int D, int heads,
                const float* attn_mask, const uint8_t* key_pad, int plan, float* out, int num_sms,
                cudaStream_t stream);

// The block loop of `transformer` on a BATCH-FIRST fp32 residual x [N, L, D], updated in place (the residual stays
// fp32 under every plan).  Arguments as `transformer`, already validated by the caller.
int transformer_blocks(float* x, const ResBlockParams* blocks, int layers, int L, int N, int D, int heads,
                       const float* attn_mask, const uint8_t* key_pad, int plan, int num_sms, cudaStream_t stream);

}  // namespace iefvad
