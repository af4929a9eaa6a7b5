#pragma once
#include "common.cuh"

namespace iefvad {

// train/loss.py:24-27: mean of the top int(len/16 + 1) values of x[row, :len] (after an optional sigmoid).
// idx (optional, [B, kmax], -1 padded): the selected positions, descending value, ties by ascending index.
int mil_topk_mean(const float* x, const long long* lengths, long long B, long long T, int apply_sigmoid, float* mean,
                  int* idx, int kmax, cudaStream_t stream);

// train/loss.py:18-30 (CLAS2): per-row means + scalar BCE loss against 1 - labels[:, 0]; idx (optional, [B, kmax]):
// the top-k positions as in mil_topk_mean, for the backward
int clas2(const float* logits, const float* labels, long long label_stride, const long long* lengths, long long B,
          long long T, float* means, float* loss, cudaStream_t stream, int* idx = nullptr, int kmax = 0);

// stable descending argsort of fp32 scores (== np.argsort(-s, kind="stable")); keys_sorted optional
int sort_scores(const float* scores, long long n, int* order, uint32_t* keys_sorted, cudaStream_t stream);

// out[0] = roc_auc_score, out[1] = average_precision_score of np.repeat(scores, repeat) against labels with pos[j]
// positives among segment j's `repeat` frames; out[2], out[3] = #positive / #negative frames.  out: device double[4].
int auc_ap(const float* scores, const int* pos, long long n, int repeat, double* out, int* order_out,
           cudaStream_t stream);

// The same for `nsub` <= 32 subsets of the segments at once (class-wise AUC / AP and Ano-AUC, train/ucf_test.py:164-178,
// 336-353): bit s of member[j] = segment j belongs to subset s; out: device double[nsub][4].  One sort for all.
int auc_ap_multi(const float* scores, const int* pos, const uint32_t* member, long long n, int repeat, int nsub,
                 double* out, int* order_out, cudaStream_t stream);

// dst[dst_off[s] + i] = src[src_off[s] + i] for i < len[s]; all index arrays on the device
int segment_copy(const float* src, const long long* src_off, float* dst, const long long* dst_off,
                 const long long* len, long long nseg, cudaStream_t stream);

}  // namespace iefvad
