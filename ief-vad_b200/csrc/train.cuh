// Internal interface of the training-step kernels (train.cu, train_attn.cu, train_loss.cu): SURVEY 8f row N3.
#pragma once
#include "common.cuh"
#include "philox.cuh"

namespace iefvad {

// Training attention (train_attn.cu).  The head sizes the kernels are built for: 32, 64, 96 and 128.
bool attn_train_supported(int dh);
// softmax(q k^T / sqrt(dh)) v with attention dropout of mode `drop` (philox.cuh: dropout_philox / dropout_torch; its T is
// set here).  qkv [B*T, 3*H*dh] fp32 (bias added, q unscaled) -> out [B*T, H*dh], lse [B, H, T]
int attn_train_fwd(const float* qkv, int B, int T, int H, int dh, DropoutDesc drop, float* out, float* lse, cudaStream_t stream);
// dqkv [B*T, 3*H*dh] from dout [B*T, H*dh]; delta_scratch: B*H*T floats
int attn_train_bwd(const float* qkv, const float* out, const float* dout, const float* lse, int B, int T, int H, int dh,
                   DropoutDesc drop, float* delta_scratch, float* dqkv, int num_sms, cudaStream_t stream);
// mask [B*H, T, T] uint8 (1 = kept) of mode `drop`: the keep decisions the attention kernels make, in torch's layout
int dropout_mask(DropoutDesc drop, int B, int H, int T, uint8_t* mask, cudaStream_t stream);

int train_colsum_blocks(long long rows, int num_sms);
// scratch: 2 * rows + 2 * train_colsum_blocks(rows) * D floats
int layernorm_bwd(const float* x, const float* gamma, const float* dy, long long rows, int D, float eps, float* dx, float* dgamma,
                  float* dbeta, float* scratch, int num_sms, cudaStream_t stream);
// out[c] = sum_r a[r, c] (* wgt[r] when wgt != null); scratch: 2 * train_colsum_blocks(rows) * D floats
int colsum(const float* a, const float* wgt, long long rows, int D, float* out, float* scratch, int num_sms, cudaStream_t stream);
// every g_* may be null (= zero upstream gradient)
int fuse_bwd(const float* mu_i, const float* mu_e, const float* lv_i, const float* lv_e, const float* g_fused, const float* g_wi,
             const float* g_we, const float* g_mu_i, const float* g_mu_e, const float* g_lv_i, const float* g_lv_e, long long n,
             float factor, float eps, float* d_mu_i, float* d_mu_e, float* d_lv_i, float* d_lv_e, int num_sms, cudaStream_t stream);
int relu_bwd(const float* dh, const float* h, long long n, float* out, int num_sms, cudaStream_t stream);
int quickgelu(const float* x, long long n, float* out, int num_sms, cudaStream_t stream);
int axpy(float* y, const float* x, float alpha, long long n, int num_sms, cudaStream_t stream);
int outer(const float* a, const float* w, long long rows, int D, float* out, int num_sms, cudaStream_t stream);
int transpose_f32(const float* src, long long rows, int cols, float* dst, long long ld_dst, cudaStream_t stream);
// dst_hi / dst_lo [cols, ld_dst] = bf16 hi / lo split of src^T (src [rows, cols] fp32), columns [rows, ld_dst) zero
int transpose_split(const float* src, long long rows, int cols, bf16* dst_hi, bf16* dst_lo, long long ld_dst, cudaStream_t stream);
int clas2_bwd(const float* logits, const float* means, const float* labels, long long label_stride, const int* idx, int B, int T,
              int kmax, const float* g_loss, float* dlogits, cudaStream_t stream);

// Training objective of train/ucf_train.py:73-102 (train_loss.cu): CLAS2 + cosine / norm regulariser + StudentT KL.
// record: [B*T, 4] float64 for the backward; slab_scratch: 2 * train_loss_slabs(B*T) doubles; D % 4 == 0, 16-byte aligned rows.
int train_loss_slabs(long long rows);
int train_loss_fwd(const float* logits, const float* labels, long long label_stride, const long long* lengths, int B, int T,
                   const float* mu_i, const float* mu_e, const float* lv_i, const float* lv_e, int D, double nu, double reg_w,
                   double kl_w, float* means, int* idx, int kmax, double* record, double* slab_scratch, float* total,
                   float* loss_cls, float* loss_reg, float* loss_kl, cudaStream_t stream);
// g_*: device scalars, null = 0; g_cls_scratch: one device float (CLAS2's coefficient g_total + g_cls)
int train_loss_bwd(const float* logits, const float* means, const float* labels, long long label_stride, const int* idx, int B,
                   int T, int kmax, const float* mu_i, const float* mu_e, const float* lv_i, const float* lv_e, int D,
                   const double* record, double nu, double reg_w, double kl_w, const float* g_total, const float* g_cls,
                   const float* g_reg, const float* g_kl, float* g_cls_scratch, float* d_logits, float* d_mu_i, float* d_mu_e,
                   float* d_lv_i, float* d_lv_e, cudaStream_t stream);

}  // namespace iefvad
