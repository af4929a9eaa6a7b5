// extern "C" surface declared in include/iefvad.h.
#include "../../include/iefvad.h"

#include <cmath>
#include <new>
#include <string>
#include <vector>

#include "attention.cuh"
#include "clip.cuh"
#include "elementwise.cuh"
#include "event.cuh"
#include "gemm.cuh"
#include "graph.cuh"
#include "locmap.cuh"
#include "model.cuh"
#include "rank.cuh"
#include "shaping.cuh"
#include "outproj_ln.cuh"
#include "train.cuh"

namespace iefvad {
const char* last_error();
}

using namespace iefvad;

struct iefvad_model {
  Model impl;
  // scratch of the host-input forward: ping-pong input buffers filled on a copy stream while the previous part computes
  DevBuf host_in[2][2], host_out[5], host_logits, host_scores;   // host_out: fused, mu x2, logvar x2 (scratch)
  cudaStream_t copy_stream = nullptr;
  cudaEvent_t ev_copied[2] = {nullptr, nullptr}, ev_consumed[2] = {nullptr, nullptr}, ev_start = nullptr;
  // optional extra outputs of the evaluation forward (iefvad_model_set_eval_outputs): compact DEVICE buffers of the caller
  float* ex_wi_mean = nullptr;
  float* ex_we_mean = nullptr;
  float* ex_wide[3] = {nullptr, nullptr, nullptr};      // fused, image_mu, event_mu
  int64_t host_part_rows = 32768;
  uint64_t host_seq = 0;          // parts issued so far: the ping-pong of the input buffers continues across calls
};

extern "C" {

int iefvad_abi_version(void) { return IEFVAD_ABI_VERSION; }
const char* iefvad_last_error(void) { return iefvad::last_error(); }

int iefvad_model_create(iefvad_model** out, int embed_dim, int num_heads, int num_layers, int num_refinement_steps,
                        float lambda_ref, int noise_model, float nu, float epsilon) {
  IEF_CHECK(out != nullptr, "iefvad_model_create: null output pointer");
  *out = nullptr;
  iefvad_model* m = new (std::nothrow) iefvad_model();
  IEF_CHECK(m != nullptr, "out of host memory");
  int rc = m->impl.init(embed_dim, num_heads, num_layers, num_refinement_steps, lambda_ref, noise_model, nu, epsilon);
  if (rc != 0) {
    m->impl.destroy();
    delete m;
    return rc;
  }
  *out = m;
  return IEFVAD_OK;
}

void iefvad_model_destroy(iefvad_model* m) {
  if (!m) return;
  m->impl.destroy();
  for (auto& pp : m->host_in) for (auto& b : pp) b.release();
  for (auto& b : m->host_out) b.release();
  if (m->copy_stream) cudaStreamDestroy(m->copy_stream);
  for (int i = 0; i < 2; ++i) {
    if (m->ev_copied[i]) cudaEventDestroy(m->ev_copied[i]);
    if (m->ev_consumed[i]) cudaEventDestroy(m->ev_consumed[i]);
  }
  if (m->ev_start) cudaEventDestroy(m->ev_start);
  m->host_logits.release();
  m->host_scores.release();
  delete m;
}

int iefvad_model_set_param(iefvad_model* m, const char* key, const float* data, int64_t numel, void* stream) {
  IEF_CHECK(m && key && data, "iefvad_model_set_param: null argument");
  return m->impl.set_param(key, data, numel, static_cast<cudaStream_t>(stream));
}

int iefvad_model_set_plan(iefvad_model* m, int plan) {
  IEF_CHECK(m, "null model");
  IEF_CHECK(plan == IEFVAD_PLAN_HH || plan == IEFVAD_PLAN_B || plan == IEFVAD_PLAN_FP32,
            "unknown precision plan %d: choose IEFVAD_PLAN_HH (56), IEFVAD_PLAN_B (6) or IEFVAD_PLAN_FP32 (-1)", plan);
  m->impl.plan = plan;
  return IEFVAD_OK;
}

int iefvad_model_get_plan(const iefvad_model* m) { return m ? m->impl.plan : 0; }

int iefvad_model_set_option(iefvad_model* m, const char* name, int64_t value) {
  IEF_CHECK(m && name, "iefvad_model_set_option: null argument");
  const std::string key(name);
  if (key == "refine_fused") {
    IEF_CHECK(value >= -1 && value <= 1, "refine_fused: -1 (auto), 0 (off), 1 (on)");
    m->impl.refine_fused = int(value);
  } else if (key == "heads_fuse") {
    IEF_CHECK(value == 0 || value == 1, "heads_fuse: 0 (heads GEMMs + fusion kernel) or 1 (one kernel)");
    m->impl.heads_fuse_mode = int(value);
  } else if (key == "outproj_ln") {
    IEF_CHECK(value == 0 || value == 1, "outproj_ln: 0 (separate GEMM + LayerNorm launches) or 1 (one kernel)");
    m->impl.outproj_ln_mode = int(value);
  } else {
    set_error("iefvad_model_set_option: unknown option '%s'", name);
    return IEFVAD_ERR_INVALID;
  }
  return IEFVAD_OK;
}

int iefvad_model_check_finite(iefvad_model* m, int* nonfinite_host, void* stream) {
  IEF_CHECK(m && nonfinite_host, "iefvad_model_check_finite: null argument");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  int flags[4] = {0, 0, 0, 0};
  IEF_CUDA(cudaMemcpyAsync(flags, m->impl.status.p, sizeof(flags), cudaMemcpyDeviceToHost, st));
  IEF_CUDA(cudaMemsetAsync(m->impl.status.p, 0, sizeof(flags), st));
  IEF_CUDA(cudaStreamSynchronize(st));
  *nonfinite_host = flags[0];
  return IEFVAD_OK;
}

int iefvad_model_set_max_rows(iefvad_model* m, int64_t max_rows) {
  IEF_CHECK(m && max_rows >= 1, "iefvad_model_set_max_rows: need a model and max_rows >= 1");
  m->impl.max_rows = max_rows;
  return IEFVAD_OK;
}

int iefvad_model_forward(iefvad_model* m, const void* img, const void* ev, int in_dtype, int64_t B, int64_t T,
                         float* fused, float* logits, float* image_mu, float* event_mu, float* image_logvar,
                         float* event_logvar, float* w_i, float* w_e, float* scores, void* stream) {
  IEF_CHECK(m, "null model");
  IEF_CHECK(in_dtype >= 0 && in_dtype <= 2, "unsupported input dtype code %d", in_dtype);
  return m->impl.forward(img, ev, in_dtype, B, T, fused, logits, image_mu, event_mu, image_logvar, event_logvar, w_i,
                         w_e, scores, static_cast<cudaStream_t>(stream));
}

// Host-input forward, pipelined: the batch is cut into parts of whole batch elements; part p + 1 travels host -> device
// on the library's copy stream into the other input buffer while part p computes on the caller's stream, so only the
// first part's copy is exposed (the copy engine outruns the forward: ~18 k rows/ms over PCIe vs ~12 k rows/ms).
static int forward_from_host(iefvad_model* m, const void* img_host, const void* ev_host, int in_dtype, int64_t B,
                             int64_t T, float* logits_host, float* scores_host, float* logits_dev, float* scores_dev,
                             cudaStream_t st, const int64_t* valid_len_host = nullptr, const int32_t* rowmap = nullptr,
                             const int64_t* chunk_start_dev = nullptr, const int32_t* chunk_valid_dev = nullptr) {
  IEF_CHECK(m && img_host && ev_host, "host-input forward: null argument");
  IEF_CHECK(in_dtype >= 0 && in_dtype <= 2, "unsupported input dtype code %d", in_dtype);
  IEF_CHECK(B >= 0 && T >= 0, "negative batch / length");
  if (B == 0 || T == 0) return IEFVAD_OK;
  const int D = m->impl.D;
  const size_t es = (in_dtype == IEFVAD_F32) ? 4 : 2;
  // Part sizes grow geometrically from a small first part (short exposed copy) to large later parts (full GEMM grids):
  // x 1.4 from host_part_rows / 4 for dense chunks (the copy engine leads the forward by about that factor), x 3 from
  // host_part_rows / 8 for ragged inputs (no pad rows on the wire: the copy is twice as fast as the forward).
  const int64_t cap_rows = m->impl.max_rows;
  std::vector<int64_t> partsB;
  {
    const bool ragged_in = chunk_start_dev != nullptr;
    double growth = ragged_in ? 3.0 : 1.4;
    double want = double(m->host_part_rows) / (ragged_in ? 8.0 : 4.0);
    // Back-to-back calls: the previous call's last part is still computing, so this call's copy hides behind it
    // whatever its size - the whole batch then travels as ONE part into the other input buffer (full GEMM grids; a
    // small first part only pays when the device is idle at the call).
    if (m->host_seq > 0 && m->ev_consumed[(m->host_seq - 1) & 1] &&
        cudaEventQuery(m->ev_consumed[(m->host_seq - 1) & 1]) == cudaErrorNotReady) {
      (void)cudaGetLastError();            // cudaErrorNotReady is a status, not a failure: keep it out of the next check
      want = double(B * T);
      growth = 1.0;
    }
    int64_t left = B;
    while (left > 0) {
      int64_t pb = int64_t(want / double(T));
      if (pb < 1) pb = 1;
      if (pb * T > cap_rows) pb = cap_rows / T > 0 ? cap_rows / T : 1;
      if (pb > left || left - pb < pb / 4) pb = left;      // fold a small tail into the last part
      if (pb * T > cap_rows && left > pb) pb = left;         // (keeps the invariant below simple)
      partsB.push_back(pb);
      left -= pb;
      want *= growth;
    }
  }
  int64_t maxB = 0;
  for (int64_t pb : partsB) maxB = pb > maxB ? pb : maxB;
  // the input buffers are sized for the one-part schedule of back-to-back calls from the start: growing them later
  // would put a cudaFree / cudaMalloc (a device-wide synchronisation) into the middle of a pipelined loop
  const int64_t fullB = (B * T <= cap_rows) ? B : maxB;
  const size_t rows = size_t(fullB > maxB ? fullB : maxB) * T;
  if (!m->copy_stream) {
    IEF_CUDA(cudaStreamCreateWithFlags(&m->copy_stream, cudaStreamNonBlocking));
    for (int i = 0; i < 2; ++i) {
      IEF_CUDA(cudaEventCreateWithFlags(&m->ev_copied[i], cudaEventDisableTiming));
      IEF_CUDA(cudaEventCreateWithFlags(&m->ev_consumed[i], cudaEventDisableTiming));
    }
    IEF_CUDA(cudaEventCreateWithFlags(&m->ev_start, cudaEventDisableTiming));
  }
  for (auto& pp : m->host_in) for (auto& b : pp) IEF_TRY(b.reserve(rows * D * es));
  for (auto& b : m->host_out) IEF_TRY(b.reserve(rows * D * 4));
  IEF_CHECK((valid_len_host == nullptr) == (rowmap == nullptr), "valid-rows mode needs both the host lengths and the device row map");
  IEF_CHECK(valid_len_host == nullptr || (logits_host == nullptr && scores_host == nullptr),
            "valid-rows mode returns compact DEVICE results");
  const bool ragged = chunk_start_dev != nullptr;
  IEF_CHECK((chunk_start_dev == nullptr) == (chunk_valid_dev == nullptr), "ragged inputs need chunk_start and chunk_valid");
  IEF_CHECK(!ragged || valid_len_host, "ragged inputs need the valid-rows descriptors");
  if (!logits_dev) IEF_TRY(m->host_logits.reserve(size_t(B) * T * 4));
  if (!scores_dev && scores_host) IEF_TRY(m->host_scores.reserve(size_t(B) * T * 4));
  float* ldev = logits_dev ? logits_dev : m->host_logits.as<float>();
  float* sdev = scores_dev ? scores_dev : (scores_host ? m->host_scores.as<float>() : nullptr);
  cudaStream_t cs = m->copy_stream;
  // The copy stream only waits for the last forward that READ the buffer it is about to overwrite (ev_consumed, which
  // persists across calls) - not for everything queued on the caller's stream - so in a loop of calls the first
  // part of call k+1 already travels while call k is still computing its last part (and the caller's metrics).
  int64_t b0 = 0;
  size_t j0 = 0;                       // compact output offset (valid-rows mode)
  for (int p = 0; p < int(partsB.size()); b0 += partsB[p], ++p) {
    const int buf = int(m->host_seq++ & 1);
    const int64_t Bs = partsB[p];
    const size_t r0 = size_t(b0) * T, nr = size_t(Bs) * T;
    ValidRows vr;
    size_t nvalid = 0;
    if (valid_len_host) {
      for (int64_t b = b0; b < b0 + Bs; ++b) nvalid += size_t(valid_len_host[b] < 0 ? 0 : valid_len_host[b]);
      vr.len_host = reinterpret_cast<const long long*>(valid_len_host) + b0;
      vr.rowmap = rowmap + j0;
      vr.row_base = static_cast<long long>(r0);
    }
    const size_t o0 = valid_len_host ? j0 : r0;
    IEF_CUDA(cudaStreamWaitEvent(cs, m->ev_consumed[buf], 0));      // no-op until the event has been recorded once
    // ragged: the host buffers hold only the valid rows, chunk after chunk - this part's rows are [j0, j0 + nvalid)
    const size_t src0 = ragged ? j0 : r0, nsrc = ragged ? nvalid : nr;
    if (ragged) {
      vr.chunk_start = reinterpret_cast<const long long*>(chunk_start_dev) + b0;
      vr.chunk_valid = chunk_valid_dev + b0;
      vr.start_base = static_cast<long long>(j0);
    }
    if (nsrc) {
      IEF_CUDA(cudaMemcpyAsync(m->host_in[buf][0].p, static_cast<const uint8_t*>(img_host) + src0 * D * es, nsrc * D * es,
                               cudaMemcpyHostToDevice, cs));
      IEF_CUDA(cudaMemcpyAsync(m->host_in[buf][1].p, static_cast<const uint8_t*>(ev_host) + src0 * D * es, nsrc * D * es,
                               cudaMemcpyHostToDevice, cs));
    }
    IEF_CUDA(cudaEventRecord(m->ev_copied[buf], cs));
    IEF_CUDA(cudaStreamWaitEvent(st, m->ev_copied[buf], 0));
    float* o[5];
    for (int i = 0; i < 5; ++i) o[i] = m->host_out[i].as<float>();
    for (int i = 0; i < 3; ++i)
      if (m->ex_wide[i]) o[i] = m->ex_wide[i] + o0 * D;               // the caller wants this tensor: write it there
    m->impl.eval_wi_mean = m->ex_wi_mean ? m->ex_wi_mean + o0 : nullptr;
    m->impl.eval_we_mean = m->ex_we_mean ? m->ex_we_mean + o0 : nullptr;
    m->impl.heads_outputs_unused = !m->ex_wide[1] && !m->ex_wide[2];      // mu / logvar land in scratch: nobody reads them
    const int frc = m->impl.forward(m->host_in[buf][0].p, m->host_in[buf][1].p, in_dtype, Bs, T, o[0], ldev + o0, o[1], o[2], o[3],
                                    o[4], nullptr, nullptr, sdev ? sdev + o0 : nullptr, st, valid_len_host ? &vr : nullptr);
    m->impl.eval_wi_mean = m->impl.eval_we_mean = nullptr;
    m->impl.heads_outputs_unused = false;
    IEF_TRY(frc);
    j0 += nvalid;
    IEF_CUDA(cudaEventRecord(m->ev_consumed[buf], st));
    if (logits_host) IEF_CUDA(cudaMemcpyAsync(logits_host + r0, ldev + r0, nr * 4, cudaMemcpyDeviceToHost, st));
    if (scores_host) IEF_CUDA(cudaMemcpyAsync(scores_host + r0, sdev + r0, nr * 4, cudaMemcpyDeviceToHost, st));
  }
  return IEFVAD_OK;
}

int iefvad_model_forward_host(iefvad_model* m, const void* img_host, const void* ev_host, int in_dtype, int64_t B,
                              int64_t T, float* logits_host, float* scores_host, void* stream) {
  IEF_CHECK(logits_host, "iefvad_model_forward_host: null logits_host");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  IEF_TRY(forward_from_host(m, img_host, ev_host, in_dtype, B, T, logits_host, scores_host, nullptr, nullptr, st));
  IEF_CUDA(cudaStreamSynchronize(st));
  return IEFVAD_OK;
}

int iefvad_model_forward_host_to_device(iefvad_model* m, const void* img_host, const void* ev_host, int in_dtype,
                                        int64_t B, int64_t T, float* logits, float* scores, void* stream) {
  IEF_CHECK(logits, "iefvad_model_forward_host_to_device: null logits");
  return forward_from_host(m, img_host, ev_host, in_dtype, B, T, nullptr, nullptr, logits, scores,
                           static_cast<cudaStream_t>(stream));
}

int iefvad_model_forward_scores_ragged(iefvad_model* m, const void* img_packed_host, const void* ev_packed_host,
                                       int in_dtype, int64_t B, int64_t T, const int64_t* valid_len_host,
                                       const int32_t* rowmap, const int64_t* chunk_start, const int32_t* chunk_valid,
                                       float* logits, float* scores, void* stream) {
  IEF_CHECK(m && img_packed_host && ev_packed_host && logits && valid_len_host && rowmap && chunk_start && chunk_valid,
            "iefvad_model_forward_scores_ragged: null argument");
  return forward_from_host(m, img_packed_host, ev_packed_host, in_dtype, B, T, nullptr, nullptr, logits, scores,
                           static_cast<cudaStream_t>(stream), valid_len_host, rowmap, chunk_start, chunk_valid);
}

int iefvad_model_forward_scores(iefvad_model* m, const void* img, const void* ev, int in_dtype, int inputs_on_host,
                                int64_t B, int64_t T, const int64_t* valid_len_host, const int32_t* rowmap,
                                float* logits, float* scores, void* stream) {
  IEF_CHECK(m && img && ev && logits, "iefvad_model_forward_scores: null argument");
  IEF_CHECK(in_dtype >= 0 && in_dtype <= 2, "unsupported input dtype code %d", in_dtype);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (inputs_on_host)
    return forward_from_host(m, img, ev, in_dtype, B, T, nullptr, nullptr, logits, scores, st, valid_len_host, rowmap);
  IEF_CHECK((valid_len_host == nullptr) == (rowmap == nullptr), "valid-rows mode needs both the host lengths and the device row map");
  IEF_CHECK(B >= 0 && T >= 0, "negative batch / length");
  if (B == 0 || T == 0) return IEFVAD_OK;
  size_t rows = size_t(B) * T;
  ValidRows vr;
  if (valid_len_host) {
    rows = 0;
    for (int64_t b = 0; b < B; ++b) rows += size_t(valid_len_host[b] < 0 ? 0 : valid_len_host[b]);
    vr.len_host = reinterpret_cast<const long long*>(valid_len_host);
    vr.rowmap = rowmap;
  }
  for (auto& b : m->host_out) IEF_TRY(b.reserve((rows ? rows : 1) * m->impl.D * 4));
  float* o[5];
  for (int i = 0; i < 5; ++i) o[i] = m->host_out[i].as<float>();
  for (int i = 0; i < 3; ++i)
    if (m->ex_wide[i]) o[i] = m->ex_wide[i];
  m->impl.eval_wi_mean = m->ex_wi_mean;
  m->impl.eval_we_mean = m->ex_we_mean;
  m->impl.heads_outputs_unused = !m->ex_wide[1] && !m->ex_wide[2];
  const int rc = m->impl.forward(img, ev, in_dtype, B, T, o[0], logits, o[1], o[2], o[3], o[4], nullptr, nullptr, scores, st,
                                 valid_len_host ? &vr : nullptr);
  m->impl.eval_wi_mean = m->impl.eval_we_mean = nullptr;
  m->impl.heads_outputs_unused = false;
  return rc;
}

int iefvad_model_set_eval_outputs(iefvad_model* m, float* wi_mean, float* we_mean, float* fused, float* image_mu,
                                  float* event_mu) {
  IEF_CHECK(m, "null model");
  IEF_CHECK((wi_mean == nullptr) == (we_mean == nullptr), "iefvad_model_set_eval_outputs: wi_mean and we_mean go together");
  m->ex_wi_mean = wi_mean;
  m->ex_we_mean = we_mean;
  m->ex_wide[0] = fused;
  m->ex_wide[1] = image_mu;
  m->ex_wide[2] = event_mu;
  return IEFVAD_OK;
}

int iefvad_model_set_pad_dedup(iefvad_model* m, int on) {
  IEF_CHECK(m, "null model");
  m->impl.pad_dedup = on != 0;
  return IEFVAD_OK;
}

int iefvad_model_set_host_part_rows(iefvad_model* m, int64_t rows) {
  IEF_CHECK(m && rows >= 1, "iefvad_model_set_host_part_rows: need a model and rows >= 1");
  m->host_part_rows = rows;
  return IEFVAD_OK;
}

// ------------------------------------------------------------------------------------------------ operators

int iefvad_fuse(const float* mu_i, const float* mu_e, const float* logvar_i, const float* logvar_e, int64_t n,
                float factor, float epsilon, float* w_i, float* w_e, float* fused, void* stream) {
  IEF_CHECK(mu_i && mu_e && logvar_i && logvar_e && w_i && w_e, "iefvad_fuse: null argument");
  int sms = 0;
  IEF_TRY(device_sms(&sms));
  return fuse(mu_i, mu_e, logvar_i, logvar_e, n, factor, epsilon, w_i, w_e, fused, nullptr, nullptr, sms,
              static_cast<cudaStream_t>(stream));
}

int iefvad_layernorm(const float* x, int64_t rows, int dim, const float* w1, const float* b1, const float* w2,
                     const float* b2, float eps, float* out, void* stream) {
  IEF_CHECK(x && out, "iefvad_layernorm: null argument");
  int sms = 0;
  IEF_TRY(device_sms(&sms));
  return layernorm(x, rows, dim, w1, b1, w2, b2, eps, out, nullptr, nullptr, sms, static_cast<cudaStream_t>(stream));
}

int iefvad_linear(const float* x, const float* w, const float* bias, const float* resid, float alpha, int act,
                  int64_t rows, int in_f, int out_f, int plan, int tile_n, float* out, void* stream) {
  IEF_CHECK(x && w && out, "iefvad_linear: null argument");
  IEF_CHECK(rows >= 0 && rows < (1LL << 31), "iefvad_linear: bad row count");
  IEF_TRY(check_plan("iefvad_linear", plan));
  if (rows == 0) return IEFVAD_OK;
  IEF_CHECK(plan < 0 || ((rows * in_f) % 8 == 0 && (int64_t(out_f) * in_f) % 8 == 0),
            "iefvad_linear: sizes must be multiples of 8");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  int sms = 0;
  IEF_TRY(device_sms(&sms));
  EpiParams ep;
  ep.bias = bias; ep.act = act; ep.resid = resid; ep.ld_resid = out_f; ep.alpha = alpha;
  ep.out_f32 = out; ep.ld_f32 = out_f;
  Scratch sc(st);
  Mat xm, wm;
  IEF_TRY(to_mat(sc, &xm, x, int(rows), in_f, in_f, int(rows), in_f, plan, sms, st));
  IEF_TRY(to_mat(sc, &wm, w, out_f, in_f, in_f, out_f, in_f, plan, sms, st));
  if (plan < 0) return gemm_plan(plan, xm, wm, int(rows), out_f, in_f, ep, nullptr, sms, st);
  GemmTcArgs g = tc_args(plan, xm, wm, int(rows), out_f, in_f);
  g.force_bn = tile_n == 512 ? 256 : tile_n;          // 512 = 256-column tiles on CTA pairs
  g.force_cg = tile_n == 512 ? 2 : (tile_n ? 1 : 0);
  return gemm_tc_split_k(g, ep, sc, sms, st);
}

int iefvad_outproj_ln(const float* ctx, const float* w, const float* bias, const float* resid, const float* ln_w,
                      const float* ln_b, const float* ln2_w, const float* ln2_b, float eps, int64_t rows,
                      const int32_t* row_map, void* out_hi_f16, void* out_lo_f16, void* stream) {
  IEF_CHECK(ctx && w && bias && resid && ln_w && ln_b && out_hi_f16, "iefvad_outproj_ln: null argument");
  IEF_CHECK(rows >= 0 && rows < (1LL << 31) - 256, "iefvad_outproj_ln: bad row count");
  if (rows == 0) return IEFVAD_OK;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  int sms = 0;
  IEF_TRY(device_sms(&sms));
  constexpr int D = kOutprojLnDim;
  Scratch sc(st);
  uint8_t *scr = nullptr, *idt = nullptr;
  bf16 *ch = nullptr, *wh = nullptr, *rh = nullptr, *rl = nullptr;
  IEF_TRY(sc.get(&idt, outproj_ln_identity_bytes()));
  IEF_TRY(outproj_ln_identity(idt, st));
  IEF_TRY(sc.get(&ch, size_t(rows) * D));
  IEF_TRY(sc.get(&wh, size_t(D) * D));
  IEF_TRY(sc.get(&rh, size_t(rows) * D));
  IEF_TRY(sc.get(&rl, size_t(rows) * D));
  IEF_TRY(sc.get(&scr, outproj_ln_scratch_bytes(rows)));
  IEF_TRY(to_half(ctx, rows * D, ch, sms, st));
  IEF_TRY(to_half(w, int64_t(D) * D, wh, sms, st));
  IEF_TRY(ingest(resid, IEFVAD_DT_F32, rows * D, nullptr, rh, rl, sms, st, 1));
  OutprojLnArgs a;
  a.ctx = ch; a.w16 = wh; a.bias = bias; a.res_hi = rh; a.res_lo = rl; a.ln_w = ln_w; a.ln_b = ln_b; a.ln2_w = ln2_w;
  a.ln2_b = ln2_b; a.eps = eps; a.out_hi = out_hi_f16; a.out_lo = out_lo_f16; a.row_map = row_map; a.M = rows; a.scratch = scr;
  a.identity = idt;
  return outproj_ln(a, sms, st);
}

int iefvad_mha(const float* x, const float* in_w, const float* in_b, const float* out_w, const float* out_b,
               int64_t B, int64_t T, int D, int num_heads, const float* attn_mask, const uint8_t* key_padding_mask,
               int plan, float* out, void* stream) {
  IEF_CHECK(x && in_w && in_b && out_w && out_b && out, "iefvad_mha: null argument");
  IEF_CHECK(num_heads > 0 && D % num_heads == 0, "iefvad_mha: heads must divide D");
  IEF_TRY(check_plan("iefvad_mha", plan));
  IEF_CHECK(B >= 0 && T >= 0 && B * T < (1LL << 31), "iefvad_mha: bad sizes");
  if (B == 0 || T == 0) return IEFVAD_OK;
  IEF_CHECK(plan < 0 || D % 64 == 0, "iefvad_mha: tensor-core plans need D %% 64 == 0");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  int sms = 0;
  IEF_TRY(device_sms(&sms));
  const int M = int(B * T);
  Scratch sc(st);
  Mat xm, iw, ow;
  AttnWork aw;
  IEF_TRY(to_mat(sc, &xm, x, M, D, D, M, D, plan, sms, st));
  IEF_TRY(to_mat(sc, &iw, in_w, 3 * D, D, D, 3 * D, D, plan, sms, st));
  IEF_TRY(to_mat(sc, &ow, out_w, D, D, D, D, D, plan, sms, st));
  IEF_TRY(alloc_attn_work(sc, &aw, plan, int(B), int(T), D, num_heads));
  return attention_sublayer(plan, xm, iw, in_b, ow, out_b, int(B), int(T), D, num_heads, attn_mask, key_padding_mask,
                            nullptr, out, aw, sms, st);
}

int iefvad_attention_core(const void* q, const void* k, const void* vt, int64_t B, int64_t T, int H, int dh, int dhp,
                          int64_t Tpad, const float* attn_mask, const uint8_t* key_pad, const int32_t* row_out,
                          const int32_t* items, int n_chunks, int fp16, void* out, int64_t ldo, void* stream) {
  IEF_CHECK(q && k && vt && out, "iefvad_attention_core: null argument");
  IEF_CHECK(((reinterpret_cast<uintptr_t>(q) | reinterpret_cast<uintptr_t>(k) | reinterpret_cast<uintptr_t>(vt) |
              reinterpret_cast<uintptr_t>(out)) & 15) == 0, "iefvad_attention_core: q, k, vt and out must be 16-byte aligned");
  IEF_CHECK(B > 0 && T > 0 && H > 0 && B * H * T < (1LL << 31), "iefvad_attention_core: bad sizes B=%lld T=%lld H=%d",
            (long long)B, (long long)T, H);
  IEF_CHECK(dh > 0 && dhp >= dh && dhp % 8 == 0, "iefvad_attention_core: need 0 < dh <= dhp, dhp %% 8 == 0 (dh=%d dhp=%d)",
            dh, dhp);
  IEF_CHECK(Tpad >= T && Tpad % 8 == 0 && Tpad < (1LL << 31), "iefvad_attention_core: Tpad=%lld must be a multiple of 8 "
            "and >= T=%lld", (long long)Tpad, (long long)T);
  IEF_CHECK(ldo >= int64_t(H) * dh && ldo % 8 == 0 && ldo < (1LL << 31), "iefvad_attention_core: ldo=%lld must be a "
            "multiple of 8 and >= H * dh", (long long)ldo);
  IEF_CHECK(fp16 == 0 || fp16 == 1, "iefvad_attention_core: fp16 must be 0 (bf16) or 1 (fp16)");
  IEF_CHECK(n_chunks >= 0 && (items != nullptr) == (n_chunks > 0), "iefvad_attention_core: items and n_chunks > 0 go "
            "together");
  IEF_CHECK(!items || (B == 1 && !attn_mask && !key_pad), "iefvad_attention_core: ragged items need B = 1 and no masks");
  AttnTcArgs at;
  at.q = static_cast<const bf16*>(q); at.k = static_cast<const bf16*>(k); at.vt = static_cast<const bf16*>(vt);
  at.out = static_cast<bf16*>(out); at.ldo = int(ldo);
  at.B = int(B); at.T = int(T); at.H = H; at.dh = dh; at.dhp = dhp; at.Tpad = int(Tpad);
  at.attn_mask = attn_mask; at.key_pad = key_pad; at.fp16 = fp16; at.row_out = row_out;
  at.items = items; at.n_chunks = n_chunks;
  return attn_tc(at, static_cast<cudaStream_t>(stream));
}

int iefvad_classifier(const float* x, int64_t rows, int dim, const float* w, const float* bias, float* logits,
                      float* scores, void* stream) {
  IEF_CHECK(x && w && bias && logits, "iefvad_classifier: null argument");
  int sms = 0;
  IEF_TRY(device_sms(&sms));
  return classifier(x, rows, dim, w, bias, logits, scores, sms, static_cast<cudaStream_t>(stream));
}

int iefvad_mil_topk_mean(const float* x, const int64_t* lengths, int64_t B, int64_t T, int apply_sigmoid, float* mean,
                         int32_t* idx, int kmax, void* stream) {
  return mil_topk_mean(x, reinterpret_cast<const long long*>(lengths), B, T, apply_sigmoid, mean, idx, kmax,
                       static_cast<cudaStream_t>(stream));
}

int iefvad_clas2(const float* logits, const float* labels, int64_t label_stride, const int64_t* lengths, int64_t B,
                 int64_t T, float* means, float* loss, void* stream) {
  return clas2(logits, labels, label_stride, reinterpret_cast<const long long*>(lengths), B, T, means, loss,
               static_cast<cudaStream_t>(stream));
}

int iefvad_sort_scores(const float* scores, int64_t n, int32_t* order, void* stream) {
  return sort_scores(scores, n, order, nullptr, static_cast<cudaStream_t>(stream));
}

int iefvad_auc_ap(const float* scores, const int32_t* pos, int64_t n, int repeat, double* out, int32_t* order,
                  void* stream) {
  return auc_ap(scores, pos, n, repeat, out, order, static_cast<cudaStream_t>(stream));
}

int iefvad_auc_ap_multi(const float* scores, const int32_t* pos, const uint32_t* member, int64_t n, int repeat,
                        int num_subsets, double* out, int32_t* order, void* stream) {
  return auc_ap_multi(scores, pos, member, n, repeat, num_subsets, out, order, static_cast<cudaStream_t>(stream));
}

int iefvad_segment_copy(const float* src, const int64_t* src_off, float* dst, const int64_t* dst_off,
                        const int64_t* len, int64_t nseg, void* stream) {
  return segment_copy(src, reinterpret_cast<const long long*>(src_off), dst,
                      reinterpret_cast<const long long*>(dst_off), reinterpret_cast<const long long*>(len), nseg,
                      static_cast<cudaStream_t>(stream));
}

// ------------------------------------------------------------------------------------------------ rows D1-D4

int iefvad_distance_adj(int64_t batch_size, int max_seqlen, float* out, void* stream) {
  return distance_adj(out, batch_size, max_seqlen, static_cast<cudaStream_t>(stream));
}

int iefvad_similarity_adj(const float* x, const float* weight0_t, const int64_t* seq_len_host, int64_t B, int T, int in_f,
                          int out_f, int plan, float* out, void* stream) {
  int sms = 0;
  IEF_TRY(device_sms(&sms));
  return similarity_adj(x, weight0_t, reinterpret_cast<const long long*>(seq_len_host), B, T, in_f, out_f, plan, out, sms,
                        static_cast<cudaStream_t>(stream));
}

int iefvad_graph_convolution(const float* x, const float* adj, const float* weight_t, const float* bias, int residual,
                             const float* conv_w, const float* conv_b, int64_t B, int T, int in_f, int out_f, int plan,
                             float* out, void* stream) {
  int sms = 0;
  IEF_TRY(device_sms(&sms));
  return graph_convolution(x, adj, weight_t, bias, residual, conv_w, conv_b, B, T, in_f, out_f, plan, out, sms,
                           static_cast<cudaStream_t>(stream));
}

int iefvad_distance_scan(const float* s, int64_t B, int T, int D, float* y, void* stream) {
  return distance_scan(s, B, T, D, y, static_cast<cudaStream_t>(stream));
}

int iefvad_transformer(const float* x, const float* const* params, int layers, int L, int N, int D, int heads,
                       const float* attn_mask, const uint8_t* key_padding_mask, int plan, float* out, void* stream) {
  IEF_CHECK(params != nullptr || layers == 0, "iefvad_transformer: null parameter table");
  IEF_CHECK(layers >= 0 && layers <= 64, "iefvad_transformer: 0..64 layers");
  int sms = 0;
  IEF_TRY(device_sms(&sms));
  std::vector<ResBlockParams> blocks(static_cast<size_t>(layers));
  for (int i = 0; i < layers; ++i) {
    const float* const* p = params + 12 * i;
    blocks[i] = ResBlockParams{p[0], p[1], p[2], p[3], p[4], p[5], p[6], p[7], p[8], p[9], p[10], p[11]};
  }
  return transformer(x, blocks.data(), layers, L, N, D, heads, attn_mask, key_padding_mask, plan, out, sms,
                     static_cast<cudaStream_t>(stream));
}

// ------------------------------------------------------------------------------------------------ row N4 (CLIP encoder)

int iefvad_clip_visual(const void* x, int dtype, int N, int resolution, int patch, int width, int layers, int heads,
                       int output_dim, const float* const* params, int plan, float* out, void* stream) {
  IEF_CHECK(params != nullptr, "iefvad_clip_visual: null parameter table");
  IEF_CHECK(layers >= 0 && layers <= 64, "iefvad_clip_visual: layers %d outside [0, 64]", layers);
  std::vector<ResBlockParams> blocks(static_cast<size_t>(layers));
  for (int i = 0; i < layers; ++i) {
    const float* const* p = params + 5 + 12 * i;
    blocks[i] = ResBlockParams{p[0], p[1], p[2], p[3], p[4], p[5], p[6], p[7], p[8], p[9], p[10], p[11]};
  }
  const float* const* tail = params + 5 + 12 * layers;
  const ClipVisualParams cp{params[0], params[1], params[2], params[3], params[4], blocks.data(), tail[0], tail[1], tail[2]};
  return clip_visual(x, dtype, N, resolution, patch, width, layers, heads, output_dim, cp, plan, out,
                     static_cast<cudaStream_t>(stream));
}

// ------------------------------------------------------------------------------------------------ row N2

int iefvad_process_split(const void* src, int dtype, const int64_t* row_off, int64_t V, int D, int length,
                         const int64_t* chunk_off, int64_t total_chunks, void* dst, int nan_to_num, void* stream) {
  IEF_CHECK(dtype >= 0 && dtype <= 2, "unsupported dtype code %d", dtype);
  return process_split(src, dtype, reinterpret_cast<const long long*>(row_off), V, D, length,
                       reinterpret_cast<const long long*>(chunk_off), total_chunks, dst, nan_to_num,
                       static_cast<cudaStream_t>(stream));
}

int iefvad_process_feat(const void* src, int dtype, const int64_t* row_off, int64_t V, int D, int length, float* dst,
                        int64_t* out_len, int nan_to_num, void* stream) {
  IEF_CHECK(dtype >= 0 && dtype <= 2, "unsupported dtype code %d", dtype);
  return process_feat(src, dtype, reinterpret_cast<const long long*>(row_off), V, D, length, dst,
                      reinterpret_cast<long long*>(out_len), nan_to_num, static_cast<cudaStream_t>(stream));
}

int iefvad_event_image(const uint8_t* frames, int64_t B, int C, int H, int W, float threshold, float clamp_max,
                       float* sum_out, float* event_out, void* stream) {
  IEF_CHECK(B >= 0 && C >= 1 && H >= 1 && W >= 1, "iefvad_event_image: bad shape");
  if (B == 0) return IEFVAD_OK;
  IEF_CHECK(frames, "iefvad_event_image: null frames");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  int sms = 0;
  IEF_TRY(device_sms(&sms));
  Scratch sc(st);
  float* cnt = nullptr;
  unsigned* mx = nullptr;
  IEF_TRY(sc.get(&cnt, size_t(B) * H * W));
  IEF_TRY(sc.get(&mx, 4));
  return event_image(frames, B, C, H, W, threshold, clamp_max, sum_out, event_out, cnt, mx, sms, st);
}

int iefvad_bench_gemm(int64_t M, int N, int K, int nsplit, int tile_n, int stages, int epi_kind, int iters,
                      float* ms_per_iter) {
  IEF_CHECK(M > 0 && M < (1LL << 31) && N > 0 && K > 0 && iters > 0 && ms_per_iter, "iefvad_bench_gemm: bad argument");
  IEF_CHECK(epi_kind >= 0 && epi_kind <= 7, "iefvad_bench_gemm: epi_kind in [0, 7]");
  int sms = 0;
  IEF_TRY(device_sms(&sms));
  cudaStream_t st = nullptr;
  Scratch sc(st);
  bf16 *ah = nullptr, *al = nullptr, *wh = nullptr, *wl = nullptr, *oh = nullptr, *ol = nullptr, *q = nullptr, *k = nullptr,
       *vt = nullptr;
  float *bias = nullptr, *resid = nullptr, *of = nullptr;
  const int H = 8, dh = N / 3 / H > 0 ? N / 3 / H : 1, dhp = (dh + 63) / 64 * 64;
  const int T = 256, Tpad = 256;
  IEF_TRY(sc.get(&ah, size_t(M) * K));
  IEF_TRY(sc.get(&al, size_t(M) * K));
  IEF_TRY(sc.get(&wh, size_t(N) * K));
  IEF_TRY(sc.get(&wl, size_t(N) * K));
  IEF_TRY(sc.get(&bias, size_t(N)));
  IEF_TRY(sc.get(&resid, size_t(M) * N));
  IEF_TRY(sc.get(&of, size_t(M) * N));
  IEF_TRY(sc.get(&oh, size_t(M) * N));
  IEF_TRY(sc.get(&ol, size_t(M) * N));
  IEF_CUDA(cudaMemsetAsync(ah, 0x3c, size_t(M) * K * 2, st));     // bf16 0x3c3c ~ 0.0115: finite, non-zero operands
  IEF_CUDA(cudaMemsetAsync(al, 0x3a, size_t(M) * K * 2, st));
  IEF_CUDA(cudaMemsetAsync(wh, 0x3c, size_t(N) * K * 2, st));
  IEF_CUDA(cudaMemsetAsync(wl, 0x3a, size_t(N) * K * 2, st));
  IEF_CUDA(cudaMemsetAsync(bias, 0, size_t(N) * 4, st));
  IEF_CUDA(cudaMemsetAsync(resid, 0, size_t(M) * N * 4, st));
  EpiParams ep;
  ep.bias = bias;
  if (epi_kind == 0) ep.mode = EPI_DISCARD;
  if (epi_kind == 1) { ep.out_f32 = of; ep.ld_f32 = N; }
  if (epi_kind == 2) {
    ep.resid = resid; ep.ld_resid = N; ep.alpha = -0.5f; ep.out_f32 = of; ep.ld_f32 = N;
    ep.out_hi = oh; ep.out_lo = ol; ep.ld_bf = N;
  }
  if (epi_kind == 3) { ep.act = ACT_RELU; ep.out_hi = oh; ep.out_lo = ol; ep.ld_bf = N; }
  if (epi_kind == 5) { ep.act = ACT_RELU; ep.out_hi = oh; ep.ld_bf = N; ep.hi_fp16 = 1; }
  if (epi_kind == 6) {
    ep.resid = resid; ep.ld_resid = N; ep.alpha = -0.5f; ep.out_f32 = of; ep.ld_f32 = N;
    ep.out_hi = oh; ep.ld_bf = N; ep.hi_fp16 = 1;
  }
  if (epi_kind == 7) {        // refinement Linear2 of the fp16 plans: fp16 pair in, fp16 pair out (in place)
    ep.resid_h16 = oh; ep.resid_l16 = ol; ep.ld_resid = N; ep.alpha = -0.5f;
    ep.out_hi = oh; ep.out_lo = ol; ep.ld_bf = N; ep.hi_fp16 = 1;
  }
  if (epi_kind == 4) {
    IEF_CHECK(N % (3 * H * 32) == 0 && M % T == 0, "iefvad_bench_gemm: qkv epilogue needs N = 3*8*dh, M %% 256 == 0");
    IEF_TRY(sc.get(&q, size_t(M) * H * dhp));
    IEF_TRY(sc.get(&k, size_t(M) * H * dhp));
    IEF_TRY(sc.get(&vt, size_t(M) * H * dh));
    ep.mode = EPI_QKV; ep.q = q; ep.k = k; ep.vt = vt; ep.T = T; ep.H = H; ep.dh = dh; ep.dhp = dhp;
    ep.Tpad = Tpad; ep.D = N / 3; ep.qscale = 0.1f;
  }
  GemmTcArgs g;
  g.A_hi = ah; g.A_lo = al; g.W_hi = wh; g.W_lo = wl;
  g.M = int(M); g.N = N; g.K = K; g.lda = K; g.ldw = K; g.nsplit = nsplit; g.force_stages = stages;
  g.force_bn = tile_n == 512 ? 256 : tile_n;
  g.force_cg = tile_n == 512 ? 2 : (tile_n ? 1 : 0);
  g.fp16 = (epi_kind >= 5) ? 1 : 0;
  for (int i = 0; i < 3; ++i) IEF_TRY(gemm_tc(g, ep, sms, st));
  cudaEvent_t e0, e1;
  IEF_CUDA(cudaEventCreate(&e0));
  IEF_CUDA(cudaEventCreate(&e1));
  IEF_CUDA(cudaEventRecord(e0, st));
  for (int i = 0; i < iters; ++i) IEF_TRY(gemm_tc(g, ep, sms, st));
  IEF_CUDA(cudaEventRecord(e1, st));
  IEF_CUDA(cudaEventSynchronize(e1));
  float ms = 0.f;
  IEF_CUDA(cudaEventElapsedTime(&ms, e0, e1));
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  *ms_per_iter = ms / iters;
  return IEFVAD_OK;
}

uint64_t iefvad_launch_count(void) { return launch_count(); }
uint64_t iefvad_alloc_generation(void) { return alloc_generation(); }
void iefvad_add_launches(uint64_t n) { count_launches(int(n)); }

int iefvad_profile_enable(int on) {
  profiler().on = on != 0;
  return IEFVAD_OK;
}

// ------------------------------------------------------------------------------------------------ training step (N3)

// the checks every training-attention entry point makes before it touches the device; `tensors`: none of its pointers is null
static int check_train_attn(const char* fn, bool tensors, int64_t B, int64_t T, int heads, int head_dim) {
  IEF_CHECK(tensors, "%s: null argument", fn);
  IEF_CHECK(B >= 0 && B < 65536 && T >= 0 && T < (1 << 24) && heads > 0, "%s: bad B / T / heads", fn);
  IEF_CHECK(attn_train_supported(head_dim), "%s: head dim %d unsupported (32, 64, 96, 128)", fn, head_dim);
  return IEFVAD_OK;
}

int iefvad_attention_train_fwd(const float* qkv, int64_t B, int64_t T, int heads, int head_dim, float p_drop, uint64_t seed,
                               float* out, float* lse, void* stream) {
  IEF_TRY(check_train_attn("iefvad_attention_train_fwd", qkv && out && lse, B, T, heads, head_dim));
  IEF_CHECK(p_drop >= 0.f && p_drop < 1.f, "attention dropout probability %f outside [0, 1)", p_drop);
  return attn_train_fwd(qkv, int(B), int(T), heads, head_dim, dropout_philox(p_drop, seed, int(T)), out, lse,
                        static_cast<cudaStream_t>(stream));
}

static int attn_train_bwd_run(const float* qkv, const float* out, const float* dout, const float* lse, int64_t B, int64_t T,
                              int heads, int head_dim, const DropoutDesc& drop, float* dqkv, void* stream) {
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  int sms = 0;
  IEF_TRY(device_sms(&sms));
  Scratch sc(st);
  float* delta = nullptr;
  IEF_TRY(sc.get(&delta, size_t(B) * heads * T));
  return attn_train_bwd(qkv, out, dout, lse, int(B), int(T), heads, head_dim, drop, delta, dqkv, sms, st);
}

int iefvad_attention_train_bwd(const float* qkv, const float* out, const float* dout, const float* lse, int64_t B, int64_t T,
                               int heads, int head_dim, float p_drop, uint64_t seed, float* dqkv, void* stream) {
  IEF_TRY(check_train_attn("iefvad_attention_train_bwd", qkv && out && dout && lse && dqkv, B, T, heads, head_dim));
  IEF_CHECK(p_drop >= 0.f && p_drop < 1.f, "attention dropout probability %f outside [0, 1)", p_drop);
  return attn_train_bwd_run(qkv, out, dout, lse, B, T, heads, head_dim, dropout_philox(p_drop, seed, int(T)), dqkv, stream);
}

// iefvad_dropout -> the kernels' descriptor, every field checked (B, heads, T already range-checked by the caller)
static int dropout_desc(const char* fn, const iefvad_dropout* d, int64_t B, int64_t heads, int64_t T, DropoutDesc* out) {
  IEF_CHECK(d, "%s: null dropout descriptor", fn);
  if (d->kind == IEFVAD_DROPOUT_PHILOX) {
    IEF_CHECK(d->p >= 0.0 && d->p < 1.0, "%s: philox dropout probability %g outside [0, 1)", fn, d->p);
    *out = dropout_philox(float(d->p), d->seed, int(T));
    return IEFVAD_OK;
  }
  IEF_CHECK(d->kind == IEFVAD_DROPOUT_TORCH, "%s: dropout kind %d is neither IEFVAD_DROPOUT_PHILOX (0) nor "
            "IEFVAD_DROPOUT_TORCH (1)", fn, int(d->kind));
  IEF_CHECK(d->p > 0.0 && d->p < 1.0, "%s: torch dropout probability %g outside (0, 1)", fn, d->p);
  IEF_CHECK(d->threads > 0 && d->threads < (int64_t(1) << 31), "%s: torch dropout threads %lld outside (0, 2^31)", fn,
            (long long)d->threads);
  IEF_CHECK(d->offset % 4 == 0, "%s: torch generator offset %llu is not a multiple of 4", fn,
            (unsigned long long)d->offset);
  const int64_t n = B * heads * T * T;
  IEF_CHECK(n % 4 == 0, "%s: B*heads*T*T = %lld is not a multiple of 4 - torch's dropout draws such sizes with a narrower "
            "vector width, which is not reproduced", fn, (long long)n);
  *out = dropout_torch(d->p, d->seed, d->offset, unsigned(d->threads), int(T));
  return IEFVAD_OK;
}

int iefvad_attention_train_fwd_dropout(const float* qkv, int64_t B, int64_t T, int heads, int head_dim,
                                       const iefvad_dropout* drop, float* out, float* lse, void* stream) {
  IEF_TRY(check_train_attn("iefvad_attention_train_fwd_dropout", qkv && out && lse, B, T, heads, head_dim));
  DropoutDesc d;
  IEF_TRY(dropout_desc("iefvad_attention_train_fwd_dropout", drop, B, heads, T, &d));
  return attn_train_fwd(qkv, int(B), int(T), heads, head_dim, d, out, lse, static_cast<cudaStream_t>(stream));
}

int iefvad_attention_train_bwd_dropout(const float* qkv, const float* out, const float* dout, const float* lse, int64_t B,
                                       int64_t T, int heads, int head_dim, const iefvad_dropout* drop, float* dqkv,
                                       void* stream) {
  IEF_TRY(check_train_attn("iefvad_attention_train_bwd_dropout", qkv && out && dout && lse && dqkv, B, T, heads, head_dim));
  DropoutDesc d;
  IEF_TRY(dropout_desc("iefvad_attention_train_bwd_dropout", drop, B, heads, T, &d));
  return attn_train_bwd_run(qkv, out, dout, lse, B, T, heads, head_dim, d, dqkv, stream);
}

int iefvad_dropout_mask(const iefvad_dropout* drop, int64_t B, int heads, int64_t T, uint8_t* mask, void* stream) {
  IEF_CHECK(mask, "iefvad_dropout_mask: null argument");
  IEF_CHECK(B >= 0 && B < 65536 && T >= 0 && T < (1 << 24) && heads > 0 && B * heads * T < (int64_t(1) << 31),
            "iefvad_dropout_mask: bad B / T / heads");
  DropoutDesc d;
  IEF_TRY(dropout_desc("iefvad_dropout_mask", drop, B, heads, T, &d));
  return dropout_mask(d, int(B), heads, int(T), mask, static_cast<cudaStream_t>(stream));
}

int iefvad_layernorm_bwd(const float* x, const float* weight, const float* dy, int64_t rows, int dim, float eps, float* dx,
                         float* dweight, float* dbias, void* stream) {
  IEF_CHECK(x && weight && dy && dx && dweight && dbias, "iefvad_layernorm_bwd: null argument");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  int sms = 0;
  IEF_TRY(device_sms(&sms));
  Scratch sc(st);
  float* scratch = nullptr;
  IEF_TRY(sc.get(&scratch, size_t(2) * rows + size_t(2) * train_colsum_blocks(rows, sms) * dim));
  return layernorm_bwd(x, weight, dy, rows, dim, eps, dx, dweight, dbias, scratch, sms, st);
}

int iefvad_colsum(const float* a, const float* row_weight, int64_t rows, int dim, float* out, void* stream) {
  IEF_CHECK(a && out, "iefvad_colsum: null argument");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  int sms = 0;
  IEF_TRY(device_sms(&sms));
  Scratch sc(st);
  float* scratch = nullptr;
  IEF_TRY(sc.get(&scratch, size_t(2) * train_colsum_blocks(rows, sms) * dim));
  return colsum(a, row_weight, rows, dim, out, scratch, sms, st);
}

int iefvad_fuse_bwd(const float* mu_i, const float* mu_e, const float* logvar_i, const float* logvar_e, const float* g_fused,
                    const float* g_wi, const float* g_we, const float* g_mu_i, const float* g_mu_e, const float* g_logvar_i,
                    const float* g_logvar_e, int64_t n, float factor, float epsilon, float* d_mu_i, float* d_mu_e,
                    float* d_logvar_i, float* d_logvar_e, void* stream) {
  IEF_CHECK(mu_i && mu_e && logvar_i && logvar_e && d_mu_i && d_mu_e && d_logvar_i && d_logvar_e, "iefvad_fuse_bwd: null argument");
  int sms = 0;
  IEF_TRY(device_sms(&sms));
  return fuse_bwd(mu_i, mu_e, logvar_i, logvar_e, g_fused, g_wi, g_we, g_mu_i, g_mu_e, g_logvar_i, g_logvar_e, n, factor, epsilon,
                  d_mu_i, d_mu_e, d_logvar_i, d_logvar_e, sms, static_cast<cudaStream_t>(stream));
}

int iefvad_relu_bwd(const float* dh, const float* h, int64_t n, float* out, void* stream) {
  IEF_CHECK(dh && h && out, "iefvad_relu_bwd: null argument");
  int sms = 0;
  IEF_TRY(device_sms(&sms));
  return relu_bwd(dh, h, n, out, sms, static_cast<cudaStream_t>(stream));
}

int iefvad_quickgelu(const float* x, int64_t n, float* out, void* stream) {
  IEF_CHECK(x && out, "iefvad_quickgelu: null argument");
  int sms = 0;
  IEF_TRY(device_sms(&sms));
  return quickgelu(x, n, out, sms, static_cast<cudaStream_t>(stream));
}

int iefvad_axpy(float* y, const float* x, float alpha, int64_t n, void* stream) {
  IEF_CHECK(y && x, "iefvad_axpy: null argument");
  int sms = 0;
  IEF_TRY(device_sms(&sms));
  return axpy(y, x, alpha, n, sms, static_cast<cudaStream_t>(stream));
}

int iefvad_outer(const float* a, const float* w, int64_t rows, int dim, float* out, void* stream) {
  IEF_CHECK(a && w && out, "iefvad_outer: null argument");
  int sms = 0;
  IEF_TRY(device_sms(&sms));
  return outer(a, w, rows, dim, out, sms, static_cast<cudaStream_t>(stream));
}

int iefvad_transpose(const float* src, int64_t rows, int cols, float* dst, int64_t ld_dst, void* stream) {
  IEF_CHECK(src && dst, "iefvad_transpose: null argument");
  return transpose_f32(src, rows, cols, dst, ld_dst, static_cast<cudaStream_t>(stream));
}

int iefvad_wgrad(const float* dy, const float* x, int64_t rows, int out_f, int in_f, float alpha, float* dw, void* stream) {
  IEF_CHECK(dy && x && dw, "iefvad_wgrad: null argument");
  IEF_CHECK(rows > 0 && rows < (1LL << 31) && out_f % 32 == 0 && in_f % 32 == 0, "iefvad_wgrad: bad sizes");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  int sms = 0;
  IEF_TRY(device_sms(&sms));
  const int64_t Mp = (rows + 63) / 64 * 64;
  Scratch sc(st);
  bf16 *yh = nullptr, *yl = nullptr, *xh = nullptr, *xl = nullptr;
  IEF_TRY(sc.get(&yh, size_t(out_f) * Mp));
  IEF_TRY(sc.get(&yl, size_t(out_f) * Mp));
  IEF_TRY(sc.get(&xh, size_t(in_f) * Mp));
  IEF_TRY(sc.get(&xl, size_t(in_f) * Mp));
  // both operands go from row-major fp32 straight to the K-major bf16 hi / lo form the GEMM reads: one pass each instead
  // of a transposition to fp32 followed by the conversion
  IEF_TRY(transpose_split(dy, rows, out_f, yh, yl, Mp, st));
  IEF_TRY(transpose_split(x, rows, in_f, xh, xl, Mp, st));
  GemmTcArgs g;
  g.A_hi = yh; g.A_lo = yl; g.W_hi = xh; g.W_lo = xl;
  g.M = out_f; g.N = in_f; g.K = int(Mp); g.lda = int(Mp); g.ldw = int(Mp); g.nsplit = 3;
  EpiParams ep;
  ep.alpha = alpha; ep.out_f32 = dw; ep.ld_f32 = in_f;
  return gemm_tc_split_k(g, ep, sc, sms, st);
}

int iefvad_clas2_bwd(const float* logits, const float* means, const float* labels, int64_t label_stride, const int32_t* idx,
                     int64_t B, int64_t T, int kmax, const float* g_loss, float* dlogits, void* stream) {
  IEF_CHECK(logits && means && labels && idx && dlogits, "iefvad_clas2_bwd: null argument");
  return clas2_bwd(logits, means, labels, label_stride, idx, int(B), int(T), kmax, g_loss, dlogits, static_cast<cudaStream_t>(stream));
}

static int train_loss_check(const char* fn, const float* logits, const float* labels, const int32_t* idx, int64_t B, int64_t T,
                            int kmax, const float* const* wide, int D, double nu) {
  IEF_CHECK(logits && labels && idx && wide[0] && wide[1] && wide[2] && wide[3], "%s: null argument", fn);
  IEF_CHECK(B >= 1 && T >= 1 && T <= 16384 && B * T < (1LL << 31), "%s: B=%lld, T=%lld out of range", fn, (long long)B,
            (long long)T);
  IEF_CHECK(kmax == int(T / 16 + 1), "%s: kmax must be T / 16 + 1 = %d, got %d", fn, int(T / 16 + 1), kmax);
  IEF_CHECK(D >= 4 && D % 4 == 0, "%s: D=%d must be a positive multiple of 4", fn, D);
  for (int i = 0; i < 4; ++i)
    IEF_CHECK(reinterpret_cast<uintptr_t>(wide[i]) % 16 == 0, "%s: the [B, T, D] tensors must be 16-byte aligned", fn);
  IEF_CHECK(nu > 0.0, "%s: nu=%g must be positive", fn, nu);
  return IEFVAD_OK;
}

int iefvad_train_loss_fwd(const float* logits, const float* labels, int64_t label_stride, const int64_t* lengths, int64_t B,
                          int64_t T, const float* mu_i, const float* mu_e, const float* logvar_i, const float* logvar_e, int D,
                          double nu, double reg_weight, double kl_weight, float* means, int32_t* idx, int kmax, double* record,
                          float* total, float* loss_cls, float* loss_reg, float* loss_kl, void* stream) {
  const float* wide[4] = {mu_i, mu_e, logvar_i, logvar_e};
  IEF_TRY(train_loss_check("iefvad_train_loss_fwd", logits, labels, idx, B, T, kmax, wide, D, nu));
  IEF_CHECK(lengths && means && record && total && loss_cls && loss_reg && loss_kl, "iefvad_train_loss_fwd: null argument");
  IEF_CHECK(reinterpret_cast<uintptr_t>(record) % 32 == 0, "iefvad_train_loss_fwd: record must be 32-byte aligned");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  Scratch sc(st);
  double* slabs = nullptr;
  IEF_TRY(sc.get(&slabs, size_t(2) * train_loss_slabs(B * T)));
  return train_loss_fwd(logits, labels, label_stride, reinterpret_cast<const long long*>(lengths), int(B), int(T), mu_i, mu_e,
                        logvar_i, logvar_e, D, nu, reg_weight, kl_weight, means, idx, kmax, record, slabs,
                        total, loss_cls, loss_reg, loss_kl, st);
}

int iefvad_train_loss_bwd(const float* logits, const float* means, const float* labels, int64_t label_stride, const int32_t* idx,
                          int64_t B, int64_t T, int kmax, const float* mu_i, const float* mu_e, const float* logvar_i,
                          const float* logvar_e, int D, const double* record, double nu, double reg_weight, double kl_weight,
                          const float* g_total, const float* g_cls, const float* g_reg, const float* g_kl, float* d_logits,
                          float* d_mu_i, float* d_mu_e, float* d_logvar_i, float* d_logvar_e, void* stream) {
  const float* wide[4] = {mu_i, mu_e, logvar_i, logvar_e};
  IEF_TRY(train_loss_check("iefvad_train_loss_bwd", logits, labels, idx, B, T, kmax, wide, D, nu));
  IEF_CHECK(means && record && d_logits && d_mu_i && d_mu_e && d_logvar_i && d_logvar_e, "iefvad_train_loss_bwd: null argument");
  const float* outs[4] = {d_mu_i, d_mu_e, d_logvar_i, d_logvar_e};
  for (int i = 0; i < 4; ++i)
    IEF_CHECK(reinterpret_cast<uintptr_t>(outs[i]) % 16 == 0, "iefvad_train_loss_bwd: the gradients must be 16-byte aligned");
  IEF_CHECK(reinterpret_cast<uintptr_t>(record) % 32 == 0, "iefvad_train_loss_bwd: record must be 32-byte aligned");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  Scratch sc(st);
  float* g_cls_total = nullptr;
  IEF_TRY(sc.get(&g_cls_total, 1));
  return train_loss_bwd(logits, means, labels, label_stride, idx, int(B), int(T), kmax, mu_i, mu_e, logvar_i, logvar_e, D, record,
                        nu, reg_weight, kl_weight, g_total, g_cls, g_reg, g_kl, g_cls_total, d_logits,
                        d_mu_i, d_mu_e, d_logvar_i, d_logvar_e, st);
}

// ------------------------------------------------------------------------------------------------ localisation mAP (N5)

int iefvad_locmap_proposals(const float* pred, const int64_t* vid_off, const int32_t* vid_len, int64_t num_videos,
                            int num_classes, int max_len, int32_t* prop_count, int32_t* prop_se, float* prop_score,
                            float* class_score, void* stream) {
  IEF_CHECK(pred && vid_off && vid_len && prop_count && prop_se && prop_score && class_score, "iefvad_locmap_proposals: null argument");
  IEF_CHECK(num_videos >= 0 && num_videos < 65536 && num_classes > 0 && num_classes < 65536, "iefvad_locmap_proposals: bad sizes");
  return locmap_proposals(pred, reinterpret_cast<const long long*>(vid_off), vid_len, int(num_videos), num_classes, max_len,
                          prop_count, prop_se, prop_score, class_score, static_cast<cudaStream_t>(stream));
}

int iefvad_locmap_match(const int32_t* prop_count, const int32_t* prop_se, const float* prop_score, int64_t num_videos,
                        int num_classes, const int32_t* gt, const int32_t* gt_off, int64_t num_gt, double iou_threshold,
                        double* ap, int32_t* n_pred, void* stream) {
  IEF_CHECK(prop_count && prop_se && prop_score && gt_off && ap && n_pred && (gt || num_gt == 0), "iefvad_locmap_match: null argument");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int cap = int(num_videos) * 8 > 8192 ? int(num_videos) * 8 : 8192;
  Scratch sc(st);
  float* ws = nullptr;
  int *wi = nullptr, *wa = nullptr;
  IEF_TRY(sc.get(&ws, size_t(num_classes) * cap * 2));      // rounded up to a power of two inside the kernel
  IEF_TRY(sc.get(&wi, size_t(num_classes) * cap * 2));
  IEF_TRY(sc.get(&wa, size_t(num_gt ? num_gt : 1)));
  return locmap_match(prop_count, prop_se, prop_score, int(num_videos), num_classes, gt, gt_off, iou_threshold, cap * 2,
                      ws, wi, wa, ap, n_pred, st);
}

int iefvad_profile_read(double* ms, double* work, int64_t* launches) {
  IEF_CHECK(ms && work && launches, "iefvad_profile_read: null argument");
  long long l[KC_COUNT];
  IEF_TRY(profiler().read(ms, work, l));
  for (int i = 0; i < KC_COUNT; ++i) launches[i] = l[i];
  return IEFVAD_OK;
}

}  // extern "C"
