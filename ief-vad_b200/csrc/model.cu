// The IEF-VAD forward (model/imf_vad.py:109-161) as a sequence of sm_100a kernels.
#include <nvtx3/nvToolsExt.h>
#include "model.cuh"

#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdlib>
#include <cstdio>
#include <cstring>

namespace iefvad {

static std::atomic<unsigned long long> g_alloc_generation{0};
unsigned long long alloc_generation() { return g_alloc_generation.load(); }

int DevBuf::reserve(size_t need) {
  if (need <= bytes) return IEFVAD_OK;
  ++g_alloc_generation;            // every address handed out before may be gone: captured CUDA graphs are stale
  if (p) {
    IEF_CUDA(cudaFree(p));
    p = nullptr;
    bytes = 0;
  }
  IEF_CUDA(cudaMalloc(&p, need));
  bytes = need;
  return IEFVAD_OK;
}

void DevBuf::release() {
  if (p) cudaFree(p);
  p = nullptr;
  bytes = 0;
}

namespace {
size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }
}  // namespace

Profiler& profiler() {
  static Profiler p;
  return p;
}

void Profiler::begin(int cls, double work, cudaStream_t st) {
  if (!on) return;
  Rec r;
  r.cls = cls;
  r.work = work;
  cudaEventCreate(&r.a);
  cudaEventCreate(&r.b);
  cudaEventRecord(r.a, st);
  recs.push_back(r);
}

void Profiler::end(cudaStream_t st) {
  if (!on || recs.empty()) return;
  cudaEventRecord(recs.back().b, st);
}

int Profiler::read(double* ms, double* work, long long* launches) {
  for (int i = 0; i < KC_COUNT; ++i) { ms[i] = 0.0; work[i] = 0.0; launches[i] = 0; }
  for (auto& r : recs) {
    IEF_CUDA(cudaEventSynchronize(r.b));
    float t = 0.f;
    IEF_CUDA(cudaEventElapsedTime(&t, r.a, r.b));
    ms[r.cls] += t;
    work[r.cls] += r.work;
    launches[r.cls] += 1;
    cudaEventDestroy(r.a);
    cudaEventDestroy(r.b);
  }
  recs.clear();
  return IEFVAD_OK;
}

// time one launch when profiling is on (no-op otherwise)
// NVTX ranges around every stage of the forward (nsys / ncu --nvtx timelines; SURVEY section 5 tracing row).  NVTX v3 is
// header-only: without an attached tool the calls are no-ops, and they are compiled in only behind IEFVAD_NVTX=1.
static const bool g_nvtx = [] { const char* e = getenv("IEFVAD_NVTX"); return e && atoi(e) != 0; }();
static const char* const kClassNames[KC_COUNT] = {"gemm_qkv", "attn_tc", "layernorm", "fuse", "classifier", "ingest", "gemm_simt",
                                                  "attn_simt", "gemm_out_proj", "gemm_heads", "gemm_refine1", "gemm_refine2",
                                                  "gather_valid_rows", "refine_fused", "heads_fuse", "outproj_ln"};

#define IEF_PROF(cls, work, call)                 \
  do {                                            \
    if (g_nvtx) nvtxRangePushA(kClassNames[cls]); \
    profiler().begin(cls, work, stream);          \
    int _prc = (call);                            \
    profiler().end(stream);                       \
    if (g_nvtx) nvtxRangePop();                   \
    if (_prc != 0) return _prc;                   \
  } while (0)

int Model::init(int embed_dim, int num_heads, int layers, int refine_steps, float lambda, int noise_model, float nu,
                float epsilon) {
  IEF_CHECK(embed_dim >= 128 && embed_dim % 128 == 0 && embed_dim <= 1024,
            "embed_dim=%d unsupported: need a multiple of 128 in [128, 1024]", embed_dim);
  IEF_CHECK(num_heads > 0 && embed_dim % num_heads == 0, "num_heads=%d must divide embed_dim=%d", num_heads, embed_dim);
  D = embed_dim; H = num_heads; L = layers; R = refine_steps;
  dh = D / H;
  IEF_CHECK(dh == 32 || dh == 64 || dh == 96 || dh == 128, "head dim %d unsupported (32, 64, 96, 128)", dh);
  dhp = (dh + 63) / 64 * 64;
  IEF_CHECK(L >= 0 && R >= 0, "negative layer / refinement count");
  lambda_ref = lambda;
  eps = epsilon;
  if (noise_model == 0) factor = 1.f;                                  // Gaussian, model/imf_vad.py:130-132
  else if (noise_model == 1) factor = (nu + 1.f) / nu;                 // StudentT, :133-136
  else { set_error("Unsupported noise_model. Choose 'Gaussian' or 'StudentT'."); return IEFVAD_ERR_INVALID; }
  IEF_CUDA(cudaGetDevice(&device));
  IEF_CUDA(cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, device));

  // ---- carve one fp32 arena (+ bf16 hi / lo and fp16 arenas mirroring the weight matrices).  The encoder's in- and
  // out-projections run one 16-bit operand pass in every plan, so only the heads and refinement weights keep a bf16 lo.
  struct Want { std::string key; long long numel; bool is_weight; float** dst; bf16** hi; bf16** lo; bf16** h16 = nullptr; };
  std::vector<Want> wants;
  const char* mods[2] = {"image", "event"};
  for (int m = 0; m < 2; ++m) {
    in_proj[m].assign(L, Linear());
    out_proj[m].assign(L, Linear());
    ln_w[m].assign(L, nullptr);
    ln_b[m].assign(L, nullptr);
  }
  ref1.assign(R, Linear());
  ref2.assign(R, Linear());
  char buf[160];
  for (int m = 0; m < 2; ++m) {
    for (int i = 0; i < L; ++i) {
      Linear& ip = in_proj[m][i];
      Linear& op = out_proj[m][i];
      ip.out = 3 * D; ip.in = D; op.out = D; op.in = D;
      snprintf(buf, sizeof(buf), "temporal.%s_attn_layers.%d.in_proj_weight", mods[m], i);
      wants.push_back({buf, 3LL * D * D, true, &ip.w, &ip.w_hi, nullptr, &ip.w_h16});
      snprintf(buf, sizeof(buf), "temporal.%s_attn_layers.%d.in_proj_bias", mods[m], i);
      wants.push_back({buf, 3LL * D, false, &ip.b, nullptr, nullptr});
      snprintf(buf, sizeof(buf), "temporal.%s_attn_layers.%d.out_proj.weight", mods[m], i);
      wants.push_back({buf, 1LL * D * D, true, &op.w, &op.w_hi, nullptr, &op.w_h16});
      snprintf(buf, sizeof(buf), "temporal.%s_attn_layers.%d.out_proj.bias", mods[m], i);
      wants.push_back({buf, D, false, &op.b, nullptr, nullptr});
      snprintf(buf, sizeof(buf), "temporal.%s_norms.%d.weight", mods[m], i);
      wants.push_back({buf, D, false, &ln_w[m][i], nullptr, nullptr});
      snprintf(buf, sizeof(buf), "temporal.%s_norms.%d.bias", mods[m], i);
      wants.push_back({buf, D, false, &ln_b[m][i], nullptr, nullptr});
    }
    snprintf(buf, sizeof(buf), "temporal.whiten_%s.weight", mods[m]);
    wants.push_back({buf, D, false, &whiten_w[m], nullptr, nullptr});
    snprintf(buf, sizeof(buf), "temporal.whiten_%s.bias", mods[m]);
    wants.push_back({buf, D, false, &whiten_b[m], nullptr, nullptr});
    heads[m].out = 2 * D; heads[m].in = D;
    // mu and logvar of one modality share their input: stored as one [2D, D] matrix (rows [0,D) = mu)
    wants.push_back({std::string("@heads_w.") + mods[m], 2LL * D * D, true, &heads[m].w, &heads[m].w_hi, &heads[m].w_lo, &heads[m].w_h16});
    wants.push_back({std::string("@heads_b.") + mods[m], 2LL * D, false, &heads[m].b, nullptr, nullptr});
  }
  for (int i = 0; i < R; ++i) {
    ref1[i].out = ref1[i].in = ref2[i].out = ref2[i].in = D;
    snprintf(buf, sizeof(buf), "temporal.refinement_blocks.%d.0.weight", i);
    wants.push_back({buf, 1LL * D * D, true, &ref1[i].w, &ref1[i].w_hi, &ref1[i].w_lo, &ref1[i].w_h16});
    snprintf(buf, sizeof(buf), "temporal.refinement_blocks.%d.0.bias", i);
    wants.push_back({buf, D, false, &ref1[i].b, nullptr, nullptr});
    snprintf(buf, sizeof(buf), "temporal.refinement_blocks.%d.2.weight", i);
    wants.push_back({buf, 1LL * D * D, true, &ref2[i].w, &ref2[i].w_hi, &ref2[i].w_lo, &ref2[i].w_h16});
    snprintf(buf, sizeof(buf), "temporal.refinement_blocks.%d.2.bias", i);
    wants.push_back({buf, D, false, &ref2[i].b, nullptr, nullptr});
  }
  wants.push_back({"temporal.classifier.weight", D, false, &cls_w, nullptr, nullptr});
  wants.push_back({"temporal.classifier.bias", 1, false, &cls_b, nullptr, nullptr});

  size_t f32_elems = 0, bf_elems = 0, lo_elems = 0, h16_elems = 0;
  for (auto& w : wants) {
    f32_elems += align_up(size_t(w.numel), 64);
    if (w.is_weight) bf_elems += align_up(size_t(w.numel), 64);
    if (w.lo) lo_elems += align_up(size_t(w.numel), 64);
    if (w.h16) h16_elems += align_up(size_t(w.numel), 64);
  }
  IEF_TRY(params_h16.reserve((h16_elems ? h16_elems : 64) * sizeof(bf16)));
  IEF_TRY(params_f32.reserve(f32_elems * sizeof(float)));
  IEF_TRY(params_hi.reserve(bf_elems * sizeof(bf16)));
  IEF_TRY(params_lo.reserve(lo_elems * sizeof(bf16)));
  IEF_CUDA(cudaMemset(params_f32.p, 0, params_f32.bytes));
  IEF_TRY(status.reserve(4 * sizeof(int)));
  IEF_CUDA(cudaMemset(status.p, 0, status.bytes));
  size_t fo = 0, bo = 0, lo_o = 0, ho = 0;
  for (auto& w : wants) {
    *w.dst = params_f32.as<float>() + fo;
    fo += align_up(size_t(w.numel), 64);
    ParamSlot s;
    s.dst = *w.dst;
    s.numel = w.numel;
    if (w.is_weight) {
      *w.hi = params_hi.as<bf16>() + bo;
      s.hi = *w.hi;
      bo += align_up(size_t(w.numel), 64);
    }
    if (w.lo) {
      *w.lo = params_lo.as<bf16>() + lo_o;
      s.lo = *w.lo;
      lo_o += align_up(size_t(w.numel), 64);
    }
    if (w.h16) {
      *w.h16 = params_h16.as<bf16>() + ho;
      s.h16 = *w.h16;
      ho += align_up(size_t(w.numel), 64);
    }
    slots[w.key] = s;
  }
  // the four head Linears alias halves of the packed [2D, D] matrices
  for (int m = 0; m < 2; ++m) {
    const ParamSlot& hw = slots[std::string("@heads_w.") + mods[m]];
    const ParamSlot& hb = slots[std::string("@heads_b.") + mods[m]];
    const char* kinds[2] = {"mu", "logvar"};
    for (int k = 0; k < 2; ++k) {
      ParamSlot sw;
      sw.dst = hw.dst + (long long)k * D * D; sw.numel = 1LL * D * D;
      sw.hi = hw.hi + (long long)k * D * D;   sw.lo = hw.lo + (long long)k * D * D;
      sw.h16 = hw.h16 + (long long)k * D * D;
      snprintf(buf, sizeof(buf), "temporal.%s_%s.weight", mods[m], kinds[k]);
      slots[buf] = sw;
      ParamSlot sb;
      sb.dst = hb.dst + (long long)k * D; sb.numel = D;
      snprintf(buf, sizeof(buf), "temporal.%s_%s.bias", mods[m], kinds[k]);
      slots[buf] = sb;
    }
    slots.erase(std::string("@heads_w.") + mods[m]);
    slots.erase(std::string("@heads_b.") + mods[m]);
  }
  refine_contig = R > 0;
  for (int i = 0; i < R; ++i) {
    if (ref2[i].w_h16 != ref1[i].w_h16 + (long long)D * D) refine_contig = false;
    if (i + 1 < R && ref1[i + 1].w_h16 != ref2[i].w_h16 + (long long)D * D) refine_contig = false;
  }
  return IEFVAD_OK;
}

int Model::set_param(const char* key, const float* dptr, long long numel, cudaStream_t stream) {
  auto it = slots.find(key);
  IEF_CHECK(it != slots.end(), "unexpected parameter key '%s'", key);
  ParamSlot& s = it->second;
  IEF_CHECK(s.numel == numel, "parameter '%s': expected %lld elements, got %lld", key, s.numel, numel);
  IEF_CUDA(cudaMemcpyAsync(s.dst, dptr, size_t(numel) * sizeof(float), cudaMemcpyDeviceToDevice, stream));
  if (s.hi) IEF_TRY(ingest(s.dst, IEFVAD_DT_F32, numel, nullptr, s.hi, s.lo, num_sms, stream));
  if (s.h16) IEF_TRY(to_half(s.dst, numel, s.h16, num_sms, stream));
  s.loaded = true;
  return IEFVAD_OK;
}

int Model::check_loaded() const {
  for (auto& kv : slots)
    if (!kv.second.loaded) {
      set_error("parameter '%s' was never uploaded (iefvad_model_set_param)", kv.first.c_str());
      return IEFVAD_ERR_STATE;
    }
  return IEFVAD_OK;
}

int Model::reserve_workspace(long long rows, int B, int T, bool fp32_plan) {
  const size_t act = size_t(rows) * D;
  IEF_TRY(x32.reserve(act * 4));
  IEF_TRY(y32.reserve(act * 4));
  if (!fp32_plan) {
    IEF_TRY(a_hi.reserve(act * 2));
    IEF_TRY(a_lo.reserve(act * 2));
    IEF_TRY(h_hi.reserve(act * 2 + size_t(256) * D * 2));      // + one 256-row tile: the fused refinement chain's scratch
    IEF_TRY(h_lo.reserve(act * 2));
    const int Tpad = (T + 7) / 8 * 8;
    IEF_TRY(qb.reserve(size_t(B) * H * T * dhp * 2));
    IEF_TRY(kb.reserve(size_t(B) * H * T * dhp * 2));
    IEF_TRY(vtb.reserve(size_t(B) * H * dh * Tpad * 2));
  } else {
    IEF_TRY(qkv32.reserve(act * 3 * 4));
    IEF_TRY(attn32.reserve(act * 4));
    IEF_TRY(h32.reserve(act * 4));
  }
  return IEFVAD_OK;
}

int Model::forward(const void* img, const void* ev, int in_dtype, long long B, long long T, float* fused, float* logits,
                   float* image_mu, float* event_mu, float* image_logvar, float* event_logvar, float* w_i, float* w_e,
                   float* scores, cudaStream_t stream, const ValidRows* vr) {
  IEF_TRY(check_loaded());
  IEF_CHECK(B >= 0 && T >= 0, "negative batch / length");
  if (B == 0 || T == 0) return IEFVAD_OK;
  struct NvtxScope {
    bool on;
    explicit NvtxScope(bool o, const char* name) : on(o) { if (on) nvtxRangePushA(name); }
    ~NvtxScope() { if (on) nvtxRangePop(); }
  } nvtx_scope(g_nvtx, vr ? "iefvad forward (valid rows)" : "iefvad forward");
  IEF_CHECK(img && ev && fused && logits && image_mu && event_mu && image_logvar && event_logvar,
            "forward: null tensor pointer");
  IEF_CHECK((w_i == nullptr) == (w_e == nullptr), "forward: w_i and w_e are written together or not at all");
  IEF_CHECK(T <= (1 << 24), "T=%lld too long", T);
  const bool fp32_plan = plan == PLAN_FP32;
  const bool f16 = plan == PLAN_HH;        // fp16 operands, one MMA pass everywhere
  const bool bsplit = plan == PLAN_B;      // bf16 operands, 3-term split for the heads and the refinement Linears
  if (vr) {
    IEF_CHECK(vr->len_host && vr->rowmap, "forward: valid-rows descriptor with null members");
    IEF_CHECK(!fp32_plan && L >= 1, "forward: the valid-rows mode needs a tensor-core plan and at least one attention layer");
  }
  const size_t in_esize = (in_dtype == IEFVAD_DT_F32) ? 4 : 2;
  long long slabB = max_rows / T;
  if (slabB < 1) slabB = 1;
  if (slabB > B) slabB = B;
  if (slabB > 65535) slabB = 65535;
  IEF_TRY(reserve_workspace(slabB * T, int(slabB), int(T), fp32_plan));
  const int Tpad = int((T + 7) / 8 * 8);
  const float qscale = 1.0f / sqrtf(float(dh));
  float* mu_out[2] = {image_mu, event_mu};
  float* lv_out[2] = {image_logvar, event_logvar};
  const void* inputs[2] = {img, ev};

  for (long long b0 = 0; b0 < B; b0 += slabB) {
    const int Bs = int((B - b0 < slabB) ? (B - b0) : slabB);
    const long long M = (long long)Bs * T;
    IEF_CHECK(M < (1LL << 31), "slab of %lld rows exceeds 2^31", M);
    const long long row0 = b0 * T;
    // valid-rows mode: Mo rows survive the last attention core; outputs are compact at offset `out0`
    long long Mo = M, out0 = row0;
    if (vr) {
      out0 = 0;
      for (long long b = 0; b < b0; ++b) out0 += vr->len_host[b];
      Mo = 0;
      for (long long b = b0; b < b0 + Bs; ++b) {
        IEF_CHECK(vr->len_host[b] >= 0 && vr->len_host[b] <= T, "forward: valid length %lld outside [0, T]", vr->len_host[b]);
        Mo += vr->len_host[b];
      }
    }
    // valid-rows mode with >= 2 layers: the producers of the last layer's out-projection inputs write compact rows
    // themselves (LayerNorm of layer L-2: fp32 residual; last attention core: context) - no gather pass
    const bool direct_compact = vr && L >= 2;
    // Out-projection + residual + LayerNorm(s) as one kernel (outproj_ln.cu) under the all-fp16 plan: y never reaches HBM.
    // Every encoder stage then works in encoder-row space (all rows, or the packed rows of the pad de-duplication); the
    // LAST layer's kernel writes its result through the inverse row map, i.e. directly as compact valid rows.
    const bool ln_fused = f16 && D == kOutprojLnDim && L >= 1 && outproj_ln_mode != 0 &&
                          (in_dtype == IEFVAD_DT_F16 || !(vr && vr->chunk_start && vr->chunk_valid));
    // Pad de-duplication (valid-rows mode, fp16 inputs, fp16 encoder, chunks of <= 256 rows): the zero-pad rows of a
    // chunk are identical, and stay identical to each other through every row-wise stage and through attention, so
    // ONE representative per chunk goes through the encoder; as an attention key it counts `mult` times (its score
    // gets + log mult, which is exactly what mult equal keys contribute to the softmax).  The encoder then works on
    // Me = sum(valid + 1) packed rows instead of B * T; chunks without valid rows vanish.  Same arithmetic as the
    // dense forward up to the rounding of that one key's probability.
    const bool dedup = direct_compact && f16 && in_dtype == IEFVAD_DT_F16 && T <= 256 && T % 32 == 0 && pad_dedup;
    long long Me = M;                       // rows the encoder stages before the valid-row cut run on
    if (dedup) {
      items_host.clear();
      aux_host.clear();
      const bool ragged_src = vr->chunk_start && vr->chunk_valid;
      long long cur = 0, src = 0, outc = 0;
      for (long long b = b0; b < b0 + Bs; ++b) {
        const int n = int(vr->len_host[b]);
        if (n > 0) {
          const bool pad = n < T;
          items_host.push_back({int(cur), n + (pad ? 1 : 0), n, pad ? int(T) - n : 0});
          aux_host.push_back({ragged_src ? src : (b - b0) * T, 0, int(outc)});
          cur = (cur + n + (pad ? 1 : 0) + 7) / 8 * 8;
        }
        src += n;
        outc += n;
      }
      Me = (cur + 31) / 32 * 32;
      if (Me < 32) Me = 32;
      for (size_t i = 0; i < items_host.size(); ++i)
        aux_host[i].span = int((i + 1 < items_host.size() ? items_host[i + 1].start : Me) - items_host[i].start);
      // longest chunks first: the persistent attention CTAs take items round-robin, so each gets a similar mix and
      // the short items (no second query tile) end up together at the end
      {
        std::vector<size_t> order(items_host.size());
        for (size_t i = 0; i < order.size(); ++i) order[i] = i;
        std::stable_sort(order.begin(), order.end(), [&](size_t a, size_t b) { return items_host[a].rows > items_host[b].rows; });
        std::vector<ChunkItem> si(order.size());
        std::vector<ChunkAux> sa(order.size());
        for (size_t i = 0; i < order.size(); ++i) { si[i] = items_host[order[i]]; sa[i] = aux_host[order[i]]; }
        items_host.swap(si);
        aux_host.swap(sa);
      }
      if (!items_host.empty()) {
        IEF_TRY(items_dev.reserve(items_host.size() * sizeof(ChunkItem)));
        IEF_TRY(aux_dev.reserve(aux_host.size() * sizeof(ChunkAux)));
        IEF_CUDA(cudaMemcpyAsync(items_dev.p, items_host.data(), items_host.size() * sizeof(ChunkItem), cudaMemcpyHostToDevice, stream));
        IEF_CUDA(cudaMemcpyAsync(aux_dev.p, aux_host.data(), aux_host.size() * sizeof(ChunkAux), cudaMemcpyHostToDevice, stream));
      }
    }
    const int n_items = dedup ? int(items_host.size()) : 0;
    double attn_flops = 4.0 * double(Me) * double(T) * D;      // executed: QK^T + PV over the keys each query really sees
    if (dedup) {
      attn_flops = 0.0;
      for (const ChunkItem& it : items_host) attn_flops += 4.0 * double(it.rows) * double(it.rows) * D;
    }
    if (dedup && n_items == 0) continue;                 // no valid row in this slab
    // heads of both modalities + fusion as one kernel (heads_fuse.cu) when the caller keeps neither mu / logvar nor the fusion
    // weights (the evaluation forward) and the refinement chain takes the fp16 pair
    const bool hf = ln_fused && vr && heads_outputs_unused && !w_i && !eval_wi_mean && R > 0 && D == kHeadsFuseDim && L >= 2 &&
                    heads_fuse_mode != 0;
    if (ln_fused) {
      IEF_TRY(ln_scratch.reserve(outproj_ln_scratch_bytes(Me)));
      if (!ln_ident.p) {
        IEF_TRY(ln_ident.reserve(outproj_ln_identity_bytes()));
        IEF_TRY(outproj_ln_identity(ln_ident.p, stream));
      }
    }
    if (direct_compact || (vr && ln_fused)) {
      IEF_TRY(inv_map.reserve(size_t(Me) * sizeof(int)));
      if (dedup) IEF_TRY(inverse_rowmap_items(items_dev.as<ChunkItem>(), aux_dev.as<ChunkAux>(), n_items, inv_map.as<int>(), stream,
                                              (vr->chunk_start && vr->chunk_valid) ? nullptr : vr->rowmap + out0, vr->row_base + row0, status.as<int>()));
      else IEF_TRY(inverse_rowmap(vr->rowmap + out0, vr->row_base + row0, Mo, M, inv_map.as<int>(), num_sms, stream));
    }
    for (int m = 0; m < 2; ++m) {
      const bool ragged = vr && vr->chunk_start && vr->chunk_valid;
      const uint8_t* in = static_cast<const uint8_t*>(inputs[m]) + (ragged ? 0 : size_t(row0) * D * in_esize);
      // fp16 inputs under an fp16-operand encoder are their own first GEMM operand AND (exactly) their own fp32
      // residual: no fp32 copy is written, a dense batch is not touched at all before the QKV GEMM
      const bool direct16 = f16 && in_dtype == IEFVAD_DT_F16 && L >= 1 && !(vr && L == 1);
      const bf16* x16 = a_hi.as<bf16>();          // layer-0 operand (and fp16 residual when direct16)
      if (dedup) {
        // dense chunks or ragged packed rows -> the packed layout (the only pass over the inputs)
        const uint8_t* src = static_cast<const uint8_t*>(inputs[m]) + (ragged ? 0 : size_t(row0) * D * in_esize);
        IEF_PROF(KC_INGEST, double(Mo) * D * 2 + double(Me) * D * 2,
                 pack_chunks(src, items_dev.as<ChunkItem>(), aux_dev.as<ChunkAux>(), n_items, D, a_hi.p, stream));
      } else if (ragged) {
        IEF_PROF(KC_INGEST, double(Mo) * D * in_esize + double(M) * D * (direct16 ? 2 : 4 + 2),
                 ingest_ragged(in, in_dtype, vr->chunk_start + b0, vr->start_base, vr->chunk_valid + b0, Bs, int(T), D,
                               direct16 ? nullptr : x32.as<float>(), a_hi.as<bf16>(), (f16 && L > 0) ? 1 : 0, num_sms, stream));
      } else if (direct16) {
        IEF_CHECK((reinterpret_cast<uintptr_t>(in) & 15) == 0, "forward: fp16 inputs must be 16-byte aligned");
        x16 = reinterpret_cast<const bf16*>(in);
      } else if (ln_fused)      // the residual stream starts as the fp16 pair (hi = first operand, lo = remainder; 0 for fp16 values)
        IEF_PROF(KC_INGEST, double(M) * D * (in_esize + 2 + 2), ingest(in, in_dtype, M * D, nullptr, a_hi.as<bf16>(), a_lo.as<bf16>(),
                       num_sms, stream, 1));
      else
      IEF_PROF(KC_INGEST, double(M) * D * (in_esize + 4 + 2), ingest(in, in_dtype, M * D, x32.as<float>(), fp32_plan ? nullptr : a_hi.as<bf16>(),
                     nullptr, num_sms, stream, (f16 && L > 0) ? 1 : 0));
      for (int i = 0; i < L; ++i) {                                   // model/imf_vad.py:114-116 / :120-122
        const Linear& ip = in_proj[m][i];
        const Linear& op = out_proj[m][i];
        const bool last = (i == L - 1);
        if (fp32_plan) {
          EpiParams e1;
          e1.bias = ip.b; e1.out_f32 = qkv32.as<float>(); e1.ld_f32 = 3 * D;
          IEF_PROF(KC_GEMM_SIMT, 6.0 * M * D * D, gemm_simt(x32.as<float>(), D, ip.w, D, int(M), 3 * D, D, e1, stream));
          IEF_PROF(KC_ATTN_SIMT, 4.0 * M * T * D, attn_simt(qkv32.as<float>(), attn32.as<float>(), Bs, int(T), H, dh, nullptr, nullptr, stream));
          EpiParams e2;
          e2.bias = op.b; e2.resid = x32.as<float>(); e2.ld_resid = D; e2.out_f32 = y32.as<float>(); e2.ld_f32 = D;
          IEF_PROF(KC_GEMM_SIMT, 2.0 * M * D * D, gemm_simt(attn32.as<float>(), D, op.w, D, int(M), D, D, e2, stream));
          IEF_PROF(KC_LAYERNORM, double(M) * D * 8, layernorm(y32.as<float>(), M, D, ln_w[m][i], ln_b[m][i], last ? whiten_w[m] : nullptr,
                            last ? whiten_b[m] : nullptr, 1e-5f, x32.as<float>(), nullptr, nullptr, num_sms, stream));
        } else {
          AttnTcArgs at;
          at.q = qb.as<bf16>(); at.k = kb.as<bf16>(); at.vt = vtb.as<bf16>(); at.out = h_hi.as<bf16>(); at.ldo = D;
          at.B = Bs; at.T = int(T); at.H = H; at.dh = dh; at.Tpad = Tpad;
          if (dedup) { at.B = 1; at.T = int(Me); at.Tpad = int(Me); at.items = items_dev.as<int>(); at.n_chunks = n_items; }
          at.fp16 = f16;
          if (direct_compact && last && !ln_fused) at.row_out = inv_map.as<int>();
          at.dhp = attn_qk_cols(at);
          EpiParams e1;
          e1.hi_fp16 = f16;
          e1.mode = EPI_QKV; e1.bias = ip.b; e1.q = qb.as<bf16>(); e1.k = kb.as<bf16>(); e1.vt = vtb.as<bf16>();
          e1.T = at.T; e1.H = H; e1.dh = dh; e1.dhp = at.dhp; e1.Tpad = at.Tpad; e1.D = D; e1.qscale = qscale;
          GemmTcArgs g1;
          g1.A_hi = (i == 0) ? x16 : a_hi.as<bf16>(); g1.W_hi = f16 ? ip.w_h16 : ip.w_hi;
          g1.M = int(Me); g1.N = 3 * D; g1.K = D; g1.lda = D; g1.ldw = D; g1.fp16 = f16;
          IEF_PROF(KC_GEMM_QKV, 6.0 * Me * D * D, gemm_tc(g1, e1, num_sms, stream));
          IEF_PROF(KC_ATTN_TC, attn_flops, attn_tc(at, stream));
          if (ln_fused) {
            OutprojLnArgs oa;
            oa.ctx = h_hi.p; oa.w16 = op.w_h16; oa.bias = op.b;
            oa.res_hi = (i == 0) ? static_cast<const void*>(x16) : a_hi.p;
            oa.res_lo = (i == 0) ? ((dedup || direct16 || ragged) ? nullptr : a_lo.p) : a_lo.p;
            oa.ln_w = ln_w[m][i]; oa.ln_b = ln_b[m][i];
            if (last) { oa.ln2_w = whiten_w[m]; oa.ln2_b = whiten_b[m]; }
            // in place (each element's residual is read by the warp that later writes it), except the row-mapped result of
            // the last layer, which lands in other rows: that one goes to h_lo
            oa.out_hi = (last && vr) ? ((hf && m == 0) ? x32.p : h_lo.p) : a_hi.p;   // heads_fuse: image rows wait in x32 (as fp16)
            oa.out_lo = last ? nullptr : a_lo.p;
            oa.row_map = (last && vr) ? inv_map.as<int>() : nullptr;
            oa.M = Me; oa.scratch = ln_scratch.p; oa.identity = ln_ident.p;
            IEF_PROF(KC_OUTPROJ_LN, double(Me) * D * (2 + (oa.res_lo ? 4 : 2) + (oa.out_lo ? 4 : 2)), outproj_ln(oa, num_sms, stream));
            continue;
          }
          // after the last attention core only the valid rows go on: gather (context, residual) into compact matrices
          const bool compact = vr && last;
          const long long Mc = compact ? Mo : Me;
          const bf16* ctx = h_hi.as<bf16>();
          const float* resid = x32.as<float>();
          float* yout = y32.as<float>();
          if (compact && direct_compact) {
            resid = x32.as<float>(); yout = y32.as<float>();       // both already compact
          } else if (compact) {
            IEF_PROF(KC_GATHER, double(Mo) * D * 12, gather_rows(h_hi.as<bf16>(), x32.as<float>(), vr->rowmap + out0,
                     vr->row_base + row0, Mo, D, h_lo.as<bf16>(), y32.as<float>(), num_sms, stream));
            ctx = h_lo.as<bf16>(); resid = y32.as<float>(); yout = x32.as<float>();
          }
          if (Mc > 0) {
            EpiParams e2;
            e2.bias = op.b; e2.resid = resid; e2.ld_resid = D; e2.out_f32 = yout; e2.ld_f32 = D;
            if (direct16 && i == 0) { e2.resid = nullptr; e2.resid_h16 = x16; }
            GemmTcArgs g2;
            g2.A_hi = ctx; g2.W_hi = f16 ? op.w_h16 : op.w_hi; g2.M = int(Mc); g2.N = D; g2.K = D; g2.lda = D; g2.ldw = D;
            g2.fp16 = f16;
            IEF_PROF(KC_GEMM_OUT, 2.0 * Mc * D * D, gemm_tc(g2, e2, num_sms, stream));
            // LN_i (+ whitening LN after the last layer, :117/:123); hi (+ lo for the split heads) feed the next GEMM
            IEF_PROF(KC_LAYERNORM, double(Mc) * D * 8, layernorm(yout, Mc, D, ln_w[m][i], ln_b[m][i], last ? whiten_w[m] : nullptr,
                              last ? whiten_b[m] : nullptr, 1e-5f, last ? nullptr : x32.as<float>(), a_hi.as<bf16>(),
                              (last && bsplit) ? a_lo.as<bf16>() : nullptr, num_sms, stream, f16 ? 1 : 0,
                              (direct_compact && i == L - 2) ? inv_map.as<int>() : nullptr));
          }
        }
      }
      if (L == 0) {
        // no attention layers: only the whitening LN (model/imf_vad.py:117)
        IEF_PROF(KC_LAYERNORM, double(M) * D * 8, layernorm(x32.as<float>(), M, D, whiten_w[m], whiten_b[m], nullptr, nullptr, 1e-5f,
                          fp32_plan ? y32.as<float>() : nullptr, fp32_plan ? nullptr : a_hi.as<bf16>(),
                          bsplit ? a_lo.as<bf16>() : nullptr, num_sms, stream, f16 ? 1 : 0));
        if (fp32_plan) IEF_CUDA(cudaMemcpyAsync(x32.p, y32.p, size_t(M) * D * 4, cudaMemcpyDeviceToDevice, stream));
      }
      // heads (:125-128): one [M, D] x [2D, D]^T GEMM per modality, mu and logvar written to the user tensors
      EpiParams eh;
      eh.bias = heads[m].b; eh.out_f32 = mu_out[m] + out0 * D; eh.out_f32_b = lv_out[m] + out0 * D; eh.ld_f32 = D;
      eh.split_col = D;
      if (Mo == 0 || hf) continue;
      if (fp32_plan) {
        IEF_PROF(KC_GEMM_SIMT, 4.0 * Mo * D * D, gemm_simt(x32.as<float>(), D, heads[m].w, D, int(Mo), 2 * D, D, eh, stream));
      } else {
        GemmTcArgs gh;
        gh.A_hi = (ln_fused && vr) ? h_lo.as<bf16>() : a_hi.as<bf16>(); gh.A_lo = a_lo.as<bf16>();
        gh.W_hi = f16 ? heads[m].w_h16 : heads[m].w_hi; gh.W_lo = heads[m].w_lo;
        gh.M = int(Mo); gh.N = 2 * D; gh.K = D; gh.lda = D; gh.ldw = D;
        gh.nsplit = bsplit ? 3 : 1;
        gh.fp16 = f16 ? 1 : 0;
        IEF_PROF(KC_GEMM_HEADS, 4.0 * Mo * D * D, gemm_tc(gh, eh, num_sms, stream));
      }
    }
    if (Mo == 0) continue;
    // uncertainty-weighted fusion (:130-144)
    float* fused_out = fused + out0 * D;
    // fp16 refinement: the residual stream lives as an fp16 pair x = hi + lo (hi is the GEMM operand anyway), so a
    // refinement step moves 7.5 KB per row through HBM instead of 12 KB (no separate fp32 copy of x)
    const bool pair16 = f16 && R > 0;
    float* xcur = (R == 0) ? fused_out : (pair16 ? nullptr : x32.as<float>());
    if (hf) {
      HeadsFuseArgs ha;
      ha.x_i = x32.p; ha.x_e = h_lo.p; ha.w_i16 = heads[0].w_h16; ha.w_e16 = heads[1].w_h16; ha.b_i = heads[0].b; ha.b_e = heads[1].b;
      ha.factor = factor; ha.eps = eps; ha.out_hi = a_hi.p; ha.out_lo = a_lo.p; ha.M = Mo;
      IEF_PROF(KC_HEADS_FUSE, 8.0 * Mo * D * D, heads_fuse(ha, num_sms, stream));
    } else {
      bf16* f_hi = (fp32_plan || R == 0) ? nullptr : a_hi.as<bf16>();
      bf16* f_lo = f_hi ? a_lo.as<bf16>() : nullptr;     // both tensor-core plans start the refinement from a hi + lo pair
      const double fuse_bytes = double(Mo) * D * (16 + (w_i ? 8 : 0) + (xcur ? 4 : 0) + (f_hi ? 2 : 0) + (f_lo ? 2 : 0));
      if (eval_wi_mean && eval_we_mean && !w_i)      // the evaluation loop's w_i.mean(-1) / w_e.mean(-1), train/ucf_test.py:124-131
        IEF_PROF(KC_FUSE, fuse_bytes, fuse_rows(image_mu + out0 * D, event_mu + out0 * D, image_logvar + out0 * D, event_logvar + out0 * D,
                 Mo, D, factor, eps, eval_wi_mean + out0, eval_we_mean + out0, xcur, f_hi, f_lo, num_sms, stream, f16 ? 1 : 0));
      else
        IEF_PROF(KC_FUSE, fuse_bytes, fuse(image_mu + out0 * D, event_mu + out0 * D, image_logvar + out0 * D, event_logvar + out0 * D, Mo * D,
                 factor, eps, w_i ? w_i + out0 * D : nullptr, w_e ? w_e + out0 * D : nullptr, xcur, f_hi, f_lo, num_sms, stream, f16 ? 1 : 0));
    }
    // iterative refinement (:146-149): x <- x - lambda * (W2 relu(W1 x + b1) + b2)
    // fp16-pair stream with enough rows: ONE persistent kernel keeps each 256-row tile on chip for all R steps
    bool chain = pair16 && D == kRefineDim && R <= kRefineMaxSteps && refine_contig && refine_fused != 0;
    if (chain && refine_fused < 0) chain = refine_chain_preferred(Mo, num_sms);
    if (chain) {
      RefineChainArgs ra;
      ra.x_hi = a_hi.p; ra.x_lo = a_lo.p; ra.w16 = ref1[0].w_h16;
      for (int i = 0; i < R; ++i) { ra.b1[i] = ref1[i].b; ra.b2[i] = ref2[i].b; }
      ra.steps = R; ra.lambda = lambda_ref; ra.M = Mo; ra.out_f32 = fused_out; ra.lo_scratch = h_hi.p;
      IEF_CHECK(refine_chain_scratch_bytes(Mo) <= h_hi.bytes, "forward: refinement scratch too small");
      IEF_PROF(KC_REFINE_FUSED, 4.0 * R * Mo * D * D, refine_chain(ra, num_sms, stream));
    }
    for (int i = 0; i < (chain ? 0 : R); ++i) {
      const bool last = (i == R - 1);
      float* xnext = last ? fused_out : x32.as<float>();
      if (fp32_plan) {
        EpiParams e1;
        e1.bias = ref1[i].b; e1.act = ACT_RELU; e1.out_f32 = h32.as<float>(); e1.ld_f32 = D;
        IEF_PROF(KC_GEMM_SIMT, 2.0 * Mo * D * D, gemm_simt(x32.as<float>(), D, ref1[i].w, D, int(Mo), D, D, e1, stream));
        EpiParams e2;
        e2.bias = ref2[i].b; e2.resid = x32.as<float>(); e2.ld_resid = D; e2.alpha = -lambda_ref;
        e2.out_f32 = xnext; e2.ld_f32 = D;
        IEF_PROF(KC_GEMM_SIMT, 2.0 * Mo * D * D, gemm_simt(h32.as<float>(), D, ref2[i].w, D, int(Mo), D, D, e2, stream));
      } else {
        EpiParams e1;
        e1.bias = ref1[i].b; e1.act = ACT_RELU; e1.out_hi = h_hi.as<bf16>(); e1.out_lo = bsplit ? h_lo.as<bf16>() : nullptr;
        e1.ld_bf = D; e1.hi_fp16 = f16 ? 1 : 0;
        GemmTcArgs g1;
        g1.A_hi = a_hi.as<bf16>(); g1.A_lo = a_lo.as<bf16>(); g1.W_hi = f16 ? ref1[i].w_h16 : ref1[i].w_hi; g1.W_lo = ref1[i].w_lo;
        g1.M = int(Mo); g1.N = D; g1.K = D; g1.lda = D; g1.ldw = D; g1.nsplit = bsplit ? 3 : 1; g1.fp16 = f16 ? 1 : 0;
        IEF_PROF(KC_GEMM_REF1, 2.0 * Mo * D * D, gemm_tc(g1, e1, num_sms, stream));
        EpiParams e2;
        e2.bias = ref2[i].b; e2.resid = x32.as<float>(); e2.ld_resid = D; e2.alpha = -lambda_ref;
        e2.out_f32 = xnext; e2.ld_f32 = D;
        if (!last) { e2.out_hi = a_hi.as<bf16>(); e2.out_lo = a_lo.as<bf16>(); e2.ld_bf = D; e2.hi_fp16 = f16 ? 1 : 0; }
        if (f16) {
          e2.resid = nullptr; e2.resid_h16 = a_hi.as<bf16>(); e2.resid_l16 = a_lo.as<bf16>();
          if (!last) e2.out_f32 = nullptr;          // x stays an fp16 pair until the last step writes `fused`
        }
        GemmTcArgs g2;
        g2.A_hi = h_hi.as<bf16>(); g2.A_lo = h_lo.as<bf16>(); g2.W_hi = f16 ? ref2[i].w_h16 : ref2[i].w_hi; g2.W_lo = ref2[i].w_lo;
        g2.M = int(Mo); g2.N = D; g2.K = D; g2.lda = D; g2.ldw = D; g2.nsplit = bsplit ? 3 : 1; g2.fp16 = f16 ? 1 : 0;
        IEF_PROF(KC_GEMM_REF2, 2.0 * Mo * D * D, gemm_tc(g2, e2, num_sms, stream));
      }
    }
    // classifier (:150) stays fp32 in every plan
    IEF_PROF(KC_CLASSIFIER, double(Mo) * D * 4, classifier(fused_out, Mo, D, cls_w, cls_b, logits + out0, scores ? scores + out0 : nullptr, num_sms, stream, status.as<int>()));
  }
  return IEFVAD_OK;
}

void Model::destroy() {
  DevBuf* all[] = {&params_f32, &params_hi, &params_lo, &params_h16, &x32, &y32, &a_hi, &a_lo, &h_hi, &h_lo,
                   &qb, &kb, &vtb, &qkv32, &attn32, &h32, &inv_map, &items_dev, &aux_dev, &status, &ln_scratch, &ln_ident};
  for (DevBuf* b : all) b->release();
}

}  // namespace iefvad
