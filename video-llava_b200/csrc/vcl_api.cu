// C ABI of libvcl.so (declared in include/vcl.h): handle, weight repacking, and the launch
// sequences for the three stages of the hot path (SURVEY.md section 3.2):
//   vcl_clip_encode    CLIP ViT over the sampled frames
//   vcl_st_pool        spatio-temporal mean pool
//   vcl_llm_prefill / vcl_llm_decode_step / vcl_llm_generate   projector + splice + LLaMA
// Host code here only sequences kernels on the caller's stream; it never synchronises on the
// compute path and never touches a CPU implementation.
#include "../../include/vcl.h"

#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <map>
#include <string>
#include <vector>

#include "common.cuh"
#include "kernels.h"

namespace vcl {

static thread_local char g_err[1024] = "";
static long long g_launches = 0;

// Every kernel launcher calls count_launches(1); graph replays add their node count.
void count_launches(long long n) { g_launches += n; }
long long launch_count() { return g_launches; }

void set_last_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

}  // namespace vcl

using namespace vcl;

namespace {

struct ClipLayerW {
  bf16 *ln1_w, *ln1_b, *wqkv, *bqkv, *wo, *bo, *ln2_w, *ln2_b, *w1, *b1, *w2, *b2;
};
struct LlmLayerW {
  bf16 *ln1, *wqkv, *wo, *ln2, *wgu, *wd;
  bf16 *wqkv_t = nullptr, *wo_t = nullptr, *wgu_t = nullptr, *wd_t = nullptr;   // tiled copies for B = 1 decode
};
enum DecodeMode { MODE_GREEDY = 0, MODE_SAMPLED = 1 };
struct GraphEntry {
  int B, S, n_new;     // S = -1: the prompt length is read on the device (h->d_pos), any S replays it
  int mode;            // DecodeMode; a sampled graph reads its parameters from h->d_sample
  cudaGraphExec_t exec;
  long long kernels;   // kernel nodes in the graph (for vcl_launch_count)
  unsigned long long last_use;
};
constexpr size_t MAX_DECODE_GRAPHS = 6;   // LRU-bounded: an instantiated graph holds ~5 000 kernel nodes

// what one decode step reads and leaves behind
struct StepIo {
  const int32_t* tok_in = nullptr; long long in_stride = 1;      // the token fed at this step ...
  bool tok_from_partials = false;                                // ... or: the arg-max of the previous step's partials
  int32_t* tok_store = nullptr; long long store_stride = 1;      // where that reduced token is recorded
  bool partials_out = false;      // leave this step's arg-max as per-CTA partials for the next step (no arg-max kernel)
  float* logits_out = nullptr;
  int32_t* tok_out = nullptr; long long out_stride = 1;
  const int* pos_dev = nullptr;   // position = pos + *pos_dev
  bool sample = false;            // tok_out is sampled with the parameters in h->d_sample instead of the arg-max
};

}  // namespace

struct vcl_handle {
  vcl_config cfg;
  int P = 0;         // patches per frame
  int KP = 0;        // padded im2col width
  int NV = 0;        // video tokens per clip = n_temporal + P
  std::vector<void*> allocs;
  bool clip_loaded = false, llm_loaded = false;
  // CLIP weights
  bf16 *patch_w = nullptr, *cls = nullptr, *pos = nullptr, *pre_w = nullptr, *pre_b = nullptr;
  std::vector<ClipLayerW> cl;
  // LLM weights
  bf16 *embed = nullptr, *norm_w = nullptr, *lm_head = nullptr, *lm_head_t = nullptr;
  bf16 *proj_w0 = nullptr, *proj_b0 = nullptr, *proj_w1 = nullptr, *proj_b1 = nullptr;
  std::vector<LlmLayerW> ll;
  // CLIP activations (rows = max_frames * (P+1))
  bf16 *v_h = nullptr, *v_x = nullptr, *v_qkv = nullptr, *v_attn = nullptr, *v_act = nullptr;
  // LLM activations (rows = max_batch * max_seq)
  bf16 *l_h = nullptr, *l_x = nullptr, *l_qkv = nullptr, *l_attn = nullptr, *l_act = nullptr;
  bf16 *l_vid = nullptr, *l_vid_tmp = nullptr;
  bf16 *kcache = nullptr, *vcache = nullptr;   // [L][B][H][s_max][128]
  bf16 *rope_cos = nullptr, *rope_sin = nullptr;
  float* logits = nullptr;                     // [max_batch, vocab]
  int32_t* tokens = nullptr;                   // [max_batch, max_seq] generated-token scratch
  // decode activations ([max_batch, .])
  bf16 *d_h = nullptr, *d_x = nullptr, *d_q = nullptr, *d_qkv = nullptr, *d_attn = nullptr,
       *d_act = nullptr;
  std::vector<GraphEntry> graphs;
  unsigned long long graph_clock = 0;
  int* d_pos = nullptr;                        // prompt length of the running decode loop (device scalar)
  SampleParams* d_sample = nullptr;            // sampling parameters of the running sampled loop
  ArgmaxPart* amax = nullptr;                  // [#SMs][max_batch] per-CTA partial arg-max of the logits kernel
  bool force_legacy_attention = false;

  size_t cache_layer_elems() const {
    return (size_t)cfg.max_batch * cfg.llm_heads * cfg.max_seq * 128;
  }
};

namespace {

template <class T>
int dalloc(vcl_handle* h, T** p, size_t n) {
  void* q = nullptr;
  cudaError_t e = cudaMalloc(&q, n * sizeof(T) + 256);
  if (e != cudaSuccess) {
    set_last_error("cudaMalloc of %zu bytes failed: %s", n * sizeof(T), cudaGetErrorString(e));
    return -2;
  }
  h->allocs.push_back(q);
  *p = reinterpret_cast<T*>(q);
  return 0;
}

typedef std::map<std::string, const vcl_tensor*> TensorMap;

const vcl_tensor* find_tensor(const TensorMap& m, const std::string& name, int ndim, long long d0,
                              long long d1 = -1, long long d2 = -1, long long d3 = -1) {
  auto it = m.find(name);
  if (it == m.end()) {
    set_last_error("missing weight '%s'", name.c_str());
    return nullptr;
  }
  const vcl_tensor* t = it->second;
  const long long want[4] = {d0, d1, d2, d3};
  bool ok = t->ndim == ndim && t->data != nullptr;
  for (int i = 0; ok && i < ndim; ++i) ok = (t->shape[i] == want[i]);
  if (!ok) {
    set_last_error("weight '%s' has shape [%lld,%lld,%lld,%lld] (ndim %d), expected [%lld,%lld,%lld,%lld] (ndim %d)",
                   name.c_str(), (long long)t->shape[0], (long long)t->shape[1],
                   (long long)t->shape[2], (long long)t->shape[3], t->ndim, d0, d1, d2, d3, ndim);
    return nullptr;
  }
  return t;
}

// allocate dst and copy a whole tensor
int load_copy(vcl_handle* h, const TensorMap& m, const std::string& name, bf16** dst, int ndim,
              long long d0, long long d1 = -1, long long d2 = -1, long long d3 = -1) {
  const vcl_tensor* t = find_tensor(m, name, ndim, d0, d1, d2, d3);
  if (!t) return -1;
  size_t n = 1;
  for (int i = 0; i < ndim; ++i) n *= (size_t)t->shape[i];
  if (dalloc(h, dst, n) != 0) return -2;
  VCL_CUDA_OK(cudaMemcpy(*dst, t->data, n * sizeof(bf16), cudaMemcpyDeviceToDevice));
  return 0;
}

int check_device() {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) {
    set_last_error("no CUDA device: %s (libvcl has no CPU fallback)", cudaGetErrorString(e));
    return -2;
  }
  int major = 0;
  VCL_CUDA_OK(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev));
  VCL_REQUIRE(major == 10, "device compute capability %d.x is not sm_100 (B200); libvcl is sm_100a only",
              major);
  return 0;
}

cudaStream_t as_stream(void* s) { return reinterpret_cast<cudaStream_t>(s); }

}  // namespace

extern "C" {

int vcl_version(void) { return VCL_VERSION; }

const char* vcl_last_error(void) { return vcl::g_err; }

int vcl_create(vcl_handle** out, const vcl_config* c) {
  VCL_REQUIRE(out != nullptr && c != nullptr, "vcl_create: null argument");
  *out = nullptr;
  if (check_device() != 0) return -2;
  VCL_REQUIRE(c->clip_hidden > 0 && c->clip_heads > 0 && c->clip_hidden == c->clip_heads * 64,
              "vcl_create: CLIP head_dim must be 64 (hidden %d, heads %d)", c->clip_hidden, c->clip_heads);
  VCL_REQUIRE(c->clip_hidden % 256 == 0 && c->clip_inter % 256 == 0,
              "vcl_create: CLIP widths must be multiples of 256");
  VCL_REQUIRE(c->patch_size > 0 && c->image_size % c->patch_size == 0, "vcl_create: image/patch mismatch");
  VCL_REQUIRE(c->llm_hidden == c->llm_heads * 128, "vcl_create: LLM head_dim must be 128 (hidden %d, heads %d)",
              c->llm_hidden, c->llm_heads);
  VCL_REQUIRE(c->llm_hidden % 256 == 0 && c->llm_inter % 64 == 0, "vcl_create: LLM widths unsupported");
  VCL_REQUIRE(c->clip_layers >= 0 && c->llm_layers >= 0 && c->vocab > 0, "vcl_create: bad layer/vocab counts");
  VCL_REQUIRE(c->max_frames > 0 && c->max_batch > 0 && c->max_seq > 0, "vcl_create: capacities must be > 0");
  VCL_REQUIRE(c->proj_type == VCL_PROJ_LINEAR || c->proj_type == VCL_PROJ_MLP2X_GELU, "vcl_create: proj_type");

  vcl_handle* h = new vcl_handle();
  h->cfg = *c;
  const int G = c->image_size / c->patch_size;
  h->P = G * G;
  h->KP = ((3 * c->patch_size * c->patch_size + 63) / 64) * 64;
  h->NV = c->n_temporal + h->P;

  int rc = 0;
  rc |= init_gemm_kernels();
  rc |= init_attention_kernels();
  rc |= init_attention_tc_kernels();
  h->force_legacy_attention = getenv("VCL_LEGACY_ATTENTION") != nullptr;
  rc |= init_gemv_kernels();
  rc |= init_gemv_tc_kernels();
  rc |= init_gemv_mma_kernels();
  rc |= init_gemv_tcw_kernels();

  const size_t C = c->clip_hidden, F = c->clip_inter;
  const size_t Mv = (size_t)c->max_frames * (h->P + 1);
  const size_t act_elems = Mv * F > (size_t)c->max_frames * h->P * h->KP ? Mv * F
                                                                          : (size_t)c->max_frames * h->P * h->KP;
  rc |= dalloc(h, &h->v_h, Mv * C);
  rc |= dalloc(h, &h->v_x, Mv * C);
  rc |= dalloc(h, &h->v_qkv, Mv * 3 * C);
  rc |= dalloc(h, &h->v_attn, Mv * C);
  rc |= dalloc(h, &h->v_act, act_elems);

  const size_t D = c->llm_hidden, LF = c->llm_inter;
  const size_t Ml = (size_t)c->max_batch * c->max_seq;
  rc |= dalloc(h, &h->l_h, Ml * D);
  rc |= dalloc(h, &h->l_x, Ml * D);
  rc |= dalloc(h, &h->l_qkv, Ml * 3 * D);
  rc |= dalloc(h, &h->l_attn, Ml * D);
  rc |= dalloc(h, &h->l_act, Ml * LF);
  rc |= dalloc(h, &h->l_vid, (size_t)c->max_batch * h->NV * D);
  rc |= dalloc(h, &h->l_vid_tmp, (size_t)c->max_batch * h->NV * D);
  rc |= dalloc(h, &h->kcache, (size_t)c->llm_layers * h->cache_layer_elems());
  rc |= dalloc(h, &h->vcache, (size_t)c->llm_layers * h->cache_layer_elems());
  rc |= dalloc(h, &h->rope_cos, (size_t)c->max_seq * 64);
  rc |= dalloc(h, &h->rope_sin, (size_t)c->max_seq * 64);
  rc |= dalloc(h, &h->logits, (size_t)c->max_batch * c->vocab);
  rc |= dalloc(h, &h->tokens, (size_t)c->max_batch * c->max_seq);
  const size_t Bm = c->max_batch;
  rc |= dalloc(h, &h->d_h, Bm * D);
  rc |= dalloc(h, &h->d_x, xwin_elems((int)Bm, (int)D) > Bm * D ? xwin_elems((int)Bm, (int)D) : Bm * D);
  rc |= dalloc(h, &h->d_q, Bm * D);
  rc |= dalloc(h, &h->d_qkv, Bm * 3 * D);
  rc |= dalloc(h, &h->d_attn, xwin_elems((int)Bm, (int)D) > Bm * D ? xwin_elems((int)Bm, (int)D) : Bm * D);
  rc |= dalloc(h, &h->d_act, xwin_elems((int)Bm, (int)LF) > Bm * LF ? xwin_elems((int)Bm, (int)LF) : Bm * LF);
  rc |= dalloc(h, &h->d_pos, 4);
  rc |= dalloc(h, &h->d_sample, 1);
  rc |= dalloc(h, &h->amax, (size_t)device_num_sms() * Bm);
  if (rc == 0) rc = launch_rope_table(h->rope_cos, h->rope_sin, c->max_seq, 128, c->rope_theta, 0);
  if (rc == 0) {
    cudaError_t e = cudaDeviceSynchronize();
    if (e != cudaSuccess) {
      set_last_error("vcl_create: %s", cudaGetErrorString(e));
      rc = -2;
    }
  }
  if (rc != 0) {
    vcl_destroy(h);
    return -2;
  }
  *out = h;
  return 0;
}

void vcl_destroy(vcl_handle* h) {
  if (!h) return;
  for (auto& g : h->graphs) cudaGraphExecDestroy(g.exec);
  for (void* p : h->allocs) cudaFree(p);
  delete h;
}

int vcl_load_clip_weights(vcl_handle* h, const vcl_tensor* tensors, int n) {
  VCL_REQUIRE(h && tensors && n > 0, "vcl_load_clip_weights: null argument");
  VCL_REQUIRE(!h->clip_loaded, "vcl_load_clip_weights: already loaded");
  TensorMap m;
  for (int i = 0; i < n; ++i)
    if (tensors[i].name) m[tensors[i].name] = &tensors[i];
  const vcl_config& c = h->cfg;
  const long long C = c.clip_hidden, F = c.clip_inter, ps = c.patch_size;
  const std::string pre = "vision_model.";
  // patch embedding [C,3,ps,ps] -> [C, KP] zero padded along K
  {
    const vcl_tensor* t = find_tensor(m, pre + "embeddings.patch_embedding.weight", 4, C, 3, ps, ps);
    if (!t) return -1;
    if (dalloc(h, &h->patch_w, (size_t)C * h->KP) != 0) return -2;
    VCL_CUDA_OK(cudaMemset(h->patch_w, 0, (size_t)C * h->KP * 2));
    const size_t k = 3 * ps * ps;
    VCL_CUDA_OK(cudaMemcpy2D(h->patch_w, (size_t)h->KP * 2, t->data, k * 2, k * 2, C,
                             cudaMemcpyDeviceToDevice));
  }
  if (load_copy(h, m, pre + "embeddings.class_embedding", &h->cls, 1, C)) return -1;
  if (load_copy(h, m, pre + "embeddings.position_embedding.weight", &h->pos, 2, h->P + 1, C)) return -1;
  if (load_copy(h, m, pre + "pre_layrnorm.weight", &h->pre_w, 1, C)) return -1;
  if (load_copy(h, m, pre + "pre_layrnorm.bias", &h->pre_b, 1, C)) return -1;
  h->cl.resize(c.clip_layers);
  for (int l = 0; l < c.clip_layers; ++l) {
    ClipLayerW& w = h->cl[l];
    const std::string lp = pre + "encoder.layers." + std::to_string(l) + ".";
    if (load_copy(h, m, lp + "layer_norm1.weight", &w.ln1_w, 1, C)) return -1;
    if (load_copy(h, m, lp + "layer_norm1.bias", &w.ln1_b, 1, C)) return -1;
    if (load_copy(h, m, lp + "layer_norm2.weight", &w.ln2_w, 1, C)) return -1;
    if (load_copy(h, m, lp + "layer_norm2.bias", &w.ln2_b, 1, C)) return -1;
    if (dalloc(h, &w.wqkv, (size_t)3 * C * C) || dalloc(h, &w.bqkv, (size_t)3 * C)) return -2;
    const char* nm[3] = {"q_proj", "k_proj", "v_proj"};
    for (int j = 0; j < 3; ++j) {
      const vcl_tensor* tw = find_tensor(m, lp + "self_attn." + nm[j] + ".weight", 2, C, C);
      const vcl_tensor* tb = find_tensor(m, lp + "self_attn." + nm[j] + ".bias", 1, C);
      if (!tw || !tb) return -1;
      VCL_CUDA_OK(cudaMemcpy(w.wqkv + (size_t)j * C * C, tw->data, (size_t)C * C * 2, cudaMemcpyDeviceToDevice));
      VCL_CUDA_OK(cudaMemcpy(w.bqkv + (size_t)j * C, tb->data, (size_t)C * 2, cudaMemcpyDeviceToDevice));
    }
    if (load_copy(h, m, lp + "self_attn.out_proj.weight", &w.wo, 2, C, C)) return -1;
    if (load_copy(h, m, lp + "self_attn.out_proj.bias", &w.bo, 1, C)) return -1;
    if (load_copy(h, m, lp + "mlp.fc1.weight", &w.w1, 2, F, C)) return -1;
    if (load_copy(h, m, lp + "mlp.fc1.bias", &w.b1, 1, F)) return -1;
    if (load_copy(h, m, lp + "mlp.fc2.weight", &w.w2, 2, C, F)) return -1;
    if (load_copy(h, m, lp + "mlp.fc2.bias", &w.b2, 1, C)) return -1;
  }
  VCL_CUDA_OK(cudaDeviceSynchronize());
  h->clip_loaded = true;
  return 0;
}

int vcl_load_llm_weights(vcl_handle* h, const vcl_tensor* tensors, int n) {
  VCL_REQUIRE(h && tensors && n > 0, "vcl_load_llm_weights: null argument");
  VCL_REQUIRE(!h->llm_loaded, "vcl_load_llm_weights: already loaded");
  TensorMap m;
  for (int i = 0; i < n; ++i)
    if (tensors[i].name) m[tensors[i].name] = &tensors[i];
  const vcl_config& c = h->cfg;
  const long long D = c.llm_hidden, F = c.llm_inter, V = c.vocab, CV = c.clip_hidden;
  if (load_copy(h, m, "model.embed_tokens.weight", &h->embed, 2, V, D)) return -1;
  if (load_copy(h, m, "model.norm.weight", &h->norm_w, 1, D)) return -1;
  if (load_copy(h, m, "lm_head.weight", &h->lm_head, 2, V, D)) return -1;
  if (c.proj_type == VCL_PROJ_LINEAR) {
    if (load_copy(h, m, "model.mm_projector.weight", &h->proj_w0, 2, D, CV)) return -1;
    if (load_copy(h, m, "model.mm_projector.bias", &h->proj_b0, 1, D)) return -1;
  } else {
    if (load_copy(h, m, "model.mm_projector.0.weight", &h->proj_w0, 2, D, CV)) return -1;
    if (load_copy(h, m, "model.mm_projector.0.bias", &h->proj_b0, 1, D)) return -1;
    if (load_copy(h, m, "model.mm_projector.2.weight", &h->proj_w1, 2, D, D)) return -1;
    if (load_copy(h, m, "model.mm_projector.2.bias", &h->proj_b1, 1, D)) return -1;
  }
  h->ll.resize(c.llm_layers);
  for (int l = 0; l < c.llm_layers; ++l) {
    LlmLayerW& w = h->ll[l];
    const std::string lp = "model.layers." + std::to_string(l) + ".";
    if (load_copy(h, m, lp + "input_layernorm.weight", &w.ln1, 1, D)) return -1;
    if (load_copy(h, m, lp + "post_attention_layernorm.weight", &w.ln2, 1, D)) return -1;
    if (dalloc(h, &w.wqkv, (size_t)3 * D * D)) return -2;
    const char* nm[3] = {"q_proj", "k_proj", "v_proj"};
    for (int j = 0; j < 3; ++j) {
      const vcl_tensor* tw = find_tensor(m, lp + "self_attn." + nm[j] + ".weight", 2, D, D);
      if (!tw) return -1;
      VCL_CUDA_OK(cudaMemcpy(w.wqkv + (size_t)j * D * D, tw->data, (size_t)D * D * 2, cudaMemcpyDeviceToDevice));
    }
    if (load_copy(h, m, lp + "self_attn.o_proj.weight", &w.wo, 2, D, D)) return -1;
    // gate/up interleaved by row: row 2j = gate_j, row 2j+1 = up_j
    const vcl_tensor* tg = find_tensor(m, lp + "mlp.gate_proj.weight", 2, F, D);
    const vcl_tensor* tu = find_tensor(m, lp + "mlp.up_proj.weight", 2, F, D);
    if (!tg || !tu) return -1;
    if (dalloc(h, &w.wgu, (size_t)2 * F * D)) return -2;
    VCL_CUDA_OK(cudaMemcpy2D(w.wgu, (size_t)2 * D * 2, tg->data, (size_t)D * 2, (size_t)D * 2, F,
                             cudaMemcpyDeviceToDevice));
    VCL_CUDA_OK(cudaMemcpy2D(w.wgu + D, (size_t)2 * D * 2, tu->data, (size_t)D * 2, (size_t)D * 2, F,
                             cudaMemcpyDeviceToDevice));
    if (load_copy(h, m, lp + "mlp.down_proj.weight", &w.wd, 2, D, F)) return -1;
  }
  // Decode-only second copy of every streamed matrix in the tile order of gemv_tc.cu (one bulk
  // copy per 16 KB slot). 13.2 GB more for the 7B model, 25.7 GB for 13B - HBM is 180 GB.
  if (getenv("VCL_NO_TILED_WEIGHTS") == nullptr && D % 32 == 0 && F % 32 == 0) {
    auto tiled = [&](const bf16* src, bf16** dst, int N, int K, bool qkv) -> int {
      if (dalloc(h, dst, gemv_tc_tiled_elems(N, K))) return -2;
      return launch_gemv_tc_repack(src, *dst, N, K, qkv, nullptr);
    };
    for (int l = 0; l < c.llm_layers; ++l) {
      LlmLayerW& w = h->ll[l];
      if (tiled(w.wqkv, &w.wqkv_t, 3 * D, D, true) || tiled(w.wo, &w.wo_t, D, D, false) ||
          tiled(w.wgu, &w.wgu_t, 2 * F, D, false) || tiled(w.wd, &w.wd_t, D, F, false)) return -2;
    }
    if (tiled(h->lm_head, &h->lm_head_t, V, D, false)) return -2;
  }
  VCL_CUDA_OK(cudaDeviceSynchronize());
  h->llm_loaded = true;
  return 0;
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------
// launch sequences
// ---------------------------------------------------------------------------------------------
namespace {

#define VCL_TRY(expr)        \
  do {                       \
    int _rc = (expr);        \
    if (_rc != 0) return _rc; \
  } while (0)

int gemm(const bf16* A, long long lda, const bf16* W, long long ldw, bf16* C, long long ldc,
         const bf16* bias, const bf16* res, long long ldr, int M, int N, int K, int act,
         cudaStream_t st, int block_n = 0, int cluster = 0) {
  GemmArgs g;
  g.cluster = cluster;
  g.A = A; g.lda = lda; g.W = W; g.ldw = ldw; g.C = C; g.ldc = ldc; g.bias = bias;
  g.residual = res; g.ldr = ldr; g.M = M; g.N = N; g.K = K; g.act = act; g.block_n = block_n;
  return launch_gemm_bf16_tn(g, st);
}

// CLIP ViT: leaves hidden_states[n_layers] in h->v_h ([n_frames, P+1, C])
int clip_forward(vcl_handle* h, const void* pixels, int fmt, int n_frames, int n_layers,
                 cudaStream_t st) {
  const vcl_config& c = h->cfg;
  VCL_REQUIRE(h->clip_loaded, "CLIP weights are not loaded");
  VCL_REQUIRE(n_frames > 0 && n_frames <= c.max_frames, "n_frames=%d outside 1..%d", n_frames, c.max_frames);
  VCL_REQUIRE(n_layers >= 0 && n_layers <= c.clip_layers, "n_layers=%d outside 0..%d", n_layers, c.clip_layers);
  VCL_REQUIRE(fmt == VCL_PIXELS_BF16_NCHW || fmt == VCL_PIXELS_U8_NHWC, "unknown pixel format %d", fmt);
  const int C = c.clip_hidden, F = c.clip_inter, P = h->P, S = P + 1;
  const int M = n_frames * S;
  bf16* patchA = h->v_act;      // [n_frames*P, KP]   (aliases the MLP buffer, dead before layer 0)
  bf16* patch_out = h->v_qkv;   // [n_frames*P, C]
  VCL_TRY(launch_im2col(pixels, fmt, patchA, n_frames, c.image_size, c.patch_size, h->KP, st));
  VCL_TRY(gemm(patchA, h->KP, h->patch_w, h->KP, patch_out, C, nullptr, nullptr, 0, n_frames * P, C,
               h->KP, ACT_NONE, st));
  VCL_TRY(launch_clip_embed_ln(patch_out, h->cls, h->pos, h->pre_w, h->pre_b, h->v_h, n_frames, P, C,
                               c.clip_ln_eps, st));
  const float scale = 0.125f;  // head_dim 64 ^ -1/2
  for (int l = 0; l < n_layers; ++l) {
    const ClipLayerW& w = h->cl[l];
    VCL_TRY(launch_layernorm(h->v_h, C, h->v_x, C, w.ln1_w, w.ln1_b, M, C, c.clip_ln_eps, st));
    VCL_TRY(gemm(h->v_x, C, w.wqkv, C, h->v_qkv, 3 * C, w.bqkv, nullptr, 0, M, 3 * C, C, ACT_NONE, st));
    AttnArgs a;
    a.q = h->v_qkv;         a.q_sb = (long long)S * 3 * C; a.q_sh = 64; a.q_ss = 3 * C;
    a.k = h->v_qkv + C;     a.k_sb = a.q_sb; a.k_sh = 64; a.k_ss = 3 * C;
    a.v = h->v_qkv + 2 * C; a.v_sb = a.q_sb; a.v_sh = 64; a.v_ss = 3 * C;
    a.o = h->v_attn;        a.o_sb = (long long)S * C; a.o_sh = 64; a.o_ss = C;
    a.B = n_frames; a.H = c.clip_heads; a.S = S; a.head_dim = 64; a.scale = scale; a.causal = 0;
    if (S >= 129 && S <= 257 && !h->force_legacy_attention) {
      VCL_TRY(launch_attention_vit_tc(h->v_qkv, h->v_attn, n_frames, S, c.clip_heads, C, st));
    } else {
      VCL_TRY(launch_attention(a, st));   // 336-px tower (S = 577): flash-style mma.sync kernel
    }
    VCL_TRY(gemm(h->v_attn, C, w.wo, C, h->v_h, C, w.bo, h->v_h, C, M, C, C, ACT_NONE, st));
    VCL_TRY(launch_layernorm(h->v_h, C, h->v_x, C, w.ln2_w, w.ln2_b, M, C, c.clip_ln_eps, st));
    VCL_TRY(gemm(h->v_x, C, w.w1, C, h->v_act, F, w.b1, nullptr, 0, M, F, C, ACT_QGELU, st));
    VCL_TRY(gemm(h->v_act, F, w.w2, F, h->v_h, C, w.b2, h->v_h, C, M, C, F, ACT_NONE, st));
  }
  return 0;
}

bf16* kc_layer(vcl_handle* h, int l) { return h->kcache + (size_t)l * h->cache_layer_elems(); }
bf16* vc_layer(vcl_handle* h, int l) { return h->vcache + (size_t)l * h->cache_layer_elems(); }

// 1..4 clips take the ring-kernel family (gemv_tc, activation vectors of all clips in shared memory)
// when every projection of the model fits its shared-memory plan; 5..16 clips use gemv_mma
static bool tc_batch(vcl_handle* h, int B) {
  if (B < 1 || B > 4 || h->lm_head_t == nullptr || h->ll.empty()) return false;
  const vcl_config& c = h->cfg;
  const int D = c.llm_hidden, F = c.llm_inter;
  const int shapes[5][2] = {{3 * D, D}, {D, D}, {2 * F, D}, {D, F}, {c.vocab, D}};
  for (const auto& nk : shapes) {
    GemvArgs g;
    g.x = h->d_h; g.ldx = nk[1]; g.W = h->lm_head; g.W_tiled = h->lm_head_t; g.B = B; g.N = nk[0]; g.K = nk[1];
    if (!gemv_tc_supported(g)) return false;
  }
  return true;
}

// final RMSNorm + lm_head on rows x[b*ldx .. ] (b < B), arg-max
// partials_out: the arg-max is left as per-CTA partials in h->amax for the next step's q|k|v kernel
// sample_pos >= 0: tok_out is sampled (parameters in h->d_sample) for sequence position sample_pos (+ *pos_dev)
int lm_head_argmax(vcl_handle* h, const bf16* x, long long ldx, int B, float* logits_out,
                   int32_t* tok_out, long long tok_stride, cudaStream_t st, bool partials_out = false,
                   int sample_pos = -1, const int* pos_dev = nullptr) {
  const vcl_config& c = h->cfg;
  if (partials_out) {
    GemvArgs g;
    g.x = x; g.ldx = ldx; g.W = h->lm_head; g.W_tiled = h->lm_head_t; g.B = B; g.N = c.vocab;
    g.K = c.llm_hidden; g.norm_w = h->norm_w; g.eps = c.rms_eps; g.amax_out = h->amax;
    return launch_gemv_tc_logits(g, nullptr, c.vocab, st);
  }
  if (B >= 2 && !tc_batch(h, B)) {
    // small batches: normalise the B rows once, then the mma.sync weight-streaming kernel
    for (int b0 = 0; b0 < B; b0 += 16) {
      const int nb = B - b0 < 16 ? B - b0 : 16;
      GemvArgs g;
      g.x = h->d_x; g.ldx = c.llm_hidden; g.W = h->lm_head; g.W_tiled = h->lm_head_t; g.B = nb; g.N = c.vocab; g.K = c.llm_hidden;
      if (gemv_tcw_supported(g)) {
        VCL_TRY(launch_xwin_norm(x + (long long)b0 * ldx, ldx, h->d_x, h->norm_w, nb, c.llm_hidden, c.rms_eps, st));
        VCL_TRY(launch_gemv_tcw_logits(g, h->logits + (size_t)b0 * c.vocab, c.vocab, st));
      } else {
        VCL_TRY(launch_rmsnorm(x + (long long)b0 * ldx, ldx, h->d_x, c.llm_hidden, h->norm_w, nb, c.llm_hidden,
                               c.rms_eps, st));
        VCL_TRY(launch_gemv_mma_logits(g, h->logits + (size_t)b0 * c.vocab, c.vocab, st));
      }
    }
  } else
  for (int b0 = 0; b0 < B; b0 += 4) {
    const int nb = B - b0 < 4 ? B - b0 : 4;
    GemvArgs g;
    g.x = x + (long long)b0 * ldx; g.ldx = ldx; g.W = h->lm_head; g.W_tiled = h->lm_head_t; g.B = nb; g.N = c.vocab;
    g.K = c.llm_hidden; g.norm_w = h->norm_w; g.eps = c.rms_eps;
    VCL_TRY(launch_gemv_logits(g, h->logits + (size_t)b0 * c.vocab, c.vocab, st));
  }
  if (logits_out != nullptr && logits_out != h->logits)
    VCL_CUDA_OK(cudaMemcpyAsync(logits_out, h->logits, (size_t)B * c.vocab * sizeof(float),
                                cudaMemcpyDeviceToDevice, st));
  if (tok_out != nullptr) {
    if (sample_pos >= 0)
      VCL_TRY(launch_sample(h->logits, c.vocab, B, c.vocab, h->d_sample, SampleParams{}, sample_pos, pos_dev, tok_out,
                            tok_stride, st));
    else
      VCL_TRY(launch_argmax(h->logits, tok_out, tok_stride, B, c.vocab, st));
  }
  return 0;
}

// start_pos > 0 continues a cached sequence: the S new tokens take positions start_pos .. start_pos+S-1
// and attend to the whole cache (multi-turn reuse; no video span in a continuation).
// states_out (optional): [n_layers + 1][B][S][D], entry i = HF's hidden_states[i] (the raw output of
// layer i; entry 0 the spliced input embeddings), copied out as the stack advances.
int llm_prefill(vcl_handle* h, const int64_t* ids, const void* video_feats, const int32_t* vid_start,
                int B, int S, int n_layers, void* hidden_out, float* logits_out, int32_t* next_tok,
                long long tok_stride, cudaStream_t st, int start_pos = 0, void* states_out = nullptr) {
  const vcl_config& c = h->cfg;
  VCL_REQUIRE(h->llm_loaded, "LLM weights are not loaded");
  VCL_REQUIRE(B > 0 && B <= c.max_batch, "B=%d outside 1..%d", B, c.max_batch);
  VCL_REQUIRE(S > 0 && start_pos >= 0 && start_pos + S <= c.max_seq, "positions %d..%d outside the cache (max_seq %d)",
              start_pos, start_pos + S - 1, c.max_seq);
  VCL_REQUIRE(n_layers >= 0 && n_layers <= c.llm_layers, "n_layers=%d outside 0..%d", n_layers, c.llm_layers);
  VCL_REQUIRE(ids != nullptr && (vid_start != nullptr || start_pos > 0), "ids / vid_start are required");
  VCL_REQUIRE(start_pos == 0 || video_feats == nullptr, "a continuation cannot carry a video span");
  VCL_REQUIRE((logits_out == nullptr && next_tok == nullptr) || n_layers == c.llm_layers,
              "logits / next token need the full stack (n_layers == %d)", c.llm_layers);
  const int D = c.llm_hidden, F = c.llm_inter, H = c.llm_heads, NV = h->NV;
  const int M = B * S;
  if (video_feats != nullptr) {
    const bf16* vf = reinterpret_cast<const bf16*>(video_feats);
    if (c.proj_type == VCL_PROJ_LINEAR) {
      VCL_TRY(gemm(vf, c.clip_hidden, h->proj_w0, c.clip_hidden, h->l_vid, D, h->proj_b0, nullptr, 0,
                   B * NV, D, c.clip_hidden, ACT_NONE, st));
    } else {
      VCL_TRY(gemm(vf, c.clip_hidden, h->proj_w0, c.clip_hidden, h->l_vid_tmp, D, h->proj_b0, nullptr, 0,
                   B * NV, D, c.clip_hidden, ACT_GELU, st));
      VCL_TRY(gemm(h->l_vid_tmp, D, h->proj_w1, D, h->l_vid, D, h->proj_b1, nullptr, 0, B * NV, D, D,
                   ACT_NONE, st));
    }
  }
  VCL_TRY(launch_embed_splice(reinterpret_cast<const long long*>(ids), h->embed, h->l_vid, vid_start,
                              h->l_h, B, S, D, video_feats ? NV : 0, c.vocab, st));
  const float scale = 0.08838834764831845f;  // 128 ^ -1/2
  auto keep_state = [&](int i) -> int {
    if (states_out == nullptr) return 0;
    VCL_CUDA_OK(cudaMemcpyAsync(reinterpret_cast<bf16*>(states_out) + (size_t)i * M * D, h->l_h, (size_t)M * D * 2,
                                cudaMemcpyDeviceToDevice, st));
    return 0;
  };
  VCL_TRY(keep_state(0));
  for (int l = 0; l < n_layers; ++l) {
    const LlmLayerW& w = h->ll[l];
    VCL_TRY(launch_rmsnorm(h->l_h, D, h->l_x, D, w.ln1, M, D, c.rms_eps, st));
    // q|k|v projection with RoPE and the KV-cache write in its epilogue: q lands (rotated) in l_qkv, k and v in
    // the cache. VCL_PREFILL_ROPE_SEPARATE=1: plain GEMM + rope_kv_prefill_kernel (A/B)
    static const bool rope_separate = getenv("VCL_PREFILL_ROPE_SEPARATE") != nullptr;
    if (!rope_separate) {
      GemmArgs g;
      g.A = h->l_x; g.lda = D; g.W = w.wqkv; g.ldw = D; g.C = h->l_qkv; g.ldc = 3 * D; g.M = M; g.N = 3 * D; g.K = D;
      g.act = ACT_ROPE;
      g.rope.cos_t = h->rope_cos; g.rope.sin_t = h->rope_sin; g.rope.kcache = kc_layer(h, l); g.rope.vcache = vc_layer(h, l);
      g.rope.S = S; g.rope.start_pos = start_pos; g.rope.H = H; g.rope.s_max = c.max_seq;
      VCL_TRY(launch_gemm_bf16_tn(g, st));
    } else {
      VCL_TRY(gemm(h->l_x, D, w.wqkv, D, h->l_qkv, 3 * D, nullptr, nullptr, 0, M, 3 * D, D, ACT_NONE, st));
      VCL_TRY(launch_rope_kv_prefill(h->l_qkv, kc_layer(h, l), vc_layer(h, l), h->rope_cos, h->rope_sin, B,
                                     S, H, 128, c.max_seq, start_pos, st));
    }
    AttnArgs a;
    a.q = h->l_qkv; a.q_sb = (long long)S * 3 * D; a.q_sh = 128; a.q_ss = 3 * D;
    a.k = kc_layer(h, l); a.k_sb = (long long)H * c.max_seq * 128; a.k_sh = (long long)c.max_seq * 128; a.k_ss = 128;
    a.v = vc_layer(h, l); a.v_sb = a.k_sb; a.v_sh = a.k_sh; a.v_ss = 128;
    a.o = h->l_attn; a.o_sb = (long long)S * D; a.o_sh = 128; a.o_ss = D;
    a.B = B; a.H = H; a.S = S; a.head_dim = 128; a.scale = scale; a.causal = 1;
    a.S_kv = start_pos + S; a.q_off = start_pos;
    VCL_TRY(launch_attention(a, st));
    VCL_TRY(gemm(h->l_attn, D, w.wo, D, h->l_h, D, nullptr, h->l_h, D, M, D, D, ACT_NONE, st));
    VCL_TRY(launch_rmsnorm(h->l_h, D, h->l_x, D, w.ln2, M, D, c.rms_eps, st));
    VCL_TRY(gemm(h->l_x, D, w.wgu, D, h->l_act, F, nullptr, nullptr, 0, M, 2 * F, D, ACT_SWIGLU, st));
    VCL_TRY(gemm(h->l_act, F, w.wd, F, h->l_h, D, nullptr, h->l_h, D, M, D, F, ACT_NONE, st));
    VCL_TRY(keep_state(l + 1));
  }
  if (hidden_out != nullptr)
    VCL_CUDA_OK(cudaMemcpyAsync(hidden_out, h->l_h, (size_t)M * D * 2, cudaMemcpyDeviceToDevice, st));
  if (logits_out != nullptr || next_tok != nullptr)
    VCL_TRY(lm_head_argmax(h, h->l_h + (size_t)(S - 1) * D, (long long)S * D, B, logits_out, next_tok,
                           tok_stride, st));
  return 0;
}

// One decode step: the token of io is fed at position pos (+ *io.pos_dev).
int llm_decode_step(vcl_handle* h, const StepIo& io, int B, int pos, cudaStream_t st) {
  const vcl_config& c = h->cfg;
  const int D = c.llm_hidden, F = c.llm_inter, H = c.llm_heads;
  const float scale = 0.08838834764831845f;
  const int* pd = io.pos_dev;
  VCL_REQUIRE(pos >= 0 && pos < c.max_seq, "decode position %d outside the cache (max_seq %d)", pos, c.max_seq);
  const bool tc = tc_batch(h, B);
  // On the ring-kernel path the embedding lookup is part of layer 0's q|k|v kernel (and with it the
  // arg-max of the previous step); every other path gathers the rows with a kernel of its own.
  const bool fused_embed = tc && c.llm_layers > 0;
  VCL_REQUIRE(fused_embed || (!io.tok_from_partials && !io.partials_out), "partial arg-max hand-off needs the ring-kernel path");
  if (!fused_embed) VCL_TRY(launch_embed_tokens(io.tok_in, io.in_stride, h->embed, h->d_h, B, D, c.vocab, st));
  for (int l = 0; l < c.llm_layers; ++l) {
    const LlmLayerW& w = h->ll[l];
    if (B >= 2 && B <= 16 && !tc) {
      GemvArgs g, go, gg, gd;
      g.x = h->d_x; g.ldx = D; g.W = w.wqkv; g.W_tiled = w.wqkv_t; g.B = B; g.N = 3 * D; g.K = D;
      go.x = h->d_attn; go.ldx = D; go.W = w.wo; go.W_tiled = w.wo_t; go.B = B; go.N = D; go.K = D;
      gg.x = h->d_x; gg.ldx = D; gg.W = w.wgu; gg.W_tiled = w.wgu_t; gg.B = B; gg.N = 2 * F; gg.K = D;
      gd.x = h->d_act; gd.ldx = F; gd.W = w.wd; gd.W_tiled = w.wd_t; gd.B = B; gd.N = D; gd.K = F;
      if (gemv_tcw_supported(g) && gemv_tcw_supported(go) && gemv_tcw_supported(gg) && gemv_tcw_supported(gd)) {
        // 5..16 clips: the ring kernel over the slot-ordered copy (gemv_tcw). Its inputs travel in the
        // window-major layout (kernels.h: xwin), written by the norm, the attention kernel and its own
        // SwiGLU epilogue; the residual stream d_h stays row-major.
        VCL_TRY(launch_xwin_norm(h->d_h, D, h->d_x, w.ln1, B, D, c.rms_eps, st));
        VCL_TRY(launch_gemv_tcw_qkv_rope(g, h->d_q, D, kc_layer(h, l), vc_layer(h, l), h->rope_cos, h->rope_sin, H,
                                         c.max_seq, pos, st, pd));
        VCL_TRY(launch_decode_attention(h->d_q, D, kc_layer(h, l), vc_layer(h, l), h->d_attn, D, B, H, 128,
                                        c.max_seq, pos + 1, scale, st, pd, /*o_xwin=*/true));
        VCL_TRY(launch_gemv_tcw_residual(go, h->d_h, D, h->d_h, D, st));
        VCL_TRY(launch_xwin_norm(h->d_h, D, h->d_x, w.ln2, B, D, c.rms_eps, st));
        VCL_TRY(launch_gemv_tcw_swiglu(gg, h->d_act, F, /*out_xwin=*/true, st));
        VCL_TRY(launch_gemv_tcw_residual(gd, h->d_h, D, h->d_h, D, st));
      } else {
        // 2..4 clips without a slot-ordered copy, and shapes the ring kernels do not take: weights straight
        // from global memory into MMA fragments (gemv_mma)
        VCL_TRY(launch_rmsnorm(h->d_h, D, h->d_x, D, w.ln1, B, D, c.rms_eps, st));
        VCL_TRY(launch_gemv_mma_qkv_rope(g, h->d_q, D, kc_layer(h, l), vc_layer(h, l), h->rope_cos, h->rope_sin,
                                         H, 128, c.max_seq, pos, st, pd));
        VCL_TRY(launch_decode_attention(h->d_q, D, kc_layer(h, l), vc_layer(h, l), h->d_attn, D, B, H, 128,
                                        c.max_seq, pos + 1, scale, st, pd));
        VCL_TRY(launch_gemv_mma_residual(go, h->d_h, D, h->d_h, D, st));
        VCL_TRY(launch_rmsnorm(h->d_h, D, h->d_x, D, w.ln2, B, D, c.rms_eps, st));
        VCL_TRY(launch_gemv_mma_swiglu(gg, h->d_act, F, st));
        VCL_TRY(launch_gemv_mma_residual(gd, h->d_h, D, h->d_h, D, st));
      }
    } else if (B <= 4) {
      GemvArgs g;
      g.x = h->d_h; g.ldx = D; g.W = w.wqkv; g.W_tiled = w.wqkv_t; g.B = B; g.N = 3 * D; g.K = D; g.norm_w = w.ln1; g.eps = c.rms_eps;
      if (fused_embed && l == 0) {
        g.x = nullptr; g.embed = h->embed; g.vocab = c.vocab; g.h_out = h->d_h;
        if (io.tok_from_partials) {
          g.amax_in = h->amax; g.amax_n = device_num_sms(); g.tok_out = io.tok_store; g.tok_out_stride = io.store_stride;
        } else {
          g.tok_in = io.tok_in; g.tok_stride = io.in_stride;
        }
      }
      VCL_TRY(launch_gemv_qkv_rope(g, h->d_q, D, kc_layer(h, l), vc_layer(h, l), h->rope_cos, h->rope_sin,
                                   H, 128, c.max_seq, pos, st, pd));
      VCL_TRY(launch_decode_attention(h->d_q, D, kc_layer(h, l), vc_layer(h, l), h->d_attn, D, B, H, 128,
                                      c.max_seq, pos + 1, scale, st, pd));
      GemvArgs go;
      go.x = h->d_attn; go.ldx = D; go.W = w.wo; go.W_tiled = w.wo_t; go.B = B; go.N = D; go.K = D;
      static const int o_slots = getenv("VCL_OPROJ_SLOTS") ? atoi(getenv("VCL_OPROJ_SLOTS")) : 0;   // A/B switch
      go.ring_slots = o_slots;
      VCL_TRY(launch_gemv_residual(go, h->d_h, D, h->d_h, D, st));
      GemvArgs gg;
      gg.x = h->d_h; gg.ldx = D; gg.W = w.wgu; gg.W_tiled = w.wgu_t; gg.B = B; gg.N = 2 * F; gg.K = D; gg.norm_w = w.ln2; gg.eps = c.rms_eps;
      VCL_TRY(launch_gemv_swiglu(gg, h->d_act, F, st));
      GemvArgs gd;
      gd.x = h->d_act; gd.ldx = F; gd.W = w.wd; gd.W_tiled = w.wd_t; gd.B = B; gd.N = D; gd.K = F;
      VCL_TRY(launch_gemv_residual(gd, h->d_h, D, h->d_h, D, st));
    } else {
      // B > 16: tensor-core path, the B new rows ride in one (mostly empty) 128-row tile and the
      // N tile is narrowed so that every SM streams a slice of the weights
      VCL_TRY(launch_rmsnorm(h->d_h, D, h->d_x, D, w.ln1, B, D, c.rms_eps, st));
      VCL_TRY(gemm(h->d_x, D, w.wqkv, D, h->d_qkv, 3 * D, nullptr, nullptr, 0, B, 3 * D, D, ACT_NONE, st));
      VCL_TRY(launch_rope_kv_prefill(h->d_qkv, kc_layer(h, l), vc_layer(h, l), h->rope_cos, h->rope_sin, B,
                                     1, H, 128, c.max_seq, pos, st, pd));
      VCL_TRY(launch_decode_attention(h->d_qkv, 3 * D, kc_layer(h, l), vc_layer(h, l), h->d_attn, D, B, H,
                                      128, c.max_seq, pos + 1, scale, st, pd));
      VCL_TRY(gemm(h->d_attn, D, w.wo, D, h->d_h, D, nullptr, h->d_h, D, B, D, D, ACT_NONE, st));
      VCL_TRY(launch_rmsnorm(h->d_h, D, h->d_x, D, w.ln2, B, D, c.rms_eps, st));
      VCL_TRY(gemm(h->d_x, D, w.wgu, D, h->d_act, F, nullptr, nullptr, 0, B, 2 * F, D, ACT_SWIGLU, st));
      VCL_TRY(gemm(h->d_act, F, w.wd, F, h->d_h, D, nullptr, h->d_h, D, B, D, F, ACT_NONE, st));
    }
  }
  VCL_REQUIRE(!(io.sample && io.partials_out), "a sampled step has no partial arg-max hand-off");
  VCL_TRY(lm_head_argmax(h, h->d_h, D, B, io.logits_out, io.tok_out, io.out_stride, st, io.partials_out,
                         io.sample ? pos + 1 : -1, pd));
  return 0;
}

// Steps 1 .. n_new-1 of a greedy loop over the token scratch tk [B][n_new] (tk[:, 0] is given).
// On the ring-kernel path no arg-max / embedding kernel runs between two steps: the logits kernel
// leaves per-CTA partials, the next step's first q|k|v kernel reduces them, records the token and
// gathers its embedding row. A sampled loop (mode MODE_SAMPLED) has no hand-off: every step writes
// full logits, the sampler writes tk[:, i] and the next step gathers the row from there.
int decode_steps(vcl_handle* h, int32_t* tk, int B, int S, int n_new, const int* pos_dev, int mode, cudaStream_t st) {
  const bool hand_off = mode == MODE_GREEDY && tc_batch(h, B) && h->cfg.llm_layers > 0;
  for (int i = 1; i < n_new; ++i) {
    StepIo io;
    io.pos_dev = pos_dev;
    io.sample = mode == MODE_SAMPLED;
    if (hand_off && i > 1) {
      io.tok_from_partials = true; io.tok_store = tk + (i - 1); io.store_stride = n_new;
    } else {
      io.tok_in = tk + (i - 1); io.in_stride = n_new;
    }
    if (hand_off && i + 1 < n_new) io.partials_out = true;
    else { io.tok_out = tk + i; io.out_stride = n_new; }
    VCL_TRY(llm_decode_step(h, io, B, (pos_dev ? 0 : S) + i - 1, st));
  }
  return 0;
}

}  // namespace

extern "C" {

int vcl_clip_encode(vcl_handle* h, const void* pixels, int pixel_format, int n_frames, int frame_h, int frame_w,
                    int n_layers, void* hidden_out, void* stream) {
  VCL_REQUIRE(h && pixels && hidden_out, "vcl_clip_encode: null argument");
  VCL_REQUIRE(frame_h == h->cfg.image_size && frame_w == h->cfg.image_size,
              "vcl_clip_encode: frames are %dx%d but the tower takes %dx%d (resize / crop them first)", frame_h,
              frame_w, h->cfg.image_size, h->cfg.image_size);
  cudaStream_t st = as_stream(stream);
  VCL_TRY(clip_forward(h, pixels, pixel_format, n_frames, n_layers, st));
  const size_t bytes = (size_t)n_frames * (h->P + 1) * h->cfg.clip_hidden * 2;
  VCL_CUDA_OK(cudaMemcpyAsync(hidden_out, h->v_h, bytes, cudaMemcpyDeviceToDevice, st));
  return 0;
}

int vcl_st_pool(const void* feats, int in_dtype, int64_t frame_stride, int64_t patch_stride, int T,
                int P, int C, int n_temporal, void* out, int out_dtype, void* stream) {
  VCL_REQUIRE(feats && out, "vcl_st_pool: null argument");
  if (check_device() != 0) return -2;
  return launch_st_pool(feats, in_dtype, frame_stride, patch_stride, T, P, C, n_temporal, out, out_dtype,
                        as_stream(stream));
}

int vcl_clip_features(vcl_handle* h, const void* pixels, int pixel_format, int n_frames, int frame_h, int frame_w,
                      void* out, int out_dtype, void* stream) {
  VCL_REQUIRE(h && pixels && out, "vcl_clip_features: null argument");
  VCL_REQUIRE(frame_h == h->cfg.image_size && frame_w == h->cfg.image_size,
              "vcl_clip_features: frames are %dx%d but the tower takes %dx%d (resize / crop them first)", frame_h,
              frame_w, h->cfg.image_size, h->cfg.image_size);
  cudaStream_t st = as_stream(stream);
  VCL_REQUIRE(n_frames <= h->cfg.n_temporal, "vcl_clip_features: %d frames exceed the %d temporal slots",
              n_frames, h->cfg.n_temporal);
  VCL_TRY(clip_forward(h, pixels, pixel_format, n_frames, h->cfg.clip_layers, st));
  const int C = h->cfg.clip_hidden;
  // drop the CLS row by starting at row 1 of every frame
  return launch_st_pool(h->v_h + C, VCL_DTYPE_BF16, (long long)(h->P + 1) * C, C, n_frames, h->P, C,
                        h->cfg.n_temporal, out, out_dtype, st);
}

int vcl_llm_prefill(vcl_handle* h, const int64_t* ids, const void* video_feats,
                    const int32_t* vid_start, int B, int S, int n_layers, void* hidden_out,
                    float* logits_out, int32_t* next_tok, void* stream) {
  VCL_REQUIRE(h != nullptr, "vcl_llm_prefill: null handle");
  return llm_prefill(h, ids, video_feats, vid_start, B, S, n_layers, hidden_out, logits_out, next_tok, 1,
                     as_stream(stream));
}

int vcl_llm_prefill_states(vcl_handle* h, const int64_t* ids, const void* video_feats,
                           const int32_t* vid_start, int B, int S, void* states_out, float* logits_out,
                           void* stream) {
  VCL_REQUIRE(h != nullptr && states_out != nullptr, "vcl_llm_prefill_states: null argument");
  return llm_prefill(h, ids, video_feats, vid_start, B, S, h->cfg.llm_layers, nullptr, logits_out, nullptr, 1,
                     as_stream(stream), 0, states_out);
}

int vcl_llm_prefill_append(vcl_handle* h, const int64_t* ids, int B, int S, int start_pos, void* hidden_out,
                           float* logits_out, int32_t* next_tok, void* stream) {
  VCL_REQUIRE(h != nullptr && ids != nullptr, "vcl_llm_prefill_append: null argument");
  VCL_REQUIRE(start_pos > 0, "vcl_llm_prefill_append: start_pos must be > 0 (use vcl_llm_prefill for a new sequence)");
  return llm_prefill(h, ids, nullptr, nullptr, B, S, h->cfg.llm_layers, hidden_out, logits_out, next_tok, 1,
                     as_stream(stream), start_pos);
}

int vcl_llm_decode_step(vcl_handle* h, const int32_t* tok_in, int B, int pos, float* logits_out,
                        int32_t* tok_out, void* stream) {
  VCL_REQUIRE(h && tok_in, "vcl_llm_decode_step: null argument");
  VCL_REQUIRE(h->llm_loaded, "LLM weights are not loaded");
  VCL_REQUIRE(B > 0 && B <= h->cfg.max_batch, "B=%d outside 1..%d", B, h->cfg.max_batch);
  StepIo io;
  io.tok_in = tok_in; io.logits_out = logits_out; io.tok_out = tok_out;
  return llm_decode_step(h, io, B, pos, as_stream(stream));
}

}  // extern "C"

namespace {

int check_sampling(const vcl_sampling* sp) {
  VCL_REQUIRE(sp != nullptr, "sampling parameters are required");
  VCL_REQUIRE(!isnan(sp->temperature), "sampling temperature is NaN");
  return 0;
}

SampleParams sample_params(const vcl_sampling* sp) { return SampleParams{sp->temperature, sp->top_k, sp->seed}; }

// vcl_llm_decode_loop (MODE_GREEDY) and vcl_llm_decode_loop_sampled (MODE_SAMPLED: h->d_sample holds the
// parameters, written on the stream before this is called)
int decode_loop(vcl_handle* h, const int32_t* first_tok, int B, int S, int n_new, int mode, int32_t* out_tokens,
                cudaStream_t st) {
  VCL_REQUIRE(h && first_tok && out_tokens, "vcl_llm_decode_loop: null argument");
  VCL_REQUIRE(h->llm_loaded, "LLM weights are not loaded");
  VCL_REQUIRE(B > 0 && B <= h->cfg.max_batch, "B=%d outside 1..%d", B, h->cfg.max_batch);
  VCL_REQUIRE(n_new >= 1 && S + n_new <= h->cfg.max_seq + 1, "S + n_new = %d exceeds max_seq %d", S + n_new,
              h->cfg.max_seq);
  int32_t* tk = h->tokens;  // [B, n_new] row-major scratch
  if (first_tok != tk)
    VCL_CUDA_OK(cudaMemcpy2DAsync(tk, (size_t)n_new * sizeof(int32_t), first_tok, sizeof(int32_t),
                                  sizeof(int32_t), B, cudaMemcpyDeviceToDevice, st));
  if (n_new > 1) {
    // One graph per (B, n_new, mode): the prompt length S reaches the kernels through h->d_pos (and the
    // sampling parameters through h->d_sample), so a new prompt length replays the same graph. Bounded
    // LRU cache (an entry holds thousands of nodes).
    GraphEntry* ge = nullptr;
    for (auto& g : h->graphs)
      if (g.B == B && g.n_new == n_new && g.S == -1 && g.mode == mode) ge = &g;
    const bool can_capture = (st != nullptr) && (st != cudaStreamLegacy);
    if (ge == nullptr && can_capture) {
      if (h->graphs.size() >= MAX_DECODE_GRAPHS) {
        size_t victim = 0;
        for (size_t i = 1; i < h->graphs.size(); ++i)
          if (h->graphs[i].last_use < h->graphs[victim].last_use) victim = i;
        cudaGraphExecDestroy(h->graphs[victim].exec);
        h->graphs.erase(h->graphs.begin() + victim);
      }
      const long long before = launch_count();
      VCL_CUDA_OK(cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
      const int rc = decode_steps(h, tk, B, S, n_new, h->d_pos, mode, st);
      cudaGraph_t graph = nullptr;
      cudaError_t e = cudaStreamEndCapture(st, &graph);
      const long long nodes = launch_count() - before;
      count_launches(-nodes);  // captured, not executed
      if (rc != 0) {
        if (graph) cudaGraphDestroy(graph);
        return rc;
      }
      if (e != cudaSuccess) {
        set_last_error("decode graph capture failed: %s", cudaGetErrorString(e));
        return -2;
      }
      cudaGraphExec_t exec = nullptr;
      e = cudaGraphInstantiate(&exec, graph, 0);
      cudaGraphDestroy(graph);
      if (e != cudaSuccess) {
        set_last_error("decode graph instantiate failed: %s", cudaGetErrorString(e));
        return -2;
      }
      h->graphs.push_back({B, -1, n_new, mode, exec, nodes, 0});
      ge = &h->graphs.back();
    }
    if (ge != nullptr) {
      ge->last_use = ++h->graph_clock;
      VCL_TRY(launch_set_int(h->d_pos, S, st));
      VCL_CUDA_OK(cudaGraphLaunch(ge->exec, st));
      count_launches(ge->kernels);
    } else {
      VCL_TRY(decode_steps(h, tk, B, S, n_new, nullptr, mode, st));
    }
  }
  VCL_CUDA_OK(cudaMemcpyAsync(out_tokens, tk, (size_t)B * n_new * sizeof(int32_t), cudaMemcpyDeviceToDevice, st));
  return 0;
}

}  // namespace

extern "C" {

int vcl_llm_decode_loop(vcl_handle* h, const int32_t* first_tok, int B, int S, int n_new,
                        int32_t* out_tokens, void* stream) {
  return decode_loop(h, first_tok, B, S, n_new, MODE_GREEDY, out_tokens, as_stream(stream));
}

int vcl_llm_decode_loop_sampled(vcl_handle* h, const int32_t* first_tok, int B, int S, int n_new,
                                const vcl_sampling* sampling, int32_t* out_tokens, void* stream) {
  VCL_REQUIRE(h != nullptr, "vcl_llm_decode_loop_sampled: null handle");
  VCL_TRY(check_sampling(sampling));
  cudaStream_t st = as_stream(stream);
  VCL_TRY(launch_set_sample_params(h->d_sample, sample_params(sampling), st));
  return decode_loop(h, first_tok, B, S, n_new, MODE_SAMPLED, out_tokens, st);
}

int vcl_llm_generate(vcl_handle* h, const int64_t* ids, const void* video_feats,
                     const int32_t* vid_start, int B, int S, int n_new, int32_t* out_tokens,
                     void* stream) {
  VCL_REQUIRE(h && out_tokens, "vcl_llm_generate: null argument");
  VCL_REQUIRE(n_new >= 1 && S + n_new <= h->cfg.max_seq + 1, "S + n_new = %d exceeds max_seq %d", S + n_new,
              h->cfg.max_seq);
  cudaStream_t st = as_stream(stream);
  VCL_TRY(llm_prefill(h, ids, video_feats, vid_start, B, S, h->cfg.llm_layers, nullptr, nullptr, h->tokens,
                      n_new, st));
  return vcl_llm_decode_loop(h, h->tokens, B, S, n_new, out_tokens, stream);
}

int vcl_llm_generate_sampled(vcl_handle* h, const int64_t* ids, const void* video_feats, const int32_t* vid_start,
                             int B, int S, int n_new, const vcl_sampling* sampling, int32_t* out_tokens,
                             void* stream) {
  VCL_REQUIRE(h && out_tokens, "vcl_llm_generate_sampled: null argument");
  VCL_TRY(check_sampling(sampling));
  VCL_REQUIRE(n_new >= 1 && S + n_new <= h->cfg.max_seq + 1, "S + n_new = %d exceeds max_seq %d", S + n_new,
              h->cfg.max_seq);
  cudaStream_t st = as_stream(stream);
  VCL_TRY(launch_set_sample_params(h->d_sample, sample_params(sampling), st));
  // the prefill leaves its last-position logits in h->logits; the first new token takes position S
  VCL_TRY(llm_prefill(h, ids, video_feats, vid_start, B, S, h->cfg.llm_layers, nullptr, h->logits, nullptr, 1, st));
  VCL_TRY(launch_sample(h->logits, h->cfg.vocab, B, h->cfg.vocab, h->d_sample, SampleParams{}, S, nullptr, h->tokens,
                        n_new, st));
  return decode_loop(h, h->tokens, B, S, n_new, MODE_SAMPLED, out_tokens, st);
}

long long vcl_launch_count(void) { return launch_count(); }

int vcl_op_sample(const float* logits, int64_t ld, int B, int V, const vcl_sampling* sampling, int pos,
                  int32_t* tok_out, void* stream) {
  VCL_REQUIRE(logits && tok_out, "vcl_op_sample: null argument");
  VCL_TRY(check_sampling(sampling));
  VCL_REQUIRE(B >= 0 && pos >= 0, "vcl_op_sample: B=%d pos=%d", B, pos);
  if (check_device() != 0) return -2;
  return launch_sample(logits, ld, B, V, nullptr, sample_params(sampling), pos, nullptr, tok_out, 1,
                       as_stream(stream));
}

// ---- single-operator entry points ----
int vcl_op_gemm(const void* A, int64_t lda, const void* W, int64_t ldw, void* C, int64_t ldc,
                const void* bias, const void* residual, int64_t ldr, int M, int N, int K, int act,
                int block_n, void* stream) {
  return vcl_op_gemm_ex(A, lda, W, ldw, C, ldc, bias, residual, ldr, M, N, K, act, block_n, 0, stream);
}

int vcl_op_gemm_ex(const void* A, int64_t lda, const void* W, int64_t ldw, void* C, int64_t ldc,
                   const void* bias, const void* residual, int64_t ldr, int M, int N, int K, int act,
                   int block_n, int cluster, void* stream) {
  if (check_device() != 0) return -2;
  static bool inited = false;
  if (!inited) {
    VCL_TRY(init_gemm_kernels());
    inited = true;
  }
  return gemm(reinterpret_cast<const bf16*>(A), lda, reinterpret_cast<const bf16*>(W), ldw,
              reinterpret_cast<bf16*>(C), ldc, reinterpret_cast<const bf16*>(bias),
              reinterpret_cast<const bf16*>(residual), ldr, M, N, K, act, as_stream(stream), block_n, cluster);
}

int vcl_op_layernorm(const void* x, void* y, const void* w, const void* b, int rows, int D, float eps,
                     void* stream) {
  if (check_device() != 0) return -2;
  return launch_layernorm(reinterpret_cast<const bf16*>(x), D, reinterpret_cast<bf16*>(y), D,
                          reinterpret_cast<const bf16*>(w), reinterpret_cast<const bf16*>(b), rows, D, eps,
                          as_stream(stream));
}

int vcl_op_rmsnorm(const void* x, void* y, const void* w, int rows, int D, float eps, void* stream) {
  if (check_device() != 0) return -2;
  return launch_rmsnorm(reinterpret_cast<const bf16*>(x), D, reinterpret_cast<bf16*>(y), D,
                        reinterpret_cast<const bf16*>(w), rows, D, eps, as_stream(stream));
}

int vcl_op_attention(const void* q, const void* k, const void* v, void* o, int B, int S, int H,
                     int head_dim, float scale, int causal, void* stream) {
  if (check_device() != 0) return -2;
  static bool inited = false;
  if (!inited) {
    VCL_TRY(init_attention_kernels());
    inited = true;
  }
  AttnArgs a;
  const long long sb = (long long)S * H * head_dim, sh = head_dim, ss = (long long)H * head_dim;
  a.q = reinterpret_cast<const bf16*>(q); a.q_sb = sb; a.q_sh = sh; a.q_ss = ss;
  a.k = reinterpret_cast<const bf16*>(k); a.k_sb = sb; a.k_sh = sh; a.k_ss = ss;
  a.v = reinterpret_cast<const bf16*>(v); a.v_sb = sb; a.v_sh = sh; a.v_ss = ss;
  a.o = reinterpret_cast<bf16*>(o); a.o_sb = sb; a.o_sh = sh; a.o_ss = ss;
  a.B = B; a.H = H; a.S = S; a.head_dim = head_dim; a.scale = scale; a.causal = causal;
  return launch_attention(a, as_stream(stream));
}

int vcl_op_attention_vit(const void* qkv, void* out, int n_frames, int S, int H, void* stream) {
  if (check_device() != 0) return -2;
  static bool inited = false;
  if (!inited) {
    VCL_TRY(init_gemm_kernels());
    VCL_TRY(init_attention_tc_kernels());
    inited = true;
  }
  return launch_attention_vit_tc(reinterpret_cast<const bf16*>(qkv), reinterpret_cast<bf16*>(out), n_frames, S, H,
                                 H * 64, as_stream(stream));
}

int vcl_op_gemv(const void* x, const void* W, void* out, const void* res, const void* norm_w,
                float eps, int B, int N, int K, void* stream) {
  if (check_device() != 0) return -2;
  static bool inited = false;
  if (!inited) {
    VCL_TRY(init_gemv_kernels());
    VCL_TRY(init_gemv_tc_kernels());
    VCL_TRY(init_gemv_tcw_kernels());
    inited = true;
  }
  GemvArgs g;
  g.x = reinterpret_cast<const bf16*>(x); g.ldx = K; g.W = reinterpret_cast<const bf16*>(W);
  g.B = B; g.N = N; g.K = K; g.norm_w = reinterpret_cast<const bf16*>(norm_w); g.eps = eps;
  // exercise the slot-ordered-copy kernels the decode loop uses. The copy is built here and kept for the
  // next call with the same matrix (this entry point is a test / micro-benchmark hook, not a hot path).
  static const void* c_W = nullptr; static int c_N = 0, c_K = 0; static bf16* c_tiled = nullptr;
  if (B <= 16 && K % 32 == 0 && N >= 16 && getenv("VCL_GEMV_LEGACY") == nullptr) {
    // (the copy is only REUSED when VCL_OP_GEMV_CACHE is set -- tools/microbench.py -- because a caller may
    // hand in a different matrix at a recycled address)
    if (c_W != W || c_N != N || c_K != K || getenv("VCL_OP_GEMV_CACHE") == nullptr) {
      cudaStreamSynchronize(as_stream(stream));
      if (c_tiled != nullptr) cudaFree(c_tiled);
      c_tiled = nullptr; c_W = nullptr;
      VCL_CUDA_OK(cudaMalloc(&c_tiled, gemv_tc_tiled_elems(N, K) * sizeof(bf16)));
      const int rc0 = launch_gemv_tc_repack(g.W, c_tiled, N, K, false, as_stream(stream));
      if (rc0 != 0) { cudaFree(c_tiled); c_tiled = nullptr; return rc0; }
      c_W = W; c_N = N; c_K = K;
    }
    g.W_tiled = c_tiled;
  }
  if (B >= 5) {
    // 5..16 rows: the wide ring kernel; its input is normalised and re-laid out (xwin) by a launch of its own,
    // as on the decode path
    static bf16* xn = nullptr; static size_t xn_elems = 0;
    if (xn_elems < xwin_elems(B, K)) {
      cudaStreamSynchronize(as_stream(stream));
      if (xn) cudaFree(xn);
      VCL_CUDA_OK(cudaMalloc(&xn, xwin_elems(B, K) * sizeof(bf16)));
      xn_elems = xwin_elems(B, K);
    }
    VCL_TRY(launch_xwin_norm(g.x, K, xn, g.norm_w, B, K, eps, as_stream(stream)));
    g.x = xn; g.norm_w = nullptr;
    VCL_REQUIRE(gemv_tcw_supported(g), "vcl_op_gemv: B=%d N=%d K=%d is outside the wide ring kernel's range", B, N, K);
    return launch_gemv_tcw_residual(g, reinterpret_cast<bf16*>(out), N, reinterpret_cast<const bf16*>(res), N, as_stream(stream));
  }
  return launch_gemv_residual(g, reinterpret_cast<bf16*>(out), N, reinterpret_cast<const bf16*>(res), N, as_stream(stream));
}

}  // extern "C"
