/* vcl.h -- C ABI of libvcl.so, the B200-native replacement for the device side of
 * PG-Video-LLaVA's video-conversation inference path.
 *
 * The reference (mbzuai-oryx/Video-LLaVA) has no FFI or operator registry: its boundary is a set
 * of Python call sites that hand tensors to PyTorch/HF modules. Each entry point below states the
 * reference call it replaces (file:line relative to the reference tree; "$TF" = the installed
 * HuggingFace transformers, where the arithmetic the reference delegates to lives).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name ends in _host; the caller owns all memory
 *     passed in; the library owns its packed weights, activations and KV cache (allocated by
 *     vcl_create / vcl_load_*), freed by vcl_destroy;
 *   - 16-bit tensors are bf16 unless a dtype code says otherwise (0 = fp16, 1 = bf16);
 *   - work is enqueued on `stream` (a cudaStream_t passed as void*) and never synchronised,
 *     except vcl_load_* which return after the repack has completed;
 *   - return value 0 = ok, negative = error; vcl_last_error() gives the message of the last
 *     failure on the calling thread's process (one handle per process/GPU, not thread-safe);
 *   - there is no CPU fallback: on a machine without an sm_100 device every compute entry point
 *     fails with an error.
 */
#ifndef VCL_H_
#define VCL_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VCL_VERSION 1

#define VCL_DTYPE_F16 0
#define VCL_DTYPE_BF16 1

#define VCL_PIXELS_BF16_NCHW 0 /* [N,3,H,W] bf16, already CLIP-normalised (inference.py:86-89)   */
#define VCL_PIXELS_U8_NHWC 1   /* [N,H,W,3] uint8 raw frames; (x/255-mean)/std applied on device */

#define VCL_PROJ_LINEAR 0     /* nn.Linear(1024, D)            video_chatgpt/model/video_chatgpt.py:51-53 */
#define VCL_PROJ_MLP2X_GELU 1 /* Linear-GELU-Linear            model/multimodal_projector/builder.py:39-46 */

typedef struct vcl_handle vcl_handle;

typedef struct vcl_config {
  /* vision tower: CLIP ViT ($TF/models/clip/modeling_clip.py:647-693) */
  int32_t clip_layers;   /* encoder layers to EXECUTE; the path consumes hidden_states[-2]
                            (inference.py:94), i.e. num_hidden_layers - 1 (23 for ViT-L/14)   */
  int32_t clip_hidden;   /* 1024 */
  int32_t clip_inter;    /* 4096 */
  int32_t clip_heads;    /* 16 (head_dim must be 64) */
  int32_t image_size;    /* 224 or 336 */
  int32_t patch_size;    /* 14 */
  float clip_ln_eps;     /* 1e-5 */
  /* language model: LLaMA/Vicuna ($TF/models/llama/modeling_llama.py:355-425) */
  int32_t llm_layers;    /* 32 (7B) / 40 (13B) */
  int32_t llm_hidden;    /* 4096 / 5120 (head_dim must be 128) */
  int32_t llm_inter;     /* 11008 / 13824 */
  int32_t llm_heads;     /* 32 / 40 (kv heads == heads) */
  int32_t vocab;         /* 32003 after the three video tokens are added (eval/model_utils.py:114-119) */
  float rms_eps;         /* 1e-5 */
  float rope_theta;      /* 10000 */
  int32_t proj_type;     /* VCL_PROJ_* */
  int32_t n_temporal;    /* 100: temporal token slots (inference.py:31) */
  /* capacities */
  int32_t max_frames;    /* frames per vcl_clip_encode call */
  int32_t max_batch;     /* clips per prefill / decode call */
  int32_t max_seq;       /* prompt + generated tokens per clip */
} vcl_config;

/* A named tensor in the layout of the HF/reference state_dict (row-major, bf16, on the device).
 * Names are the state_dict keys listed in SURVEY.md section 8a ("weight-name contract"). */
typedef struct vcl_tensor {
  const char* name;
  const void* data;
  int32_t ndim;
  int64_t shape[4];
} vcl_tensor;

int vcl_version(void);
const char* vcl_last_error(void);

/* Replaces the module construction in video_chatgpt/eval/model_utils.py:104-105,134-136. */
int vcl_create(vcl_handle** out, const vcl_config* cfg);
void vcl_destroy(vcl_handle* h);

/* Replace CLIPVisionModel.from_pretrained / VideoChatGPTLlamaForCausalLM.from_pretrained +
 * load_state_dict (eval/model_utils.py:104,122-127,134): repack into the kernel layouts
 * (fused q|k|v, interleaved gate/up, K-padded patch-embed matrix). Unknown names are ignored
 * (e.g. vision_model.post_layernorm.*, unused by the path); a missing required name is an error.
 * vcl_load_llm_weights additionally builds a decode-only copy of the streamed matrices in the slot
 * order of the single-clip decode kernel (+1x the LLM weight bytes; VCL_NO_TILED_WEIGHTS=1 in the
 * environment skips it and decode falls back to the row-major kernels). */
int vcl_load_clip_weights(vcl_handle* h, const vcl_tensor* tensors, int n);
int vcl_load_llm_weights(vcl_handle* h, const vcl_tensor* tensors, int n);

/* vision_tower(pixel_values, output_hidden_states=True).hidden_states[k]
 * (video_chatgpt/inference.py:93-94, scripts/save_spatio_temporal_clip_features.py:116-120).
 * Runs `n_layers` encoder layers (<= clip_layers; pass clip_layers for hidden_states[-2]; 0 gives
 * hidden_states[0], the post-pre_layrnorm embeddings). hidden_out is [n_frames, 1+P, C] bf16 with
 * the CLS row kept, as in HF; callers slice [:, 1:]. frame_h / frame_w are the height and width of
 * the frames behind `pixels`: they must equal image_size (the image processor of the reference
 * resizes and crops, inference.py:86; raw frames of another size are an error, never read out of bounds). */
int vcl_clip_encode(vcl_handle* h, const void* pixels, int pixel_format, int n_frames, int frame_h, int frame_w,
                    int n_layers, void* hidden_out, void* stream);

/* get_spatio_temporal_features_torch (video_chatgpt/inference.py:13-44) and its numpy twin
 * get_spatio_temporal_features (scripts/save_spatio_temporal_clip_features.py:46-57).
 * feats element (t,p,c) at feats + t*frame_stride + p*patch_stride + c (strides in elements), so a
 * [T,1+P,C] hidden state can be pooled in place by pointing at row 1. out is [n_temporal+P, C]. */
int vcl_st_pool(const void* feats, int in_dtype, int64_t frame_stride, int64_t patch_stride, int T,
                int P, int C, int n_temporal, void* out, int out_dtype, void* stream);

/* vcl_clip_encode(clip_layers) + CLS drop + vcl_st_pool in one call: the per-video body of
 * scripts/save_spatio_temporal_clip_features.py:105-123 and inference.py:93-95. */
int vcl_clip_features(vcl_handle* h, const void* pixels, int pixel_format, int n_frames, int frame_h, int frame_w,
                      void* out, int out_dtype, void* stream);

/* VideoChatGPTLlamaForCausalLM.forward on a full prompt (video_chatgpt/model/video_chatgpt.py:82-175,
 * 193-251): token embedding, mm_projector on video_feats [B, n_temporal+P, 1024], splice after
 * <vid_start> (vid_start[b] = index of the row after which the video rows go: the <vid_start> token, or
 * -1 when the patch tokens start the row without one; VCL_NO_VIDEO marks a text-only row), n_layers
 * decoder layers filling the KV cache at positions [0, S).
 *   hidden_out  optional [B,S,D] bf16: output of decoder layer n_layers (n_layers = 0: the spliced
 *               input embeddings), i.e. HF hidden_states[n_layers]
 *   logits_out  optional [B,vocab] fp32: lm_head(norm(h)) at the LAST position only, rounded to
 *               bf16 like the reference's logits tensor (requires n_layers == llm_layers)
 *   next_tok    optional [B] int32: arg-max of those logits (lowest index wins ties) */
int vcl_llm_prefill(vcl_handle* h, const int64_t* ids, const void* video_feats,
                    const int32_t* vid_start, int B, int S, int n_layers, void* hidden_out,
                    float* logits_out, int32_t* next_tok, void* stream);
#define VCL_NO_VIDEO (-2147483647 - 1)

/* forward(..., output_hidden_states=True) (video_chatgpt/model/video_chatgpt.py:205-218): the same
 * full-depth prefill, keeping every hidden state: states_out is [llm_layers + 1][B][S][D] bf16, entry i
 * = the raw output of decoder layer i (entry 0: the spliced input embeddings). HF returns the LAST
 * entry after the final RMSNorm; the caller applies it (vcl_op_rmsnorm with model.norm.weight). */
int vcl_llm_prefill_states(vcl_handle* h, const int64_t* ids, const void* video_feats,
                           const int32_t* vid_start, int B, int S, void* states_out, float* logits_out,
                           void* stream);

/* Continue a cached sequence: S more token ids per clip (text only, no video span) take positions
 * [start_pos, start_pos + S) and attend to everything already in the KV cache. This is the building
 * block for multi-turn conversations about one video: the reference re-runs the vision tower and the
 * whole prompt on every turn (video_chatgpt/chat.py:137-154, inference.py:86-112); with the cache of
 * the previous turn only the new question is prefilled. Outputs as in vcl_llm_prefill (hidden_out
 * [B,S,D] of the new positions; logits / next token at the last new position). start_pos must be the
 * number of positions the cache of every clip already holds (> 0). */
int vcl_llm_prefill_append(vcl_handle* h, const int64_t* ids, int B, int S, int start_pos, void* hidden_out,
                           float* logits_out, int32_t* next_tok, void* stream);

/* One cached decoding step (the `input_ids.shape[1] == 1` branch, model/video_chatgpt.py:103,
 * 253-257): tok_in [B] int32 are fed at position `pos` (= tokens already in the cache).
 * logits_out / tok_out as above. Used for teacher-forced parity checks. */
int vcl_llm_decode_step(vcl_handle* h, const int32_t* tok_in, int B, int pos, float* logits_out,
                        int32_t* tok_out, void* stream);

/* model.generate(input_ids, video_spatio_temporal_features=..., do_sample=False,
 * max_new_tokens=n_new) with EOS ignored (video_chatgpt/inference.py:105-112; greedy is the
 * benchmark's setting, BASELINE.md section 5): prefill + (n_new-1) decode steps, tokens chained on
 * the device, the decode loop replayed from a CUDA graph. out_tokens is [B, n_new] int32 (new
 * tokens only; the Python shim prepends the prompt as HF does).
 * The graph is captured once per (B, n_new) on a non-default stream: the prompt length S reaches the
 * kernels through device memory, so any S replays it; at most 6 graphs are kept (least recently used
 * first out). With 1-4 clips no arg-max / embedding kernel runs between two steps (the logits kernel
 * leaves per-CTA partial arg-max, the next step's first q|k|v kernel reduces them and gathers the row). */
int vcl_llm_generate(vcl_handle* h, const int64_t* ids, const void* video_feats,
                     const int32_t* vid_start, int B, int S, int n_new, int32_t* out_tokens,
                     void* stream);

/* The decode half of vcl_llm_generate on its own (so a caller can time prefill and decode
 * separately): first_tok [B] int32 is the token produced by the prefill; runs n_new-1 cached steps
 * at positions S, S+1, ... and writes [B, n_new] (first_tok included) to out_tokens. */
int vcl_llm_decode_loop(vcl_handle* h, const int32_t* first_tok, int B, int S, int n_new,
                        int32_t* out_tokens, void* stream);

/* ---- sampling (do_sample=True): temperature -> top-k -> softmax -> multinomial on the device ----
 * The reference's callers sample (inference.py:105-112: do_sample=True, temperature=0.2, HF's default
 * top-k 50). HF applies TemperatureLogitsWarper, TopKLogitsWarper ($TF/generation/logits_process.py),
 * softmax and torch.multinomial; the contract here, for row b and the fp32 logits l[0..V) the logits
 * kernels write (bf16-rounded values), is:
 *   - temperature <= 0: the arg-max, lowest index winning (the token vcl_llm_generate would produce);
 *   - k = top_k if 1 <= top_k < V, else V (0: no filter); tau = the k-th largest logit counting
 *     multiplicity; the kept set is K = {i : l_i >= tau} (every tie at tau stays, so |K| can exceed k);
 *     NaN counts as -inf;
 *   - weights w_i = exp(((double)l_i - (double)max l) / (double)T) in fp64 (HF's softmax is fp32: the
 *     probabilities differ by ~1e-7 relative, in exchange for an exact host restatement);
 *   - u in [0,1), t = u * sum_K w_i; the token is the smallest id of K, walking ids in ascending order,
 *     whose running sum exceeds t (the largest id of K if rounding leaves none). The device sums in a
 *     different association than a sequential walk, so a draw within ~1e-16 Z of a bin edge may land on the
 *     neighbouring id;
 *   - u = (w0 >> 11) * 2^-53, w0 = word 0 of Philox4x64-10 with key (seed, 0) at counter (pos, b, 0, 0),
 *     pos = the sequence position the sampled token will occupy (the first new token after an S-token
 *     prompt is at S), b = the row within the call. The stream therefore does not depend on chunking,
 *     graph or eager launches, or the decode kernel family. (numpy.random.Philox(key=[seed, 0],
 *     counter=[pos - 1, b, 0, 0]).random_raw(4)[0] is the same word: numpy increments before generating.)
 * A row without a finite maximum yields the lowest id at its maximum (id 0 when every logit is -inf or NaN).
 * vcl_sampling is a HOST struct, read when the call is made. */
typedef struct vcl_sampling {
  float temperature;
  int32_t top_k;
  uint64_t seed;
} vcl_sampling;

/* vcl_llm_generate with sampling: prefill, the first token sampled at position S, n_new-1 sampled decode
 * steps from a CUDA graph kept per (B, n_new, mode) under the same LRU bound (one sampled graph serves every
 * temperature, top-k, seed and prompt length). Sampled steps hand full logits to the sampler, so there is
 * no partial arg-max hand-off on this path. */
int vcl_llm_generate_sampled(vcl_handle* h, const int64_t* ids, const void* video_feats, const int32_t* vid_start,
                             int B, int S, int n_new, const vcl_sampling* sampling, int32_t* out_tokens,
                             void* stream);
/* vcl_llm_decode_loop with sampling: first_tok [B] is the token at position S; token i of the output takes
 * position S + i. */
int vcl_llm_decode_loop_sampled(vcl_handle* h, const int32_t* first_tok, int B, int S, int n_new,
                                const vcl_sampling* sampling, int32_t* out_tokens, void* stream);
/* tok_out[b] = the token sampled from logits row b (fp32, row pitch ld elements, V columns) for sequence
 * position pos (row b uses counter (pos, b)): the first token after vcl_llm_prefill_append, and the tests. */
int vcl_op_sample(const float* logits, int64_t ld, int B, int V, const vcl_sampling* sampling, int pos,
                  int32_t* tok_out, void* stream);

/* Number of kernels of this library launched so far in the process (CUDA-graph replays count the
 * kernel nodes they contain). Evidence for bench.py's "gpu_launches". */
long long vcl_launch_count(void);

/* ---- single-operator entry points (unit tests / profiling of the individual kernels) ---- */
/* C[M,N] = act(A[M,K] . W[N,K]^T + bias) (+ residual); act: 0 none, 1 quick_gelu, 2 gelu(erf),
 * 3 swiglu over interleaved rows (C is [M,N/2]). block_n: 0 = auto, or 32/64/128/256. */
int vcl_op_gemm(const void* A, int64_t lda, const void* W, int64_t ldw, void* C, int64_t ldc,
                const void* bias, const void* residual, int64_t ldr, int M, int N, int K, int act,
                int block_n, void* stream);
/* same with an explicit thread-block-cluster size along M (1, 2 or 4): the CTAs of a cluster share
 * each weight tile through TMA multicast; cluster = -2: CTA pairs (tcgen05 cta_group::2, one M = 256 MMA
 * per pair, each CTA stages half of the weight tile; block_n 256 or 128) */
int vcl_op_gemm_ex(const void* A, int64_t lda, const void* W, int64_t ldw, void* C, int64_t ldc,
                   const void* bias, const void* residual, int64_t ldr, int M, int N, int K, int act,
                   int block_n, int cluster, void* stream);
int vcl_op_layernorm(const void* x, void* y, const void* w, const void* b, int rows, int D, float eps,
                     void* stream);
int vcl_op_rmsnorm(const void* x, void* y, const void* w, int rows, int D, float eps, void* stream);
/* q,k,v,o: [B,S,H,hd] contiguous bf16 */
int vcl_op_attention(const void* q, const void* k, const void* v, void* o, int B, int S, int H,
                     int head_dim, float scale, int causal, void* stream);
/* ViT attention on the fused projection output: qkv [n_frames*S, 3*H*64] (q|k|v) -> out
 * [n_frames*S, H*64]; tcgen05 kernel, 129 <= S <= 257, non-causal, scale 64^-1/2 */
int vcl_op_attention_vit(const void* qkv, void* out, int n_frames, int S, int H, void* stream);
/* out[b,n] = x[b,:].W[n,:] (+res) with optional RMSNorm of x: B <= 4 the ring kernel of the single-clip
 * decode path (fused norm), 5 <= B <= 16 the wide ring kernel (norm + window-major re-layout by a launch of
 * its own, as on the decode path) */
int vcl_op_gemv(const void* x, const void* W, void* out, const void* res, const void* norm_w,
                float eps, int B, int N, int K, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* VCL_H_ */
