// Internal launcher prototypes shared between the kernel translation units and vcl_api.cu.
// Everything here enqueues on the stream it is given and never synchronises.
#pragma once

#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace vcl {

typedef __nv_bfloat16 bf16;

enum Act { ACT_NONE = 0, ACT_QGELU = 1, ACT_GELU = 2, ACT_SWIGLU = 3, ACT_ROPE = 4 };
// ACT_ROPE: the GEMM is the LLaMA q|k|v projection of a prefill (N = 3 * H * 128, rows = [clip][position]).
// The epilogue rotates q and k (RoPE, every product and the sum rounded to bf16 like the reference), writes q to
// C (columns [0, H * 128)), k and v straight into the KV cache; the k | v columns of C are not written.
struct RopeEpilogue {
  const bf16* cos_t = nullptr; const bf16* sin_t = nullptr;    // [s_max][64]
  bf16* kcache = nullptr; bf16* vcache = nullptr;              // [clip][head][s_max][128] of this layer
  int S = 0, start_pos = 0, H = 0, s_max = 0;                  // rows per clip, position of row 0, heads
};

void set_last_error(const char* fmt, ...);
void count_launches(long long n);
long long launch_count();
int device_num_sms();

// ---- gemm_tc.cu : C[M,N] = epi(A[M,K] . W[N,K]^T), tcgen05 + TMA -------------------------------
struct GemmArgs {
  const bf16* A = nullptr;  long long lda = 0;   // activations, row pitch in elements
  const bf16* W = nullptr;  long long ldw = 0;   // weights [N,K] (nn.Linear layout)
  bf16* C = nullptr;        long long ldc = 0;   // output (width N, or N/2 for ACT_SWIGLU)
  const bf16* bias = nullptr;                    // [N] or null
  const bf16* residual = nullptr; long long ldr = 0;  // [M,N] or null; may alias C
  int M = 0, N = 0, K = 0;
  int act = ACT_NONE;
  int block_n = 0;     // 0 = choose
  int cluster = 0;     // CTAs per cluster along M sharing multicast weight tiles: 0/1, 2 or 4
  int max_ctas = 0;    // 0 = one per SM
  RopeEpilogue rope;   // act == ACT_ROPE only
};
int launch_gemm_bf16_tn(const GemmArgs& g, cudaStream_t stream);
int init_gemm_kernels();
// 2-D bf16 tensor map [rows, cols] with row pitch ld (elements); box = [box_rows, 64], 128-B swizzle
int make_tmap_2d(CUtensorMap* out, const void* ptr, long long rows, long long cols, long long ld,
                 int box_rows);

// ---- elementwise.cu ---------------------------------------------------------------------------
// y = LayerNorm(x) * w + b   (rows x D, fp32 statistics, one bf16 rounding)
int launch_layernorm(const bf16* x, long long ldx, bf16* y, long long ldy, const bf16* w,
                     const bf16* b, int rows, int D, float eps, cudaStream_t stream);
// y = w * bf16(x * rsqrt(mean(x^2)+eps))   (LlamaRMSNorm rounding order)
int launch_rmsnorm(const bf16* x, long long ldx, bf16* y, long long ldy, const bf16* w, int rows,
                   int D, float eps, cudaStream_t stream);
// pixels -> patch matrix [N*P, KP] (k = c*ps*ps + i*ps + j, zero padded to KP)
//   mode 0: bf16 NCHW already normalised;  mode 1: uint8 NHWC raw, CLIP mean/std applied here
int launch_im2col(const void* pixels, int mode, bf16* out, int n_frames, int image, int patch,
                  int KP, cudaStream_t stream);
// h[n, 0] = LN(cls + pos[0]); h[n, 1+p] = LN(patch[n*P+p] + pos[1+p])
int launch_clip_embed_ln(const bf16* patch_out, const bf16* cls, const bf16* pos, const bf16* ln_w,
                         const bf16* ln_b, bf16* h, int n_frames, int P, int D, float eps,
                         cudaStream_t stream);
// token-embedding gather with the projected video rows spliced in after <vid_start>
int launch_embed_splice(const long long* ids, const bf16* table, const bf16* vid, const int* vid_start,
                        bf16* h, int B, int S, int D, int n_vid, int vocab, cudaStream_t stream);
// cos/sin tables [max_pos, head_dim/2] rounded to bf16 (stored as bf16)
int launch_rope_table(bf16* cos_t, bf16* sin_t, int max_pos, int head_dim, float theta,
                      cudaStream_t stream);
// prefill: rotate q (in place inside qkv) and k, write k/v into the cache at [pos0, pos0+S)
// (pos_dev != null: the position is pos0 + *pos_dev, read on the device -- a captured decode graph then
// serves every prompt length; the same convention holds for every `pos_dev` below)
int launch_rope_kv_prefill(bf16* qkv, bf16* kcache, bf16* vcache, const bf16* cos_t,
                           const bf16* sin_t, int B, int S, int H, int head_dim, int s_max, int pos0,
                           cudaStream_t stream, const int* pos_dev = nullptr);
// h[b,:] = table[tok[b*tok_stride]]  (decode-time embedding lookup, tokens live on the device)
int launch_embed_tokens(const int* tok, long long tok_stride, const bf16* table, bf16* h, int B,
                        int D, int vocab, cudaStream_t stream);
int launch_argmax(const float* logits, int* out, long long out_stride, int B, int V,
                  cudaStream_t stream);
int launch_set_int(int* dst, int value, cudaStream_t stream);

// ---- sample.cu : temperature / top-k sampling, the contract of vcl_sampling (include/vcl.h) ----------
struct SampleParams { float temperature; int top_k; unsigned long long seed; };   // layout of vcl_sampling
// out[b * out_stride] = the token sampled from row b of logits (pitch ld) for sequence position
// pos (+ *pos_dev); the parameters are read from params_dev when it is non-null, else taken from params
int launch_sample(const float* logits, long long ld, int B, int V, const SampleParams* params_dev,
                  const SampleParams& params, int pos, const int* pos_dev, int* out, long long out_stride,
                  cudaStream_t stream);
int launch_set_sample_params(SampleParams* dst, const SampleParams& p, cudaStream_t stream);

// ---- st_pool.cu ---------------------------------------------------------------------------------
// dtype codes: 0 = fp16, 1 = bf16
int launch_st_pool(const void* feats, int in_dtype, long long frame_stride, long long patch_stride,
                   int T, int P, int C, int n_temporal, void* out, int out_dtype,
                   cudaStream_t stream);

// ---- attention.cu -------------------------------------------------------------------------------
// softmax(Q K^T * scale [+ causal]) V for S_q == S_kv, bf16, fp32 softmax; element (b,h,s,d) of
// each operand lives at base + b*sb + h*sh + s*ss + d.
struct AttnArgs {
  const bf16* q; long long q_sb, q_sh, q_ss;
  const bf16* k; long long k_sb, k_sh, k_ss;
  const bf16* v; long long v_sb, v_sh, v_ss;
  bf16* o;       long long o_sb, o_sh, o_ss;
  int B, H, S, head_dim;
  float scale;
  int causal;
  int S_kv = 0;      // number of keys (0: = S); > S when the queries continue a cached sequence
  int q_off = 0;     // absolute position of query 0 for the causal mask (S_kv - S for a continuation)
};
int launch_attention(const AttnArgs& a, cudaStream_t stream);     // dispatches to the tcgen05 prefill kernel when it applies
int init_attention_kernels();
// ---- attention_prefill_tc.cu : tcgen05 causal attention (hd 128, <= 512 keys) -----------------------
bool attention_prefill_tc_supported(const AttnArgs& a);
int launch_attention_prefill_tc(const AttnArgs& a, cudaStream_t stream);
int init_attention_prefill_tc_kernels();
// ---- attention_tc.cu : tcgen05 attention for the ViT (hd 64, 129 <= S <= 257, non-causal) ----------
int launch_attention_vit_tc(const bf16* qkv, bf16* out, int n_frames, int S, int H, int C,
                            cudaStream_t stream);
int init_attention_tc_kernels();
// single-query attention against the cache: q [B, H*hd] -> o [B, H*hd]; kv_len keys per clip
int launch_decode_attention(const bf16* q, long long q_ld, const bf16* kcache, const bf16* vcache,
                            bf16* o, long long o_ld, int B, int H, int head_dim, int s_max,
                            int kv_len, float scale, cudaStream_t stream, const int* pos_dev = nullptr,
                            bool o_xwin = false);   // o_xwin: the output [B][H*hd] is written in xwin layout

// ---- gemv.cu : decode-time weight streaming (M = B <= 8 rows) ------------------------------------
// per-CTA partial arg-max of the logits kernel: the next step's q|k|v kernel reduces the grid's
// partials itself (lowest index wins ties), so no arg-max kernel runs between two decode steps
struct ArgmaxPart { float v; int idx; };

struct GemvArgs {
  const bf16* x = nullptr; long long ldx = 0;   // [B, K]
  const bf16* W = nullptr;                      // [N, K]
  const bf16* W_tiled = nullptr;                // optional decode-only tiled copy (gemv_tc.cu), B = 1
  int ring_slots = 0;                           // gemv_tc: deeper shared-memory ring than the default (0 = default)
  int B = 0, N = 0, K = 0;
  const bf16* norm_w = nullptr; float eps = 0;  // optional fused RMSNorm prologue
  // gemv_tc only. q|k|v with a fused token-embedding gather: x is row `token` of `embed` [vocab, K],
  // the token read from tok_in[b * tok_stride] or reduced from the previous step's arg-max partials
  // (amax_in [amax_n][B]); CTA 0 then stores the token (tok_out) and the raw row (h_out [B][K], the
  // residual stream). Logits: amax_out [grid][B] receives the per-CTA partial arg-max.
  const bf16* embed = nullptr; int vocab = 0;
  const int* tok_in = nullptr; long long tok_stride = 0;
  const ArgmaxPart* amax_in = nullptr; int amax_n = 0;
  int* tok_out = nullptr; long long tok_out_stride = 0;
  bf16* h_out = nullptr;
  ArgmaxPart* amax_out = nullptr;
};
// out[b, n] = bf16(bf16(x.W[n]) + res[b, n])      (res may alias out; res == null -> plain)
int launch_gemv_residual(const GemvArgs& g, bf16* out, long long ldo, const bf16* res,
                         long long ldr, cudaStream_t stream);
// W rows interleaved (2j gate, 2j+1 up): out[b, j] = silu(gate)*up,  N = 2*F
int launch_gemv_swiglu(const GemvArgs& g, bf16* out, long long ldo, cudaStream_t stream);
// fused q/k/v projection + RoPE + cache write for one new token per clip at position pos
int launch_gemv_qkv_rope(const GemvArgs& g, bf16* q_out, long long ldq, bf16* kcache, bf16* vcache,
                         const bf16* cos_t, const bf16* sin_t, int H, int head_dim, int s_max,
                         int pos, cudaStream_t stream, const int* pos_dev = nullptr);
int init_gemv_kernels();

// ---- gemv_tc.cu : 1..4 clips (bulk-copy ring over a slot-ordered weight copy + mma.sync) ---------
// The launch_gemv_* entry points above route to these when gemv_tc_supported(g).
int init_gemv_tc_kernels();
enum { TC_MODE_RES = 0, TC_MODE_SWIGLU = 1, TC_MODE_QKV = 2, TC_MODE_LOGITS = 3 };
struct TcPhase {
  int mode = TC_MODE_RES;
  const bf16* W_tiled = nullptr; int N = 0, K = 0;   // slot-ordered copy of the [N, K] matrix
  const bf16* x = nullptr; long long ldx = 0;        // [B][ldx] input (written by the previous phase / kernel)
  int B = 1;                                         // clips (1..4; chains of several phases: 1)
  const bf16* norm_w = nullptr;                      // optional fused RMSNorm of x
  int ring_slots = 0;                                // 0 = default ring depth
  bf16* out = nullptr; long long ldo = 0;            // RES: out[B][N] (+res); SWIGLU: out[B][N/2]
  const bf16* res = nullptr; long long ldr = 0;
  bf16* q_out = nullptr; long long ldq = 0;          // QKV: q [B][ldq], cache base of the layer [B][H][S][128]
  bf16* kcache = nullptr; bf16* vcache = nullptr;
  float* logits = nullptr; long long ldl = 0;        // LOGITS: [B][ldl] bf16-rounded fp32 (null: not stored)
  ArgmaxPart* amax_out = nullptr;                    // LOGITS: [grid][B] per-CTA partial arg-max
  // QKV with a fused embedding gather (see GemvArgs)
  const bf16* embed = nullptr; int vocab = 0;
  const int* tok_in = nullptr; long long tok_stride = 0;
  const ArgmaxPart* amax_in = nullptr; int amax_n = 0;
  int* tok_out = nullptr; long long tok_out_stride = 0;
  bf16* h_out = nullptr;
};
struct TcChainCommon {
  float eps = 0.f;
  const bf16* cos_t = nullptr; const bf16* sin_t = nullptr;
  int H = 0, s_max = 0, pos = 0;
  const int* pos_dev = nullptr;                      // position = pos + *pos_dev
};
bool gemv_tc_chain_supported(const TcPhase* ph, int n);
int launch_gemv_tc_chain(const TcPhase* ph, int n, const TcChainCommon& c, cudaStream_t stream);
bool gemv_tc_supported(const GemvArgs& g);
size_t gemv_tc_tiled_elems(int N, int K);     // elements of the tiled copy of an [N, K] matrix
// qkv_pairs: rows are taken in the order of the fused q/k/v kernel (RoPE pairs adjacent)
int launch_gemv_tc_repack(const bf16* W, bf16* dst, int N, int K, bool qkv_pairs, cudaStream_t stream);
int launch_gemv_tc_residual(const GemvArgs& g, bf16* out, long long ldo, const bf16* res, long long ldr,
                            cudaStream_t stream);
int launch_gemv_tc_swiglu(const GemvArgs& g, bf16* out, long long ldo, cudaStream_t stream);
int launch_gemv_tc_qkv_rope(const GemvArgs& g, bf16* q_out, long long ldq, bf16* kcache, bf16* vcache,
                            const bf16* cos_t, const bf16* sin_t, int H, int s_max, int pos, cudaStream_t stream,
                            const int* pos_dev = nullptr);
int launch_gemv_tc_logits(const GemvArgs& g, float* logits, long long ldl, cudaStream_t stream);
// logits (bf16-rounded, stored fp32) [B, N]
int launch_gemv_logits(const GemvArgs& g, float* logits, long long ldl, cudaStream_t stream);

// ---- gemv_tcw.cu : 5..16 clips over the slot-ordered weight copy (chunk-major K walk); the activations
// g.x are already normalised (norm_w must be null) and stored window-major ("xwin"): element (b, k) of a
// [B][K] activation lives at xwin_offset(b, k, B); a buffer holds xwin_elems(B, K) elements ----
constexpr int XWIN_KC = 512, XWIN_PITCH = 544;        // 512 k per window row + 32 elements (64 B) of padding
__host__ __device__ inline size_t xwin_offset(int b, int k, int B) {
  return ((size_t)(k / XWIN_KC) * B + b) * XWIN_PITCH + (k % XWIN_KC);
}
inline size_t xwin_elems(int B, int K) { return (size_t)((K + XWIN_KC - 1) / XWIN_KC) * B * XWIN_PITCH; }
// y (xwin layout) = x [B][ldx] rows, RMS-normalised when w != null (LlamaRMSNorm rounding order)
int launch_xwin_norm(const bf16* x, long long ldx, bf16* y, const bf16* w, int B, int K, float eps, cudaStream_t stream);
int init_gemv_tcw_kernels();
bool gemv_tcw_supported(const GemvArgs& g);
int launch_gemv_tcw_residual(const GemvArgs& g, bf16* out, long long ldo, const bf16* res, long long ldr,
                             cudaStream_t stream);
int launch_gemv_tcw_swiglu(const GemvArgs& g, bf16* out, long long ldo, bool out_xwin, cudaStream_t stream);
int launch_gemv_tcw_qkv_rope(const GemvArgs& g, bf16* q_out, long long ldq, bf16* kcache, bf16* vcache,
                             const bf16* cos_t, const bf16* sin_t, int H, int s_max, int pos, cudaStream_t stream,
                             const int* pos_dev = nullptr);
int launch_gemv_tcw_logits(const GemvArgs& g, float* logits, long long ldl, cudaStream_t stream);

// ---- gemv_mma.cu : small-batch (2..16) decode projections on mma.sync, input already normalised ----
int init_gemv_mma_kernels();
int launch_gemv_mma_residual(const GemvArgs& g, bf16* out, long long ldo, const bf16* res, long long ldr,
                             cudaStream_t stream);
int launch_gemv_mma_swiglu(const GemvArgs& g, bf16* out, long long ldo, cudaStream_t stream);
int launch_gemv_mma_qkv_rope(const GemvArgs& g, bf16* q_out, long long ldq, bf16* kcache, bf16* vcache,
                             const bf16* cos_t, const bf16* sin_t, int H, int head_dim, int s_max, int pos,
                             cudaStream_t stream, const int* pos_dev = nullptr);
int launch_gemv_mma_logits(const GemvArgs& g, float* logits, long long ldl, cudaStream_t stream);


}  // namespace vcl
