"""ctypes binding of libvcl.so (include/vcl.h). PyTorch is used only as the owner of device
memory and streams: every call passes raw device pointers and the current CUDA stream.

There is no fallback: if the shared library is missing or the device is not an sm_100 GPU the
calls raise.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, Structure, c_char_p, c_float, c_int, c_int32, c_int64, c_uint64, c_void_p

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libvcl.so")

DTYPE_F16, DTYPE_BF16 = 0, 1
PIXELS_BF16_NCHW, PIXELS_U8_NHWC = 0, 1
PROJ_LINEAR, PROJ_MLP2X_GELU = 0, 1
NO_VIDEO = -2 ** 31          # vid_start value of a text-only row (VCL_NO_VIDEO)
ACT_NONE, ACT_QGELU, ACT_GELU, ACT_SWIGLU = 0, 1, 2, 3


class VclError(RuntimeError):
    pass


class vcl_config(Structure):
    _fields_ = [
        ("clip_layers", c_int32), ("clip_hidden", c_int32), ("clip_inter", c_int32),
        ("clip_heads", c_int32), ("image_size", c_int32), ("patch_size", c_int32),
        ("clip_ln_eps", c_float),
        ("llm_layers", c_int32), ("llm_hidden", c_int32), ("llm_inter", c_int32),
        ("llm_heads", c_int32), ("vocab", c_int32), ("rms_eps", c_float), ("rope_theta", c_float),
        ("proj_type", c_int32), ("n_temporal", c_int32),
        ("max_frames", c_int32), ("max_batch", c_int32), ("max_seq", c_int32),
    ]


class vcl_tensor(Structure):
    _fields_ = [("name", c_char_p), ("data", c_void_p), ("ndim", c_int32), ("shape", c_int64 * 4)]


class vcl_sampling(Structure):
    _fields_ = [("temperature", c_float), ("top_k", c_int32), ("seed", c_uint64)]


def sampling(temperature: float, top_k, seed: int) -> vcl_sampling:
    """The vcl_sampling struct (include/vcl.h); top_k None or 0 means no top-k filter."""
    return vcl_sampling(float(temperature), int(top_k or 0), int(seed) & (2 ** 64 - 1))


# name -> (restype, argtypes); mirrors include/vcl.h one to one
_SIGNATURES = {
    "vcl_version": (c_int, []),
    "vcl_last_error": (c_char_p, []),
    "vcl_create": (c_int, [POINTER(c_void_p), POINTER(vcl_config)]),
    "vcl_destroy": (None, [c_void_p]),
    "vcl_load_clip_weights": (c_int, [c_void_p, POINTER(vcl_tensor), c_int]),
    "vcl_load_llm_weights": (c_int, [c_void_p, POINTER(vcl_tensor), c_int]),
    "vcl_clip_encode": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "vcl_st_pool": (c_int, [c_void_p, c_int, c_int64, c_int64, c_int, c_int, c_int, c_int, c_void_p,
                            c_int, c_void_p]),
    "vcl_clip_features": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_int, c_void_p]),
    "vcl_llm_prefill": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p,
                                c_void_p, c_void_p, c_void_p]),
    "vcl_llm_prefill_states": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "vcl_llm_prefill_append": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p]),
    "vcl_llm_decode_step": (c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "vcl_llm_generate": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p,
                                 c_void_p]),
    "vcl_llm_decode_loop": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p]),
    "vcl_llm_generate_sampled": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int,
                                         POINTER(vcl_sampling), c_void_p, c_void_p]),
    "vcl_llm_decode_loop_sampled": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, POINTER(vcl_sampling), c_void_p,
                                            c_void_p]),
    "vcl_op_sample": (c_int, [c_void_p, c_int64, c_int, c_int, POINTER(vcl_sampling), c_int, c_void_p, c_void_p]),
    "vcl_launch_count": (ctypes.c_longlong, []),
    "vcl_op_gemm": (c_int, [c_void_p, c_int64, c_void_p, c_int64, c_void_p, c_int64, c_void_p, c_void_p,
                            c_int64, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "vcl_op_gemm_ex": (c_int, [c_void_p, c_int64, c_void_p, c_int64, c_void_p, c_int64, c_void_p, c_void_p,
                               c_int64, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "vcl_op_layernorm": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_float, c_void_p]),
    "vcl_op_rmsnorm": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_float, c_void_p]),
    "vcl_op_attention": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int,
                                 c_float, c_int, c_void_p]),
    "vcl_op_attention_vit": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    "vcl_op_gemv": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_float, c_int, c_int,
                            c_int, c_void_p]),
}

EXPORTED_SYMBOLS = tuple(_SIGNATURES)

_lib = None


def lib() -> ctypes.CDLL:
    """Load libvcl.so (built in-tree by build.py). Fails loudly if it is absent."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise VclError(f"{LIB_PATH} is missing: run `python video-llava_b200/build.py` "
                           "(there is no CPU or PyTorch fallback for this path)")
        l = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(l, name)
            fn.restype = res
            fn.argtypes = args
        _lib = l
    return _lib


def check(rc: int) -> None:
    if rc != 0:
        raise VclError(f"libvcl error {rc}: {lib().vcl_last_error().decode()}")


def ptr(t) -> c_void_p:
    if t is None:
        return c_void_p(0)
    assert t.is_cuda and t.is_contiguous(), "vcl needs contiguous CUDA tensors"
    return c_void_p(t.data_ptr())


def cur_stream() -> c_void_p:
    return c_void_p(torch.cuda.current_stream().cuda_stream)


def _dtype_code(dt: torch.dtype) -> int:
    if dt == torch.float16:
        return DTYPE_F16
    if dt == torch.bfloat16:
        return DTYPE_BF16
    raise VclError(f"unsupported dtype {dt} (fp16 / bf16 only)")


# ---------------------------------------------------------------------------------------------
# stateless operators
# ---------------------------------------------------------------------------------------------
def st_pool(features: torch.Tensor, n_temporal: int = 100, out_dtype: torch.dtype = torch.float16):
    """[T,P,C] (fp16|bf16, last dim contiguous) -> [n_temporal+P, C]; see vcl_st_pool."""
    T, P, C = features.shape
    assert features.is_cuda and features.stride(2) == 1
    out = torch.empty(n_temporal + P, C, dtype=out_dtype, device=features.device)
    check(lib().vcl_st_pool(c_void_p(features.data_ptr()), _dtype_code(features.dtype),
                            features.stride(0), features.stride(1), T, P, C, n_temporal,
                            ptr(out), _dtype_code(out_dtype), cur_stream()))
    return out


def op_gemm(a, w, bias=None, residual=None, act=ACT_NONE, block_n=0, out=None, cluster=0):
    M, K = a.shape
    N = w.shape[0]
    n_out = N // 2 if act == ACT_SWIGLU else N
    if out is None:
        out = torch.empty(M, n_out, dtype=torch.bfloat16, device=a.device)
    check(lib().vcl_op_gemm_ex(ptr(a), a.stride(0), ptr(w), w.stride(0), ptr(out), out.stride(0), ptr(bias),
                               ptr(residual), residual.stride(0) if residual is not None else 0, M, N, K,
                               act, block_n, cluster, cur_stream()))
    return out


def op_layernorm(x, w, b, eps):
    y = torch.empty_like(x)
    check(lib().vcl_op_layernorm(ptr(x), ptr(y), ptr(w), ptr(b), x.shape[0], x.shape[1], eps, cur_stream()))
    return y


def op_rmsnorm(x, w, eps):
    y = torch.empty_like(x)
    check(lib().vcl_op_rmsnorm(ptr(x), ptr(y), ptr(w), x.shape[0], x.shape[1], eps, cur_stream()))
    return y


def op_attention(q, k, v, scale, causal):
    """q,k,v: [B,S,H,hd] contiguous bf16."""
    B, S, H, hd = q.shape
    o = torch.empty_like(q)
    check(lib().vcl_op_attention(ptr(q), ptr(k), ptr(v), ptr(o), B, S, H, hd, scale, int(causal), cur_stream()))
    return o


def op_attention_vit(qkv, n_frames, S, H):
    """qkv: [n_frames*S, 3*H*64] bf16 -> [n_frames*S, H*64] (tcgen05 ViT attention)."""
    out = torch.empty(n_frames * S, H * 64, dtype=torch.bfloat16, device=qkv.device)
    check(lib().vcl_op_attention_vit(ptr(qkv), ptr(out), n_frames, S, H, cur_stream()))
    return out


def op_gemv(x, w, res=None, norm_w=None, eps=0.0):
    B, K = x.shape
    N = w.shape[0]
    out = torch.empty(B, N, dtype=torch.bfloat16, device=x.device)
    check(lib().vcl_op_gemv(ptr(x), ptr(w), ptr(out), ptr(res), ptr(norm_w), eps, B, N, K, cur_stream()))
    return out


def op_sample(logits, temperature, top_k, seed, pos):
    """[B, V] fp32 logits (row stride may exceed V) -> [B] int32 tokens for sequence position `pos`
    (the contract of vcl_sampling)."""
    B, V = logits.shape
    assert logits.is_cuda and logits.dtype == torch.float32 and logits.stride(1) == 1
    tok = torch.empty(B, dtype=torch.int32, device=logits.device)
    sp = sampling(temperature, top_k, seed)
    check(lib().vcl_op_sample(c_void_p(logits.data_ptr()), logits.stride(0), B, V, ctypes.byref(sp), int(pos),
                              ptr(tok), cur_stream()))
    return tok


# ---------------------------------------------------------------------------------------------
# engine handle
# ---------------------------------------------------------------------------------------------
def _tensor_array(state: dict, keep: list):
    """Pack a {name: cuda bf16 tensor} dict into a vcl_tensor array (tensors kept alive in `keep`)."""
    arr = (vcl_tensor * len(state))()
    for i, (name, t) in enumerate(state.items()):
        t = t.detach()
        if t.dtype != torch.bfloat16 or not t.is_cuda or not t.is_contiguous():
            t = t.to(device="cuda", dtype=torch.bfloat16).contiguous()
        keep.append(t)
        arr[i].name = name.encode()
        arr[i].data = t.data_ptr()
        arr[i].ndim = t.dim()
        for d in range(t.dim()):
            arr[i].shape[d] = t.shape[d]
    return arr


def launch_count() -> int:
    return int(lib().vcl_launch_count())


class Engine:
    """Owns one vcl_handle (one per process / GPU)."""

    def __init__(self, cfg: vcl_config):
        self.cfg = cfg
        self._h = c_void_p()
        check(lib().vcl_create(ctypes.byref(self._h), ctypes.byref(cfg)))
        g = cfg.image_size // cfg.patch_size
        self.P = g * g
        self.NV = cfg.n_temporal + self.P

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            lib().vcl_destroy(self._h)
            self._h = c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- weights ----
    def load_clip(self, state: dict):
        keep: list = []
        arr = _tensor_array(state, keep)
        torch.cuda.synchronize()
        check(lib().vcl_load_clip_weights(self._h, arr, len(state)))

    def load_llm(self, state: dict):
        keep: list = []
        arr = _tensor_array(state, keep)
        torch.cuda.synchronize()
        check(lib().vcl_load_llm_weights(self._h, arr, len(state)))

    # ---- vision ----
    @staticmethod
    def _pixels(pixels: torch.Tensor):
        """-> (contiguous tensor, format code, frame height, frame width); the layout is told by the
        dtype: uint8 = raw [N,H,W,3] frames, floating = normalised [N,3,H,W] pixel_values."""
        if pixels.dim() != 4:
            raise VclError(f"pixels must be 4-D, got shape {tuple(pixels.shape)}")
        if pixels.dtype == torch.uint8:
            if pixels.shape[3] != 3:
                raise VclError(f"uint8 frames must be [N,H,W,3] (channels last), got {tuple(pixels.shape)}")
            return pixels.contiguous(), PIXELS_U8_NHWC, pixels.shape[1], pixels.shape[2]
        if pixels.shape[1] != 3:
            raise VclError(f"pixel_values must be [N,3,H,W], got {tuple(pixels.shape)}")
        return pixels.to(torch.bfloat16).contiguous(), PIXELS_BF16_NCHW, pixels.shape[2], pixels.shape[3]

    def clip_encode(self, pixels: torch.Tensor, n_layers: int | None = None) -> torch.Tensor:
        """pixels: [N,3,H,W] bf16 (normalised) or [N,H,W,3] uint8 -> hidden_states[n_layers] [N,1+P,C]."""
        pixels, fmt, fh, fw = self._pixels(pixels)
        n = pixels.shape[0]
        nl = self.cfg.clip_layers if n_layers is None else n_layers
        out = torch.empty(n, self.P + 1, self.cfg.clip_hidden, dtype=torch.bfloat16, device=pixels.device)
        check(lib().vcl_clip_encode(self._h, ptr(pixels), fmt, n, fh, fw, nl, ptr(out), cur_stream()))
        return out

    def clip_features(self, pixels: torch.Tensor, out_dtype=torch.float16, out=None) -> torch.Tensor:
        pixels, fmt, fh, fw = self._pixels(pixels)
        if out is None:
            out = torch.empty(self.NV, self.cfg.clip_hidden, dtype=out_dtype, device=pixels.device)
        else:
            out_dtype = out.dtype
            assert out.shape == (self.NV, self.cfg.clip_hidden)
        check(lib().vcl_clip_features(self._h, ptr(pixels), fmt, pixels.shape[0], fh, fw, ptr(out),
                                      _dtype_code(out_dtype), cur_stream()))
        return out

    # ---- language model ----
    def prefill(self, ids, video_feats, vid_start, n_layers=None, want_hidden=False, want_logits=False,
                want_token=True, tok_out=None):
        B, S = ids.shape
        nl = self.cfg.llm_layers if n_layers is None else n_layers
        dev = ids.device
        hidden = torch.empty(B, S, self.cfg.llm_hidden, dtype=torch.bfloat16, device=dev) if want_hidden else None
        logits = torch.empty(B, self.cfg.vocab, dtype=torch.float32, device=dev) if want_logits else None
        tok = tok_out if tok_out is not None else (
            torch.empty(B, dtype=torch.int32, device=dev) if want_token else None)
        vf = None
        if video_feats is not None:
            vf = video_feats.to(torch.bfloat16).contiguous()
            assert vf.shape == (B, self.NV, self.cfg.clip_hidden), vf.shape
        check(lib().vcl_llm_prefill(self._h, ptr(ids.contiguous()), ptr(vf), ptr(vid_start.contiguous()), B, S,
                                    nl, ptr(hidden), ptr(logits), ptr(tok), cur_stream()))
        return hidden, logits, tok

    def prefill_states(self, ids, video_feats, vid_start, want_logits=False):
        """Full-depth prefill keeping every hidden state: ([L+1, B, S, D] bf16 raw layer outputs,
        last-position logits [B, vocab] | None)."""
        B, S = ids.shape
        dev = ids.device
        states = torch.empty(self.cfg.llm_layers + 1, B, S, self.cfg.llm_hidden, dtype=torch.bfloat16, device=dev)
        logits = torch.empty(B, self.cfg.vocab, dtype=torch.float32, device=dev) if want_logits else None
        vf = None
        if video_feats is not None:
            vf = video_feats.to(torch.bfloat16).contiguous()
            assert vf.shape == (B, self.NV, self.cfg.clip_hidden), vf.shape
        check(lib().vcl_llm_prefill_states(self._h, ptr(ids.contiguous()), ptr(vf), ptr(vid_start.contiguous()), B, S,
                                           ptr(states), ptr(logits), cur_stream()))
        return states, logits

    def prefill_append(self, ids, start_pos, want_hidden=False, want_logits=False, want_token=True):
        """Continue the cached sequences with `ids` [B, S] (text only) at positions start_pos.. ;
        returns (hidden [B,S,D] | None, logits [B,vocab] | None, next token [B] | None)."""
        B, S = ids.shape
        dev = ids.device
        hidden = torch.empty(B, S, self.cfg.llm_hidden, dtype=torch.bfloat16, device=dev) if want_hidden else None
        logits = torch.empty(B, self.cfg.vocab, dtype=torch.float32, device=dev) if want_logits else None
        tok = torch.empty(B, dtype=torch.int32, device=dev) if want_token else None
        check(lib().vcl_llm_prefill_append(self._h, ptr(ids.contiguous()), B, S, int(start_pos), ptr(hidden),
                                           ptr(logits), ptr(tok), cur_stream()))
        return hidden, logits, tok

    def decode_step(self, tok_in, pos, want_logits=False):
        B = tok_in.shape[0]
        logits = torch.empty(B, self.cfg.vocab, dtype=torch.float32, device=tok_in.device) if want_logits else None
        tok = torch.empty(B, dtype=torch.int32, device=tok_in.device)
        check(lib().vcl_llm_decode_step(self._h, ptr(tok_in.contiguous()), B, pos, ptr(logits), ptr(tok),
                                        cur_stream()))
        return logits, tok

    def decode_loop(self, first_tok, S, n_new, out=None):
        B = first_tok.shape[0]
        if out is None:
            out = torch.empty(B, n_new, dtype=torch.int32, device=first_tok.device)
        check(lib().vcl_llm_decode_loop(self._h, ptr(first_tok.contiguous()), B, S, n_new, ptr(out), cur_stream()))
        return out

    def generate(self, ids, video_feats, vid_start, n_new):
        B, S = ids.shape
        out = torch.empty(B, n_new, dtype=torch.int32, device=ids.device)
        vf = None
        if video_feats is not None:
            vf = video_feats.to(torch.bfloat16).contiguous()
        check(lib().vcl_llm_generate(self._h, ptr(ids.contiguous()), ptr(vf), ptr(vid_start.contiguous()), B, S,
                                     n_new, ptr(out), cur_stream()))
        return out

    def generate_sampled(self, ids, video_feats, vid_start, n_new, temperature, top_k, seed):
        B, S = ids.shape
        out = torch.empty(B, n_new, dtype=torch.int32, device=ids.device)
        vf = None
        if video_feats is not None:
            vf = video_feats.to(torch.bfloat16).contiguous()
        sp = sampling(temperature, top_k, seed)
        check(lib().vcl_llm_generate_sampled(self._h, ptr(ids.contiguous()), ptr(vf), ptr(vid_start.contiguous()), B,
                                             S, n_new, ctypes.byref(sp), ptr(out), cur_stream()))
        return out

    def decode_loop_sampled(self, first_tok, S, n_new, temperature, top_k, seed, out=None):
        B = first_tok.shape[0]
        if out is None:
            out = torch.empty(B, n_new, dtype=torch.int32, device=first_tok.device)
        sp = sampling(temperature, top_k, seed)
        check(lib().vcl_llm_decode_loop_sampled(self._h, ptr(first_tok.contiguous()), B, S, n_new, ctypes.byref(sp),
                                                ptr(out), cur_stream()))
        return out
