"""Drop-in for the reference's multimodal model classes on the inference path
(reference: video_chatgpt/model/video_chatgpt.py:16-325 and the bare HF CLIPVisionModel the
reference uses as its vision tower, video_chatgpt/eval/model_utils.py:134-136).

    VisionConfig, VideoChatGPTConfig            :16-34
    VideoChatGPTLlamaModel                      :37-175   (embed + mm_projector + splice + LLaMA stack)
    VideoChatGPTLlamaForCausalLM                :178-321  (forward, generate, prepare_inputs_for_generation)
    CLIPVisionTower                             HF calling convention tower(x, output_hidden_states=True)

All device work goes through one libvcl handle (vcl_native.Engine) shared by the tower and the
language model; these classes only keep state_dicts until the first call, validate inputs the way
the reference does (same ValueError texts for malformed video spans) and translate call
conventions. Differences from the reference, all documented where they occur:
  * compute dtype is bf16 (BASELINE.json); `.half()` is accepted and ignored;
  * `forward` returns logits for the LAST position only, shape [B,1,V] (the reference materialises
    [B,S,V] and every caller on this path reads [:, -1]);
  * the vision tower's `hidden_states` are lazy: an entry is computed when indexed (the path reads [-2]);
    the language model's `hidden_states` are the L+1 tensors HF returns (the last one after the final
    RMSNorm), produced by ONE prefill pass.
"""
from __future__ import annotations

import json
import os
import sys
from types import SimpleNamespace

import torch

_PKG = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
if _PKG not in sys.path:
    sys.path.insert(0, _PKG)
import vcl_native as vn  # noqa: E402

from ..constants import (DEFAULT_VID_END_TOKEN, DEFAULT_VID_START_TOKEN,  # noqa: E402
                         DEFAULT_VIDEO_PATCH_TOKEN)
from .multimodal_projector.builder import build_vision_projector  # noqa: E402


def _host_sampling() -> bool:
    """VCL_HOST_SAMPLING=1: sampling and stopping criteria take one C-ABI step per token with host-side
    sampling (torch.topk / softmax / multinomial) instead of the device sampler and chunked decode loops."""
    return os.environ.get("VCL_HOST_SAMPLING") == "1"


class VisionConfig:
    def __init__(self, frame_size=224, patch_size=14, hidden_size=1024):
        self.frame_size = frame_size
        self.patch_size = patch_size
        self.hidden_size = hidden_size
        self.use_vid_start_end = None
        self.vid_start_token = None
        self.vid_end_token = None
        self.vid_patch_token = None


_CLIP_DEFAULTS = dict(hidden_size=1024, intermediate_size=4096, num_hidden_layers=24, num_attention_heads=16,
                      image_size=224, patch_size=14, layer_norm_eps=1e-5, hidden_act="quick_gelu")


def _clip_config(src) -> SimpleNamespace:
    """CLIP vision config from a dict, an object with attributes, or a directory with config.json."""
    d = dict(_CLIP_DEFAULTS)
    if src is None:
        pass
    elif isinstance(src, dict):
        d.update(src.get("vision_config", src))
    elif isinstance(src, str):
        path = os.path.join(src, "config.json")
        if not os.path.exists(path):
            raise FileNotFoundError(f"mm_vision_tower='{src}' must be a local directory with config.json "
                                    "(no network access on this path)")
        j = json.load(open(path))
        d.update(j.get("vision_config", j))
    else:
        for k in d:
            if hasattr(src, k):
                d[k] = getattr(src, k)
    if d["hidden_act"] != "quick_gelu":
        raise ValueError("libvcl implements the quick_gelu ViT MLP only")
    return SimpleNamespace(**d)


class VideoChatGPTConfig:
    """LLaMA config + the multimodal fields the reference adds (model_type 'VideoChatGPT')."""
    model_type = "VideoChatGPT"

    def __init__(self, **kw):
        self.hidden_size = kw.pop("hidden_size", 4096)
        self.intermediate_size = kw.pop("intermediate_size", 11008)
        self.num_hidden_layers = kw.pop("num_hidden_layers", 32)
        self.num_attention_heads = kw.pop("num_attention_heads", 32)
        self.num_key_value_heads = kw.pop("num_key_value_heads", self.num_attention_heads)
        self.vocab_size = kw.pop("vocab_size", 32000)
        self.rms_norm_eps = kw.pop("rms_norm_eps", 1e-5)
        self.rope_theta = kw.pop("rope_theta", 10000.0)
        self.max_position_embeddings = kw.pop("max_position_embeddings", 2048)
        self.use_cache = kw.pop("use_cache", True)
        for k, v in kw.items():          # mm_vision_tower, use_mm_proj, mm_hidden_size, mm_projector_type, ...
            setattr(self, k, v)
        if self.num_key_value_heads != self.num_attention_heads:
            raise ValueError("libvcl implements multi-head attention only (kv heads == heads), as Vicuna uses")

    @classmethod
    def from_pretrained(cls, path, **kw):
        j = json.load(open(os.path.join(path, "config.json")))
        j.update(kw)
        return cls(**j)


class _LazyStates:
    """Tuple-like view of hidden states; entry i is produced on first access."""

    def __init__(self, n, fn):
        self._n, self._fn, self._cache = n, fn, {}

    def __len__(self):
        return self._n

    def __getitem__(self, i):
        if isinstance(i, slice):
            return tuple(self[j] for j in range(*i.indices(self._n)))
        if i < 0:
            i += self._n
        if not 0 <= i < self._n:
            raise IndexError(i)
        if i not in self._cache:
            self._cache[i] = self._fn(i)
        return self._cache[i]


class _Engines:
    """One vcl handle per process/GPU, created when both configs are known."""

    def __init__(self):
        self.engine = None


class CLIPVisionTower:
    """The vision tower with HF's calling convention (the reference holds a bare CLIPVisionModel):

        outs = tower(pixel_values, output_hidden_states=True)
        feats = outs.hidden_states[-2][:, 1:]          # video_chatgpt/inference.py:93-94

    pixel_values: [N,3,H,W] float (normalised by the image processor) or [N,H,W,3] uint8 raw frames
    (normalised on the device). hidden_states has num_hidden_layers+1 entries like HF; entries are
    computed on access; index -1 needs the last encoder layer, which is only loaded when the tower
    was built with run_layers = num_hidden_layers (the path itself never reads it)."""

    def __init__(self, owner: "VideoChatGPTLlamaForCausalLM"):
        self._owner = owner
        self.config = owner.clip_config
        self.dtype = torch.bfloat16
        self.device = torch.device("cuda")

    def eval(self): return self
    def cuda(self, *a, **k): return self
    def half(self): return self
    def to(self, *a, **k): return self

    def load_state_dict(self, sd, strict=True):
        self._owner._clip_state = {k: v for k, v in sd.items()}
        return SimpleNamespace(missing_keys=[], unexpected_keys=[])

    @torch.no_grad()
    def __call__(self, pixel_values, output_hidden_states=True, **kw):
        eng = self._owner._ensure_engine(need_clip=True)
        n_states = self.config.num_hidden_layers + 1
        px = pixel_values.cuda()

        def state(i):
            if i > eng.cfg.clip_layers:
                raise vn.VclError(f"hidden_states[{i}] needs encoder layer {i}; only {eng.cfg.clip_layers} layers are "
                                  "loaded (the path consumes hidden_states[-2])")
            return eng.clip_encode(px, n_layers=i)

        hs = _LazyStates(n_states, state)
        return SimpleNamespace(hidden_states=hs if output_hidden_states else None)

    forward = __call__


class VideoChatGPTLlamaModel:
    def __init__(self, owner, config):
        self._owner = owner
        self.config = config
        if hasattr(config, "mm_vision_tower") or owner.clip_config is not None:
            cc = owner.clip_config
            self.vision_config = VisionConfig(cc.image_size, cc.patch_size, cc.hidden_size)
        if getattr(config, "use_mm_proj", False):
            if not hasattr(config, "mm_hidden_size"):
                config.mm_hidden_size = self.vision_config.hidden_size
            if self.vision_config.frame_size == 224:       # LLaVA-v1.1-Lightning: plain linear
                config.mm_projector_type = "linear"
            self.mm_projector = build_vision_projector(config)

    def initialize_vision_modules(self, pretrain_mm_mlp_adapter=None, tune_mm_mlp_adapter=False):
        vc = self.vision_config
        self.config.use_mm_proj = True
        self.config.mm_hidden_size = vc.hidden_size
        if not hasattr(self, "mm_projector"):
            if vc.frame_size == 224:
                self.config.mm_projector_type = "linear"
            self.mm_projector = build_vision_projector(self.config)
        if pretrain_mm_mlp_adapter is not None:
            w = torch.load(pretrain_mm_mlp_adapter, map_location="cpu")
            self._owner.load_state_dict({k: v for k, v in w.items() if "mm_projector" in k}, strict=False)
        return dict(num_patches=(vc.frame_size // vc.patch_size) ** 2, vision_config=vc)


class VideoChatGPTLlamaForCausalLM:
    config_class = VideoChatGPTConfig

    def __init__(self, config: VideoChatGPTConfig, clip_config=None, max_batch: int = 1, max_seq: int | None = None,
                 clip_run_layers: int | None = None):
        self.config = config
        self.clip_config = _clip_config(clip_config if clip_config is not None
                                        else getattr(config, "mm_vision_tower", None))
        self.model = VideoChatGPTLlamaModel(self, config)
        self._state: dict = {}
        self._clip_state: dict | None = None
        self._engine = None
        self._max_batch = max_batch
        self._max_seq = max_seq or config.max_position_embeddings
        self._clip_run_layers = clip_run_layers
        self._pos = 0              # tokens in the KV cache after the last forward
        self.training = False
        self.dtype = torch.bfloat16
        self.device = torch.device("cuda")

    # ---- construction / state -----------------------------------------------------------
    @classmethod
    def from_pretrained(cls, model_name, **kw):
        """Local directory with config.json and *.safetensors / pytorch_model*.bin (no hub access)."""
        kw.pop("low_cpu_mem_usage", None); kw.pop("torch_dtype", None)
        use_cache = kw.pop("use_cache", True)
        config = VideoChatGPTConfig.from_pretrained(model_name, use_cache=use_cache)
        m = cls(config, **kw)
        files = sorted(f for f in os.listdir(model_name) if f.endswith((".safetensors", ".bin")) and "training" not in f)
        if not files:
            raise FileNotFoundError(f"no weight files in {model_name}")
        for f in files:
            path = os.path.join(model_name, f)
            if f.endswith(".safetensors"):
                from safetensors.torch import load_file
                m.load_state_dict(load_file(path), strict=False)
            else:
                m.load_state_dict(torch.load(path, map_location="cpu"), strict=False)
        return m

    def get_model(self): return self.model
    def get_vision_tower(self): return CLIPVisionTower(self)
    def eval(self): return self
    def cuda(self, *a, **k): return self
    def half(self): return self
    def to(self, *a, **k): return self
    def parameters(self): return iter(self._state.values())

    def state_dict(self):
        return dict(self._state)

    def load_state_dict(self, sd, strict=True):
        if self._engine is not None:
            raise vn.VclError("weights are already resident in libvcl; load_state_dict must precede the first forward")
        known = lambda k: k.startswith(("model.", "lm_head."))
        unexpected = [k for k in sd if not known(k)]
        for k, v in sd.items():
            if known(k):
                self._state[k] = v
        if strict and unexpected:
            raise RuntimeError(f"Unexpected key(s) in state_dict: {unexpected}")
        return SimpleNamespace(missing_keys=[], unexpected_keys=unexpected)

    def resize_token_embeddings(self, n: int):
        """Grow embed_tokens / lm_head to n rows; new rows start as the mean of the old ones (HF's
        mean-resizing default) and are normally overwritten by the projection checkpoint that the
        reference loads right after (eval/model_utils.py:119-127)."""
        for key in ("model.embed_tokens.weight", "lm_head.weight"):
            w = self._state.get(key)
            if w is None or w.shape[0] == n:
                continue
            if w.shape[0] > n:
                self._state[key] = w[:n].clone()
            else:
                extra = w.float().mean(0, keepdim=True).to(w.dtype).expand(n - w.shape[0], -1)
                self._state[key] = torch.cat([w, extra], 0)
        self.config.vocab_size = n

    def initialize_vision_tokenizer(self, mm_use_vid_start_end, tokenizer, device=None,
                                    tune_mm_mlp_adapter=False, pretrain_mm_mlp_adapter=None):
        vc = self.get_model().vision_config
        vc.use_vid_start_end = mm_use_vid_start_end
        tokenizer.add_tokens([DEFAULT_VIDEO_PATCH_TOKEN], special_tokens=True)
        self.resize_token_embeddings(len(tokenizer))
        if mm_use_vid_start_end:
            tokenizer.add_tokens([DEFAULT_VID_START_TOKEN, DEFAULT_VID_END_TOKEN], special_tokens=True)
            self.resize_token_embeddings(len(tokenizer))
            vc.vid_start_token, vc.vid_end_token = tokenizer.convert_tokens_to_ids(
                [DEFAULT_VID_START_TOKEN, DEFAULT_VID_END_TOKEN])
        vc.vid_patch_token = tokenizer.convert_tokens_to_ids([DEFAULT_VIDEO_PATCH_TOKEN])[0]

    # ---- engine ---------------------------------------------------------------------------
    def _ensure_engine(self, need_clip=False, need_llm=False):
        if self._engine is None:
            c, cc = self.config, self.clip_config
            k = vn.vcl_config()
            k.clip_layers = cc.num_hidden_layers - 1 if self._clip_run_layers is None else self._clip_run_layers
            k.clip_hidden, k.clip_inter, k.clip_heads = cc.hidden_size, cc.intermediate_size, cc.num_attention_heads
            k.image_size, k.patch_size, k.clip_ln_eps = cc.image_size, cc.patch_size, cc.layer_norm_eps
            k.llm_layers, k.llm_hidden, k.llm_inter = c.num_hidden_layers, c.hidden_size, c.intermediate_size
            k.llm_heads, k.vocab = c.num_attention_heads, c.vocab_size
            k.rms_eps, k.rope_theta = c.rms_norm_eps, c.rope_theta
            kind = getattr(c, "mm_projector_type", "linear")
            k.proj_type = vn.PROJ_LINEAR if kind == "linear" else vn.PROJ_MLP2X_GELU
            k.n_temporal = 100
            k.max_frames, k.max_batch, k.max_seq = 100, self._max_batch, self._max_seq
            self._engine = vn.Engine(k)
            self._clip_loaded = self._llm_loaded = False
        if need_clip and not self._clip_loaded:
            if not self._clip_state:
                raise vn.VclError("vision tower weights were never loaded (CLIPVisionTower.load_state_dict)")
            self._engine.load_clip(self._clip_state)
            self._clip_state, self._clip_loaded = None, True
        if need_llm and not self._llm_loaded:
            self._engine.load_llm(self._state)
            self._llm_loaded = True
        return self._engine

    # ---- validation (same errors as video_chatgpt.py:119-128,150-157) ---------------------
    def _video_spans(self, input_ids: torch.Tensor, n_vid: int) -> list:
        """Index of the row after which the projected video rows are spliced, per sample (-1: none)."""
        vc = self.get_model().vision_config
        ids = input_ids.cpu()
        starts = []
        for row in ids:
            if (row == vc.vid_patch_token).sum() == 0:
                starts.append(vn.NO_VIDEO)             # text-only sample
                continue
            if vc.use_vid_start_end:
                if (row == vc.vid_start_token).sum() != (row == vc.vid_end_token).sum():
                    raise ValueError("The number of video start tokens and video end tokens should be the same.")
                pos = torch.where(row == vc.vid_start_token)[0]
                if len(pos) != 1:
                    raise ValueError("libvcl supports exactly one video span per sample")
                s = int(pos[0])
                if s + n_vid + 1 >= len(row) or row[s + n_vid + 1] != vc.vid_end_token:
                    raise ValueError("The video end token should follow the video start token.")
                starts.append(s)
            else:
                if (row == vc.vid_patch_token).sum() != n_vid:
                    raise ValueError("The number of video patch tokens should be the same as the number of video patches.")
                idx = torch.where(row == vc.vid_patch_token)[0]
                s0 = int(idx[0])
                if (idx != torch.arange(s0, s0 + n_vid)).any():
                    raise ValueError("The video patch tokens should be consecutive.")
                starts.append(s0 - 1)                  # rows s0 .. s0+n_vid-1 are replaced (-1: from row 0)
        return starts

    def _spans_dev(self, ids, feats, n_vid):
        starts = self._video_spans(ids, n_vid) if feats is not None else [vn.NO_VIDEO] * ids.shape[0]
        return torch.tensor(starts, dtype=torch.int32, device="cuda")

    # ---- forward / generate ----------------------------------------------------------------
    @torch.no_grad()
    def forward(self, input_ids=None, attention_mask=None, past_key_values=None, inputs_embeds=None, labels=None,
                use_cache=None, output_attentions=None, output_hidden_states=None,
                video_spatio_temporal_features=None, return_dict=None):
        if inputs_embeds is not None or labels is not None or output_attentions:
            raise NotImplementedError("inference path only: input_ids in, logits out")
        eng = self._ensure_engine(need_llm=True)
        ids = input_ids.cuda().to(torch.int64)
        B, S = ids.shape
        if S == 1 and past_key_values is not None:
            # cached single-token step: the video features are ignored, as in the reference (:103)
            logits, _ = eng.decode_step(ids[:, 0].to(torch.int32).contiguous(), self._pos, want_logits=True)
            self._pos += 1
            hs = None
        else:
            feats = video_spatio_temporal_features
            vs = self._spans_dev(ids, feats, eng.NV)
            if feats is not None:
                feats = feats.cuda()
            hs = None
            if output_hidden_states:
                # HF's tuple: [0] the spliced input embeddings, [i] the output of layer i, and the
                # LAST entry after the final RMSNorm ($TF/models/llama/modeling_llama.py:411-425)
                states, logits = eng.prefill_states(ids, feats, vs, want_logits=True)
                L, D = self.config.num_hidden_layers, self.config.hidden_size
                norm_w = self._state["model.norm.weight"].to(device="cuda", dtype=torch.bfloat16).contiguous()
                last = vn.op_rmsnorm(states[L].reshape(B * S, D), norm_w, self.config.rms_norm_eps).view(B, S, D)
                hs = tuple(states[i] for i in range(L)) + (last,)
            else:
                _, logits, _ = eng.prefill(ids, feats, vs, want_logits=True, want_token=False)
            self._pos = S
        return SimpleNamespace(loss=None, logits=logits.to(torch.bfloat16)[:, None, :], past_key_values=self._pos,
                               hidden_states=hs, attentions=None)

    __call__ = forward

    def prepare_inputs_for_generation(self, input_ids, past_key_values=None, attention_mask=None,
                                      inputs_embeds=None, **kwargs):
        """Same contract as the reference (:253-273), with the cache test made explicit: only a
        NON-EMPTY cache narrows input_ids to the last token (the reference's truthiness test breaks
        under transformers 5.x, SURVEY.md 8c)."""
        if past_key_values:
            input_ids = input_ids[:, -1:]
        return {"input_ids": input_ids, "past_key_values": past_key_values, "use_cache": kwargs.get("use_cache"),
                "attention_mask": attention_mask,
                "video_spatio_temporal_features": kwargs.get("video_spatio_temporal_features")}

    _GREEDY_CHUNK = 32      # tokens per device-side decode loop between two host-side EOS checks

    def _eos_pad(self, eos_token_id, pad_token_id):
        """HF generate's defaults: eos from the (generation) config -- LLaMA / Vicuna: 2 -- and padding
        of finished rows with pad_token_id, which falls back to the eos id. Pass eos_token_id=None to
        decode a fixed number of tokens (the benchmark does)."""
        if eos_token_id == "config":
            eos_token_id = getattr(self.config, "eos_token_id", 2)
            if isinstance(eos_token_id, (list, tuple)):
                eos_token_id = eos_token_id[0] if eos_token_id else None
        if pad_token_id is None:
            pad_token_id = getattr(self.config, "pad_token_id", None)
        if pad_token_id is None:
            pad_token_id = eos_token_id
        return eos_token_id, pad_token_id

    @torch.no_grad()
    def generate(self, input_ids, video_spatio_temporal_features=None, do_sample=False, temperature=1.0,
                 max_new_tokens=32, stopping_criteria=None, eos_token_id="config", pad_token_id=None, top_k=50,
                 **kw):
        """Returns [B, S+n] int64 INCLUDING the prompt, like HF generate (inference.py:105-120), and
        like HF it stops at EOS (config.eos_token_id unless eos_token_id is given; None disables it):
        finished rows are padded, the call returns when every row has finished.
        Everything runs on the device: prefill + CUDA-graph decode loops of 32 tokens with one host-side
        check per loop (a single loop of exactly max_new_tokens for greedy decoding without EOS or
        stopping criteria). Sampling (temperature, top-k 50 as HF defaults) uses the device sampler
        (include/vcl.h, vcl_sampling) with a seed drawn from torch's default CPU generator, so
        torch.manual_seed makes runs reproducible. Stopping criteria are called after each loop, exactly
        as a per-token loop would call them (_replay). VCL_HOST_SAMPLING=1 in the environment keeps the
        per-token C-ABI step with host-side sampling and checks (_stepwise) for sampling and criteria."""
        eng = self._ensure_engine(need_llm=True)
        ids = input_ids.cuda().to(torch.int64)
        B, S = ids.shape
        feats = video_spatio_temporal_features
        vs = self._spans_dev(ids, feats, eng.NV)
        if feats is not None:
            feats = feats.cuda()
        n = min(max_new_tokens, self._max_seq - S)
        if n <= 0:
            raise ValueError(f"prompt length {S} leaves no room in max_seq {self._max_seq}")
        eos, pad = self._eos_pad(eos_token_id, pad_token_id)
        if (do_sample or stopping_criteria) and _host_sampling():
            _, logits, _ = eng.prefill(ids, feats, vs, want_logits=True, want_token=False)
            self._pos = S
            self._last_out = self._stepwise(eng, ids, logits, n, do_sample, temperature, stopping_criteria, eos, pad,
                                            top_k)
            return self._last_out
        if (do_sample and temperature > 0) or stopping_criteria:
            sp = self._sampling(do_sample, temperature, top_k)
            if sp is None:
                first_chunk = lambda c: eng.generate(ids, feats, vs, c)
            else:
                first_chunk = lambda c: eng.generate_sampled(ids, feats, vs, c, *sp)
            self._last_out = self._device_decode(eng, ids, first_chunk, n, sp, stopping_criteria, eos, pad)
            return self._last_out
        if eos is None:
            new = eng.generate(ids, feats, vs, n).to(torch.int64)
            self._pos = S + n - 1
            self._last_out = torch.cat([ids, new], dim=1)
            return self._last_out
        # greedy with EOS: device loops of _GREEDY_CHUNK tokens, EOS looked for between them
        c = min(n, self._GREEDY_CHUNK)
        new = eng.generate(ids, feats, vs, c).to(torch.int64)
        while True:
            new, done = self._mask_finished(new, eos, pad)
            k = new.shape[1]
            if done or k >= n:
                break
            m = min(self._GREEDY_CHUNK, n - k)
            more = eng.decode_loop(new[:, -1].to(torch.int32).contiguous(), S + k - 1, m + 1)
            new = torch.cat([new, more[:, 1:].to(torch.int64)], dim=1)
        self._pos = S + new.shape[1] - 1
        self._last_out = torch.cat([ids, new], dim=1)
        return self._last_out

    @staticmethod
    def _mask_finished(new, eos, pad):
        """Pad every row after its first EOS; when all rows have one, cut at the longest row."""
        is_eos = new == eos
        seen = torch.cumsum(is_eos.to(torch.int32), dim=1)
        after = (seen - is_eos.to(torch.int32)) > 0            # strictly after the first EOS
        new = torch.where(after, torch.full_like(new, pad), new)
        if bool((seen[:, -1] > 0).all()):
            first = is_eos.to(torch.int32).argmax(dim=1)
            return new[:, : int(first.max()) + 1], True
        return new, False

    def generate_continue(self, new_input_ids, do_sample=False, temperature=1.0, max_new_tokens=32,
                          stopping_criteria=None, eos_token_id="config", pad_token_id=None, top_k=50):
        """Next turn about the SAME video(s): `new_input_ids` [B, S_new] follow everything generated
        so far. Only the tokens the KV cache does not hold yet (the last generated token and the new
        text) are prefilled (vcl_llm_prefill_append); the reference re-runs the tower and the whole
        prompt every turn (chat.py:137-154). Returns the full sequence [B, S_total + n] like generate."""
        if getattr(self, "_last_out", None) is None:
            raise ValueError("generate_continue: no previous generate() to continue")
        eng = self._ensure_engine(need_llm=True)
        prev = self._last_out
        tail = torch.cat([prev[:, self._pos:], new_input_ids.cuda().to(torch.int64)], dim=1)
        start = self._pos
        ctx = torch.cat([prev, new_input_ids.cuda().to(torch.int64)], dim=1)
        n = min(max_new_tokens, self._max_seq - ctx.shape[1])
        if n <= 0:
            raise ValueError(f"context length {ctx.shape[1]} leaves no room in max_seq {self._max_seq}")
        eos, pad = self._eos_pad(eos_token_id, pad_token_id)
        if _host_sampling():
            _, logits, _ = eng.prefill_append(tail, start, want_logits=True, want_token=False)
            self._pos = ctx.shape[1]
            self._last_out = self._stepwise(eng, ctx, logits, n, do_sample, temperature, stopping_criteria, eos, pad,
                                            top_k)
            return self._last_out
        sp = self._sampling(do_sample, temperature, top_k)
        P0 = ctx.shape[1]                                       # position of the first new token
        if sp is None:
            _, _, first = eng.prefill_append(tail, start, want_token=True)
            first_chunk = lambda c: eng.decode_loop(first, P0, c)
        else:
            _, logits, _ = eng.prefill_append(tail, start, want_logits=True, want_token=False)
            first = vn.op_sample(logits, *sp, pos=P0)
            first_chunk = lambda c: eng.decode_loop_sampled(first, P0, c, *sp)
        self._last_out = self._device_decode(eng, ctx, first_chunk, n, sp, stopping_criteria, eos, pad)
        return self._last_out

    @staticmethod
    def _sampling(do_sample, temperature, top_k):
        """(temperature, top_k, seed) for the device sampler, None for greedy decoding. The seed comes from
        torch's default CPU generator, one draw per call."""
        if not (do_sample and temperature > 0):
            return None
        seed = int(torch.randint(0, 2 ** 63 - 1, (1,)))
        return float(temperature), int(top_k or 0), seed

    def _device_decode(self, eng, out, first_chunk, n, sp, stopping_criteria, eos, pad):
        """Up to n new tokens after `out` [B, P0] in device loops of _GREEDY_CHUNK tokens; first_chunk(c) gives
        the first c tokens ([B, c] int32, token 0 at position P0), later loops continue from the last token.
        After each loop _replay makes the calls _stepwise would have made, in the same order, and cuts `out`
        where _stepwise would have stopped. Tokens computed past that point stay in the KV cache as dead rows:
        decode attention reads only pos + 1 keys and the next prefill (generate_continue) overwrites them."""
        P0 = out.shape[1]
        unfinished = torch.ones(out.shape[0], dtype=torch.bool)
        new = first_chunk(min(n, self._GREEDY_CHUNK))
        k = 0
        while True:
            out, unfinished, stopped = self._replay(out, new, unfinished, stopping_criteria, eos, pad)
            k += new.shape[1]
            if stopped or k >= n:
                break
            m = min(self._GREEDY_CHUNK, n - k)
            last = new[:, -1].to(torch.int32).contiguous()
            more = (eng.decode_loop(last, P0 + k - 1, m + 1) if sp is None
                    else eng.decode_loop_sampled(last, P0 + k - 1, m + 1, *sp))
            new = more[:, 1:]
        self._pos = out.shape[1] - 1
        return out

    @staticmethod
    def _replay(out, new, unfinished, stopping_criteria, eos, pad):
        """_stepwise's per-token bookkeeping over the device tokens `new` [B, c]: append each token (pad if
        its row has finished), update `unfinished`, stop when no row is left, else call every criterion on
        the prefix and stop at the first True. Returns (out, unfinished, stopped)."""
        new_h = new.to(device="cpu", dtype=torch.int64)
        cols = []
        stopped = False
        for j in range(new_h.shape[1]):
            nxt = new_h[:, j]
            if eos is not None:
                nxt = torch.where(unfinished, nxt, torch.full_like(nxt, pad))
            cols.append(nxt)
            if stopping_criteria:
                out = torch.cat([out, nxt[:, None].to(out.device)], dim=1)   # the prefix the criteria see
            if eos is not None:
                unfinished = unfinished & (nxt != eos)
                if not bool(unfinished.any()):
                    stopped = True
                    break
            if stopping_criteria and any(c(out, None) for c in stopping_criteria):
                stopped = True
                break
        if not stopping_criteria:
            out = torch.cat([out, torch.stack(cols, dim=1).to(out.device)], dim=1)
        return out, unfinished, stopped

    def _stepwise(self, eng, out, logits, n, do_sample, temperature, stopping_criteria, eos, pad, top_k=50):
        """One token per C-ABI call (VCL_HOST_SAMPLING=1). After the loop the cache holds every returned token but the last
        (self._pos = out.shape[1] - 1), the state generate_continue starts from."""
        unfinished = torch.ones(out.shape[0], dtype=torch.bool, device=out.device)
        for step in range(n):
            if do_sample and temperature > 0:
                lg = logits / temperature
                if top_k and top_k < lg.shape[-1]:            # HF's default warpers: temperature, then top-k 50
                    kth = torch.topk(lg, top_k, dim=-1).values[:, -1:]
                    lg = lg.masked_fill(lg < kth, float("-inf"))
                nxt = torch.multinomial(torch.softmax(lg, dim=-1), 1)[:, 0]
            else:
                nxt = logits.argmax(-1)
            if eos is not None:
                nxt = torch.where(unfinished, nxt, torch.full_like(nxt, pad))
            out = torch.cat([out, nxt[:, None].to(torch.int64)], dim=1)
            if eos is not None:
                unfinished = unfinished & (nxt != eos)
                if not bool(unfinished.any()):
                    break
            if stopping_criteria and any(c(out, None) for c in stopping_criteria):
                break
            if step + 1 == n or self._pos >= self._max_seq:
                break
            logits, _ = eng.decode_step(nxt.to(torch.int32).contiguous(), self._pos, want_logits=True)
            self._pos += 1
        return out
