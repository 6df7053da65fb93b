"""Generate the golden fixtures in this directory by running THE REFERENCE ITSELF.

It needs a checkout of PG-Video-LLaVA (mbzuai-oryx/Video-LLaVA); the tests only read the fixtures:

    python tests/golden/make_golden.py <reference checkout>

What is executed (nothing from this repo's product code, and no copy of reference source):
  * <reference>/video_chatgpt/model/video_chatgpt.py : VideoChatGPTLlamaForCausalLM.forward
    (embedding splice, mm_projector, lm_head) on top of the installed transformers LlamaModel
  * <reference>/video_chatgpt/inference.py : get_spatio_temporal_features_torch
  * <reference>/scripts/save_spatio_temporal_clip_features.py : get_spatio_temporal_features
  * transformers.CLIPVisionModel (what the reference instantiates for its vision tower,
    video_chatgpt/eval/model_utils.py:134), attn_implementation="eager"
all in fp32 on CPU, with the seeded synthetic weights/inputs of oracle/vcl_oracle.py
(random_clip_state / random_llm_state / make_frames / make_prompt_ids), so that the oracle, the
reference and libvcl.so can be fed identical bytes. Greedy decoding uses the hand-rolled loop of
SURVEY.md 9.2 because model.generate is broken under transformers 5.x with the reference's
prepare_inputs_for_generation (video_chatgpt.py:253-257).

Outputs (all small; see tests/test_oracle_cpu.py and tests/test_parity_gpu.py for their use):
  clip_tiny.npz   3-layer ViT (full width 1024), 3 frames: slices + row norms of hidden_states[0..2]
  pool.npz        reference torch and numpy pooling of seeded fp16 features, T=8 (padded) and T=100;
                  the numpy results are stored as the XOR of their fp16 bit patterns with the torch
                  results (*_xor_torch), which keeps the file small (tests/_util.py: load_pool_golden)
  config1.npz     BASELINE config 1: 8 frames, full 24-layer ViT-L/14 -> pooled [356,1024] (fp32 run)
  llm_tiny.npz    2-layer LLaMA (hidden 512, 4 heads), B=2, S=448: last-row logits, hidden slices,
                  8 greedy tokens per clip; plus the malformed-span error behaviour
  bf16_tiny.npz   the same two tiny models cast to bf16 (the benchmark dtype) and run by the reference /
                  HF on CPU: hidden states, logits and greedy ids stored as raw bf16 bit patterns
                  (uint16), so the oracle's bf16 ROUNDING POINTS are pinned bit for bit, not just its
                  fp32 arithmetic. `rotary_emb.inv_freq` stays fp32, as `from_pretrained(torch_dtype=
                  bf16)` leaves it (a blanket `.to(bf16)` would round the rotary frequencies too).
"""
import importlib.util
import os
import sys
import tempfile
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
if len(sys.argv) != 2:
    sys.exit("usage: python tests/golden/make_golden.py <reference checkout>")
REF = os.path.abspath(sys.argv[1])
sys.path.insert(0, ROOT)
sys.path.insert(0, REF)

# the reference imports decord at module import time (eval/model_utils.py:4); it is not installed
sys.modules.setdefault("decord", types.SimpleNamespace(VideoReader=None, cpu=None))

from transformers import CLIPVisionConfig, CLIPVisionModel  # noqa: E402

from oracle import vcl_oracle as O  # noqa: E402
from video_chatgpt.inference import get_spatio_temporal_features_torch  # noqa: E402  (reference)
from video_chatgpt.model.video_chatgpt import (VideoChatGPTConfig,  # noqa: E402  (reference)
                                               VideoChatGPTLlamaForCausalLM)

_spec = importlib.util.spec_from_file_location(
    "ref_save_features", os.path.join(REF, "scripts", "save_spatio_temporal_clip_features.py"))


def _load_ref_numpy_pool():
    # the script imports decord/tqdm at the top; both are stubbed / present
    mod = importlib.util.module_from_spec(_spec)
    _spec.loader.exec_module(mod)
    return mod.get_spatio_temporal_features


def build_clip(cfg: O.ClipCfg, sd: dict) -> CLIPVisionModel:
    hf = CLIPVisionConfig(hidden_size=cfg.hidden, intermediate_size=cfg.inter, num_hidden_layers=cfg.layers,
                          num_attention_heads=cfg.heads, image_size=cfg.image, patch_size=cfg.patch,
                          projection_dim=768, hidden_act="quick_gelu", layer_norm_eps=cfg.eps,
                          attn_implementation="eager")
    m = CLIPVisionModel(hf).eval()
    full = dict(sd)
    full["vision_model.post_layernorm.weight"] = torch.ones(cfg.hidden)
    full["vision_model.post_layernorm.bias"] = torch.zeros(cfg.hidden)
    missing, unexpected = m.load_state_dict(full, strict=False)
    assert not unexpected, unexpected
    assert all("position_ids" in k for k in missing), missing
    return m


def build_llm(cfg: O.LlmCfg, sd: dict, clip_cfg: O.ClipCfg) -> VideoChatGPTLlamaForCausalLM:
    d = tempfile.mkdtemp()
    CLIPVisionConfig(hidden_size=clip_cfg.hidden, intermediate_size=clip_cfg.inter, num_hidden_layers=clip_cfg.layers,
                     num_attention_heads=clip_cfg.heads, image_size=clip_cfg.image, patch_size=clip_cfg.patch,
                     projection_dim=768).save_pretrained(d)
    c = VideoChatGPTConfig(hidden_size=cfg.hidden, intermediate_size=cfg.inter, num_hidden_layers=cfg.layers,
                           num_attention_heads=cfg.heads, num_key_value_heads=cfg.heads, vocab_size=cfg.vocab,
                           rms_norm_eps=cfg.rms_eps, rope_theta=cfg.rope_theta, max_position_embeddings=4096,
                           attn_implementation="eager", tie_word_embeddings=False)
    c.mm_vision_tower = d
    c.use_mm_proj = True
    c.mm_hidden_size = cfg.mm_hidden
    if cfg.proj_type != "linear":
        c.mm_projector_type = cfg.proj_type
    m = VideoChatGPTLlamaForCausalLM(c).eval()
    missing, unexpected = m.load_state_dict(sd, strict=False)
    assert not unexpected and not missing, (missing, unexpected)
    vc = m.get_model().vision_config
    vc.vid_patch_token, vc.vid_start_token, vc.vid_end_token = cfg.vid_patch_token, cfg.vid_start_token, cfg.vid_end_token
    vc.use_vid_start_end = True
    return m


def ref_greedy(m, ids, feats, n_new):
    """SURVEY.md 9.2 work-around (i): prefill with use_cache, then last-token steps."""
    toks, logs = [], []
    out = m(input_ids=ids, video_spatio_temporal_features=feats, use_cache=True)
    for i in range(n_new):
        lg = out.logits[:, -1].float()
        logs.append(lg)
        nxt = lg.argmax(-1)
        toks.append(nxt)
        if i + 1 == n_new:
            break
        out = m(input_ids=nxt[:, None], past_key_values=out.past_key_values,
                video_spatio_temporal_features=feats, use_cache=True)
    return torch.stack(toks, 1), torch.stack(logs, 0)


def rownorm(x):
    return x.float().norm(dim=-1).numpy()


@torch.no_grad()
def main():
    torch.set_num_threads(os.cpu_count())
    ref_numpy_pool = _load_ref_numpy_pool()

    # ---------------- clip_tiny ----------------
    ccfg = O.ClipCfg(hidden=1024, inter=1024, heads=16, layers=3)
    csd = O.random_clip_state(ccfg, seed=11)
    clip = build_clip(ccfg, csd)
    px = O.preprocess_frames(O.make_frames(7, 3))
    hs = clip(px, output_hidden_states=True).hidden_states
    np.savez_compressed(os.path.join(HERE, "clip_tiny.npz"),
                        **{f"h{i}_slice": hs[i][:, :6, :96].numpy().astype(np.float32) for i in range(3)},
                        **{f"h{i}_rownorm": rownorm(hs[i]) for i in range(3)},
                        n_hidden_states=np.int64(len(hs)))
    print("clip_tiny: hidden_states", len(hs), [tuple(h.shape) for h in hs[:1]])

    # ---------------- pool ----------------
    g = torch.Generator().manual_seed(5)
    f8 = torch.randn(8, 256, 1024, generator=g).half()
    f100 = torch.randn(100, 256, 1024, generator=g).half()
    pool = {
        "t8_torch": get_spatio_temporal_features_torch(f8).numpy(),
        "t8_numpy": ref_numpy_pool(f8.numpy()),
        "t100_torch_rows": get_spatio_temporal_features_torch(f100).numpy()[::7],     # every 7th row
        "t100_numpy_rows": ref_numpy_pool(f100.numpy())[::7],
        # bf16 input (what the bf16 benchmark model feeds), as the reference function handles it
        "t100_bf16_rows": get_spatio_temporal_features_torch(f100.bfloat16()).numpy()[::7],
    }
    print("pool:", {k: (v.shape, v.dtype) for k, v in pool.items()})
    # the two reference variants agree in (nearly) every bit: stored as bit differences they compress to
    # almost nothing, where a second full copy would double the file
    for k in ("t8_numpy", "t100_numpy_rows"):
        torch_k = k.replace("numpy", "torch")
        pool[k + "_xor_torch"] = pool.pop(k).view(np.uint16) ^ pool[torch_k].view(np.uint16)
    np.savez_compressed(os.path.join(HERE, "pool.npz"), **pool)

    # ---------------- config 1 (BASELINE.json configs[0]) ----------------
    fcfg = O.ClipCfg()
    fsd = O.random_clip_state(fcfg, seed=0)
    fclip = build_clip(fcfg, fsd)
    frames = np.random.default_rng(0).integers(0, 256, (8, 224, 224, 3), dtype=np.uint8)
    hsf = fclip(O.preprocess_frames(frames), output_hidden_states=True).hidden_states
    feats = hsf[-2][:, 1:]
    pooled = get_spatio_temporal_features_torch(feats)
    np.savez_compressed(os.path.join(HERE, "config1.npz"), pooled=pooled.numpy(),
                        penult_rownorm=rownorm(hsf[-2]), penult_slice=hsf[-2][:, :4, :64].numpy())
    print("config1: pooled", tuple(pooled.shape), pooled.dtype, "rows 8..99 zero:", bool((pooled[8:100] == 0).all()))

    # ---------------- llm_tiny ----------------
    lcfg = O.LlmCfg(hidden=512, inter=1024, heads=4, layers=2)
    lsd = O.random_llm_state(lcfg, seed=21)
    llm = build_llm(lcfg, lsd, fcfg)
    ids = O.make_prompt_ids(lcfg, 356, seed=1, batch=2)
    gf = torch.Generator().manual_seed(9)
    vfe = (torch.randn(2, 356, 1024, generator=gf) * 0.5).half().float()   # fp16-representable features
    out = llm(input_ids=ids, video_spatio_temporal_features=vfe, output_hidden_states=True, use_cache=True)
    toks, logs = ref_greedy(llm, ids, vfe, 8)
    # single-clip run must agree with the batched one (per-sample independence)
    out1 = llm(input_ids=ids[:1], video_spatio_temporal_features=vfe[:1])
    assert torch.allclose(out1.logits[0, -1], out.logits[0, -1], atol=1e-4)
    err = ""
    bad = ids.clone()
    bad[0, 64 + 357] = 5  # overwrite <vid_end>
    try:
        llm(input_ids=bad, video_spatio_temporal_features=vfe)
    except ValueError as e:
        err = str(e)
    hsl = out.hidden_states
    np.savez_compressed(
        os.path.join(HERE, "llm_tiny.npz"),
        logits_last=out.logits[:, -1].numpy(),
        h0_rows=hsl[0][:, 60:72].numpy(),              # around <vid_start> (index 64): splice boundary
        h0_rownorm=rownorm(hsl[0]), h1_rownorm=rownorm(hsl[1]), h2_rownorm=rownorm(hsl[2]),
        h2_last=hsl[2][:, -1].numpy(), h1_slice=hsl[1][:, ::37, :64].numpy(),
        greedy_tokens=toks.numpy(), greedy_logits_top=torch.topk(logs, 4, dim=-1).values.numpy(),
        n_hidden_states=np.int64(len(hsl)), bad_span_error=np.array(err))
    print("llm_tiny: tokens", toks.tolist(), "error text:", err)

    # ---------------- bf16_tiny: the same models in the benchmark dtype ----------------
    bits = lambda t: t.contiguous().view(torch.int16).numpy().view(np.uint16)
    inv = [m_.inv_freq.clone() for m_ in llm.modules() if hasattr(m_, "inv_freq")]
    llm_b = llm.to(torch.bfloat16)
    for m_, f in zip([m_ for m_ in llm_b.modules() if hasattr(m_, "inv_freq")], inv):
        m_.inv_freq = f                                   # keep the rotary frequencies fp32
        if hasattr(m_, "original_inv_freq"):
            m_.original_inv_freq = f
    vfb = vfe.bfloat16()
    outb = llm_b(input_ids=ids, video_spatio_temporal_features=vfb, output_hidden_states=True, use_cache=True)
    toksb, logsb = ref_greedy(llm_b, ids, vfb, 8)
    clip_b = clip.to(torch.bfloat16)
    hsb = clip_b(px.bfloat16(), output_hidden_states=True).hidden_states
    np.savez_compressed(
        os.path.join(HERE, "bf16_tiny.npz"),
        llm_logits_last=bits(outb.logits[:, -1]),
        llm_h0_rows=bits(outb.hidden_states[0][:, 60:72]), llm_h1_slice=bits(outb.hidden_states[1][:, ::37, :64]),
        llm_h2_last=bits(outb.hidden_states[2][:, -1]),
        llm_greedy_tokens=toksb.numpy(), llm_greedy_top4=bits(torch.topk(logsb.bfloat16(), 4, dim=-1).values),
        **{f"clip_h{i}_slice": bits(hsb[i][:, :6, :96]) for i in range(3)},
        clip_h2_rows=bits(hsb[2][:, ::64, ::8]))
    print("bf16_tiny: tokens", toksb.tolist())


if __name__ == "__main__":
    main()
