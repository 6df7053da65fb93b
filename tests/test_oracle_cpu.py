"""CPU tests: the oracle restatement (oracle/vcl_oracle.py) against the golden fixtures that
tests/golden/make_golden.py produced by running the reference itself. These pin the oracle; the
GPU parity tests then compare libvcl.so with the oracle (and with the same fixtures)."""
import os

import numpy as np
import pytest
import torch

from oracle import vcl_oracle as O

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _load(name):
    return np.load(os.path.join(G, name))


def _close(a, b, rtol, atol):
    a = torch.as_tensor(np.asarray(a)).float()
    b = torch.as_tensor(np.asarray(b)).float()
    assert a.shape == b.shape, (a.shape, b.shape)
    assert torch.allclose(a, b, rtol=rtol, atol=atol), (a - b).abs().max().item()


@torch.no_grad()
def test_clip_tiny_matches_hf_reference():
    g = _load("clip_tiny.npz")
    cfg = O.ClipCfg(hidden=1024, inter=1024, heads=16, layers=3)
    sd = O.random_clip_state(cfg, seed=11)
    px = O.preprocess_frames(O.make_frames(7, 3))
    hs = O.clip_hidden_states(sd, cfg, px, n_layers=2)
    assert int(g["n_hidden_states"]) == 4          # HF returns layers+1 states; the path uses [-2]
    for i in range(3):
        _close(hs[i][:, :6, :96], g[f"h{i}_slice"], 1e-4, 1e-4)
        _close(hs[i].norm(dim=-1), g[f"h{i}_rownorm"], 1e-4, 1e-3)


def test_pool_torch_and_numpy_bit_exact():
    from _util import load_pool_golden
    g = load_pool_golden(os.path.join(G, "pool.npz"))
    gen = torch.Generator().manual_seed(5)
    f8 = torch.randn(8, 256, 1024, generator=gen).half()
    f100 = torch.randn(100, 256, 1024, generator=gen).half()
    o8 = O.st_pool_torch(f8)
    assert o8.dtype == torch.float16 and o8.shape == (356, 1024)
    assert (o8[8:100] == 0).all()
    assert np.array_equal(o8.numpy(), g["t8_torch"])
    assert np.array_equal(O.st_pool_numpy(f8.numpy()), g["t8_numpy"])
    assert np.array_equal(O.st_pool_torch(f100).numpy()[::7], g["t100_torch_rows"])
    assert np.array_equal(O.st_pool_numpy(f100.numpy())[::7], g["t100_numpy_rows"])
    assert np.array_equal(O.st_pool_torch(f100.bfloat16()).numpy()[::7], g["t100_bf16_rows"])
    # the two reference variants agree to one fp16 ulp (different fp32 summation trees)
    d = np.abs(g["t8_torch"].astype(np.float32) - g["t8_numpy"].astype(np.float32))
    assert d.max() <= 2 ** -10 * np.abs(g["t8_torch"].astype(np.float32)).max()


def test_pool_edge_cases():
    f1 = torch.arange(2 * 3 * 8, dtype=torch.float32).reshape(1, 6, 8).half()   # T = 1
    o = O.st_pool_torch(f1)
    assert o.shape == (106, 8) and (o[1:100] == 0).all()
    assert torch.equal(o[100:], f1[0])                                             # mean over one frame
    f = torch.randn(100, 4, 8).half()                                              # T = 100: no padding
    assert O.st_pool_torch(f).shape == (104, 8)


@torch.no_grad()
def test_config1_full_vit_pooled():
    """BASELINE.json configs[0]: 8 frames, full ViT-L/14, pooled [356,1024] (fp32 run of the reference)."""
    g = _load("config1.npz")
    cfg = O.ClipCfg()
    sd = O.random_clip_state(cfg, seed=0, n_layers=23)    # layer 24 is dead work for the path
    frames = np.random.default_rng(0).integers(0, 256, (8, 224, 224, 3), dtype=np.uint8)
    hs = O.clip_hidden_states(sd, cfg, O.preprocess_frames(frames))
    assert len(hs) == 24
    _close(hs[-1][:, :4, :64], g["penult_slice"], 1e-3, 1e-3)
    pooled = O.st_pool_torch(hs[-1][:, 1:])
    assert (pooled[8:100] == 0).all()
    ref = torch.as_tensor(g["pooled"]).float()
    err = ((pooled.float() - ref).norm() / ref.norm()).item()
    assert err < 1e-3, err


@torch.no_grad()
def test_llm_tiny_matches_reference_forward():
    g = _load("llm_tiny.npz")
    cfg = O.LlmCfg(hidden=512, inter=1024, heads=4, layers=2)
    sd = O.random_llm_state(cfg, seed=21)
    ids = O.make_prompt_ids(cfg, 356, seed=1, batch=2)
    assert ids.shape == (2, 448)
    gf = torch.Generator().manual_seed(9)
    vf = (torch.randn(2, 356, 1024, generator=gf) * 0.5).half().float()
    logits, hs, _ = O.llm_forward(sd, cfg, ids, vf)
    assert int(g["n_hidden_states"]) == 3
    _close(hs[0][:, 60:72], g["h0_rows"], 1e-5, 1e-5)             # splice boundary at <vid_start> = 64
    for i in range(3):
        _close(hs[i].norm(dim=-1), g[f"h{i}_rownorm"], 1e-4, 1e-3)
    _close(hs[2][:, -1], g["h2_last"], 1e-3, 1e-3)                # [-1] is post final norm
    _close(hs[1][:, ::37, :64], g["h1_slice"], 1e-3, 1e-3)
    _close(logits[:, -1], g["logits_last"], 1e-3, 2e-3)
    toks, logs = O.greedy_generate(sd, cfg, ids, vf, 8)
    assert np.array_equal(toks.numpy(), g["greedy_tokens"])       # fp32 on the same CPU: bit-exact ids
    _close(torch.topk(logs, 4, dim=-1).values, g["greedy_logits_top"], 1e-3, 2e-3)


def test_splice_errors_match_reference():
    g = _load("llm_tiny.npz")
    cfg = O.LlmCfg(hidden=512, inter=1024, heads=4, layers=2)
    sd = {"model.embed_tokens.weight": torch.zeros(cfg.vocab, 8),
          "model.mm_projector.weight": torch.zeros(8, 1024), "model.mm_projector.bias": torch.zeros(8)}
    ids = O.make_prompt_ids(cfg, 356, seed=1, batch=1)
    bad = ids.clone()
    bad[0, 64 + 357] = 5
    with pytest.raises(ValueError) as e:
        O.splice_embeddings(sd, cfg, bad, torch.zeros(1, 356, 1024))
    assert str(e.value) == str(g["bad_span_error"])
    shifted = ids.clone()                                          # <vid_end> not right after the span
    shifted[0, 64 + 357] = cfg.vid_patch_token
    shifted[0, 64 + 358] = cfg.vid_end_token
    with pytest.raises(ValueError):
        O.splice_embeddings(sd, cfg, shifted, torch.zeros(1, 356, 1024))


@torch.no_grad()
def test_bf16_rounding_points_bit_exact_vs_reference():
    """bf16_tiny.npz holds raw bf16 bit patterns produced by the REFERENCE forward / HF CLIP in bf16 on
    this CPU (rotary inv_freq kept fp32). The oracle run in bf16 must reproduce them bit for bit: this
    pins every bf16 rounding point of the restatement, which is what the GPU kernels are built to match."""
    g = _load("bf16_tiny.npz")
    bits = lambda t: t.contiguous().view(torch.int16).numpy().view(np.uint16)
    bf = lambda sd: {k: v.bfloat16() for k, v in sd.items()}
    cfg = O.LlmCfg(hidden=512, inter=1024, heads=4, layers=2)
    sd = bf(O.random_llm_state(cfg, seed=21))
    ids = O.make_prompt_ids(cfg, 356, seed=1, batch=2)
    vf = (torch.randn(2, 356, 1024, generator=torch.Generator().manual_seed(9)) * 0.5).half().float().bfloat16()
    logits, hs, _ = O.llm_forward(sd, cfg, ids, vf)
    assert np.array_equal(bits(hs[0][:, 60:72]), g["llm_h0_rows"])
    assert np.array_equal(bits(hs[1][:, ::37, :64]), g["llm_h1_slice"])
    assert np.array_equal(bits(hs[2][:, -1]), g["llm_h2_last"])
    assert np.array_equal(bits(logits[:, -1]), g["llm_logits_last"])
    toks, logs = O.greedy_generate(sd, cfg, ids, vf, 8)
    assert np.array_equal(toks.numpy(), g["llm_greedy_tokens"])
    assert np.array_equal(bits(torch.topk(logs.bfloat16(), 4, dim=-1).values), g["llm_greedy_top4"])
    ccfg = O.ClipCfg(hidden=1024, inter=1024, heads=16, layers=3)
    csd = bf(O.random_clip_state(ccfg, seed=11))
    hsc = O.clip_hidden_states(csd, ccfg, O.preprocess_frames(O.make_frames(7, 3)).bfloat16(), n_layers=2)
    for i in range(3):
        assert np.array_equal(bits(hsc[i][:, :6, :96]), g[f"clip_h{i}_slice"]), i
    assert np.array_equal(bits(hsc[2][:, ::64, ::8]), g["clip_h2_rows"])
