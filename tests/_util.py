"""Helpers shared by the tests: build a vcl Engine from oracle configs, load the golden fixtures."""
import numpy as np
import torch

import vcl_native as vn
from oracle import vcl_oracle as O


def make_engine(clip: O.ClipCfg | None = None, llm: O.LlmCfg | None = None, clip_run_layers=None,
                max_frames=1, max_batch=1, max_seq=512):
    clip = clip or O.ClipCfg()
    llm = llm or O.LlmCfg(hidden=512, inter=1024, heads=4, layers=0)
    c = vn.vcl_config()
    c.clip_layers = (clip.layers - 1) if clip_run_layers is None else clip_run_layers
    c.clip_hidden, c.clip_inter, c.clip_heads = clip.hidden, clip.inter, clip.heads
    c.image_size, c.patch_size, c.clip_ln_eps = clip.image, clip.patch, clip.eps
    c.llm_layers, c.llm_hidden, c.llm_inter, c.llm_heads = llm.layers, llm.hidden, llm.inter, llm.heads
    c.vocab, c.rms_eps, c.rope_theta = llm.vocab, llm.rms_eps, llm.rope_theta
    c.proj_type = vn.PROJ_LINEAR if llm.proj_type == "linear" else vn.PROJ_MLP2X_GELU
    c.n_temporal = 100
    c.max_frames, c.max_batch, c.max_seq = max_frames, max_batch, max_seq
    return vn.Engine(c)


def load_pool_golden(path):
    """golden/pool.npz as a dict, with the reference's numpy-pooling results rebuilt from the stored XOR of
    their fp16 bit patterns with the torch-pooling results (golden/make_golden.py)."""
    g = dict(np.load(path))
    for k in ("t8_numpy", "t100_numpy_rows"):
        torch_bits = g[k.replace("numpy", "torch")].view(np.uint16)
        g[k] = (torch_bits ^ g.pop(k + "_xor_torch")).view(np.float16)
    return g


def to_dev(sd, dtype=torch.bfloat16, device="cuda"):
    return {k: v.to(device=device, dtype=dtype) for k, v in sd.items()}


def relerr(a, b):
    a = a.float()
    b = b.float().to(a.device)
    return ((a - b).norm() / b.norm().clamp_min(1e-30)).item()


def vid_start_of(ids, llm: O.LlmCfg):
    """index of <vid_start> per row (VCL_NO_VIDEO if absent), int32 on the ids' device"""
    out = []
    for row in ids.tolist():
        out.append(row.index(llm.vid_start_token) if llm.vid_start_token in row else vn.NO_VIDEO)
    return torch.tensor(out, dtype=torch.int32, device=ids.device)


def bar(ours, ref_bf16, gold, what):
    e_ours, e_ref = relerr(ours, gold), relerr(ref_bf16, gold)
    print(f"[parity] {what}: ours-vs-gold {e_ours:.3e}  oracle(bf16)-vs-gold {e_ref:.3e}  ours-vs-oracle(bf16) {relerr(ours, ref_bf16):.3e}")
    assert e_ours <= 1.3 * e_ref + 1e-3, (what, e_ours, e_ref)



def teacher_forced_check(eng, sd_b, cfg, ids, vf, n_new, what, verbose=False, oracle=None):
    """Greedy ids of the bf16 oracle; our engine is teacher-forced with them. Rule (SURVEY.md 7):
    identical arg-max wherever the oracle's top-1/top-2 margin is >= 3 bf16 ulps; at a near-tie our token
    must be one of the tied candidates (its oracle logit within 3 ulps of the top). `oracle` = (tokens, logits) of a greedy_generate already run; verbose prints the margin
    (in bf16 ulps of the top logit) of every step."""
    B, S = ids.shape
    o_toks, o_logits = oracle if oracle is not None else O.greedy_generate(sd_b, cfg, ids, vf.bfloat16(), n_new)
    vs = vid_start_of(ids, cfg)
    _, lg, tok = eng.prefill(ids, vf, vs, want_logits=True)
    ours_logits = [lg.clone()]
    ours_toks = [tok.clone()]
    for i in range(1, n_new):
        lg, tok = eng.decode_step(o_toks[:, i - 1].to(torch.int32).contiguous(), S + i - 1, want_logits=True)
        ours_logits.append(lg.clone())
        ours_toks.append(tok.clone())
    ours_toks = torch.stack(ours_toks, 1).long()
    n_strict = n_ok = 0
    for i in range(n_new):
        top = torch.topk(o_logits[i], 2, dim=-1)
        ulp = top.values[:, 0].abs().clamp_min(2 ** -6) * 2 ** -7
        margin_ulps = (top.values[:, 0] - top.values[:, 1]) / ulp
        if verbose:
            print(f"[parity] {what}: step {i:2d} oracle margin (ulps) {[round(float(m), 1) for m in margin_ulps]} "
                  f"ours {ours_toks[:, i].tolist()} oracle {o_toks[:, i].tolist()}")
        for b in range(B):
            if margin_ulps[b] >= 3:
                n_strict += 1
                assert ours_toks[b, i] == o_toks[b, i], (what, i, b, margin_ulps[b].item())
                n_ok += 1
            else:
                # a near-tie by the oracle's own logits: our token must be one of the tied candidates, i.e. its
                # oracle logit lies within 3 ulps of the oracle's top logit (with more than two candidates inside
                # one ulp, "top-2 membership" alone would reject a legitimate third)
                gap_ulps = ((top.values[b, 0] - o_logits[i][b, ours_toks[b, i]]) / ulp[b]).item()
                assert gap_ulps < 3, (what, i, b, "our token's oracle logit is %.2f ulps below the top" % gap_ulps)
        e = relerr(ours_logits[i], o_logits[i])
        assert e < 3e-2, (what, i, e)
    print(f"[parity] {what}: teacher-forced {n_ok}/{n_strict} strict steps identical; "
          f"free-running agreement {(ours_toks == o_toks).float().mean().item():.2f}")
    return o_toks


