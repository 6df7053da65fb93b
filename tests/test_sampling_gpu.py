"""The device sampler (sample.cu, vcl_sampling in include/vcl.h) and the sampled decode path on the GPU:
token-for-token against the host restatement, its distribution, the sampled graph loop against single steps,
chunking, the greedy limit, reproducibility under torch.manual_seed, and the drop-in callers."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import vcl_oracle as O  # noqa: E402

import _sampling_oracle as SO  # noqa: E402

V = 32003


def _model(max_batch=1, max_seq=640, seed=21):
    from video_chatgpt.model import VideoChatGPTConfig, VideoChatGPTLlamaForCausalLM
    lcfg = O.LlmCfg(hidden=512, inter=1024, heads=4, layers=2)
    cfg = VideoChatGPTConfig(hidden_size=lcfg.hidden, intermediate_size=lcfg.inter, num_hidden_layers=lcfg.layers,
                             num_attention_heads=lcfg.heads, vocab_size=lcfg.vocab, use_mm_proj=True, mm_hidden_size=1024)
    clip = dict(hidden_size=1024, intermediate_size=1024, num_hidden_layers=3, num_attention_heads=16)
    m = VideoChatGPTLlamaForCausalLM(cfg, clip_config=clip, max_batch=max_batch, max_seq=max_seq)
    vc = m.get_model().vision_config
    vc.vid_patch_token, vc.vid_start_token, vc.vid_end_token, vc.use_vid_start_end = 32000, 32001, 32002, True
    m.load_state_dict(O.random_llm_state(lcfg, seed=seed))
    return m, lcfg


def _inputs(lcfg, B, seed=4):
    feats = (torch.randn(B, 356, 1024, generator=torch.Generator().manual_seed(seed)) * 0.5).half().cuda()
    ids = O.make_prompt_ids(lcfg, 356, seed=seed, batch=B).cuda()
    return ids, feats


def _logits(kind, B=16, seed=0):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(B, V, generator=g) * 2.5
    if kind == "bf16":                                   # bf16-rounded: ties everywhere, also at tau
        x = x.bfloat16().float()
    x[3, ::4] = float("-inf")                            # a row with -inf entries
    x[3, 17] = float("nan")
    return x


@pytest.mark.parametrize("kind", ["random", "bf16"])
def test_sampler_matches_reference(kind):
    x = _logits(kind)
    wide = torch.zeros(16, V + 61, device="cuda")        # a row pitch larger than V
    wide[:, :V] = x.cuda()
    dev = wide[:, :V]
    checked = mismatches = near_edge = 0
    for B in (1, 5, 16):
        for T in (0.2, 1.0, 2.0):
            for k in (1, 50, 1024, 0):
                seed, pos = 1000 * B + int(10 * T) + k, 448 + B
                got = vn_op_sample(dev[:B], T, k, seed, pos).cpu().numpy()
                want, margin = SO.sample_reference(x[:B].numpy(), T, k, seed, pos, with_margin=True)
                bad = got != want
                near_edge += int((bad & (margin < 1e-9)).sum())
                mismatches += int((bad & (margin >= 1e-9)).sum())
                checked += B
    print(f"[sampling] {kind} logits: {checked} rows, {near_edge} mismatches within 1e-9 Z of a bin edge, "
          f"{mismatches} elsewhere")
    assert mismatches == 0


def vn_op_sample(logits, T, k, seed, pos):
    import vcl_native as vn
    return vn.op_sample(logits, T, k, seed, pos)


def test_sampler_greedy_limit_and_distribution():
    x = _logits("bf16")
    dev = x.cuda()
    am = torch.nan_to_num(dev, nan=float("-inf")).argmax(-1).to(torch.int32)   # the first maximal index
    for T in (0.0, -1.0):
        assert torch.equal(vn_op_sample(dev, T, 50, 3, 500), am)
    # 65 536 draws from one row at T = 1, k = 50: chi-square against the exact probabilities
    row = torch.randn(V, generator=torch.Generator().manual_seed(9)).cuda()
    rows = row[None].expand(16, V).contiguous()
    K, p = SO.sample_probs(row.cpu().numpy(), 1.0, 50)
    toks = torch.cat([vn_op_sample(rows, 1.0, 50, 12345, pos) for pos in range(1, 4097)]).cpu().numpy()
    assert toks.size == 65536
    assert np.isin(toks, K).all()
    counts = np.array([(toks == i).sum() for i in K])
    from scipy.stats import chisquare
    pv = chisquare(counts, p * toks.size).pvalue
    print(f"[sampling] 65536 draws, |K| = {len(K)}, chi-square p = {pv:.3g}")
    assert pv > 1e-4


@pytest.mark.parametrize("B", [1, 6])
@pytest.mark.parametrize("graph", [True, False])
@torch.no_grad()
def test_sampled_loop_equals_single_steps(B, graph):
    """Each token of the sampled decode loop equals vcl_op_sample on vcl_llm_decode_step's logits fed the
    same tokens: B = 1 takes the ring kernels, B = 6 the wide ring kernels; on a side stream the loop is a
    CUDA graph, on the default stream eager launches."""
    m, lcfg = _model(max_batch=6)
    eng = m._ensure_engine(need_llm=True)
    ids, feats = _inputs(lcfg, B)
    vs = m._spans_dev(ids, feats, eng.NV)
    S, n, T, k, seed = ids.shape[1], 12, 1.0, 50, 2024
    st = torch.cuda.Stream() if graph else torch.cuda.default_stream()
    with torch.cuda.stream(st):
        _, lg, _ = eng.prefill(ids, feats, vs, want_logits=True, want_token=False)
        first = vn_op_sample(lg, T, k, seed, S)
        loop = eng.decode_loop_sampled(first, S, n, T, k, seed)
        direct = eng.generate_sampled(ids, feats, vs, n, T, k, seed)
        steps = [first]
        for i in range(1, n):
            lg_i, _ = eng.decode_step(loop[:, i - 1].contiguous(), S + i - 1, want_logits=True)
            steps.append(vn_op_sample(lg_i, T, k, seed, S + i))
    st.synchronize()
    ref = torch.stack(steps, 1)
    assert torch.equal(loop, ref), (loop, ref)
    assert torch.equal(direct, loop)
    assert len(set(loop.flatten().tolist())) > n // 2          # T = 1 over random logits: not stuck on one id


@torch.no_grad()
def test_chunks_equal_one_loop_and_generate():
    m, lcfg = _model()
    eng = m._ensure_engine(need_llm=True)
    ids, feats = _inputs(lcfg, 1)
    vs = m._spans_dev(ids, feats, eng.NV)
    S, T, k = ids.shape[1], 1.0, 50
    torch.manual_seed(7)
    seed = int(torch.randint(0, 2 ** 63 - 1, (1,)))
    st = torch.cuda.Stream()
    with torch.cuda.stream(st):
        one = eng.generate_sampled(ids, feats, vs, 64, T, k, seed)
        a = eng.generate_sampled(ids, feats, vs, 32, T, k, seed)
        b = eng.decode_loop_sampled(a[:, -1].contiguous(), S + 31, 33, T, k, seed)
        torch.manual_seed(7)
        out = m.generate(ids, video_spatio_temporal_features=feats, do_sample=True, temperature=T, top_k=k,
                         max_new_tokens=64, eos_token_id=None)
    st.synchronize()
    assert torch.equal(torch.cat([a, b[:, 1:]], 1), one)
    assert torch.equal(out[:, S:].to(torch.int32), one) and torch.equal(out[:, :S], ids)
    assert m._pos == S + 63


@pytest.mark.parametrize("B", [1, 6])
@torch.no_grad()
def test_temperature_zero_is_the_greedy_path(B, monkeypatch):
    m, lcfg = _model(max_batch=6)
    eng = m._ensure_engine(need_llm=True)
    ids, feats = _inputs(lcfg, B, seed=5)
    vs = m._spans_dev(ids, feats, eng.NV)
    st = torch.cuda.Stream()
    with torch.cuda.stream(st):
        greedy = eng.generate(ids, feats, vs, 40)
        sampled = eng.generate_sampled(ids, feats, vs, 40, 0.0, 50, 99)
        cont = eng.decode_loop_sampled(greedy[:, -1].contiguous(), ids.shape[1] + 39, 9, 0.0, 0, 5)
        cont_greedy = eng.decode_loop(greedy[:, -1].contiguous(), ids.shape[1] + 39, 9)
    st.synchronize()
    assert torch.equal(sampled, greedy) and torch.equal(cont, cont_greedy)

    # greedy with stopping criteria: the device path gives today's (per-token) tokens, and stops at the same place
    class StopAt:
        def __init__(self, n): self.n, self.calls = n, 0
        def __call__(self, out, scores):
            self.calls += 1
            return self.calls >= self.n
    outs = []
    for host in ("0", "1"):
        monkeypatch.setenv("VCL_HOST_SAMPLING", host)
        crit = StopAt(23)
        outs.append((m.generate(ids, video_spatio_temporal_features=feats, do_sample=False, max_new_tokens=40,
                                stopping_criteria=[crit], eos_token_id=None), crit.calls, m._pos))
    assert torch.equal(outs[0][0], outs[1][0]) and outs[0][1:] == outs[1][1:]
    assert outs[0][0].shape[1] == ids.shape[1] + 23
    assert torch.equal(outs[0][0][:, ids.shape[1]:].to(torch.int32), greedy[:, :23])


@torch.no_grad()
def test_manual_seed_reproduces_generate():
    m, lcfg = _model()
    ids, feats = _inputs(lcfg, 1, seed=6)
    runs = []
    for s in (11, 11, 12):
        torch.manual_seed(s)
        runs.append(m.generate(ids, video_spatio_temporal_features=feats[0:1], do_sample=True, temperature=1.0,
                               max_new_tokens=40, eos_token_id=None))
    assert torch.equal(runs[0], runs[1])
    assert not torch.equal(runs[0], runs[2])


@torch.no_grad()
def test_generate_continue_samples_on_the_device(monkeypatch):
    m, lcfg = _model()
    ids, feats = _inputs(lcfg, 1, seed=8)
    eng = m._ensure_engine(need_llm=True)
    monkeypatch.setattr(eng, "decode_step", lambda *a, **k: pytest.fail("per-token step on the device path"))
    torch.manual_seed(3)
    turn1 = m.generate(ids, video_spatio_temporal_features=feats, do_sample=True, temperature=0.2, max_new_tokens=8,
                       eos_token_id=None)
    q2 = torch.randint(3, 32000, (1, 11), generator=torch.Generator().manual_seed(8)).cuda()
    turn2 = m.generate_continue(q2, do_sample=True, temperature=0.2, max_new_tokens=8, eos_token_id=None)
    S = ids.shape[1]
    assert turn2.shape == (1, S + 8 + 11 + 8)
    assert torch.equal(turn2[:, :S + 8], turn1) and torch.equal(turn2[:, S + 8:S + 19], q2)
    assert m._pos == turn2.shape[1] - 1


@torch.no_grad()
def test_video_chatgpt_infer_defaults_run_on_the_device(tmp_path, monkeypatch):
    """The reference's hard-coded settings (do_sample=True, temperature=0.2, the stop-string criterion, EOS): no
    per-token C-ABI step, and the output ends where the per-token loop would have ended
    given the same tokens."""
    from PIL import Image
    from _checkpoint import make_tiny_checkpoint
    from video_chatgpt.eval.model_utils import initialize_model
    from video_chatgpt.inference import video_chatgpt_infer
    from video_chatgpt.model.utils import KeywordsStoppingCriteria
    ck = make_tiny_checkpoint(tmp_path)
    model, tower, tok, ip, vlen = initialize_model(ck["model_dir"], max_batch=1, max_seq=1024)
    frames = [Image.fromarray(f) for f in O.make_frames(21, 6)]
    eng = model._ensure_engine(need_llm=True)
    monkeypatch.setattr(eng, "decode_step", lambda *a, **k: pytest.fail("per-token step on the device path"))
    seen = {}
    orig = model.generate

    def spy(input_ids, **kw):
        out = orig(input_ids, **kw)
        seen.update(ids=input_ids, kw=kw, out=out)
        return out
    monkeypatch.setattr(model, "generate", spy)
    torch.manual_seed(0)
    # the reference's settings except the length: 48 new tokens keep every position below 512
    text = video_chatgpt_infer(frames, "w10 w11 w12 w13", "pg-video-llava", model, tower, tok, ip, vlen,
                               max_new_tokens=48)
    assert isinstance(text, str)
    kw, out, ids = seen["kw"], seen["out"], seen["ids"]
    assert kw["do_sample"] is True and kw["temperature"] == 0.2 and kw["max_new_tokens"] == 48
    S = ids.shape[1]
    n = min(48, 1024 - S)
    new = out[0, S:].tolist()
    print(f"[sampling] video_chatgpt_infer: {len(new)} new tokens of at most {n}; text {text[:60]!r}")
    # the per-token loop over the same tokens: EOS, then the criterion on every prefix, then the length limit
    crit = KeywordsStoppingCriteria([kw["stopping_criteria"][0].keywords[0]], tok, ids)
    eos = kw["eos_token_id"]
    stop = None
    for j in range(len(new)):
        if new[j] == eos or crit(out[:, :S + j + 1], None):
            stop = j + 1
            break
    assert len(new) == (stop if stop is not None else n)
