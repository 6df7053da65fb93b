"""CPU tests of the sampling contract (include/vcl.h, vcl_sampling) and of the host side of the device
decode path: the Philox4x64-10 restatement against numpy, the fp64 sampler against an HF-style one, and the
replay of stopping criteria over device-sized chunks against the per-token loop."""
import os
import sys

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import _sampling_oracle as SO  # noqa: E402

M64 = 2 ** 64 - 1


def _np_philox(seed, counter):
    return tuple(int(w) for w in np.random.Philox(key=np.array([seed, 0], dtype=np.uint64),
                                                  counter=np.array(counter, dtype=np.uint64)).random_raw(4))


@pytest.mark.parametrize("seed", [0, 1, 12345, 2 ** 63 - 2, 0xDEADBEEFCAFEF00D])
def test_philox4x64_matches_numpy(seed):
    # numpy increments the 256-bit counter before generating: its counter c gives our block at c + 1
    for pos, b in [(1, 0), (448, 0), (449, 15), (2 ** 31 - 1, 3), (2 ** 64 - 1, 7)]:
        assert _np_philox(seed, [pos - 1, b, 0, 0]) == SO.philox4x64((seed, 0), (pos, b, 0, 0)), (seed, pos, b)
    # counter carry: word 0 wraps into word 1
    assert _np_philox(seed, [M64, 4, 0, 0]) == SO.philox4x64((seed, 0), (0, 5, 0, 0))
    assert _np_philox(seed, [M64, M64, 2, 0]) == SO.philox4x64((seed, 0), (0, 0, 3, 0))
    u = SO.uniform(seed, 448, 2)
    assert 0.0 <= u < 1.0


def _hf_probs(row: torch.Tensor, T: float, k):
    """HF's warpers in fp32: logits / T, keep >= the k-th largest, softmax."""
    lg = row[None].float() / T
    if k and k < lg.shape[-1]:
        kth = torch.topk(lg, k, dim=-1).values[:, -1:]
        lg = lg.masked_fill(lg < kth, float("-inf"))
    return torch.softmax(lg, dim=-1)[0].double().numpy()


def _logit_rows():
    g = torch.Generator().manual_seed(0)
    rows = [torch.randn(4096, generator=g) * 3,
            (torch.randn(4096, generator=g) * 2).bfloat16().float(),      # bf16-rounded: many ties
            torch.round(torch.randn(512, generator=g) * 2) / 2]            # coarse grid: ties at tau for sure
    r = torch.randn(1000, generator=g)
    r[::3] = float("-inf")
    r[5] = float("nan")
    rows.append(r)
    return rows


@pytest.mark.parametrize("T", [0.2, 1.0, 2.0])
@pytest.mark.parametrize("k", [1, 50, 1024, 0])
def test_sample_probs_match_hf_warpers(T, k):
    for row in _logit_rows():
        K, p = SO.sample_probs(row.numpy(), T, k)
        hf = _hf_probs(torch.nan_to_num(row, nan=float("-inf")), T, k)
        kept_hf = np.nonzero(hf > 0)[0]
        x = torch.nan_to_num(row, nan=float("-inf")).numpy()
        if k and k < len(x):
            tau = np.sort(x)[::-1][k - 1]
            assert set(K) == set(np.nonzero(x >= tau)[0])                  # every tie at tau kept
            assert len(K) >= min(k, np.isfinite(x).sum())
        # HF's kept set, minus ids whose fp32 probability underflows to 0
        assert set(kept_hf) <= set(K)
        full = np.zeros(len(x))
        full[K] = p
        assert np.abs(full - hf).max() < 1e-6
        assert abs(p.sum() - 1.0) < 1e-12


def test_sample_reference_is_inverse_cdf_over_ascending_ids():
    rows = _logit_rows()
    V = 512
    L = np.stack([r.numpy()[:V] for r in rows])
    seed, pos = 77, 450
    for T in (0.2, 1.0):
        for k in (1, 50, 0):
            toks, margin = SO.sample_reference(L, T, k, seed, pos, with_margin=True)
            for b in range(L.shape[0]):
                K, p = SO.sample_probs(L[b], T, k)
                u = SO.uniform(seed, pos, b)
                j = min(int(np.searchsorted(np.cumsum(p), u, side="right")), len(K) - 1)
                assert toks[b] == K[j] or margin[b] < 1e-12
                assert toks[b] in set(K)
    # temperature <= 0: the arg-max, lowest index winning
    tie = np.array([[0.5, 2.0, 2.0, -1.0]], dtype=np.float32)
    assert SO.sample_reference(tie, 0.0, 50, 1, 9)[0] == 1
    assert SO.sample_reference(np.full((1, 8), -np.inf, dtype=np.float32), 1.0, 0, 1, 9)[0] == 0


def test_sample_reference_empirical_distribution():
    row = (torch.randn(256, generator=torch.Generator().manual_seed(3)) * 1.5).numpy()[None]
    K, p = SO.sample_probs(row[0], 1.0, 8)
    n = 4000
    toks = np.array([SO.sample_reference(row, 1.0, 8, seed=s, pos=100)[0] for s in range(n)])
    counts = np.array([(toks == i).sum() for i in K])
    assert counts.sum() == n                                               # nothing outside K
    from scipy.stats import chisquare
    assert chisquare(counts, p * n).pvalue > 1e-4


# ---- chunked replay of stopping criteria vs the per-token loop --------------------------------------------
class _Engine:
    """Scripted tokens: row b's token at sequence position P0 + i is script[b, i], whatever is fed."""

    def __init__(self, script, P0, V=64):
        self.script, self.P0, self.V = script, P0, V
        self.steps = self.loops = 0

    def logits_for(self, pos):
        lg = torch.full((self.script.shape[0], self.V), float("-inf"))
        lg[torch.arange(self.script.shape[0]), self.script[:, pos - self.P0]] = 0.0
        return lg

    def decode_step(self, tok, pos, want_logits=True):
        self.steps += 1
        return self.logits_for(pos + 1), None

    def decode_loop(self, first, S, n_new):
        self.loops += 1
        out = self.script[:, S - self.P0: S - self.P0 + n_new].to(torch.int32).clone()
        out[:, 0] = first
        return out

    def decode_loop_sampled(self, first, S, n_new, T, k, seed):
        return self.decode_loop(first, S, n_new)


class _Recorder:
    def __init__(self, log, name, stop_len=None):
        self.log, self.name, self.stop_len = log, name, stop_len

    def __call__(self, out, scores):
        self.log.append((self.name, out.shape[1], out[:, -1].tolist()))
        return self.stop_len is not None and out.shape[1] >= self.stop_len


def _model():
    from video_chatgpt.model import VideoChatGPTConfig, VideoChatGPTLlamaForCausalLM
    cfg = VideoChatGPTConfig(hidden_size=512, intermediate_size=1024, num_hidden_layers=2, num_attention_heads=4,
                             vocab_size=64, use_mm_proj=True, mm_hidden_size=1024)
    return VideoChatGPTLlamaForCausalLM(cfg, clip_config={}, max_seq=4096)


def _script(B, N, eos_at):
    g = torch.Generator().manual_seed(5)
    s = torch.randint(3, 60, (B, N), generator=g)
    for b, i in eos_at.items():
        s[b, i] = 2
    return s


@pytest.mark.parametrize("case", ["eos", "criteria_mid_chunk", "max_new_tokens", "eos_no_criteria"])
@pytest.mark.parametrize("do_sample", [False, True])
def test_chunked_replay_makes_the_stepwise_calls(case, do_sample):
    B, P0, n = 3, 20, 70
    eos_at = {"eos": {0: 5, 1: 40, 2: 33}, "eos_no_criteria": {0: 1, 1: 64, 2: 31}}.get(case, {})
    script = _script(B, n + 1, eos_at)
    prompt = torch.randint(3, 60, (B, P0), generator=torch.Generator().manual_seed(1))
    stop_len = P0 + 45 if case == "criteria_mid_chunk" else None
    eos = 2 if case in ("eos", "eos_no_criteria") else None
    results = []
    for path in ("stepwise", "chunked"):
        log = []
        crits = [] if case == "eos_no_criteria" else [_Recorder(log, "a", stop_len), _Recorder(log, "b")]
        m = _model()
        eng = _Engine(script, P0)
        m._pos = P0
        if path == "stepwise":
            out = m._stepwise(eng, prompt.clone(), eng.logits_for(P0), n, do_sample, 0.7, crits, eos, 0, 50)
        else:
            sp = (0.7, 50, 123) if do_sample else None
            first = script[:, 0].to(torch.int32)
            out = m._device_decode(eng, prompt.clone(), lambda c: eng.decode_loop(first, P0, c), n, sp, crits, eos, 0)
            assert eng.steps == 0 and eng.loops >= 1
        results.append((out, m._pos, log))
    (o1, p1, l1), (o2, p2, l2) = results
    assert torch.equal(o1, o2), (o1[:, P0:], o2[:, P0:])
    assert p1 == p2 == o1.shape[1] - 1
    assert l1 == l2
    if case == "criteria_mid_chunk":
        assert o1.shape[1] == stop_len and l1[-1][0] == "a"                 # "b" is not called after "a" says stop
    if case == "max_new_tokens":
        assert o1.shape[1] == P0 + n and len(l1) == 2 * n
    if case == "eos":
        assert o1.shape[1] == P0 + 41 and (o1[0, P0 + 6:] == 0).all()
