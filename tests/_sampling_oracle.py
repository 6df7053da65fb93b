"""Host restatement of the device sampler's contract (include/vcl.h, above vcl_sampling), for the tests.

    philox4x64(key, counter)                       Philox4x64-10, hand-written (Salmon et al., SC'11)
    sample_probs(row, temperature, top_k)          kept set K and the fp64 probabilities over it
    sample_reference(logits, temperature, top_k, seed, pos)   the token of every row, fp64, sequential walk

HF's order (TemperatureLogitsWarper -> TopKLogitsWarper -> softmax -> multinomial, $TF/generation/
logits_process.py) with two stated differences: the weights are fp64 rather than fp32, and the uniform
draw comes from Philox4x64-10 at counter (pos, b, 0, 0) under key (seed, 0), so that a token depends only on
the seed, its sequence position and its row.
"""
from __future__ import annotations

import numpy as np

M64 = (1 << 64) - 1
PHILOX_M = (0xD2E7470EE14C6C93, 0xCA5A826395121157)
PHILOX_W = (0x9E3779B97F4A7C15, 0xBB67AE8584CAA73B)


def philox4x64(key, counter, rounds: int = 10):
    """The four 64-bit words of Philox4x64-`rounds` at `counter` (4 ints) under `key` (2 ints)."""
    k0, k1 = key[0] & M64, key[1] & M64
    x0, x1, x2, x3 = (c & M64 for c in counter)
    for r in range(rounds):
        if r > 0:
            k0, k1 = (k0 + PHILOX_W[0]) & M64, (k1 + PHILOX_W[1]) & M64
        p0, p1 = PHILOX_M[0] * x0, PHILOX_M[1] * x2
        x0, x1, x2, x3 = ((p1 >> 64) ^ x1 ^ k0, p1 & M64, (p0 >> 64) ^ x3 ^ k1, p0 & M64)
    return x0, x1, x2, x3


def uniform(seed: int, pos: int, b: int) -> float:
    """u in [0, 1) of row b for the token at sequence position pos."""
    return (philox4x64((seed, 0), (pos, b, 0, 0))[0] >> 11) * 2.0 ** -53


def _row(row) -> np.ndarray:
    x = np.asarray(row, dtype=np.float32).copy()
    x[np.isnan(x)] = -np.inf                        # NaN counts as -inf
    return x


def kept_set(row, top_k) -> np.ndarray:
    """Ids of K in ascending order: every logit >= the k-th largest (ties at tau included)."""
    x = _row(row)
    V = x.shape[0]
    k = top_k if top_k is not None and 1 <= top_k < V else V
    tau = np.sort(x)[::-1][k - 1]
    return np.nonzero(x >= tau)[0]


def sample_probs(row, temperature: float, top_k):
    """(K, p): the kept ids and their probabilities, weights exp((l - max) / T) in fp64."""
    x = _row(row)
    K = kept_set(x, top_k)
    w = np.exp((x[K].astype(np.float64) - np.float64(x.max())) / np.float64(np.float32(temperature)))
    return K, w / w.sum()


def sample_reference(logits, temperature: float, top_k, seed: int, pos: int, with_margin: bool = False):
    """Tokens [B] (int64) for sequence position pos, the contract of vcl_sampling. with_margin: also the
    distance of t to the nearest bin edge of the running sum, over Z (a draw that close to an edge may land
    on the neighbouring id when the sums are associated differently)."""
    L = np.asarray(logits, dtype=np.float32)
    toks, margins = [], []
    for b in range(L.shape[0]):
        x = _row(L[b])
        mx = x.max()
        if np.float32(temperature) <= 0 or not np.isfinite(mx):
            toks.append(int(np.argmax(x)) if np.isfinite(mx) or mx == np.inf else 0)
            margins.append(np.inf)
            continue
        K = kept_set(x, top_k)
        w = np.exp((x[K].astype(np.float64) - np.float64(mx)) / np.float64(np.float32(temperature)))
        c = np.cumsum(w)                             # sequential running sum in ascending id order
        Z = c[-1]
        t = uniform(seed, pos, b) * Z
        j = int(np.searchsorted(c, t, side="right"))  # first running sum > t
        toks.append(int(K[j]) if j < len(K) else int(K[-1]))
        margins.append(float(np.min(np.abs(c - t)) / Z))
    toks = np.asarray(toks, dtype=np.int64)
    return (toks, np.asarray(margins)) if with_margin else toks
