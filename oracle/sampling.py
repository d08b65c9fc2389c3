"""fp64 restatement of ``dots_sample_advance`` (tests only): Philox4x32-10, the warper chain with its tie rule, and the
Gumbel-max draw.  Given a logits row, its parameters, seed and step, ``replay`` names the token the kernel must pick.

Warper chain (transformers ``generation/logits_process.py``, HF's order): temperature, then top-k (keep l >= the k-th
largest; ties kept, as ``TopKLogitsWarper``), then top-p over the survivors (keep l iff the softmax(l / T) mass of
strictly larger logits is < p: the whole run of ties at the cut-off is kept, where HF cuts it at a sort position).
"""
from __future__ import annotations

import numpy as np

_M0, _M1 = 0xD2511F53, 0xCD9E8D57
_W0, _W1 = 0x9E3779B9, 0xBB67AE85
_MASK = 0xFFFFFFFF
GREEDY_BELOW = 1e-5


def philox4x32_10(ctr, key):
    """Scalar Philox4x32-10: counter (4 x u32), key (2 x u32) -> 4 x u32 (Random123's known-answer vectors hold)."""
    c0, c1, c2, c3 = (int(x) & _MASK for x in ctr)
    k0, k1 = (int(x) & _MASK for x in key)
    for _ in range(10):
        p0, p1 = _M0 * c0, _M1 * c2
        c0, c1, c2, c3 = ((p1 >> 32) ^ c1 ^ k0) & _MASK, p1 & _MASK, ((p0 >> 32) ^ c3 ^ k1) & _MASK, p0 & _MASK
        k0, k1 = (k0 + _W0) & _MASK, (k1 + _W1) & _MASK
    return c0, c1, c2, c3


def philox_words(n_groups: int, step: int, seed: int) -> np.ndarray:
    """Vectorised Philox for counters (g, step, 0, 0), g < n_groups: uint32 [n_groups * 4] in token order (word i & 3 of
    group i >> 2 belongs to token i)."""
    c0 = np.arange(n_groups, dtype=np.uint64)
    c1 = np.full(n_groups, step & _MASK, dtype=np.uint64)
    c2 = np.zeros(n_groups, dtype=np.uint64)
    c3 = np.zeros(n_groups, dtype=np.uint64)
    k0, k1 = np.uint64(seed & _MASK), np.uint64((seed >> 32) & _MASK)
    m32 = np.uint64(_MASK)
    for _ in range(10):
        p0 = np.uint64(_M0) * c0
        p1 = np.uint64(_M1) * c2
        c0, c1, c2, c3 = ((p1 >> np.uint64(32)) ^ c1 ^ k0) & m32, p1 & m32, ((p0 >> np.uint64(32)) ^ c3 ^ k1) & m32, p0 & m32
        k0, k1 = (k0 + np.uint64(_W0)) & m32, (k1 + np.uint64(_W1)) & m32
    return np.stack([c0, c1, c2, c3], axis=1).reshape(-1).astype(np.uint32)


def uniforms(V: int, step: int, seed: int) -> np.ndarray:
    """u_i = ((x_i >> 8) + 0.5) * 2^-24 in fp64, i < V."""
    x = philox_words((V + 3) // 4, step, seed)[:V]
    return ((x >> 8).astype(np.float64) + 0.5) * 2.0 ** -24


def kept_mask(logits, temperature: float, top_p: float = 1.0, top_k: int = 0, return_margin: bool = False):
    """Boolean mask of the tokens that survive top-k then top-p (fp64 arithmetic on the given values).  With
    ``return_margin``: also the relative distance of the top-p threshold p * Z from the nearest cumulative mass
    (inf when top-p is off), the quantity the kernel's fixed-point sums could round across."""
    l = np.asarray(logits, dtype=np.float64)
    V = l.shape[0]
    keep = np.ones(V, dtype=bool)
    if 0 < top_k < V:
        kth = np.sort(l)[::-1][top_k - 1]
        keep &= l >= kth
    margin = np.inf
    if top_p < 1.0:
        t = float(temperature)
        vals = np.unique(l[keep])[::-1]                   # distinct surviving values, descending
        w = np.exp((l[keep] - vals[0]) / t)
        Z = w.sum()
        mass_per_val = np.bincount(np.searchsorted(-vals, -l[keep]), weights=w, minlength=vals.size)
        above = np.concatenate([[0.0], np.cumsum(mass_per_val)[:-1]])   # mass strictly larger than each value
        thr = float(np.float32(top_p)) * Z
        ok = above < thr
        cut = vals[ok].min()
        keep &= l >= cut
        margin = float(np.min(np.abs(above[1:] - thr)) / Z) if vals.size > 1 else np.inf
    return (keep, margin) if return_margin else keep


def gumbel_keys(logits, temperature: float, step: int, seed: int) -> np.ndarray:
    l = np.asarray(logits, dtype=np.float64)
    u = uniforms(l.shape[0], step, seed)
    return l / float(np.float32(temperature)) - np.log(-np.log(u))


def replay(logits, temperature: float, top_p: float = 1.0, top_k: int = 0, seed: int = 0, step: int = 0, return_info: bool = False):
    """The token ``dots_sample_advance`` picks for one row.  ``return_info``: (token, info) with info = dict(gap = relative
    distance between the two largest Gumbel keys, p_margin = see ``kept_mask``, kept = the kept mask)."""
    l = np.asarray(logits, dtype=np.float64)
    if float(np.float32(temperature)) < GREEDY_BELOW:
        tok = int(np.argmax(l))
        return (tok, dict(gap=np.inf, p_margin=np.inf, kept=None)) if return_info else tok
    keep, margin = kept_mask(l, float(np.float32(temperature)), float(np.float32(top_p)), int(top_k), return_margin=True)
    g = np.where(keep, gumbel_keys(l, temperature, step, seed), -np.inf)
    tok = int(np.argmax(g))
    if not return_info:
        return tok
    top2 = np.sort(g[keep])[-2:] if keep.sum() > 1 else np.array([-np.inf, g[tok]])
    gap = float(abs(top2[1] - top2[0]) / max(abs(top2[1]), 1e-30))
    return tok, dict(gap=gap, p_margin=margin, kept=keep)


def distribution(logits, temperature: float, top_p: float = 1.0, top_k: int = 0) -> np.ndarray:
    """Exact fp64 probabilities of the draw: softmax(l / T) restricted to the kept set."""
    l = np.asarray(logits, dtype=np.float64)
    keep = kept_mask(l, temperature, top_p, top_k)
    z = np.where(keep, (l - l[keep].max()) / float(np.float32(temperature)), -np.inf)
    p = np.exp(z)
    return p / p.sum()
