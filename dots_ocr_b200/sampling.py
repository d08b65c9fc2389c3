"""Per-request sampling parameters and the serving policy that decides whether requests may use them.

Decoding is greedy unless a caller asks for sampling.  A sampled row runs HF's warper chain (transformers
``generation/logits_process.py``: Temperature -> TopK -> TopP) and a Gumbel-max draw on the device, in
``dots_sample_advance`` (csrc/sampling.cu; DESIGN.md section 3):

* ``temperature < 1e-5`` is greedy (vLLM's threshold), bit-identical to ``dots_argmax_advance``;
* ``top_k > 0`` keeps the logits >= the k-th largest, ties at the cut-off included (HF's rule);
* ``top_p < 1`` keeps, among those, every token whose softmax mass of STRICTLY larger logits is < p.  Every token tied with
  the last kept value is kept: HF and vLLM cut inside a run of tied logits at an arbitrary sort position, and bf16 logits do
  tie; keeping the whole run needs no sort and does not depend on the batch;
* the random numbers come from Philox4x32-10 keyed by the row's 64-bit seed with counter (token index >> 2, step, 0, 0),
  so a row's token depends on its logits, parameters, seed and step only -- not on the batch size, its position in the
  batch, graph or eager execution, or the other rows.  Nothing random lives on the host.

A request without a seed gets one drawn once, at submission, from torch's default CPU generator, so ``torch.manual_seed``
makes in-process runs reproducible as it does for HF ``generate``.
"""
from __future__ import annotations

import math
import os
from dataclasses import dataclass, replace
from typing import List, Optional, Sequence, Union

GREEDY_BELOW = 1e-5         # temperatures below this decode greedily (vLLM's _SAMPLING_EPS)
POLICIES = ("greedy", "request")


def sampling_policy() -> str:
    """Whether the serving fronts honour the sampling fields of a request: environment ``DOTS_B200_SAMPLING`` =
    ``greedy`` (default: every request decodes greedily, its sampling fields are ignored) or ``request``."""
    v = os.environ.get("DOTS_B200_SAMPLING", "greedy").strip().lower() or "greedy"
    if v not in POLICIES:
        raise ValueError(f"DOTS_B200_SAMPLING must be one of {POLICIES}, got {v!r}")
    return v


@dataclass(frozen=True)
class SamplingParams:
    temperature: float = 1.0
    top_p: float = 1.0
    top_k: int = 0              # 0 = off
    seed: Optional[int] = None  # u64; None = drawn at submission (``with_seed``)

    def __post_init__(self):
        for name in ("temperature", "top_p"):
            v = getattr(self, name)
            if isinstance(v, bool) or not isinstance(v, (int, float)):
                raise ValueError(f"{name} must be a number, got {v!r}")
        if isinstance(self.top_k, bool) or not isinstance(self.top_k, int):
            raise ValueError(f"top_k must be an integer, got {self.top_k!r}")
        if self.seed is not None and (isinstance(self.seed, bool) or not isinstance(self.seed, int)):
            raise ValueError(f"seed must be an integer, got {self.seed!r}")
        if not (math.isfinite(self.temperature) and self.temperature >= 0):
            raise ValueError(f"temperature must be finite and >= 0, got {self.temperature}")
        if not (0 < self.top_p <= 1):
            raise ValueError(f"top_p must be in (0, 1], got {self.top_p}")
        if self.top_k < 0:
            raise ValueError(f"top_k must be >= 0 (0 = off), got {self.top_k}")
        if self.seed is not None and not (0 <= self.seed < 1 << 64):
            raise ValueError(f"seed must fit in an unsigned 64-bit integer, got {self.seed}")

    @property
    def greedy(self) -> bool:
        return self.temperature < GREEDY_BELOW

    def with_seed(self) -> "SamplingParams":
        """These parameters with a seed: their own, or one drawn now from torch's default CPU generator."""
        if self.seed is not None:
            return self
        import torch
        s = int(torch.randint(-(1 << 63), (1 << 63) - 1, (1,), dtype=torch.int64).item())
        return replace(self, seed=s & ((1 << 64) - 1))


GREEDY = SamplingParams(temperature=0.0, seed=0)


def from_hf_kwargs(kw: dict) -> Optional[SamplingParams]:
    """HF ``generate`` keyword arguments -> parameters (HF defaults: temperature 1.0, top_p 1.0, top_k 50), or None when
    ``do_sample`` is absent or false (HF then decodes greedily and ignores the others)."""
    if not kw.get("do_sample"):
        return None
    pick = lambda k, d: d if kw.get(k) is None else kw[k]          # noqa: E731
    return SamplingParams(temperature=float(pick("temperature", 1.0)), top_p=float(pick("top_p", 1.0)), top_k=int(pick("top_k", 50)))


def per_row(sampling: Union[SamplingParams, Sequence[SamplingParams]], n: int) -> List[SamplingParams]:
    """One set of parameters for every row, or a sequence of ``n``; every row gets a seed (drawn now where missing)."""
    rows = [sampling] * n if isinstance(sampling, SamplingParams) else list(sampling)
    if len(rows) != n or not all(isinstance(r, SamplingParams) for r in rows):
        raise ValueError(f"sampling: need one SamplingParams or a sequence of {n}, got {sampling!r}")
    return [r.with_seed() for r in rows]              # one seedless SamplingParams for all rows: a distinct draw per row


def host_arrays(rows: Sequence[SamplingParams]):
    """(temperature f32, top_p f32, top_k i32, seed i64 holding the u64 bits) CPU tensors, the layout
    ``dots_sample_advance`` reads.  Every row must have a seed."""
    import torch
    seeds = [r.seed - (1 << 64) if r.seed >= 1 << 63 else r.seed for r in rows]
    return (torch.tensor([r.temperature for r in rows], dtype=torch.float32),
            torch.tensor([r.top_p for r in rows], dtype=torch.float32),
            torch.tensor([r.top_k for r in rows], dtype=torch.int32),
            torch.tensor(seeds, dtype=torch.int64))
