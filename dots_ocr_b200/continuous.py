"""Continuous batching behind the one-page call surface (SURVEY.md section 8f N2, second step).

``BatchingRunner`` (batching.py) forms a batch, runs it to its LONGEST page and only then looks at the queue again: a row
that stops after 300 tokens idles while its neighbour writes 4000, and pages that arrive meanwhile wait for the whole batch.
Here the decode state is a fixed set of SLOTS (rows of one KV cache / one captured decode graph).  The scheduler alternates

    admit    free slots <- queued pages: ViT + prefill write the new rows of the cache, first token selected
    decode   ``chunk`` steps for every slot (one graph replay per step)
    harvest  rows that produced a stop id or used up their own token budget are answered and their slots freed

so a finished row is refilled at the next chunk boundary while the other rows keep their context.  No kernel knows about
slots: prefill addresses cache rows through ``seq_of_tok`` (dots_llm_rope_kv_append), every decode kernel already works on
per-row ``pos`` / ``ctx_len`` / ``step`` / ``finished`` arrays, and between chunks the host rewrites those few ints.

Two parts:

* ``ContinuousBatcher`` -- the scheduler (threads, queue, slot table, budgets).  Pure host logic; tested on CPU against a
  simulated backend that enforces the row bounds (tests/test_continuous_cpu.py).
* ``EngineSlots`` -- the backend over ``Engine`` (GPU cases: tests/test_zzz_continuous_gpu.py).

Row bounds the scheduler guarantees to the backend (``chunk`` = steps between harvests, ``max_new`` = largest budget):
an occupied row is harvested at the first chunk boundary with ``step >= budget``, so ``step < budget + chunk``; idle rows are
re-armed (step 0, pos 0) at every boundary, so they never pass ``chunk``.  Hence ``out_ids`` needs ``max_new + chunk`` columns
and the cache ``max_prompt + max_new + chunk`` positions.
"""
from __future__ import annotations

import queue
import threading
import time
from concurrent.futures import Future
from typing import List, Optional, Sequence, Tuple

from .batching import page_vit_tokens


# =====================================================================================================================
# backend over the CUDA engine
# =====================================================================================================================
class EngineSlots:
    """Slot backend over ``Engine``: one KV cache of ``n_slots`` rows and one captured decode graph for the session."""

    def __init__(self, engine, tokenizer, n_slots: int = 64, max_prompt: int = 2048, max_new: int = 2048, chunk: int = 32,
                 min_pixels=None, max_pixels=None):
        import torch
        from .engine import _round_up
        self.engine, self.tokenizer = engine, tokenizer
        self.n_slots, self.max_prompt, self.max_new, self.chunk = int(n_slots), int(max_prompt), int(max_new), int(chunk)
        self.min_pixels, self.max_pixels = min_pixels, max_pixels
        assert 1 <= self.n_slots <= 256 and self.chunk >= 1
        self.n_cols = self.max_new + self.chunk
        self.ctx_max = _round_up(self.max_prompt + self.max_new + self.chunk, 64)
        dev = engine.device
        stops = list(getattr(tokenizer, "stop_ids", ())) or ([] if tokenizer.eos_token_id is None else [tokenizer.eos_token_id])
        self.stops = [int(x) for x in stops]              # any of these finishes a row on the device (dots_argmax_advance)
        self.pad = int(tokenizer.pad_token_id)
        with torch.no_grad(), torch.cuda.device(dev):
            kc, vc = engine._alloc_cache(self.n_slots, self.ctx_max)
            lens = torch.ones(self.n_slots, dtype=torch.int64, device=dev)
            self.st = engine._new_decode_state(self.n_slots, lens, kc, vc, self.ctx_max, self.n_cols, self.stops, self.pad)
        self.rearm(list(range(self.n_slots)))
        self._graph = None
        self._warm = False

    # -- admission ------------------------------------------------------------------------------------------------------
    def prepare(self, image, prompt: str, sampling=None):
        """Host half of admission (runs in the scheduler thread before the GPU is touched): uint8 page + prompt ids +
        the page's sampling parameters (None: greedy)."""
        from .processing import page_to_u8, model_image_tokens
        page = page_to_u8(image)                               # original size: the resize runs on the GPU at admission
        n_img = model_image_tokens(int(page.shape[0]), int(page.shape[1]), self.min_pixels, self.max_pixels)
        ids = self.tokenizer.encode_chat(prompt, n_img)
        if len(ids) > self.max_prompt:
            raise ValueError(f"prompt of {len(ids)} tokens exceeds the session's max_prompt {self.max_prompt}")
        return page, ids, sampling

    def _enable_sampling(self) -> None:
        """First sampled page of the session: add the per-row parameter arrays (every row greedy until admitted with
        parameters) and drop the captured graph, so that the next step captures it with dots_sample_advance.  A session
        that only ever sees greedy pages keeps the greedy kernel."""
        import torch
        st, n, dev = self.st, self.n_slots, self.engine.device
        st["temperature"] = torch.zeros(n, device=dev, dtype=torch.float32)
        st["top_p"] = torch.ones(n, device=dev, dtype=torch.float32)
        st["top_k"] = torch.zeros(n, device=dev, dtype=torch.int32)
        st["seed"] = torch.zeros(n, device=dev, dtype=torch.int64)
        self._graph = None

    def admit(self, slots: Sequence[int], prepared: Sequence) -> None:
        """ViT + prefill of the new pages into cache rows ``slots``; selects each row's first token."""
        import torch
        from . import ops
        from .sampling import GREEDY, host_arrays
        eng, st, dev = self.engine, self.st, self.engine.device
        t = eng.cfg.text
        params = [item[2] if len(item) > 2 else None for item in prepared]
        if "temperature" not in st and any(p is not None for p in params):
            self._enable_sampling()
        with torch.no_grad(), torch.cuda.device(dev):
            pages = [item[0].to(dev, non_blocking=True) for item in prepared]
            rows = [item[1] for item in prepared]
            seq_lens = [len(r) for r in rows]
            ids_packed = torch.tensor([i for r in rows for i in r], dtype=torch.int64, device=dev)
            positions = torch.cat([torch.arange(n, dtype=torch.int32) for n in seq_lens]).to(dev)
            seq_of_tok = torch.cat([torch.full((n,), int(s), dtype=torch.int32) for n, s in zip(seq_lens, slots)]).to(dev)
            lens = torch.tensor(seq_lens, dtype=torch.int64, device=dev)
            cu = torch.zeros(len(rows) + 1, dtype=torch.int32, device=dev)
            cu[1:] = lens.cumsum(0).to(torch.int32)
            image_embeds = eng.encode_pages_u8(pages, min_pixels=self.min_pixels, max_pixels=self.max_pixels)
            img_slots, count = ops.image_slots(ids_packed, eng.cfg.image_token_id)
            if int(count.item()) != image_embeds.shape[0]:
                raise ValueError(f"image tokens in the prompts ({int(count.item())}) != image embedding rows ({image_embeds.shape[0]})")
            x = eng._prefill(ids_packed, img_slots, image_embeds, cu, seq_lens, positions, seq_of_tok, st["kc"], st["vc"], self.ctx_max)
            hl = ops.gather_rows(x, (cu[1:] - 1).to(torch.int32))
            normed = ops.rmsnorm(hl, eng.final_norm, t.rms_norm_eps)
            n = len(rows)
            logits = torch.empty((n, t.vocab_size), device=dev, dtype=torch.bfloat16)
            ops.gemm_skinny(normed, eng.lm_head, 1, out_bf16=logits)
            # first token through the same kernel, on row-compact temporaries, then scattered into the session's rows
            last = torch.zeros(n, dtype=torch.int64, device=dev)
            out = torch.full((n, self.n_cols), self.pad, dtype=torch.int64, device=dev)
            step = torch.zeros(n, dtype=torch.int32, device=dev)
            pos = (lens - 1).to(torch.int32)
            ctx = lens.to(torch.int32)
            fin = torch.zeros(n, dtype=torch.int32, device=dev)
            idx = torch.tensor(list(slots), dtype=torch.int64, device=dev)
            if "temperature" in st:
                arrs = [a.to(dev) for a in host_arrays([GREEDY if p is None else p.with_seed() for p in params])]
                ops.sample_advance(logits, last, *arrs, out, step, pos, ctx, fin, tuple(self.stops[: ops.MAX_STOP_IDS]), self.pad, None)
                for name, a in zip(("temperature", "top_p", "top_k", "seed"), arrs):
                    st[name].index_copy_(0, idx, a)
            else:
                ops.argmax_advance(logits, last, out, step, pos, ctx, fin, tuple(self.stops[: ops.MAX_STOP_IDS]), self.pad, None)
            eng.launches += 5
            st["last"].index_copy_(0, idx, last)
            st["out_ids"].index_copy_(0, idx, out)
            st["step"].index_copy_(0, idx, step)
            st["pos"].index_copy_(0, idx, pos)
            st["ctx_len"].index_copy_(0, idx, ctx)
            st["finished"].index_copy_(0, idx, fin)

    # -- decode ---------------------------------------------------------------------------------------------------------
    def step(self, k: int) -> None:
        """``k`` decode steps for every slot (idle rows run along on a pad token)."""
        import torch
        from . import ops
        eng, st = self.engine, self.st
        with torch.no_grad(), torch.cuda.device(eng.device):
            done = 0
            if not self._warm:
                eng._decode_step(st)                     # eager once: warms every kernel variant before capture
                self._warm = True
                done = 1
            if done < k and self._graph is None:
                cap = torch.cuda.Stream(device=eng.device)
                cap.wait_stream(torch.cuda.current_stream())
                with torch.cuda.stream(cap):
                    g = ops.capture(lambda: eng._decode_step(st))
                torch.cuda.current_stream().wait_stream(cap)
                self._graph = g
            for _ in range(k - done):
                self._graph.launch()
            eng.launches += eng.launches_per_decode_step(self.n_slots) * k

    def poll(self) -> Tuple[List[int], List[int]]:
        """(tokens generated so far, finished flag) per slot: one device->host read of 2 x n_slots ints."""
        import torch
        both = torch.stack([self.st["step"], self.st["finished"]]).cpu()
        return both[0].tolist(), both[1].tolist()

    def take(self, slot: int, n: int) -> List[int]:
        return self.st["out_ids"][slot, :n].tolist()

    def rearm(self, slots: Sequence[int]) -> None:
        """Park rows: finished, at position 0 with one visible key, so that running along stays inside their cache row;
        greedy, so that a parked row costs the sampling kernel its argmax pass only."""
        import torch
        if not slots:
            return
        st, dev = self.st, self.engine.device
        idx = torch.tensor(list(slots), dtype=torch.int64, device=dev)
        st["finished"].index_fill_(0, idx, 1)
        st["step"].index_fill_(0, idx, 0)
        st["pos"].index_fill_(0, idx, 0)
        st["ctx_len"].index_fill_(0, idx, 1)
        st["last"].index_fill_(0, idx, self.pad)
        if "temperature" in st:
            st["temperature"].index_fill_(0, idx, 0.0)

    def decode_text(self, ids: List[int]) -> str:
        return self.tokenizer.decode(ids)


# =====================================================================================================================
# scheduler
# =====================================================================================================================
class _Req:
    __slots__ = ("image", "prompt", "budget", "future", "tokens", "arrived", "sampling")

    def __init__(self, image, prompt, budget, future, tokens, sampling=None):
        self.image, self.prompt, self.budget, self.future, self.tokens = image, prompt, budget, future, tokens
        self.sampling = sampling                   # SamplingParams with its seed, or None (greedy)
        self.arrived = time.monotonic()


class ContinuousBatcher:
    """``infer(image, prompt, max_new_tokens)`` for many threads over a slot backend.

    backend: ``n_slots``, ``chunk``, ``max_new`` attributes and ``prepare / admit / step / poll / take / rearm /
    decode_text`` methods (see ``EngineSlots``).  ``max_admit_tokens`` bounds the ViT patch tokens prefetched in one admission
    (a long admission stalls the rows that are decoding)."""

    def __init__(self, backend, max_admit_tokens: int = 64 * 5476, idle_wait_ms: float = 5.0):
        self.backend = backend
        self.engine = getattr(backend, "engine", None)
        self.tokenizer = getattr(backend, "tokenizer", None)
        self.max_admit_tokens = int(max_admit_tokens)
        self.idle_wait = float(idle_wait_ms) / 1e3
        self._q: "queue.Queue" = queue.Queue()
        self._closed = False
        self._carry: Optional[_Req] = None
        self._active = {}                                    # slot -> _Req
        self.stats = {"admissions": 0, "chunks": 0, "pages": 0, "max_active": 0}
        self._worker = threading.Thread(target=self._loop, name="dots-b200-continuous", daemon=True)
        self._worker.start()

    # -- caller side ------------------------------------------------------------------------------------------------
    def submit(self, image, prompt: str, max_new_tokens: int = 512, sampling=None) -> Future:
        """sampling: None (greedy) or a ``SamplingParams``; a missing seed is drawn here, at submission."""
        if self._closed:
            raise RuntimeError("ContinuousBatcher is closed")
        fut: Future = Future()
        budget = max(1, min(int(max_new_tokens), int(self.backend.max_new)))
        self._q.put(_Req(image, prompt, budget, fut, max(1, page_vit_tokens(image)), None if sampling is None else sampling.with_seed()))
        return fut

    def infer(self, image, prompt: str, max_new_tokens: int = 512, sampling=None) -> str:
        return self.submit(image, prompt, max_new_tokens, sampling).result()

    def infer_batch(self, images, prompts, max_new_tokens: int = 512, sampling=None) -> List[str]:
        futs = [self.submit(im, pr, max_new_tokens, sampling) for im, pr in zip(images, prompts)]
        return [f.result() for f in futs]

    def close(self, timeout: Optional[float] = 30.0) -> None:
        """Stop taking requests; everything already submitted is still answered."""
        self._closed = True
        self._q.put(None)
        self._worker.join(timeout)

    # -- worker -----------------------------------------------------------------------------------------------------
    def _next_request(self, block: bool):
        if self._carry is not None:
            r, self._carry = self._carry, None
            return r
        try:
            return self._q.get(timeout=self.idle_wait) if block else self._q.get_nowait()
        except queue.Empty:
            return False

    def _admit(self, draining: bool) -> bool:
        """Fill free slots from the queue.  Returns True once the shutdown marker has been seen."""
        b = self.backend
        free = [s for s in range(b.n_slots) if s not in self._active]
        picked: List[_Req] = []
        tokens = 0
        while len(picked) < len(free):
            r = self._next_request(block=not self._active and not picked and not draining)
            if r is False:
                break
            if r is None:
                draining = True
                continue
            if picked and tokens + r.tokens > self.max_admit_tokens:
                self._carry = r
                break
            picked.append(r)
            tokens += r.tokens
        if not picked:
            return draining
        ready, slots = [], []
        for r in picked:
            try:
                ready.append((r, b.prepare(r.image, r.prompt) if r.sampling is None else b.prepare(r.image, r.prompt, sampling=r.sampling)))
            except Exception as e:      # noqa: BLE001 -- this page's caller gets the error; the others go on
                r.future.set_exception(e)
        if ready:
            slots = free[: len(ready)]
            try:
                b.admit(slots, [p for _, p in ready])
            except Exception as e:      # noqa: BLE001
                for r, _ in ready:
                    r.future.set_exception(e)
                b.rearm(slots)
                return draining
            for s, (r, _) in zip(slots, ready):
                self._active[s] = r
            self.stats["admissions"] += 1
            self.stats["max_active"] = max(self.stats["max_active"], len(self._active))
        return draining

    def _harvest(self) -> None:
        b = self.backend
        steps, fin = b.poll()
        for s in list(self._active):
            r = self._active[s]
            if fin[s] or steps[s] >= r.budget:
                n = min(int(steps[s]), r.budget)
                try:
                    r.future.set_result(b.decode_text(b.take(s, n)))
                except Exception as e:  # noqa: BLE001
                    r.future.set_exception(e)
                del self._active[s]
                self.stats["pages"] += 1
        # every row without a page is parked again: it ran along for `chunk` steps and must not drift out of its cache row
        b.rearm([s for s in range(b.n_slots) if s not in self._active])

    def _loop(self) -> None:
        draining = False
        while True:
            try:
                draining = self._admit(draining)
                if not self._active:
                    if draining and self._carry is None and self._q.empty():
                        return
                    continue
                self.backend.step(self.backend.chunk)
                self.stats["chunks"] += 1
                self._harvest()
            except Exception as e:      # noqa: BLE001 -- a backend failure answers every page in flight, then the loop goes on
                for r in self._active.values():
                    if not r.future.done():
                        r.future.set_exception(e)
                self._active.clear()
                try:
                    self.backend.rearm(list(range(self.backend.n_slots)))
                except Exception:       # noqa: BLE001
                    pass


def serving_front(page_runner, kind: Optional[str] = None, max_batch: int = 64, max_prompt: int = 16384, max_new: int = 8192, chunk: int = 32):
    """The request front behind the one-page call surface (``inference_with_vllm``, the HTTP endpoint, the per-GPU workers).

    ``kind`` (default: environment ``DOTS_B200_BATCHER``, else ``continuous``):
      * ``continuous``  ContinuousBatcher over EngineSlots: ``max_batch`` decode slots, finished pages leave and queued pages enter
                        between chunks of ``chunk`` decode steps (the server-side behaviour the reference's 64-thread fan-out expects
                        from vLLM, dots_ocr/parser.py:282-290).  ``max_prompt`` / ``max_new`` size the session's KV cache
                        (28 672 B per token and slot at full size: 64 x 24.6 k tokens = 45 GB of the 180 GB).
      * ``batching``    BatchingRunner: batches formed at arrival, each run to its longest page.
    Falls back to ``batching`` for runners that have no CUDA engine (CPU stand-ins in tests)."""
    import os
    kind = (kind or os.environ.get("DOTS_B200_BATCHER", "continuous")).lower()
    eng = getattr(page_runner, "engine", None)
    if kind == "continuous" and eng is not None and hasattr(eng, "_new_decode_state"):
        slots = EngineSlots(eng, page_runner.tokenizer, n_slots=min(int(max_batch), 256), max_prompt=max_prompt, max_new=max_new, chunk=chunk,
                            min_pixels=getattr(page_runner, "min_pixels", None), max_pixels=getattr(page_runner, "max_pixels", None))
        return ContinuousBatcher(slots)
    from .batching import BatchingRunner
    return BatchingRunner(page_runner, max_batch=max_batch)
