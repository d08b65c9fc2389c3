"""Request batching behind the one-page call surface (SURVEY.md section 8f N2).

The reference fans pages out from up to ``num_thread`` (default 64) worker threads, each calling
``inference_with_vllm(image, prompt, ...)`` for ONE page (``dots_ocr/parser.py:282-290``); the vLLM server batches them.  In process
the same threads would serialise on the engine lock, one page per ``generate``.  ``BatchingRunner`` gives them the server's
behaviour: callers block on a future while a single worker thread drains the queue into batches of up to ``max_batch`` pages
(it waits at most ``max_wait_ms`` for stragglers, counted from the arrival of the batch's first request) and runs one
``PageRunner.infer_batch`` per batch, so concurrent callers share the ViT / prefill / decode launches.  A batch is also closed
when the next page would push its ViT token count (from the image size through ``smart_resize``) past ``max_batch_tokens``:
64 pages of 1024x1024 are 350 k patch tokens, 64 pages of 1960x1960 would be 1.25 M; that page opens the next batch.
"""
from __future__ import annotations

import queue
import threading
import time
from concurrent.futures import Future
from typing import List, Optional


def page_vit_tokens(image, min_pixels=None, max_pixels=None) -> int:
    """Patch tokens the vision tower will see for this page (0 when the size cannot be told, e.g. a test stand-in)."""
    size = getattr(image, "size", None)
    if not (isinstance(size, tuple) and len(size) == 2):
        return 0
    from .utils.image_utils import token_counts
    kw = {}
    if min_pixels is not None:
        kw["min_pixels"] = min_pixels
    if max_pixels is not None:
        kw["max_pixels"] = max_pixels
    try:
        return token_counts(int(size[1]), int(size[0]), **kw)[0]
    except ValueError:            # absurd aspect ratio: let the runner raise it for this caller
        return 0


class BatchingRunner:
    def __init__(self, runner, max_batch: int = 64, max_wait_ms: float = 20.0, max_batch_tokens: int = 64 * 5476):
        self.runner = runner                      # anything with infer_batch(images, prompts, max_new_tokens) -> List[str]
        self.max_batch_tokens = int(max_batch_tokens)
        self.engine = getattr(runner, "engine", None)
        self.tokenizer = getattr(runner, "tokenizer", None)
        self.max_batch = int(max_batch)
        self.max_wait = float(max_wait_ms) / 1e3
        import inspect
        try:
            self._takes_budgets = "budgets" in inspect.signature(runner.infer_batch).parameters      # per-caller token budgets
        except (TypeError, ValueError):
            self._takes_budgets = False
        self._q: "queue.Queue" = queue.Queue()
        self._closed = False
        self.batches: List[int] = []              # sizes of the batches run so far (observability / tests)
        self._worker = threading.Thread(target=self._loop, name="dots-b200-batcher", daemon=True)
        self._worker.start()

    # -- caller side ------------------------------------------------------------------------------------------------
    def submit(self, image, prompt: str, max_new_tokens: int = 512, sampling=None) -> Future:
        """sampling: None (greedy) or a ``SamplingParams``; a missing seed is drawn here, at submission."""
        if self._closed:
            raise RuntimeError("BatchingRunner is closed")
        fut: Future = Future()
        self._q.put((image, prompt, int(max_new_tokens), fut, None if sampling is None else sampling.with_seed()))
        return fut

    def infer(self, image, prompt: str, max_new_tokens: int = 512, sampling=None) -> str:
        return self.submit(image, prompt, max_new_tokens, sampling).result()

    def infer_batch(self, images, prompts, max_new_tokens: int = 512, sampling=None) -> List[str]:
        futs = [self.submit(im, pr, max_new_tokens, sampling) for im, pr in zip(images, prompts)]
        return [f.result() for f in futs]

    def close(self, timeout: Optional[float] = 5.0) -> None:
        self._closed = True
        self._q.put(None)
        self._worker.join(timeout)

    # -- worker -----------------------------------------------------------------------------------------------------
    def _tokens(self, item) -> int:
        return page_vit_tokens(item[0], getattr(self.runner, "min_pixels", None), getattr(self.runner, "max_pixels", None))

    def _loop(self) -> None:
        carry = None                              # a request that did not fit the previous batch's token budget
        while True:
            first = carry if carry is not None else self._q.get()
            carry = None
            if first is None:
                return
            batch = [first]
            tokens = self._tokens(first)
            deadline = time.monotonic() + self.max_wait
            stop = False
            while len(batch) < self.max_batch:
                try:
                    item = self._q.get(timeout=max(0.0, deadline - time.monotonic()))
                except queue.Empty:
                    break
                if item is None:
                    stop = True
                    break
                t = self._tokens(item)
                if tokens + t > self.max_batch_tokens:
                    carry = item
                    break
                batch.append(item)
                tokens += t
            self._run(batch)
            if stop:
                if carry is not None:
                    self._run([carry])
                return

    def _run(self, batch) -> None:
        # one generate for the whole batch at the largest token budget; every caller gets its own budget back
        n_new = max(b[2] for b in batch)
        self.batches.append(len(batch))
        try:
            kw = {"budgets": [b[2] for b in batch]} if self._takes_budgets else {}
            if any(b[4] is not None for b in batch):
                # per-row parameters; the pages that did not ask for sampling decode greedily beside the others
                from .sampling import GREEDY
                kw["sampling"] = [GREEDY if b[4] is None else b[4] for b in batch]
            texts = self.runner.infer_batch([b[0] for b in batch], [b[1] for b in batch], max_new_tokens=n_new, **kw)
        except Exception as e:          # noqa: BLE001 -- the error belongs to the callers, not to the worker thread
            if len(batch) == 1:
                batch[0][3].set_exception(e)
                return
            # One bad page (aspect ratio above 200, unreadable image, over-long prompt ...) must not fail its up-to-63
            # neighbours: run the pages of the failed batch one by one, so only the page that raises gets the error.
            for b in batch:
                self._run([b])
            return
        for b, text in zip(batch, texts):
            b[3].set_result(text)
