"""Pages over the GPUs of one box: one worker PROCESS per GPU, model replicated, no collective on the data path
(SURVEY.md section 8e).  ``bench.py`` measures this layout under torchrun; this module is the same layout behind the
one-page call surface (``infer(image, prompt, max_new_tokens)``), so the parser's thread fan-out or the HTTP endpoint can
drive every GPU of the box.

The front process keeps no CUDA context.  Each request goes to the worker with the least outstanding work, counted in ViT
patch tokens (a 1960x1960 page weighs 3.6 pages of 1024x1024); inside a worker a ``BatchingRunner`` groups what arrives into
batched ``generate`` calls.  Results come back on one queue and resolve the callers' futures.
"""
from __future__ import annotations

import itertools
import multiprocessing as mp
import threading
import traceback
from concurrent.futures import Future
from typing import Callable, List, Optional, Sequence

from .batching import page_vit_tokens


def b200_worker(rank: int, weights_dir: str = "./weights/DotsOCR", preset: Optional[str] = None, max_batch: int = 64):
    """Default worker factory: the engine on ``cuda:<rank>`` behind a request batcher."""
    import torch
    from .continuous import serving_front
    from .runner import PageRunner
    torch.cuda.set_device(rank)
    return serving_front(PageRunner.from_default(device=f"cuda:{rank}", weights_dir=weights_dir, preset=preset), max_batch=max_batch)


class _Echo:
    """CPU stand-in used by the tests (must live in an importable module: workers are spawned, not forked)."""

    def __init__(self, rank: int, delay: float, fail_on: str):
        self.rank, self.delay, self.fail_on = rank, delay, fail_on

    def infer(self, image, prompt, max_new_tokens=512, sampling=None):
        import time
        time.sleep(self.delay)
        if "die" in prompt:
            import os
            os._exit(3)                                # a worker lost to a device fault
        if self.fail_on and self.fail_on in prompt:
            raise ValueError(f"worker {self.rank} refuses {prompt!r}")
        out = f"rank{self.rank}|{getattr(image, 'size', image)}|{prompt}|{max_new_tokens}"
        return out if sampling is None else f"{out}|{sampling!r}"


def echo_worker(rank: int, delay: float = 0.0, fail_on: str = "", die_at_start: int = -1):
    if rank == die_at_start:
        raise RuntimeError(f"worker {rank} cannot start")
    return _Echo(rank, delay, fail_on)


def _portable(exc: BaseException) -> BaseException:
    import pickle
    try:
        pickle.loads(pickle.dumps(exc))
        return exc
    except Exception:
        return RuntimeError(f"{type(exc).__name__}: {exc}")


def _worker_main(rank: int, factory: Callable, factory_args: tuple, req_q, res_q) -> None:
    try:
        runner = factory(rank, *factory_args)
    except Exception as e:          # noqa: BLE001 -- reported to the front process, which raises it
        res_q.put((rank, None, False, RuntimeError(f"worker {rank} failed to start: {type(e).__name__}: {e}\n"
                                                   + traceback.format_exc(limit=5))))
        return
    res_q.put((rank, None, True, "ready"))
    submit = getattr(runner, "submit", None)
    pool = None
    if submit is None:
        from concurrent.futures import ThreadPoolExecutor
        pool = ThreadPoolExecutor(max_workers=64, thread_name_prefix=f"dots-w{rank}")
        submit = lambda im, pr, n, **kw: pool.submit(runner.infer, im, pr, max_new_tokens=n, **kw)        # noqa: E731

    def done(req_id, fut):
        e = fut.exception()
        res_q.put((rank, req_id, e is None, fut.result() if e is None else _portable(e)))

    while True:
        item = req_q.get()
        if item is None:
            break
        req_id, image, prompt, n_new, sampling = item
        try:
            kw = {} if sampling is None else {"sampling": sampling}        # only a request that carries parameters passes them on
            submit(image, prompt, n_new, **kw).add_done_callback(lambda f, r=req_id: done(r, f))
        except Exception as e:      # noqa: BLE001
            res_q.put((rank, req_id, False, _portable(e)))
    if pool is not None:
        pool.shutdown(wait=True)
    close = getattr(runner, "close", None)
    if close is not None:
        close()


class MultiGpuRunner:
    def __init__(self, n_workers: int, factory: Callable = b200_worker, factory_args: Sequence = (), start_timeout: float = 600.0):
        assert n_workers >= 1
        ctx = mp.get_context("spawn")              # never fork a process that may hold a CUDA context
        self._res = ctx.Queue()
        self._reqs = [ctx.Queue() for _ in range(n_workers)]
        self._procs = [ctx.Process(target=_worker_main, args=(k, factory, tuple(factory_args), self._reqs[k], self._res),
                                   name=f"dots-b200-gpu{k}", daemon=True) for k in range(n_workers)]
        for p in self._procs:
            p.start()
        self._lock = threading.Lock()
        self._ids = itertools.count(1)
        self._pending = {}                          # req_id -> (future, worker, weight)
        self._load = [0] * n_workers                # outstanding ViT tokens per worker
        self.served = [0] * n_workers               # pages answered per worker (observability / tests)
        self._closed = False
        self._dead = set()                          # workers whose process has exited unexpectedly
        ready = 0
        try:
            while ready < n_workers:
                rank, req_id, ok, payload = self._res.get(timeout=start_timeout)
                if not ok:
                    raise payload
                ready += 1
        except BaseException:
            self._terminate()
            raise
        self._collector = threading.Thread(target=self._collect, name="dots-b200-collector", daemon=True)
        self._collector.start()

    # -- caller side ------------------------------------------------------------------------------------------------
    def submit(self, image, prompt: str, max_new_tokens: int = 512, sampling=None) -> Future:
        """sampling: None (greedy) or a ``SamplingParams``; a missing seed is drawn here, in the front process."""
        if self._closed:
            raise RuntimeError("MultiGpuRunner is closed")
        weight = max(1, page_vit_tokens(image))
        fut: Future = Future()
        with self._lock:
            alive = [i for i in range(len(self._load)) if i not in self._dead]
            if not alive:
                raise RuntimeError("every GPU worker process has died")
            k = min(alive, key=lambda i: (self._load[i], i))
            rid = next(self._ids)
            self._pending[rid] = (fut, k, weight)
            self._load[k] += weight
        self._reqs[k].put((rid, image, prompt, int(max_new_tokens), None if sampling is None else sampling.with_seed()))
        return fut

    def infer(self, image, prompt: str, max_new_tokens: int = 512, sampling=None) -> str:
        return self.submit(image, prompt, max_new_tokens, sampling).result()

    def infer_batch(self, images, prompts, max_new_tokens: int = 512, sampling=None) -> List[str]:
        futs = [self.submit(im, pr, max_new_tokens, sampling) for im, pr in zip(images, prompts)]
        return [f.result() for f in futs]

    def close(self, timeout: float = 10.0) -> None:
        if self._closed:
            return
        self._closed = True
        for q in self._reqs:
            q.put(None)
        for p in self._procs:
            p.join(timeout)
        self._res.put(None)
        self._collector.join(timeout)
        self._terminate()

    # -- internals --------------------------------------------------------------------------------------------------
    def _terminate(self) -> None:
        for p in self._procs:
            if p.is_alive():
                p.terminate()

    def _reap(self) -> None:
        """A worker process that exited while it owed answers: fail those callers instead of letting them wait forever."""
        for k, p in enumerate(self._procs):
            if k in self._dead or p.is_alive() or self._closed:
                continue
            with self._lock:
                self._dead.add(k)
                lost = [(rid, v[0]) for rid, v in self._pending.items() if v[1] == k]
                for rid, _ in lost:
                    del self._pending[rid]
                self._load[k] = 0
            for _, fut in lost:
                fut.set_exception(RuntimeError(f"GPU worker {k} exited with code {p.exitcode} while serving this page"))

    def _collect(self) -> None:
        import queue as _queue
        import time as _time
        last_reap = _time.monotonic()
        while True:
            # look for dead workers every 0.5 s whether or not results keep arriving (a steady stream from the survivors must
            # not hide a worker that died owing answers)
            if _time.monotonic() - last_reap >= 0.5:
                self._reap()
                last_reap = _time.monotonic()
            try:
                item = self._res.get(timeout=0.5)
            except _queue.Empty:
                continue
            if item is None:
                return
            rank, rid, ok, payload = item
            with self._lock:
                fut, k, weight = self._pending.pop(rid, (None, rank, 0))
                self._load[k] -= weight
                self.served[k] += 1
            if fut is None:
                continue
            if ok:
                fut.set_result(payload)
            else:
                fut.set_exception(payload)
