#!/usr/bin/env python
"""Headline benchmark: pages/sec for the dots.ocr page-parsing hot path on B200.

One "step" = one pass of the whole hot path over one batch of synthetic pages on every rank:
ViT encode (42 blocks, 5476 patch tokens per 1024x1024 page) -> embed + image scatter -> LLM prefill
(T = 1625) -> greedy decode of NEW_TOKENS tokens (EOS disabled: random weights never emit it).
Workload = BASELINE.json configs[2] ("batch=64 synthetic 1024x1024 pages, bf16, greedy, 1xB200");
at N GPUs every rank runs its own 64-page shard (pages are independent: weak scaling, no collective
on the data path; configs[3] = 512 pages on 8 GPUs).

    python bench.py --gpus 1 --steps 3 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference            # the HF/PyTorch CPU path (oracle port) on the host cores
    python bench.py --gpus 1 --steps 3 --warmup 3 --dump-outputs DIR    # also write the last timed step's outputs to DIR

Prints ONE JSON line (rank 0).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

PAGE_HW = (1024, 1024)
TEXT_TOKENS = 256
METRIC = "pages/sec (1024x1024 doc images, greedy)"
NCCL_LOG_PREFIX = os.path.join(tempfile.gettempdir(), "dots_ocr_b200_nccl_debug.")
DUMP_BYTES = 64 << 20           # --dump-outputs: at most this much in all, half for the sequences, half for the embedding sample


def _peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return dict(hbm_gbs=float(p["hbm_gbs"]), tf_burst=float(p["bf16_tflops"]),
                    tf_sustained=float(p.get("bf16_tflops_sustained", p["bf16_tflops"])), source="measured")
    except Exception:
        return dict(hbm_gbs=6650.0, tf_burst=1590.0, tf_sustained=1400.0, source="fallback")


def _page_tokens(cfg):
    from dots_ocr_b200.utils.image_utils import token_counts
    return token_counts(*PAGE_HW, patch=cfg.vision.patch_size, merge=cfg.vision.spatial_merge_size)


def _prompt_len():
    from dots_ocr_b200.utils.image_utils import token_counts
    return token_counts(*PAGE_HW)[1] + TEXT_TOKENS


def _prompt_ids(cfg, batch, t_img, seed=7):
    import torch
    g = torch.Generator().manual_seed(seed)
    vocab_text = min(cfg.text.vocab_size, 151643)
    front = TEXT_TOKENS // 2
    rows = []
    for _ in range(batch):
        txt = torch.randint(0, vocab_text, (TEXT_TOKENS,), generator=g)
        rows.append(torch.cat([txt[:front], torch.full((t_img,), cfg.image_token_id), txt[front:]]))
    return torch.stack(rows)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def usable_cpu_threads() -> int:
    """Host threads this process may really use: the scheduler affinity mask, capped by a cgroup CPU quota if one is set
    (os.cpu_count() reports the machine, not the container: oversubscribing a quota makes PyTorch's CPU path crawl)."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:
            quota, period = f.read().split()[:2]
        if quota != "max":
            n = min(n, max(1, int(float(quota) / float(period))))
    except Exception:
        try:
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                n = min(n, max(1, q // per))
        except Exception:
            pass
    return max(1, n)


# --------------------------------------------------------------------------------------- CPU arm
def cpu_reference(new_tokens: int, threads: int, ck=None, cfg=None):
    """The reference's HF CPU float32 path (oracle port: restated ViT + HF Qwen2ForCausalLM.generate, greedy) on the host
    cores: ONE page of the benchmark workload at FULL depth (42 ViT blocks, 28 decoder layers, `new_tokens` greedy steps with
    a KV cache), timed directly from pixel_values to the last token -- no per-layer extrapolation.  About a minute on 16
    threads.  `ck`: an already generated bf16 checkpoint (any device) to convert, else the seeded synthetic one is drawn here."""
    import torch
    from dots_ocr_b200 import config, weights
    from oracle.model import DotsOracle
    torch.set_num_threads(threads)
    full = cfg or config.full()
    s_vit, t_img = _page_tokens(full)
    t0 = time.perf_counter()
    if ck is None:
        ck = weights.make_synthetic_checkpoint(full, 0, "random", device="cpu")
    else:
        ck = {k: v.to("cpu") for k, v in ck.items()}
    orc = DotsOracle(full, ck, torch.float32, "cpu")
    del ck
    t_build = time.perf_counter() - t0
    g = torch.Generator().manual_seed(1234)
    pv = torch.randn(s_vit, full.vision.patch_dim, generator=g)
    from dots_ocr_b200.utils.image_utils import vit_grid
    gh, gw = vit_grid(*PAGE_HW)
    grid = torch.tensor([[1, gh, gw]])
    ids = _prompt_ids(full, 1, t_img)
    with torch.no_grad():
        # warm-up: thread pool, allocator and code paths, on a sliver of the work (one 8x8-patch image, 4 tokens)
        wpv = torch.randn(64, full.vision.patch_dim, generator=g)
        wids = torch.cat([ids[0, :4], torch.full((16,), full.image_token_id), ids[0, -4:]]).unsqueeze(0)
        orc.generate(wids, pixel_values=wpv, image_grid_thw=torch.tensor([[1, 8, 8]]), max_new_tokens=4)
        t0 = time.perf_counter()
        emb = orc.inputs_embeds(ids, pv, grid)                                   # ViT (42 blocks) + embed + masked_scatter
        t_vit = time.perf_counter() - t0
        out = orc.llm.generate(inputs_embeds=emb, attention_mask=torch.ones_like(ids), max_new_tokens=new_tokens, min_new_tokens=new_tokens,
                               do_sample=False, pad_token_id=0)
        total = time.perf_counter() - t0
    assert out.shape[1] == new_tokens, out.shape
    return dict(pages_per_sec=1.0 / total, seconds=total, t_vit=t_vit, t_llm=total - t_vit, t_build=t_build,
                sample=(f"1 page {PAGE_HW[0]}x{PAGE_HW[1]} at full depth (42 ViT blocks + 28 decoder layers, fp32, {threads} threads), prefill T={ids.shape[1]} + "
                        f"{new_tokens} greedy tokens through HF generate, timed directly ({total:.1f} s)"))


def run_reference(args):
    """`--impl reference`: the CPU arm alone.  The K timed steps together process exactly ONE page (a step = 1/K of that
    page's work), so ms_per_step x steps is the time really spent; warm-up is a sliver of work, not W more pages."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = usable_cpu_threads()
    r = cpu_reference(args.new_tokens, threads)
    v = r["pages_per_sec"]
    cfgd = _config(args, 1)
    cfgd["reference_arm"] = (f"one full-depth page timed directly in {r['seconds']:.1f} s; the {args.steps} reported steps are equal shares of that "
                             "page (a CPU page costs about a minute: K whole pages would not fit the time box); warm-up = one 8x8-patch image + 4 tokens")
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": "pages/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1000.0 * r["seconds"] / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": cfgd,
            "cpu_baseline": {"value": v, "unit": "pages/s", "cores": threads, "kind": "port", "sample": r["sample"],
                             "t_vit_s": round(r["t_vit"], 2), "t_llm_s": round(r["t_llm"], 2)},
            "e2e": {"value": v, "unit": "pages/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def _config(args, world):
    return {"workload": f"batch={args.batch} synthetic {PAGE_HW[0]}x{PAGE_HW[1]} pages per GPU, ViT encode + prefill(T={_prompt_len()}) + "
                        f"greedy decode N={args.new_tokens} (BASELINE configs[2]; x{world} GPUs = configs[3] sharding)",
            "pages_per_gpu": args.batch, "global_pages": args.batch * world, "new_tokens": args.new_tokens,
            "prompt_tokens": _prompt_len(), "parallelism": f"dp{world} (page shards, model replicated, no collective)",
            "l2": "inputs larger than L2 (pixel_values 824 MB fp32 per step; weights 6.1 GB streamed every decode step)",
            "weights": "synthetic N(0,0.02) seed 0, real architecture (ViT 1.26B + LLM 1.78B)"}


# --------------------------------------------------------------------------------------- GPU arm
def ids_checksum(new_ids) -> str:
    """Order-sensitive 64-bit checksum of a [B, N] block of generated ids (tests/test_bench_config_gpu.py reproduces it from the
    ids it has verified against the oracle; tests/golden/bench_ids_checksum.json pins it)."""
    import torch
    x = new_ids.to(torch.int64).reshape(-1).cpu()
    idx = torch.arange(1, x.numel() + 1, dtype=torch.int64)
    mod = (1 << 61) - 1
    h = int(((x + 1) * (idx % 1000003 + 7919)).remainder(mod).sum().item()) % mod
    return f"{h:016x}"


def dump_outputs(out, dump_dir: str) -> dict:
    """Write what one generate() call returned under `dump_dir`: sequences.npy [B, T + N] (prompt + generated ids, exact in
    float64), image_embeds.npy (float32, a sample of rows drawn with a fixed seed) and image_embeds_rows.npy (their indices).
    The sample depends on the shape alone, so two builds run with the same arguments can be compared array for array."""
    import numpy as np
    import torch
    seq = out.sequences.cpu().numpy().astype(np.float64)
    assert seq.nbytes <= DUMP_BYTES // 2, f"sequences are {seq.nbytes} bytes: too large to dump"
    emb = out.image_embeds
    n, h = emb.shape
    rows = torch.randperm(n, generator=torch.Generator().manual_seed(2718))[:min(n, (DUMP_BYTES // 2) // (4 * h + 8))].sort().values
    arrays = {"sequences": seq, "image_embeds": emb[rows.to(emb.device)].float().cpu().numpy(),
              "image_embeds_rows": rows.numpy().astype(np.float64)}
    os.makedirs(dump_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(dump_dir, f"{name}.npy"), a)
    return {"dir": dump_dir, "shapes": {name: list(a.shape) for name, a in arrays.items()}}


def make_workload(cfg, batch: int, rank: int, dev):
    """The benchmark's synthetic pages and prompts (shared with the parity test of this exact workload): pixel_values ~ N(0, 1)
    drawn on the device with seed 1234 + rank, prompts = 128 text ids + image pads + 128 text ids (seed 7)."""
    import torch
    from dots_ocr_b200.utils.image_utils import vit_grid
    s_vit, t_img = _page_tokens(cfg)
    gh, gw = vit_grid(*PAGE_HW)
    grid = torch.tensor([[1, gh, gw]] * batch)
    g = torch.Generator(device=dev).manual_seed(1234 + rank)
    pv = torch.randn((batch * s_vit, cfg.vision.patch_dim), generator=g, device=dev)
    ids = _prompt_ids(cfg, batch, t_img)
    return pv, grid, ids


def _decode_traffic():
    """DRAM bytes of one decode step from the committed ncu capture (profiles/decode_traffic_*.json), or None."""
    import glob
    best = None
    for f in sorted(glob.glob(os.path.join(ROOT, "profiles", "decode_traffic_*.json"))):
        try:
            with open(f) as fh:
                best = dict(json.load(fh), file=os.path.basename(f))
        except Exception:
            pass
    return best


def run_gpu(args):
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world} (launch with torch.distributed.run)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # NCCL_DEBUG is left as the caller set it; its output is routed to a file (NCCL_DEBUG_FILE, one per process) unless the caller
        # chose one, because NCCL keeps logging at process exit and the JSON must stay the LAST line of stdout
        if os.environ.get("NCCL_DEBUG") and not os.environ.get("NCCL_DEBUG_FILE"):
            os.environ["NCCL_DEBUG_FILE"] = NCCL_LOG_PREFIX + "%h.%p.log"
        dist.init_process_group("nccl", device_id=dev)

    from dots_ocr_b200 import config, weights, ops
    from dots_ocr_b200.engine import Engine
    if args.attn_impl:
        ops.ATTN_IMPL = args.attn_impl
    if args.no_pdl:
        ops.set_pdl(False)
    if args.gemm_pair is not None:
        ops.set_gemm_pair(bool(args.gemm_pair))
    cfg = config.PRESETS[args.preset]()
    ck = weights.make_synthetic_checkpoint(cfg, 0, "random", device=dev)
    eng = Engine(cfg, ck, dev)
    if args.decode_mode:
        eng.decode_mode = args.decode_mode
    if args.attn_splits:
        eng.attn_splits = args.attn_splits
    ck_cpu = {k: v.to("cpu") for k, v in ck.items()} if (world == 1 and not args.no_cpu_baseline and args.preset == "full") else None
    del ck
    torch.cuda.empty_cache()

    B, N = args.batch, args.new_tokens
    pv_dev, grid, ids = make_workload(cfg, B, rank, dev)
    ids_dev = ids.to(dev)
    pv_host = torch.empty(pv_dev.shape, dtype=torch.float32, pin_memory=True)
    pv_host.copy_(pv_dev)
    ids_host = ids.pin_memory()
    last = {}

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step_device():
        last["out"] = eng.generate(ids_dev, pixel_values=pv_dev, image_grid_thw=grid, max_new_tokens=N)

    def step_e2e():
        pv = pv_host.to(dev, non_blocking=True)
        idd = ids_host.to(dev, non_blocking=True)
        out = eng.generate(idd, pixel_values=pv, image_grid_thw=grid, max_new_tokens=N)
        last["e2e_ids"] = out.sequences[:, idd.shape[1]:].cpu()

    # third leg: the same batch as RAW uint8 pages (1024 x 1024 x 3 on pinned host memory): H2D of 3.1 MB per page, then the whole
    # image processor on the GPU (bicubic resize to 1036 x 1036 bit-identical to the CPU processor, rescale, normalise, patchify)
    gu8 = torch.Generator().manual_seed(4321 + rank)
    pages_host = [torch.randint(0, 256, (PAGE_HW[0], PAGE_HW[1], 3), generator=gu8, dtype=torch.uint8).pin_memory() for _ in range(B)]

    def step_e2e_u8():
        pgs = [p.to(dev, non_blocking=True) for p in pages_host]
        idd = ids_host.to(dev, non_blocking=True)
        out = eng.generate(idd, pages_u8=pgs, max_new_tokens=N)
        last["u8_ids"] = out.sequences[:, idd.shape[1]:].cpu()

    per_step = {}

    def timed(fn, k, name=None):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        marks = []
        for _ in range(k):
            fn()
            marks.append(torch.cuda.Event(enable_timing=True))
            marks[-1].record()
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
        # per-step times of this rank (diagnostic only: the reported number is the whole region, max over ranks)
        per_step[name or fn.__name__] = [round(a.elapsed_time(b), 1) for a, b in zip([e0] + marks[:-1], marks)]
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    for _ in range(args.warmup):
        step_device()
    # ---- timed region 1 (`value`): inputs resident in HBM, no per-launch instrumentation (events between PDL-chained
    #      kernels would serialise them); only the two always-on events around each decode loop
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    l0 = eng.launches
    eng.decode_log.clear()
    ms_total = timed(step_device, args.steps)
    launches = eng.launches - l0
    dec_log = list(eng.decode_log)
    new_ids = last["out"].sequences[:, ids_dev.shape[1]:]
    checksum = ids_checksum(new_ids)
    dumped = dump_outputs(last["out"], args.dump_outputs) if args.dump_outputs and rank == 0 else None
    # ---- timed region 2 (`e2e`): the public call with pinned host buffers, H2D and D2H inside
    ms_e2e = None
    if not args.no_e2e:
        step_e2e()
        ms_e2e = timed(step_e2e, args.steps)
        assert ids_checksum(last["e2e_ids"]) == checksum, "host-buffer leg produced different ids than the device-resident leg"
    ms_u8 = None
    if not args.no_e2e:
        step_e2e_u8()
        ms_u8 = timed(step_e2e_u8, args.steps)
    clocks = sampler.stop() if rank == 0 else None
    # ---- separate pass: CUDA events around every prefill-side launch (kernel classes and their share of a step)
    ops.PROFILE = prof = []
    ms_prof = timed(step_device, 1, "instrumented_step")
    ops.PROFILE = None

    pages = B * world * args.steps
    value = pages / (ms_total / 1e3)
    e2e_v = pages / (ms_e2e / 1e3) if ms_e2e else None
    h2d = pv_host.numel() * 4 + ids_host.numel() * 8
    d2h = B * N * 8

    peaks = _peaks()
    torch.cuda.synchronize()
    # ---- roofline of the dominant phase: the decode loop (HBM-bound), from the events around the decode loops of the timed steps
    roof = None
    dec_ms_per_step_total = 0.0
    if dec_log:
        by = sum(d[0] for d in dec_log)
        steps_dec = sum(d[1] for d in dec_log)
        ms = sum(d[2].elapsed_time(d[3]) for d in dec_log)
        dec_ms_per_step_total = ms / len(dec_log)
        ach = by / (ms / 1e3) / 1e9
        tr = _decode_traffic()
        roof = {"kernel": ("decode step = one CUDA-graph launch: " + ("cluster split-K tcgen05 GEMMs (reduction, residual, RMSNorm on chip) + "
                           "cluster-merged KV attention + gate|up SwiGLU GEMM + lm_head + argmax" if eng._decode_plan(B)["mode"] == "fused" else
                           "skinny swap-AB tcgen05 GEMMs (split-K) + KV attention + finalize kernels" +
                           (", operands pre-tiled in HBM and bulk-copied" if eng._decode_plan(B)["mode"] == "tiled" else ""))),
                "bound": "hbm", "achieved": round(ach, 1), "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": round(ach / peaks["hbm_gbs"], 4),
                "peak_source": peaks["source"] + " (copy bandwidth)",
                "launch": "one decode step (graph replay)", "algorithmic_bytes_per_launch": round(by / max(1, steps_dec)),
                "avg_launch_ms": round(ms / max(1, steps_dec), 4), "launches": steps_dec, "share_of_step": round(ms / ms_total, 4),
                "traffic": (tr or {}).get("dram_bytes_per_step"), "traffic_source": (tr or {}).get("file")}
    # ---- prefill-side kernel classes from the instrumented pass
    agg = {}
    for name, work, e0, e1 in prof:
        a = agg.setdefault(name, [0.0, 0.0, 0])
        a[0] += work; a[1] += e0.elapsed_time(e1); a[2] += 1
    by_kernel = {}
    for name, (work, ms, n) in agg.items():
        by_kernel[name] = {"launches": n, "ms": round(ms, 3), "share_of_step": round(ms / ms_prof, 4)}
    roof_gemm = roof_attn = None
    if "gemm_bf16_tcgen05" in agg:
        fl, ms, n = agg["gemm_bf16_tcgen05"]
        ach = fl / (ms / 1e3) / 1e12
        roof_gemm = {"kernel": "gemm2_bf16_tcgen05_kernel / gemm_bf16_tcgen05_kernel (ViT + LLM prefill linears)", "bound": "tensor",
                     "achieved": round(ach, 1), "peak": peaks["tf_sustained"], "unit": "TFLOP/s", "frac": round(ach / peaks["tf_sustained"], 4),
                     "peak_source": f"{peaks['source']} (sustained cuBLAS bf16; burst {peaks['tf_burst']})", "launches": n,
                     "avg_launch_ms": round(ms / n, 4), "share_of_step": round(ms / ms_prof, 4)}
    if "attn_fwd_vit" in agg:
        fl, ms, n = agg["attn_fwd_vit"]
        ach = fl / (ms / 1e3) / 1e12
        roof_attn = {"kernel": "attn_fwd_tcgen05_kernel<0> (ViT bidirectional attention)", "bound": "tensor", "achieved": round(ach, 1),
                     "peak": peaks["tf_sustained"], "unit": "TFLOP/s", "frac": round(ach / peaks["tf_sustained"], 4), "launches": n,
                     "avg_launch_ms": round(ms / n, 4), "share_of_step": round(ms / ms_prof, 4)}

    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return
    threads = usable_cpu_threads()
    cpu = None
    if ck_cpu is not None:
        try:
            r = cpu_reference(N, threads, ck=ck_cpu, cfg=cfg)
            cpu = {"value": r["pages_per_sec"], "unit": "pages/s", "cores": threads, "kind": "port", "sample": r["sample"],
                   "t_vit_s": round(r["t_vit"], 2), "t_llm_s": round(r["t_llm"], 2)}
        except Exception as e:      # the baseline must never take the GPU number down with it
            cpu = {"value": None, "unit": "pages/s", "cores": threads, "kind": "port", "sample": f"failed: {e!r}"}
    golden = None
    try:
        with open(os.path.join(ROOT, "tests", "golden", "bench_ids_checksum.json")) as f:
            golden = json.load(f).get(f"b{B}_n{N}_p{PAGE_HW[0]}_rank0")
    except Exception:
        pass
    line = {"metric": METRIC, "value": round(value, 3), "unit": "pages/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": round(ms_total / args.steps, 2), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "bf16", "data": "synthetic", "config": _config(args, world),
            "e2e": {"value": round(e2e_v, 3) if e2e_v else None, "unit": "pages/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
            "e2e_u8": {"value": round(pages / (ms_u8 / 1e3), 3) if ms_u8 else None, "unit": "pages/s",
                       "h2d_bytes_per_step": B * PAGE_HW[0] * PAGE_HW[1] * 3 + ids_host.numel() * 8, "d2h_bytes_per_step": d2h,
                       "input": "raw uint8 pages on pinned host memory; resize + rescale + normalise + patchify on the GPU"},
            "gpu_launches": launches, "clocks": clocks, "roofline": roof, "roofline_gemm": roof_gemm, "roofline_vit_attention": roof_attn,
            "phases_ms": {"decode_loop": round(dec_ms_per_step_total, 2), "step": round(ms_total / args.steps, 2),
                          "instrumented_step": round(ms_prof, 2), "per_step_rank0": per_step},
            "kernels": by_kernel, "ids_checksum": {"value": checksum, "golden": golden, "matches_golden": (checksum == golden) if golden else None},
            "cpu_baseline": cpu}
    if dumped:
        line["outputs_dumped"] = dumped
    if world > 1:
        # NCCL's log of this run (routed to files above) is echoed on STDERR so that whoever reads the run's output still sees the
        # communicator's rank count; stdout carries nothing after the JSON line
        if str(os.environ.get("NCCL_DEBUG_FILE", "")).startswith(NCCL_LOG_PREFIX):
            import glob
            for f in sorted(glob.glob(f"{NCCL_LOG_PREFIX}*.{os.getpid()}.log")):
                try:
                    with open(f) as fh:
                        sys.stderr.write(fh.read())
                except OSError:
                    pass
            sys.stderr.flush()
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--new-tokens", dest="new_tokens", type=int, default=512)
    ap.add_argument("--preset", default="full")
    ap.add_argument("--page", type=int, default=1024, help="synthetic page edge in pixels (1024 = the headline workload; 1960 with "
                    "--batch 4 --new-tokens 2048 = BASELINE configs[4], the long-context case)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", dest="no_e2e", action="store_true", help="skip the host-buffer leg (profiling runs only)")
    ap.add_argument("--gemm-pair", dest="gemm_pair", type=int, default=None, choices=[0, 1],
                    help="CTA-pair (cta_group::2) kernel for the large prefill GEMMs (default: the library default)")
    ap.add_argument("--no-pdl", dest="no_pdl", action="store_true", help="plain stream order between kernels (A/B runs)")
    ap.add_argument("--decode-mode", dest="decode_mode", default=None, choices=["tiled", "fused", "perop"],
                    help="decode layer variant (default: the engine default); see Engine.decode_mode")
    ap.add_argument("--attn-splits", dest="attn_splits", type=int, default=0, help="force the key-split count of the decode attention")
    ap.add_argument("--attn-impl", dest="attn_impl", default=None, choices=["tc", "mma"])
    ap.add_argument("--dump-outputs", dest="dump_outputs", default=None, metavar="DIR",
                    help="after the timed steps, write what the last one returned (rank 0's pages) to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the GPU path")
    global PAGE_HW
    PAGE_HW = (args.page, args.page)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
