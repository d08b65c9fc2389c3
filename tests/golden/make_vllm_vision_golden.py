"""Golden vectors from vLLM's OWN ``DotsVisionTransformer`` (vllm/model_executor/models/dots_ocr.py:476-611 -- the
implementation the reference tells users to serve with, README "vLLM inference"), executed in THIS container on CPU in fp32
with the seeded synthetic tiny-config weights.  They pin the plain-PyTorch restatement in ``oracle/vision.py``.

    python tests/golden/make_vllm_vision_golden.py      # -> tests/golden/vllm_vision_tiny.npz

How the CUDA build of vLLM is made to run its model code on a GPU-less box (nothing is patched inside vLLM):
  * ``vllm.platforms.current_platform`` is set to ``CpuPlatform()`` before any model module is imported (platform
    detection finds no device here and would otherwise refuse to build a config);
  * a world-size-1 gloo process group stands in for tensor parallelism;
  * every Linear gets ``cpu_linear = torch.nn.functional.linear``, vLLM's own fallback GEMM
    (vllm/model_executor/layers/utils.py:234) -- the tuned CPU kernels live in a vllm._C this build does not carry;
  * checkpoint tensors are copied by name; ``mlp.fc13`` = cat(fc1, fc3), the stacking vLLM's loader performs
    (dots_ocr.py:359-362).
RMSNorm runs vLLM's native implementation, attention its torch-SDPA path, rotary its native apply.

Outputs per case: the patch-embed output, every block's output, and the merged image embeddings.  The merged embeddings are
stored whole; each per-layer output keeps a seeded sample of TAP_KEEP of its rows, with their indices under ``<name>_rows``,
so that the file stays below 1 MB.
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

CASES = {                       # name -> image grids (t, h, w) in 14-px patches; h, w even (2x2 merge)
    "two_pages": [(1, 8, 12), (1, 6, 6)],
    "three_pages": [(1, 16, 16), (1, 4, 10), (1, 2, 2)],
}
SEED_W, SEED_X = 0, 3
WIDE_GRIDS = [(1, 4, 6), (1, 2, 2)]      # full-width case: 1536 wide, 12 heads x 128, SwiGLU 4224, two blocks
TAP_KEEP, SEED_ROWS = 0.25, 17


def sample_rows(out, name, t):
    """Store a seeded, sorted sample of the rows of the per-layer output `t` as `name`, and their indices as `name`_rows."""
    t = t.reshape(-1, t.shape[-1]).numpy().astype(np.float32)
    n = t.shape[0]
    rows = np.sort(np.random.default_rng([SEED_ROWS, n, t.shape[1]]).choice(n, max(1, round(n * TAP_KEEP)), replace=False))
    out[name], out[f"{name}_rows"] = t[rows], rows.astype(np.int64)


def wide_config():
    """The real tower's widths (so the 12-way head split and the 4x1536 merger are exercised) with two blocks."""
    from dots_ocr_b200 import config
    return config.DotsConfig(vision=config.VisionConfig(num_hidden_layers=2), name="dots.ocr-wide-vision")


def vision_only_checkpoint(cfg, seed):
    """Seeded bf16-rounded vision-tower tensors (same value recipe as weights.make_synthetic_checkpoint, vision part only:
    the full-width decoder would add 1.8 B parameters this case does not need)."""
    from dots_ocr_b200 import weights
    g = torch.Generator().manual_seed(seed)
    out = {}
    for name, shape, kind in weights._specs(cfg):
        if not name.startswith("vision_tower."):
            break
        w = torch.randn(shape, generator=g)
        out[name] = ((1.0 + 0.1 * w) if kind == "norm" else 0.02 * w).to(torch.bfloat16)
    return out


def case_inputs(cfg, grids, seed=SEED_X):
    g = torch.Generator().manual_seed(seed)
    S = sum(t * h * w for t, h, w in grids)
    return torch.randn(S, cfg.vision.patch_dim, generator=g), torch.tensor(grids)


def build_vllm_tower(cfg, ckpt, ctx=None):
    if ctx is None:
        import vllm.platforms as P
        from vllm.platforms.cpu import CpuPlatform
        P.current_platform = CpuPlatform()
        from vllm.config import VllmConfig, set_current_vllm_config
        from vllm.distributed import init_distributed_environment, initialize_model_parallel
        vc = VllmConfig()
        ctx = set_current_vllm_config(vc)
        ctx.__enter__()
        init_distributed_environment(world_size=1, rank=0, distributed_init_method="tcp://127.0.0.1:29591", local_rank=0,
                                     backend="gloo")
        initialize_model_parallel(1, 1)
    from vllm.model_executor.models.dots_ocr import DotsVisionTransformer
    from vllm.transformers_utils.configs.dotsocr import DotsVisionConfig
    v = cfg.vision
    vcfg = DotsVisionConfig(embed_dim=v.embed_dim, hidden_size=v.hidden_size, intermediate_size=v.intermediate_size,
                            num_hidden_layers=v.num_hidden_layers, num_attention_heads=v.num_attention_heads,
                            num_channels=v.num_channels, patch_size=v.patch_size, spatial_merge_size=v.spatial_merge_size,
                            temporal_patch_size=v.temporal_patch_size, rms_norm_eps=v.rms_norm_eps)
    tower = DotsVisionTransformer(vcfg, quant_config=None, prefix="vision_tower").float().eval()
    src = {k[len("vision_tower."):]: w.float() for k, w in ckpt.items() if k.startswith("vision_tower.")}
    used = set()
    with torch.no_grad():
        for name, p in tower.named_parameters():
            if name.endswith("mlp.fc13.weight"):
                a, b = name.replace("fc13", "fc1"), name.replace("fc13", "fc3")
                w = torch.cat([src[a], src[b]], 0)
                used.update((a, b))
            else:
                w = src[name]
                used.add(name)
            assert w.shape == p.shape, (name, tuple(w.shape), tuple(p.shape))
            p.copy_(w)
    assert used == set(src), sorted(set(src) - used)
    for mod in tower.modules():
        if hasattr(mod, "quant_method") and hasattr(mod, "weight"):
            mod.cpu_linear = torch.nn.functional.linear
    return tower, ctx


def run_tower(tower, pv, grid):
    taps = {}
    hooks = [tower.patch_embed.register_forward_hook(lambda m, i, o: taps.__setitem__("patch_embed", o.detach().clone()))]
    for li, blk in enumerate(tower.blocks):
        hooks.append(blk.register_forward_hook(lambda m, i, o, li=li: taps.__setitem__(f"block_{li}", o.detach().clone())))
    with torch.no_grad():
        out = tower(pv, grid_thw=grid.tolist())
    for h in hooks:
        h.remove()
    return out, taps


def main():
    torch.set_num_threads(1)
    import vllm
    from dots_ocr_b200 import config, weights
    cfg = config.tiny()
    ckpt = weights.make_synthetic_checkpoint(cfg, SEED_W, "random")
    tower, ctx = build_vllm_tower(cfg, ckpt)
    out = {"vllm_version": np.array(vllm.__version__)}
    for name, grids in CASES.items():
        pv, grid = case_inputs(cfg, grids)
        y, taps = run_tower(tower, pv, grid)
        out[f"{name}_grid"] = grid.numpy()
        out[f"{name}_image_embeds"] = y.numpy().astype(np.float32)
        for k, t in taps.items():
            sample_rows(out, f"{name}_{k}", t)
    # full-width case: a second tower object under the same vLLM context
    wcfg = wide_config()
    wck = vision_only_checkpoint(wcfg, SEED_W + 1)
    wide, _ = build_vllm_tower(wcfg, wck, ctx)
    pv, grid = case_inputs(wcfg, WIDE_GRIDS)
    y, taps = run_tower(wide, pv, grid)
    out["wide_grid"] = grid.numpy()
    out["wide_image_embeds"] = y.numpy().astype(np.float32)
    sample_rows(out, "wide_block_1", taps["block_1"])
    ctx.__exit__(None, None, None)
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "vllm_vision_tiny.npz")
    np.savez_compressed(path, **out)
    print({k: v.shape for k, v in out.items()}, os.path.getsize(path))


if __name__ == "__main__":
    main()
