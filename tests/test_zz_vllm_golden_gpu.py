"""The CUDA vision path against vectors produced by vLLM's own DotsVisionTransformer (fp32, CPU;
tests/golden/make_vllm_vision_golden.py) -- the same comparison test_engine_gpu.py makes against the oracle restatement,
with the third-party implementation's numbers as the target.  Tolerance: bf16 pipeline vs fp32 target, 3e-2 of the
tensor's range per layer (as in test_vision_tower_layers)."""
import os
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
TOL = 3e-2


def test_engine_vision_tower_matches_vllm_vectors():
    from dots_ocr_b200 import config, weights
    from dots_ocr_b200.engine import Engine
    sys.path.insert(0, GOLD)
    import make_vllm_vision_golden as G
    d = np.load(os.path.join(GOLD, "vllm_vision_tiny.npz"))
    cfg = config.tiny()
    eng = Engine(cfg, weights.make_synthetic_checkpoint(cfg, G.SEED_W, "random"), DEV)
    for name, grids in G.CASES.items():
        pv, grid = G.case_inputs(cfg, grids)
        out, layers = eng.encode_images(pv.to(DEV), grid, return_layers=True)
        want = [f"{name}_patch_embed"] + [f"{name}_block_{i}" for i in range(cfg.vision.num_hidden_layers)]
        assert len(layers) == len(want)
        for i, (a, k) in enumerate(zip(layers, want)):
            a, b = a.float().cpu()[torch.from_numpy(d[f"{k}_rows"])], torch.from_numpy(d[k])
            assert a.shape == b.shape
            err = float((a - b).abs().max() / b.abs().max())
            assert err < TOL, (name, i, err)
        ref = torch.from_numpy(d[f"{name}_image_embeds"])
        err = float((out.float().cpu() - ref).abs().max() / ref.abs().max())
        assert err < TOL, (name, err)
