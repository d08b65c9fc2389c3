"""PageRunner: image + prompt -> generated text on one GPU.

This is the body that replaces ``DotsOCRParser._load_hf_model`` / ``_inference_with_hf``
(``dots_ocr/parser.py:62-117``): processor call -> H2D -> ``generate`` -> trim prompt -> decode.
A lock serialises callers (the reference fans pages out from up to 64 threads,
``parser.py:282-290``; the C ABI is re-entrant per stream, not per engine object).
"""
from __future__ import annotations

import os
import threading
from typing import List, Optional, Sequence


from . import config as _config
from . import weights as _weights
from .processing import SyntheticTokenizer, build_inputs


class PageRunner:
    def __init__(self, engine, tokenizer, min_pixels=None, max_pixels=None, max_new_tokens_cap: int = 24000):
        self.engine = engine
        self.tokenizer = tokenizer
        self.min_pixels = min_pixels
        self.max_pixels = max_pixels
        self.cap = max_new_tokens_cap
        self._lock = threading.Lock()

    @classmethod
    def from_default(cls, device: str = "cuda:0", weights_dir: str = "./weights/DotsOCR", preset: Optional[str] = None):
        """Real checkpoint if ``./weights/DotsOCR`` exists (parser.py:67), else the seeded synthetic one."""
        if os.path.isdir(weights_dir):
            return cls.from_checkpoint(weights_dir, device)
        from .engine import Engine
        preset = preset or os.environ.get("DOTS_B200_PRESET", "full")
        cfg = _config.PRESETS[preset]()
        ckpt = _weights.make_synthetic_checkpoint(cfg, 0, "peaked", device=device)
        return cls(Engine(cfg, ckpt, device), SyntheticTokenizer(cfg))

    @classmethod
    def from_checkpoint(cls, weights_dir: str, device: str = "cuda:0", engine_factory=None):
        """A HF ``weights/DotsOCR`` directory: ``config.json`` -> DotsConfig (unsupported options refused),
        ``*.safetensors`` -> HBM (validated against the config), tokenizer + ``generation_config.json`` -> HFTokenizer.
        A directory with tensors only (no config / tokenizer files) runs with the published architecture and the
        byte-level stand-in tokenizer."""
        cfg = _config.from_hf_dir(weights_dir) if os.path.isfile(os.path.join(weights_dir, "config.json")) else _config.full()
        ckpt = _weights.load_safetensors_dir(weights_dir, device=device)
        _weights.validate_checkpoint(cfg, ckpt)
        has_tok = any(os.path.isfile(os.path.join(weights_dir, f)) for f in ("tokenizer.json", "tokenizer_config.json", "vocab.json"))
        if has_tok:
            from .processing import HFTokenizer
            tokenizer = HFTokenizer(weights_dir, image_token_id=cfg.image_token_id)
        else:
            tokenizer = SyntheticTokenizer(cfg)
        if engine_factory is None:
            from .engine import Engine
            engine_factory = Engine
        return cls(engine_factory(cfg, ckpt, device), tokenizer)

    def infer_batch(self, images: Sequence, prompts: Sequence[str], max_new_tokens: int = 512, gpu_preprocess: bool = True,
                    budgets: Optional[Sequence[int]] = None, sampling=None) -> List[str]:
        """sampling: None (greedy), one ``SamplingParams`` for every page or one per page (dots_ocr_b200/sampling.py).
        gpu_preprocess: the whole image processor (resize, rescale / normalise / patchify) on the GPU (3 B per pixel over PCIe instead of
        12); False = the reference's host processor output (fp32 pixel_values) as `generate` input."""
        n_new = max(1, min(int(max_new_tokens), self.cap))
        if gpu_preprocess:
            # host: RGB conversion only; resize + rescale + normalise + patchify run on the GPU (bit-identical to the CPU processor)
            from .processing import page_to_u8, model_image_tokens, build_text_inputs
            pages = [page_to_u8(im) for im in images]
            inputs = build_text_inputs(self.tokenizer, [model_image_tokens(int(p.shape[0]), int(p.shape[1]), self.min_pixels, self.max_pixels)
                                                        for p in pages], prompts)
        else:
            inputs = build_inputs(self.tokenizer, images, prompts, self.min_pixels, self.max_pixels)
        with self._lock:
            dev = self.engine.device
            kw = dict(pages_u8=[p.pin_memory().to(dev, non_blocking=True) for p in pages], min_pixels=self.min_pixels, max_pixels=self.max_pixels) \
                if gpu_preprocess else \
                dict(pixel_values=inputs["pixel_values"].to(dev), image_grid_thw=inputs["image_grid_thw"])
            # every stop id of the checkpoint's generation config when the tokenizer knows them (HF accepts a list too)
            stops = list(getattr(self.tokenizer, "stop_ids", ())) or self.tokenizer.eos_token_id
            if sampling is not None:
                kw["sampling"] = sampling
            out = self.engine.generate(input_ids=inputs["input_ids"].to(dev), attention_mask=inputs["attention_mask"].to(dev),
                                       max_new_tokens=n_new, eos_token_id=stops,
                                       pad_token_id=self.tokenizer.pad_token_id, **kw)
            seq = out.sequences.cpu()
        T = inputs["input_ids"].shape[1]
        # trim the prompt (parser.py:111-113); a batched caller may carry a smaller token budget than the batch ran with
        lim = [n_new] * len(seq) if budgets is None else [max(1, min(int(b), n_new)) for b in budgets]
        return [self.tokenizer.decode(row[T:T + k].tolist()) for row, k in zip(seq, lim)]

    def infer(self, image, prompt: str, max_new_tokens: int = 512, sampling=None) -> str:
        return self.infer_batch([image], [prompt], max_new_tokens, sampling=sampling)[0]
