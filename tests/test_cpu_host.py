"""CPU suite: oracle vs golden vectors, host logic, and the C-ABI library's exported surface."""
import ctypes
import inspect
import json
import os
import sys

import numpy as np
import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
GOLD = os.path.join(HERE, "golden")


# ------------------------------------------------------------------ smart_resize (pinned against the reference itself)
def test_smart_resize_matches_reference_golden():
    from dots_ocr_b200.utils.image_utils import smart_resize
    cases = json.load(open(os.path.join(GOLD, "smart_resize.json")))
    assert len(cases) > 1000
    for c in cases:
        try:
            got = list(smart_resize(c["h"], c["w"], **c["kw"]))
        except ValueError:
            got = "ValueError"
        assert got == c["out"], c


def test_token_counts_of_the_baseline_pages():
    from dots_ocr_b200.utils.image_utils import smart_resize, token_counts
    assert smart_resize(1024, 1024) == (1036, 1036)
    assert token_counts(1024, 1024) == (5476, 1369)
    assert token_counts(1960, 1960) == (19600, 4900)
    assert token_counts(2250, 1700) == (19520, 4880)          # demo_image1.jpg (h, w)
    assert token_counts(3360, 3360) == (57600, 14400)         # MAX_PIXELS
    with pytest.raises(ValueError):
        smart_resize(10, 2001)


# ------------------------------------------------------------------ image pre-processing vs the stock HF processor
def test_preprocess_image_equals_hf_processor():
    from PIL import Image
    from transformers import Qwen2VLImageProcessor
    from dots_ocr_b200.processing import preprocess_image
    rng = np.random.default_rng(5)
    proc = Qwen2VLImageProcessor(patch_size=14, temporal_patch_size=1, merge_size=2,
                                 size={"shortest_edge": 3136, "longest_edge": 11289600})
    for (h, w) in [(300, 200), (1024, 1024), (57, 400)]:
        arr = np.full((h, w, 3), 255, np.uint8)
        for _ in range(30):                                  # document-like: dark rectangles on white
            y, x = rng.integers(0, h - 4), rng.integers(0, w - 4)
            arr[y:y + rng.integers(2, 40), x:x + rng.integers(2, 120)] = rng.integers(0, 90, 3)
        im = Image.fromarray(arr)
        ref = proc(images=[im], return_tensors="pt")
        pv, grid = preprocess_image(im)
        assert torch.equal(grid, ref["image_grid_thw"])
        assert torch.equal(pv, ref["pixel_values"])
    pv, grid = preprocess_image(Image.fromarray(np.zeros((1024, 1024, 3), np.uint8)))
    assert pv.shape == (5476, 588) and grid.tolist() == [[1, 74, 74]]


def test_build_inputs_left_pads_and_counts_image_tokens():
    from PIL import Image
    from dots_ocr_b200 import config
    from dots_ocr_b200.processing import SyntheticTokenizer, build_inputs
    cfg = config.tiny()
    tok = SyntheticTokenizer(cfg)
    ims = [Image.new("RGB", (112, 112), "white"), Image.new("RGBA", (56, 168), (0, 0, 0, 0))]
    out = build_inputs(tok, ims, ["hello", "a longer prompt"])
    assert out["pixel_values"].shape[1] == 588
    n_img = int((out["input_ids"] == cfg.image_token_id).sum())
    assert n_img == out["pixel_values"].shape[0] // 4
    assert out["attention_mask"][0, 0] == 0 or out["attention_mask"][1, 0] == 0       # the shorter row is left-padded
    assert (out["attention_mask"][:, -1] == 1).all()
    assert tok.decode(tok.encode_chat("héllo", 0)) == "héllo"


# ------------------------------------------------------------------ oracle
def test_oracle_decoder_is_stock_hf_qwen2():
    """build_qwen2 (meta init + assign) must equal a normally constructed Qwen2ForCausalLM with the same weights
    (regression: non-persistent rotary inv_freq must be rebuilt in fp32)."""
    from transformers import Qwen2Config, Qwen2ForCausalLM
    from dots_ocr_b200 import config, weights
    from oracle.model import build_qwen2
    t = config.tiny().text
    ck = weights.make_synthetic_checkpoint(config.tiny(), 0, "random")
    m = build_qwen2(t, ck, torch.float32, torch.device("cpu"))
    hf = Qwen2Config(vocab_size=t.vocab_size, hidden_size=t.hidden_size, intermediate_size=t.intermediate_size,
                     num_hidden_layers=t.num_hidden_layers, num_attention_heads=t.num_attention_heads,
                     num_key_value_heads=t.num_key_value_heads, max_position_embeddings=t.max_position_embeddings,
                     rms_norm_eps=t.rms_norm_eps, rope_theta=t.rope_theta, tie_word_embeddings=False, attn_implementation="sdpa")
    m2 = Qwen2ForCausalLM(hf).eval()
    m2.load_state_dict({k: v.float() for k, v in ck.items() if not k.startswith("vision_tower.")}, strict=True)
    ids = torch.randint(0, 2000, (2, 33), generator=torch.Generator().manual_seed(0))
    with torch.no_grad():
        assert torch.equal(m(input_ids=ids).logits, m2(input_ids=ids).logits)
    mb = build_qwen2(t, ck, torch.bfloat16, torch.device("cpu"))
    assert mb.model.rotary_emb.inv_freq.dtype == torch.float32
    assert torch.equal(mb.model.rotary_emb.inv_freq, m2.model.rotary_emb.inv_freq)


def test_oracle_matches_golden_vectors():
    import sys
    sys.path.insert(0, GOLD)
    from make_oracle_golden import golden_inputs, N_NEW
    from dots_ocr_b200 import config, weights
    from oracle.model import DotsOracle
    cfg = config.tiny()
    gold = np.load(os.path.join(GOLD, "oracle_tiny.npz"))
    pv, grid, ids, mask = golden_inputs(cfg)
    for fl in ("peaked", "random"):
        ck = weights.make_synthetic_checkpoint(cfg, 0, fl)
        o = DotsOracle(cfg, ck, torch.float32, "cpu")
        img = o.vision.forward(pv, grid)
        ref = torch.from_numpy(gold[f"{fl}_image_embeds"])
        assert float((img - ref).abs().max() / ref.abs().max()) < 1e-4
        if fl == "peaked":            # well-posed argmax: ids are reproducible across BLAS builds / thread counts
            seq = o.generate(ids, attention_mask=mask, pixel_values=pv, image_grid_thw=grid, max_new_tokens=N_NEW)
            assert np.array_equal(seq.numpy(), gold["peaked_sequences"])
            T = ids.shape[1]
            for b in range(ids.shape[0]):     # and they follow the successor map baked into the checkpoint
                chain = [int(ids[b, -1])]
                for _ in range(N_NEW):
                    chain.append(weights.peaked_next_token(cfg, chain[-1]))
                assert seq[b, T:].tolist() == chain[1:]


def test_vision_oracle_matches_vllm_own_vision_tower():
    """oracle/vision.py against vectors produced by vLLM's DotsVisionTransformer itself, run on CPU in fp32 on the same
    seeded weights and inputs (tests/golden/make_vllm_vision_golden.py): patch embed, every block (on the stored sample of
    rows), merged embeddings.  fp32 both sides, so only summation order differs: 2e-5 of the tensor's range."""
    from dots_ocr_b200 import config, weights
    from oracle.vision import VisionOracle
    sys.path.insert(0, GOLD)
    import make_vllm_vision_golden as G
    d = np.load(os.path.join(GOLD, "vllm_vision_tiny.npz"))
    cfg = config.tiny()
    o = VisionOracle(cfg.vision, weights.make_synthetic_checkpoint(cfg, G.SEED_W, "random"), torch.float32, "cpu")
    for name, grids in G.CASES.items():
        pv, grid = G.case_inputs(cfg, grids)
        assert np.array_equal(d[f"{name}_grid"], grid.numpy())
        out, layers = o.forward(pv, grid, return_layers=True)
        want = [f"{name}_patch_embed"] + [f"{name}_block_{i}" for i in range(cfg.vision.num_hidden_layers)]
        assert len(layers) == len(want)
        for i, (a, k) in enumerate(zip(layers, want)):
            a, b = a[torch.from_numpy(d[f"{k}_rows"])], torch.from_numpy(d[k])
            assert a.shape == b.shape
            assert float((a - b).abs().max()) <= 2e-5 * float(b.abs().max()), (name, i)
        ref = torch.from_numpy(d[f"{name}_image_embeds"])
        assert out.shape == ref.shape and float((out - ref).abs().max()) <= 2e-5 * float(ref.abs().max()), name
    # the real widths (1536, 12 heads x 128, SwiGLU 4224, 6144-wide merger), two blocks
    wcfg = G.wide_config()
    ow = VisionOracle(wcfg.vision, G.vision_only_checkpoint(wcfg, G.SEED_W + 1), torch.float32, "cpu")
    pv, grid = G.case_inputs(wcfg, G.WIDE_GRIDS)
    out, layers = ow.forward(pv, grid, return_layers=True)
    for a, b in ((layers[-1][torch.from_numpy(d["wide_block_1_rows"])], d["wide_block_1"]), (out, d["wide_image_embeds"])):
        b = torch.from_numpy(b)
        assert a.shape == b.shape and float((a - b).abs().max()) <= 2e-5 * float(b.abs().max())


def test_vision_pos_ids_and_rope_known_answers():
    from oracle.vision import vision_pos_ids, rot_pos_emb
    p = vision_pos_ids([[1, 4, 4]], 2)
    # first merge block = (0,0),(0,1),(1,0),(1,1); second block starts at column 2
    assert p[:4].tolist() == [[0, 0], [0, 1], [1, 0], [1, 1]]
    assert p[4:8].tolist() == [[0, 2], [0, 3], [1, 2], [1, 3]]
    assert p[8].tolist() == [2, 0]
    ang = rot_pos_emb([[1, 4, 6]], 2, 128, 10000.0, "cpu")
    assert ang.shape == (24, 64)
    inv = 1.0 / (10000.0 ** (torch.arange(0, 64, 2).float() / 64))
    pos = vision_pos_ids([[1, 4, 6]], 2)
    assert torch.equal(ang[:, :32], pos[:, :1].float() * inv) and torch.equal(ang[:, 32:], pos[:, 1:].float() * inv)


def test_teacher_forced_logits_reproduce_generate():
    from dots_ocr_b200 import config, weights
    from oracle.model import DotsOracle
    cfg = config.tiny()
    o = DotsOracle(cfg, weights.make_synthetic_checkpoint(cfg, 0, "random"))
    ids = torch.randint(0, 2000, (2, 9), generator=torch.Generator().manual_seed(4))
    seq = o.generate(ids, max_new_tokens=5)
    lg = o.teacher_forced_logits(ids, seq[:, 9:])
    assert torch.equal(lg.argmax(-1), seq[:, 9:])


# ------------------------------------------------------------------ host logic
def test_param_counts_match_the_survey():
    from dots_ocr_b200 import config, weights
    c = weights.param_count(config.full())
    assert c["vision"] == 1_262_091_264 and c["text"] == 1_777_088_000       # SURVEY.md: 1.2621 B / 1.7771 B
    names = weights.tensor_names(config.full())
    assert "vision_tower.blocks.41.mlp.fc3.weight" in names and "model.layers.27.self_attn.q_proj.bias" in names


def test_pick_splits_is_valid_and_fills_the_sms():
    from dots_ocr_b200.ops import pick_splits
    for tiles, kb in [(16, 24), (12, 24), (12, 140), (140, 24), (1187, 24), (8, 12), (6, 16), (1, 1), (3, 7)]:
        s = pick_splits(tiles, kb, 148)
        per = -(-kb // s)
        assert -(-kb // per) == s and tiles * s <= max(148, tiles)
    assert pick_splits(12, 140) == 12 and pick_splits(140, 24) == 1


def test_gate_up_interleave_layout():
    from dots_ocr_b200.engine import _interleave_gate_up
    g = torch.arange(256 * 2, dtype=torch.float32).reshape(256, 2)
    u = -g
    w = _interleave_gate_up(g, u)
    assert w.shape == (512, 2)
    # [64 gate | 64 up] per 128 rows (layout shared by the prefill SWIGLU epilogue and the decode swap-AB epilogue)
    for blk in range(4):
        assert torch.equal(w[blk * 128: blk * 128 + 64], g[blk * 64: blk * 64 + 64])
        assert torch.equal(w[blk * 128 + 64: blk * 128 + 128], u[blk * 64: blk * 64 + 64])


def test_engine_refuses_cpu_and_missing_library(monkeypatch):
    from dots_ocr_b200 import config, _lib
    from dots_ocr_b200.engine import Engine
    with pytest.raises(RuntimeError):
        Engine(config.tiny(), {}, "cpu")
    monkeypatch.setattr(_lib, "_lib", None)
    monkeypatch.setattr(_lib, "LIB_PATH", "/nonexistent/libdots_ocr_b200.so")
    with pytest.raises(_lib.DotsLibraryError):
        _lib.load()


def test_parser_keeps_the_reference_constructor_surface():
    from dots_ocr_b200 import DotsOCRParser
    from dots_ocr_b200.model.inference import inference_with_vllm
    ref_ctor = ["protocol", "ip", "port", "model_name", "temperature", "top_p", "max_completion_tokens", "num_thread", "dpi",
                "output_dir", "min_pixels", "max_pixels", "use_hf"]                       # dots_ocr/parser.py:22-36
    got = list(inspect.signature(DotsOCRParser.__init__).parameters)[1:]
    assert got[: len(ref_ctor)] == ref_ctor
    sig = inspect.signature(DotsOCRParser.__init__).parameters
    assert sig["temperature"].default == 0.1 and sig["top_p"].default == 1.0 and sig["max_completion_tokens"].default == 16384
    assert sig["num_thread"].default == 64 and sig["dpi"].default == 200 and sig["use_hf"].default is False
    ref_inf = ["image", "prompt", "protocol", "ip", "port", "temperature", "top_p", "max_completion_tokens", "model_name",
               "system_prompt"]                                                            # dots_ocr/model/inference.py:7-18
    assert list(inspect.signature(inference_with_vllm).parameters) == ref_inf
    for m in ("parse_file", "parse_image", "parse_pdf", "get_prompt", "_inference_with_hf", "_inference_with_vllm"):
        assert hasattr(DotsOCRParser, m)
    from dots_ocr_b200.utils import dict_promptmode_to_prompt
    assert len(dict_promptmode_to_prompt) == 8 and "prompt_layout_all_en" in dict_promptmode_to_prompt


def test_parser_plumbing_with_a_fake_runner(tmp_path):
    from PIL import Image
    from dots_ocr_b200 import DotsOCRParser

    class Fake:
        def infer(self, image, prompt, max_new_tokens=0):
            self.seen = (image.size, prompt, max_new_tokens)
            return '[{"bbox": [1, 2, 3, 4], "category": "Text", "text": "x"}]'
    fake = Fake()
    p = DotsOCRParser(output_dir=str(tmp_path), runner=fake)
    img = tmp_path / "page.png"
    Image.new("RGBA", (120, 90), (255, 0, 0, 128)).save(img)
    res = p.parse_file(str(img), prompt_mode="prompt_layout_only_en")
    assert res[0]["page_no"] == 0 and os.path.exists(res[0]["layout_info_path"]) and os.path.exists(res[0]["layout_image_path"])
    assert "md_content_path" not in res[0]                         # detection only: no Markdown (parser.py:219)
    assert (res[0]["input_height"], res[0]["input_width"]) == (84, 112)
    assert fake.seen[0] == (120, 90) and "layout" in fake.seen[1]
    res = p.parse_file(str(img), prompt_mode="prompt_layout_all_en")
    import json as _json
    cells = _json.load(open(res[0]["layout_info_path"]))
    assert cells == [{"bbox": [1, 2, 3, 4], "category": "Text", "text": "x"}]          # 112/120 and 84/90 scales truncate back to the same ints
    assert open(res[0]["md_content_path"]).read() == "x" and open(res[0]["md_content_nohf_path"]).read() == "x"
    fake.infer = lambda image, prompt, max_new_tokens=0: '[{"bbox": [1, 2, 3, 4], "category": "Text", "text": "kept"}, {"bbox": [5, 6, 7, 8], "category": "Text", "text": "cut o'
    res = p.parse_file(str(img), prompt_mode="prompt_layout_all_en")
    assert res[0].get("filtered") is True and open(res[0]["md_content_path"]).read() == "kept"      # OutputCleaner drops the unfinished cell
    with pytest.raises(ValueError):
        p.parse_file(str(tmp_path / "x.tiff"))


def test_command_line_keeps_the_reference_flags(tmp_path):
    """python -m dots_ocr_b200.parser: the reference CLI's options (dots_ocr/parser.py:325-407), pages served by the
    process-wide runner in both modes."""
    from PIL import Image
    from dots_ocr_b200 import parser as P
    from dots_ocr_b200.model import inference

    class Fake:
        def __init__(self):
            self.seen = []

        def infer(self, image, prompt, max_new_tokens=0):
            self.seen.append((image.size, max_new_tokens))
            return '[{"bbox": [1, 2, 30, 40], "category": "Text", "text": "hello"}]'
    fake = Fake()
    old = inference._state["runner"]
    inference.set_default_runner(fake)
    try:
        img = tmp_path / "scan.png"
        Image.new("RGB", (200, 100), "white").save(img)
        res = P.main([str(img), "--output", str(tmp_path / "o1"), "--max_completion_tokens", "321", "--num_thread", "2",
                      "--no_fitz_preprocess"])
        assert open(res[0]["md_content_path"]).read() == "hello" and fake.seen[-1] == ((200, 100), 321)
        res = P.main([str(img), "--output", str(tmp_path / "o2"), "--use_hf", "true", "--prompt", "prompt_ocr", "--min_pixels", "3136"])
        assert open(res[0]["md_content_path"]).read().startswith('[{"bbox"')        # prompt_ocr: raw response is the Markdown
        with pytest.raises(SystemExit):
            P.main([str(img), "--prompt", "no_such_prompt"])
    finally:
        inference.set_default_runner(old)


class _FakeFitz:
    """Stand-in for PyMuPDF: a "PDF" is a list of (width_pt, height_pt) page sizes; rendering scales them by the matrix."""

    def __init__(self, pages):
        import types
        self.pages = pages
        self.renders = []
        fz = self

        class Matrix:
            def __init__(self, a, b):
                self.a, self.b = a, b

        class Page:
            def __init__(self, idx, wh):
                self.idx, self.wh = idx, wh

            def get_pixmap(self, matrix, alpha=False):
                w, h = int(self.wh[0] * matrix.a), int(self.wh[1] * matrix.b)
                fz.renders.append((self.idx, matrix.a))
                return types.SimpleNamespace(width=w, height=h, samples=bytes([self.idx * 40 % 256]) * (w * h * 3))

        class Doc:
            page_count = len(pages)

            def __getitem__(self, i):
                return Page(i, pages[i])

            def __enter__(self):
                return self

            def __exit__(self, *a):
                return False

        self.module = types.ModuleType("fitz")
        self.module.Matrix = Matrix
        self.module.open = lambda *a, **k: Doc()


def test_pdf_pages_fan_out_into_the_runner(tmp_path, monkeypatch):
    """parse_file on a .pdf: pages rendered at dpi (72 dpi when the render would pass 4500 px), fanned out over threads,
    results ordered by page, outputs named <file>_page_<i>.*, and the jsonl index written (parser.py:261-322)."""
    import json as _json
    import sys
    import threading
    from dots_ocr_b200 import DotsOCRParser
    from dots_ocr_b200.utils import doc_utils

    if "fitz" not in sys.modules:
        monkeypatch.setitem(sys.modules, "fitz", None)                # "import fitz" -> ImportError
        monkeypatch.setitem(sys.modules, "pymupdf", None)
        with pytest.raises(doc_utils.RasteriserUnavailable, match="parse_pages"):
            doc_utils.load_images_from_pdf("whatever.pdf")

    fz = _FakeFitz([(200, 300), (300, 200), (2000, 1000), (100, 100), (120, 80)])
    monkeypatch.setitem(sys.modules, "fitz", fz.module)
    imgs = doc_utils.load_images_from_pdf("doc.pdf", dpi=144)
    assert [im.size for im in imgs] == [(400, 600), (600, 400), (4000, 2000), (200, 200), (240, 160)]   # 4000 px wide: still under 4500
    fz.renders.clear()
    imgs = doc_utils.load_images_from_pdf("doc.pdf", dpi=216, start_page_id=1, end_page_id=2)
    assert [im.size for im in imgs] == [(900, 600), (2000, 1000)]            # page 2 at 216 dpi = 6000 px -> native 72 dpi
    assert fz.renders == [(1, 3.0), (2, 3.0), (2, 1.0)]
    assert len(doc_utils.load_images_from_pdf("doc.pdf", end_page_id=99)) == 5

    class Fake:
        def __init__(self):
            self.lock, self.seen, self.live, self.peak = threading.Lock(), [], 0, 0

        def infer(self, image, prompt, max_new_tokens=0):
            import time
            with self.lock:
                self.live += 1
                self.peak = max(self.peak, self.live)
                self.seen.append(image.size)
            time.sleep(0.05)
            with self.lock:
                self.live -= 1
            return '[{"bbox": [0, 0, 10, 10], "category": "Text", "text": "w%d"}]' % image.size[0]
    fake = Fake()
    p = DotsOCRParser(output_dir=str(tmp_path), runner=fake, num_thread=4, dpi=144)
    res = p.parse_file("/somewhere/report.pdf")
    assert [r["page_no"] for r in res] == [0, 1, 2, 3, 4] and all(r["file_path"] == "/somewhere/report.pdf" for r in res)
    assert sorted(fake.seen) == sorted([(400, 600), (600, 400), (4000, 2000), (200, 200), (240, 160)])
    assert 2 <= fake.peak <= 4                                           # pages in flight together, capped by num_thread
    for i, r in enumerate(res):
        assert r["layout_info_path"].endswith(f"report_page_{i}.json") and os.path.exists(r["md_content_path"])
    assert open(res[2]["md_content_path"]).read() == "w4000"
    lines = open(tmp_path / "report.jsonl").read().splitlines()
    assert [_json.loads(ln)["page_no"] for ln in lines] == [0, 1, 2, 3, 4]
    assert p.parse_pages([], "empty", "prompt_layout_all_en", str(tmp_path)) == []


# ------------------------------------------------------------------ C ABI surface (no GPU compute)
def test_library_exports_every_declared_symbol():
    from dots_ocr_b200 import _lib
    lib = _lib.load()
    names = _lib.declared_symbols()
    assert len(names) >= 25
    for n in names:
        assert hasattr(lib, n), n
    assert lib.dots_abi_version() == _lib.header_constants()["DOTS_ABI_VERSION"]


def test_argument_validation_happens_before_any_cuda_call():
    from dots_ocr_b200 import _lib
    lib = _lib.load()
    rc = lib.dots_gemm_bf16(None, ctypes.c_longlong(8), None, ctypes.c_longlong(8), None, ctypes.c_longlong(8), 16, 16, 7, 0,
                            None, None, ctypes.c_longlong(0), None)
    assert rc == -1 and b"multiples of 8" in lib.dots_last_error()
    rc = lib.dots_attn_varlen_fwd(None, ctypes.c_longlong(0), None, ctypes.c_longlong(0), None, ctypes.c_longlong(0), None,
                                  ctypes.c_longlong(0), None, 1, 1, 12, 12, 64, 0, ctypes.c_float(1.0), None)
    assert rc == -1 and b"head_dim" in lib.dots_last_error()
    rc = lib.dots_rmsnorm(None, ctypes.c_longlong(8), None, None, ctypes.c_longlong(8), ctypes.c_longlong(4), 4100,
                          ctypes.c_float(1e-6), None)
    assert rc == -1


def test_u8_preprocessing_host_half_matches_full_processor():
    """preprocess_image_u8 (resize only) + the normalise/patchify arithmetic == preprocess_image (what dots_patchify_u8 does on the GPU)."""
    from dots_ocr_b200.processing import preprocess_image, preprocess_image_u8, build_text_inputs, SyntheticTokenizer, CLIP_MEAN, CLIP_STD
    from dots_ocr_b200 import config
    g = torch.Generator().manual_seed(3)
    img = torch.randint(0, 256, (100, 150, 3), generator=g, dtype=torch.uint8).numpy()     # not a multiple of 28: exercises the resize
    pv, grid = preprocess_image(img)
    u8 = preprocess_image_u8(img)
    gh, gw = int(grid[0, 1]), int(grid[0, 2])
    assert u8.shape == (gh * 14, gw * 14, 3) and u8.dtype == torch.uint8
    x = u8.permute(2, 0, 1).float()
    mean = torch.tensor(CLIP_MEAN, dtype=torch.float32) * 255.0
    std = torch.tensor(CLIP_STD, dtype=torch.float32) * 255.0
    x = (x - mean[:, None, None]) / std[:, None, None]
    x = x.view(3, gh // 2, 2, 14, gw // 2, 2, 14).permute(1, 4, 2, 5, 0, 3, 6).reshape(gh * gw, 588)
    assert torch.equal(x, pv)
    tok = SyntheticTokenizer(config.tiny())
    t = build_text_inputs(tok, [gh * gw // 4, 3], ["ab", "c"])
    assert t["input_ids"].shape == t["attention_mask"].shape and int(t["attention_mask"][0].sum()) == gh * gw // 4 + 5 + len("ab")
    assert int((t["input_ids"][0] == tok.image_token_id).sum()) == gh * gw // 4


def test_batching_runner_groups_concurrent_callers():
    """64 threads, one page each (the reference parser's fan-out) -> a few batched infer_batch calls, every caller gets ITS result."""
    import threading
    import time
    from dots_ocr_b200.batching import BatchingRunner

    class FakeRunner:
        def __init__(self):
            self.calls = []

        def infer_batch(self, images, prompts, max_new_tokens=512):
            self.calls.append((len(images), max_new_tokens))
            time.sleep(0.05)                                   # a "generate" during which more requests queue up
            return [f"{im}|{pr}|{max_new_tokens}" for im, pr in zip(images, prompts)]

    fake = FakeRunner()
    br = BatchingRunner(fake, max_batch=16, max_wait_ms=30)
    out = {}

    def work(i):
        out[i] = br.infer(f"img{i}", f"p{i}", max_new_tokens=8 + (i % 3))
    ts = [threading.Thread(target=work, args=(i,)) for i in range(64)]
    for t in ts:
        t.start()
    for t in ts:
        t.join(20)
    br.close()
    assert len(out) == 64 and all(out[i].startswith(f"img{i}|p{i}|") for i in range(64))
    assert sum(n for n, _ in fake.calls) == 64 and max(n for n, _ in fake.calls) <= 16
    assert len(fake.calls) <= 12, fake.calls                   # batched, not 64 single-page calls
    assert all(m == 10 for n, m in fake.calls if n >= 3)       # a batch runs at its largest token budget

    class Boom:
        def infer_batch(self, images, prompts, max_new_tokens=512):
            raise ValueError("engine failed")
    br2 = BatchingRunner(Boom(), max_batch=4, max_wait_ms=5)
    with pytest.raises(ValueError):
        br2.infer("a", "b")
    br2.close()


def test_batching_runner_closes_a_batch_on_the_vit_token_budget():
    """Pages are grouped up to a ViT-token budget: four 1024x1024 pages (5476 tokens each) fit 22 000, the 1960x1960 page
    (19 600) opens its own batch, and order of results is per caller."""
    import time
    from PIL import Image
    from dots_ocr_b200.batching import BatchingRunner, page_vit_tokens

    class FakeRunner:
        min_pixels = max_pixels = None

        def __init__(self):
            self.calls = []

        def infer_batch(self, images, prompts, max_new_tokens=512):
            self.calls.append([im.size for im in images])
            time.sleep(0.02)
            return [f"{im.size[0]}:{pr}" for im, pr in zip(images, prompts)]

    small, big = Image.new("RGB", (1024, 1024)), Image.new("RGB", (1960, 1960))
    assert page_vit_tokens(small) == 5476 and page_vit_tokens(big) == 19600 and page_vit_tokens("not an image") == 0
    assert page_vit_tokens(Image.new("RGB", (10000, 10))) == 0          # aspect ratio > 200: left for the runner to refuse
    fake = FakeRunner()
    br = BatchingRunner(fake, max_batch=64, max_wait_ms=200, max_batch_tokens=22000)
    futs = [br.submit(im, f"p{i}") for i, im in enumerate([small, small, small, big, small, small])]
    got = [f.result(timeout=20) for f in futs]
    br.close()
    assert got == ["1024:p0", "1024:p1", "1024:p2", "1960:p3", "1024:p4", "1024:p5"]
    assert [len(c) for c in fake.calls] == [3, 1, 2] and fake.calls[1] == [(1960, 1960)], fake.calls
    # the wait for stragglers is counted from the first request, not restarted by every arrival
    fake2 = FakeRunner()
    br2 = BatchingRunner(fake2, max_batch=64, max_wait_ms=150)
    t0 = time.monotonic()
    f0 = br2.submit(small, "a")
    for k in range(4):
        time.sleep(0.06)
        br2.submit(small, f"late{k}")
    f0.result(timeout=20)
    assert time.monotonic() - t0 < 0.6
    br2.close()
    assert sum(len(c) for c in fake2.calls) == 5 and len(fake2.calls[0]) < 5


# ------------------------------------------------------------------ stop ids / early exit (host half of generate)
def test_finalize_new_tokens_equals_hf_generate_with_several_stop_ids():
    """finalize_new_tokens applied to the un-stopped greedy continuation must give what HF's own generate returns when
    it is handed the same eos list and pad id (rows are independent under left padding)."""
    from dots_ocr_b200 import config, weights
    from dots_ocr_b200.engine import finalize_new_tokens, stop_list
    from oracle.model import build_qwen2
    cfg = config.tiny()
    m = build_qwen2(cfg.text, weights.make_synthetic_checkpoint(cfg, 0, "random"), torch.float32, torch.device("cpu"))
    T, N, pad = 7, 12, 0
    ids = torch.randint(1, 2000, (3, T), generator=torch.Generator().manual_seed(11))
    kw = dict(do_sample=False, pad_token_id=pad, attention_mask=torch.ones_like(ids))
    with torch.no_grad():
        raw = m.generate(input_ids=ids, max_new_tokens=N, min_new_tokens=N, **kw)[:, T:]
        assert raw.shape == (3, N)
        cases = [
            [int(raw[0, 3]), int(raw[1, 5]), int(raw[2, 2])],      # every row stops, at different steps, on different ids
            [int(raw[0, 3]), int(raw[1, 5])],                      # one row never stops: no trimming, two rows padded
            [int(raw[2, 0])],                                      # single id, first token
            [5000],                                                # never produced
        ]
        for stops in cases:
            want = m.generate(input_ids=ids, max_new_tokens=N, eos_token_id=stops, **kw)[:, T:]
            got = raw.clone()
            # the device pads after the primary stop id; emulate that before the host finalisation
            prim = (got == stops[0])
            first = torch.where(prim.any(1), prim.int().argmax(1), torch.full((3,), N))
            got = torch.where(torch.arange(N)[None, :] > first[:, None], torch.full_like(got, pad), got)
            got = finalize_new_tokens(got, stop_list(stops), pad)
            assert torch.equal(got, want), (stops, got, want)
    assert stop_list(None) == [] and stop_list(7) == [7] and stop_list([7, 9, 7]) == [7, 9]
    assert stop_list(torch.tensor([3, 4])) == [3, 4]
    assert finalize_new_tokens(raw, [], pad) is raw


def test_replay_steps_checks_every_k_and_stops_early():
    from dots_ocr_b200.engine import replay_steps
    log = []
    assert replay_steps(lambda: log.append("L"), 10, 0, lambda: log.append("C") or True) == 10
    assert log == ["L"] * 10                                        # every=0: never asks
    log.clear()
    done_at = {"n": 0}

    def finished():
        log.append("C")
        return log.count("L") >= done_at["n"]

    done_at["n"] = 7
    assert replay_steps(lambda: log.append("L"), 20, 4, finished) == 8      # asked at 4 (no) and 8 (yes)
    assert log.count("C") == 2
    log.clear()
    done_at["n"] = 100
    assert replay_steps(lambda: log.append("L"), 8, 4, finished) == 8       # no question after the last launch
    assert log.count("C") == 1
    assert replay_steps(lambda: None, 0, 4, lambda: True) == 0


def test_one_bad_page_does_not_fail_its_batch():
    """ADVICE round 1: a page whose preprocessing raises must fail only its own caller, not the up-to-63 other pages that
    happened to share its batch."""
    from dots_ocr_b200.batching import BatchingRunner

    class Fake:
        def __init__(self):
            self.calls = []

        def infer_batch(self, images, prompts, max_new_tokens=512):
            self.calls.append(len(images))
            if any(im == "bad" for im in images):
                raise ValueError("absolute aspect ratio must be smaller than 200")
            return [f"{im}:{pr}" for im, pr in zip(images, prompts)]

    fake = Fake()
    br = BatchingRunner(fake, max_batch=8, max_wait_ms=300)
    futs = [br.submit(im, f"p{i}", 16) for i, im in enumerate(["a", "b", "bad", "c"])]
    br.close(10)
    assert [f.result(5) for i, f in enumerate(futs) if i != 2] == ["a:p0", "b:p1", "c:p3"]
    with pytest.raises(ValueError, match="aspect ratio"):
        futs[2].result(5)
    assert fake.calls[0] == 4 and sorted(fake.calls[1:]) == [1, 1, 1, 1]       # the batch, then each page on its own


def test_grounding_prompt_bbox_uses_the_reference_rounding():
    """parser.get_prompt scales the grounding bbox with pre_process_bboxes (int(x / (origin_w / w))), as the reference does
    (dots_ocr/parser.py:135-139); x=85, origin width 204, model width 1092 is a case where int(x * (w / origin_w)) is off by one."""
    from PIL import Image
    from dots_ocr_b200.parser import DotsOCRParser
    from dots_ocr_b200.utils.layout_utils import pre_process_bboxes
    from dots_ocr_b200.utils.prompts import dict_promptmode_to_prompt
    origin = Image.new("RGB", (204, 204))
    image = Image.new("RGB", (1092, 1092))
    p = DotsOCRParser.__new__(DotsOCRParser)
    got = p.get_prompt("prompt_grounding_ocr", bbox=[85, 85, 120, 130], origin_image=origin, image=image, min_pixels=3136, max_pixels=11289600)
    want = pre_process_bboxes(origin, [[85, 85, 120, 130]], input_width=1092, input_height=1092, min_pixels=3136, max_pixels=11289600)[0]
    assert got == dict_promptmode_to_prompt["prompt_grounding_ocr"] + str(want)
    assert want[0] == 455 and int(85 * (1092 / 204)) == 454


def test_bench_roofline_traffic_comes_from_the_committed_ncu_capture():
    """bench.py fills `roofline.traffic` from profiles/decode_traffic_*.json (the ncu `dram__bytes` of one decode step) and ties its ids
    to the parity test through tests/golden/bench_ids_checksum.json: both files must be present and well formed."""
    import json
    import os
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.path.insert(0, root)
    import bench
    tr = bench._decode_traffic()
    assert tr is not None and tr["file"].startswith("decode_traffic_") and tr["steps"] >= 1
    # one step moves at least the decoder weights + lm_head (3.09 GB) and not absurdly more than the algorithmic 6.54 GB at B=64, ctx 1.9k
    assert 3.0e9 < tr["dram_bytes_per_step"] < 2 * 6.54e9
    with open(os.path.join(root, "tests", "golden", "bench_ids_checksum.json")) as f:
        g = json.load(f)
    assert isinstance(g["b64_n512_p1024_rank0"], str) and len(g["b64_n512_p1024_rank0"]) == 16
    ids = __import__("torch").arange(12).view(3, 4)
    assert bench.ids_checksum(ids) == bench.ids_checksum(ids.clone()) != bench.ids_checksum(ids + 1)


def test_bench_dump_outputs_writes_float_arrays_within_budget(tmp_path):
    """bench.py --dump-outputs: sequences whole and exact, the image embeddings as a seeded sample of rows that the same shape
    always draws the same way, every array float32 or float64, 64 MB in all at the headline shape."""
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    import bench
    from dots_ocr_b200.engine import GenerateOutput
    seqs = torch.randint(0, 151643, (64, 1625 + 512))
    emb = torch.randn(64 * 1369, 1536).to(torch.bfloat16)
    info = bench.dump_outputs(GenerateOutput(sequences=seqs, image_embeds=emb), str(tmp_path / "a"))
    bench.dump_outputs(GenerateOutput(sequences=seqs, image_embeds=emb.clone()), str(tmp_path / "b"))
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == ["image_embeds.npy", "image_embeds_rows.npy", "sequences.npy"]
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= 64 << 20
    got = {f[:-4]: np.load(tmp_path / "a" / f) for f in files}
    assert all(a.dtype in (np.float32, np.float64) for a in got.values())
    assert np.array_equal(got["sequences"], seqs.numpy()) and info["shapes"]["sequences"] == [64, 2137]
    rows = got["image_embeds_rows"].astype(np.int64)
    assert 1000 < rows.size < emb.shape[0] and np.all(np.diff(rows) > 0)
    assert np.array_equal(got["image_embeds"], emb.float().numpy()[rows])
    for f in files:
        assert np.array_equal(got[f[:-4]], np.load(tmp_path / "b" / f))
