"""Sampling without a GPU: the fp64 oracle (oracle/sampling.py) against Random123's Philox known answers and against
transformers' own warpers, ``SamplingParams`` validation and seeding, and the plumbing of per-request parameters through the
HTTP endpoint, the batchers, the multi-GPU front, the in-process client and the parser (recording stand-ins; the kernel
itself is checked in tests/test_sampling_gpu.py)."""
import json
import threading
import urllib.error
import urllib.request

import numpy as np
import pytest
import torch
from PIL import Image

from dots_ocr_b200.sampling import GREEDY, SamplingParams, from_hf_kwargs, host_arrays, per_row, sampling_policy
from oracle import sampling as osamp


# ---------------------------------------------------------------------------------------------------------------- oracle
@pytest.mark.parametrize("ctr,key,want", [
    ((0, 0, 0, 0), (0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
    ((0xffffffff,) * 4, (0xffffffff,) * 2, (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
    ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0), (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1)),
])
def test_philox_known_answers(ctr, key, want):
    assert osamp.philox4x32_10(ctr, key) == want


def test_vectorised_philox_and_uniforms():
    seed, step = 0xFEDCBA9876543210, 77
    words = osamp.philox_words(5, step, seed)
    for g in range(5):
        assert tuple(int(w) for w in words[4 * g:4 * g + 4]) == osamp.philox4x32_10((g, step, 0, 0), (seed & 0xFFFFFFFF, seed >> 32))
    u = osamp.uniforms(18, step, seed)
    assert u.shape == (18,) and np.all((u > 0) & (u < 1))
    assert np.array_equal(u, ((words[:18] >> 8).astype(np.float64) + 0.5) * 2.0 ** -24)


def _hf_kept(row, T, top_p=1.0, top_k=0):
    from transformers.generation.logits_process import TemperatureLogitsWarper, TopKLogitsWarper, TopPLogitsWarper
    x = torch.tensor(row, dtype=torch.float64).unsqueeze(0)
    x = TemperatureLogitsWarper(T)(None, x)
    if top_k:
        x = TopKLogitsWarper(top_k)(None, x)
    if top_p < 1.0:
        x = TopPLogitsWarper(top_p)(None, x)
    return torch.isfinite(x[0]).numpy()


def _rows(rng):
    V = 2048
    yield "randn", rng.standard_normal(V) * 2.0
    yield "ties", np.round(rng.standard_normal(V) * 4.0) / 4.0                      # coarse grid: long runs of ties
    bf = torch.tensor(rng.standard_normal(V) * 3.0).to(torch.bfloat16).double().numpy()
    yield "bf16", bf


def test_oracle_top_k_matches_transformers():
    rng = np.random.default_rng(0)
    for name, row in _rows(rng):
        for T in (0.1, 0.7, 1.0, 2.5):
            for k in (1, 5, 50, 2047, 2048, 5000):                                       # k >= V keeps everything
                assert np.array_equal(osamp.kept_mask(row, T, 1.0, k), _hf_kept(row, T, top_k=k)), (name, T, k)


def _check_top_p(row, T, p, k=0):
    ours, hf = osamp.kept_mask(row, T, p, k), _hf_kept(row, T, p, k)
    assert np.all(ours >= hf), "the oracle must keep everything HF keeps"
    extra = ours & ~hf
    if extra.any():                                  # HF cut inside a run of ties: only tokens tied with its last kept value
        assert np.all(row[extra] == row[hf].min()), (row[extra][:5], row[hf].min())
    return int(extra.sum())


def test_oracle_top_p_matches_transformers_up_to_ties():
    rng = np.random.default_rng(1)
    extra = 0
    for name, row in _rows(rng):
        for T in (0.1, 0.7, 1.0, 2.0):
            for p in (1e-6, 0.1, 0.5, 0.8, 0.9, 0.95, 0.999):
                extra += _check_top_p(row, T, p)
                extra += _check_top_p(row, T, p, k=20)                                 # k and p together
                extra += _check_top_p(row, T, p, k=4096)                               # k larger than the vocab
    assert extra > 0, "the tied rows never exercised the tie rule"


def test_oracle_top_p_at_cumulative_mass_boundaries():
    rng = np.random.default_rng(2)
    row = rng.standard_normal(512) * 1.5
    T = 0.8
    w = np.exp((np.sort(row)[::-1] - row.max()) / T)
    cum = np.cumsum(w) / w.sum()
    for j in (0, 1, 5, 40, 300):
        c32 = np.float32(cum[j])                      # the kernel reads p as fp32: one fp32 step either side of the boundary
        for pf in (float(np.nextafter(c32, np.float32(0))), float(c32), float(np.nextafter(c32, np.float32(1)))):
            _check_top_p(row, T, pf)
            keep = osamp.kept_mask(row, T, pf)
            # mass of strictly larger logits < p: exactly the tokens whose exclusive cumulative mass is below p
            want = int(np.sum(np.concatenate([[0.0], cum[:-1]]) < pf))
            assert keep.sum() == want, (j, pf, keep.sum(), want)


def test_replay_is_gumbel_max_over_the_kept_set():
    rng = np.random.default_rng(3)
    row = torch.tensor(rng.standard_normal(4096) * 2).to(torch.bfloat16).double().numpy()
    for T, p, k in ((1.0, 1.0, 0), (0.7, 0.8, 20), (1.0, 1.0, 50), (0.1, 0.9, 0)):
        tok, info = osamp.replay(row, T, p, k, seed=123, step=9, return_info=True)
        assert info["kept"][tok]
        g = osamp.gumbel_keys(row, T, 9, 123)
        assert tok == int(np.argmax(np.where(info["kept"], g, -np.inf)))
    assert osamp.replay(row, 0.0, seed=5) == int(np.argmax(row))
    assert osamp.replay(row, 0.9e-5, 0.5, 3, seed=5) == int(np.argmax(row))        # below the greedy threshold


# ------------------------------------------------------------------------------------------------------ host parameters
def test_sampling_params_validation():
    SamplingParams()
    SamplingParams(temperature=0.0, top_p=1e-9, top_k=0, seed=(1 << 64) - 1)
    for kw in (dict(temperature=-0.1), dict(temperature=float("inf")), dict(temperature=float("nan")), dict(top_p=0.0),
               dict(top_p=1.01), dict(top_p=float("nan")), dict(top_k=-1), dict(top_k=2.5), dict(seed=-1), dict(seed=1 << 64),
               dict(seed=1.0), dict(temperature="1"), dict(top_k=True)):
        with pytest.raises(ValueError):
            SamplingParams(**kw)
    assert SamplingParams(temperature=0.0).greedy and SamplingParams(temperature=0.9e-5).greedy
    assert not SamplingParams(temperature=1e-5).greedy


def test_missing_seed_is_drawn_once_and_follows_torch_manual_seed():
    torch.manual_seed(1234)
    a = SamplingParams(temperature=0.5).with_seed()
    b = SamplingParams(temperature=0.5).with_seed()
    torch.manual_seed(1234)
    assert SamplingParams(temperature=0.5).with_seed() == a and a.seed != b.seed
    assert a.with_seed() is a and 0 <= a.seed < 1 << 64
    torch.manual_seed(7)
    rows = per_row(SamplingParams(top_k=3), 4)
    assert len({r.seed for r in rows}) == 4 and all(r.top_k == 3 for r in rows)
    torch.manual_seed(7)
    assert per_row(SamplingParams(top_k=3), 4) == rows
    assert per_row(SamplingParams(seed=9), 2) == [SamplingParams(seed=9)] * 2
    with pytest.raises(ValueError):
        per_row([SamplingParams()], 2)


def test_host_arrays_carry_the_u64_seed_bits():
    T, p, k, s = host_arrays([SamplingParams(0.5, 0.9, 7, (1 << 64) - 1), GREEDY, SamplingParams(seed=1 << 63)])
    assert T.dtype == torch.float32 and p.dtype == torch.float32 and k.dtype == torch.int32 and s.dtype == torch.int64
    assert T.tolist() == [0.5, 0.0, 1.0] and k.tolist() == [7, 0, 0]
    assert [int(x) & ((1 << 64) - 1) for x in s.tolist()] == [(1 << 64) - 1, 0, 1 << 63]


def test_hf_kwargs_map_onto_sampling_params():
    assert from_hf_kwargs({}) is None and from_hf_kwargs({"do_sample": False, "temperature": 0.7}) is None
    assert from_hf_kwargs({"do_sample": True}) == SamplingParams(1.0, 1.0, 50)
    assert from_hf_kwargs({"do_sample": True, "temperature": 0.7, "top_p": 0.9, "top_k": None}) == SamplingParams(0.7, 0.9, 50)


def test_policy_comes_from_the_environment(monkeypatch):
    monkeypatch.delenv("DOTS_B200_SAMPLING", raising=False)
    assert sampling_policy() == "greedy"
    monkeypatch.setenv("DOTS_B200_SAMPLING", "Request")
    assert sampling_policy() == "request"
    monkeypatch.setenv("DOTS_B200_SAMPLING", "nucleus")
    with pytest.raises(ValueError):
        sampling_policy()


# ------------------------------------------------------------------------------------------------------------- server
class _Recorder:
    def __init__(self):
        self.calls = []
        self.lock = threading.Lock()

    def infer(self, image, prompt, max_new_tokens=512, **kw):
        with self.lock:
            self.calls.append((prompt, max_new_tokens, kw))
        return f"{prompt}|{kw.get('sampling')!r}"


def _body(prompt="p", **fields):
    from dots_ocr_b200.server import IMAGE_PREFIX
    from dots_ocr_b200.utils.image_utils import PILimage_to_base64
    img = Image.new("RGB", (20, 20), (9, 9, 9))
    return dict(messages=[{"role": "user", "content": [{"type": "image_url", "image_url": {"url": PILimage_to_base64(img)}},
                                                       {"type": "text", "text": IMAGE_PREFIX + prompt}]}], **fields)


def _post(base, obj):
    req = urllib.request.Request(base + "/v1/chat/completions", data=json.dumps(obj).encode(),
                                 headers={"Content-Type": "application/json"}, method="POST")
    try:
        with urllib.request.urlopen(req, timeout=10) as resp:
            return resp.status, json.loads(resp.read())
    except urllib.error.HTTPError as e:
        return e.code, json.loads(e.read())


@pytest.fixture(params=["greedy", "request"])
def endpoint(request):
    from dots_ocr_b200.server import serve_in_thread
    r = _Recorder()
    srv, _ = serve_in_thread(r, sampling=request.param)
    yield request.param, r, f"http://127.0.0.1:{srv.server_address[1]}"
    srv.shutdown()
    srv.server_close()


def test_server_sampling_fields(endpoint):
    mode, r, base = endpoint
    code, _ = _post(base, _body("a", temperature=0.7, top_p=0.8, top_k=20, seed=5, max_tokens=9))
    assert code == 200
    code, _ = _post(base, _body("b"))
    assert code == 200
    code, _ = _post(base, _body("c", top_k=-1, temperature=0))
    assert code == 200
    if mode == "greedy":                             # exactly today's call: no sampling argument at all
        assert [c[2] for c in r.calls] == [{}, {}, {}] and r.calls[0][:2] == ("a", 9)
    else:
        assert r.calls[0][2]["sampling"] == SamplingParams(0.7, 0.8, 20, 5)
        s = r.calls[1][2]["sampling"]                 # OpenAI defaults, seed drawn on arrival
        assert (s.temperature, s.top_p, s.top_k) == (1.0, 1.0, 0) and s.seed is not None
        assert r.calls[2][2]["sampling"].top_k == 0 and r.calls[2][2]["sampling"].greedy
    n = len(r.calls)
    bad = [dict(temperature=-1), dict(temperature="hot"), dict(top_p=0), dict(top_p=1.5), dict(top_k=-2), dict(top_k=2.5),
           dict(seed=-3), dict(seed="x"), dict(seed=1 << 64), dict(temperature=True)]
    for fields in bad:
        code, body = _post(base, _body("z", **fields))
        if mode == "greedy":
            assert code == 200, fields               # ignored, as before
        else:
            assert code == 400 and body["error"]["type"] == "invalid_request_error", (fields, body)
    assert len(r.calls) == n + (len(bad) if mode == "greedy" else 0)


def test_server_cli_policy_default(monkeypatch):
    from dots_ocr_b200.server import make_server
    monkeypatch.setenv("DOTS_B200_SAMPLING", "request")
    srv = make_server(_Recorder(), port=0)
    try:
        assert srv.RequestHandlerClass.sampling == "request"
    finally:
        srv.server_close()
    with pytest.raises(ValueError):
        make_server(_Recorder(), port=0, sampling="nucleus")


# ------------------------------------------------------------------------------------------------------------ batchers
class _BatchRecorder:
    def __init__(self):
        self.calls = []

    def infer_batch(self, images, prompts, max_new_tokens=512, budgets=None, **kw):
        self.calls.append((list(prompts), kw))
        return [f"{p}" for p in prompts]


def test_batching_runner_forwards_per_row_params():
    from dots_ocr_b200.batching import BatchingRunner
    rec = _BatchRecorder()
    br = BatchingRunner(rec, max_batch=8, max_wait_ms=200)
    s = SamplingParams(temperature=1.0, top_k=5, seed=11)
    futs = [br.submit("i0", "a"), br.submit("i1", "b", 4, sampling=s), br.submit("i2", "c", 4, sampling=SamplingParams(0.5))]
    assert [f.result(timeout=30) for f in futs] == ["a", "b", "c"]
    assert br.infer("i3", "d") == "d"
    br.close()
    prompts, kw = rec.calls[0]
    assert prompts == ["a", "b", "c"]
    rows = kw["sampling"]
    assert rows[0] == GREEDY and rows[1] == s and rows[2].temperature == 0.5 and rows[2].seed is not None
    assert rec.calls[1] == (["d"], {})               # a greedy-only batch is called as before


def test_continuous_batcher_hands_params_to_prepare():
    from test_continuous_cpu import SimSlots, _want
    from dots_ocr_b200.continuous import ContinuousBatcher

    class SamplingSim(SimSlots):
        def __init__(self, **kw):
            super().__init__(**kw)
            self.seen = {}

        def prepare(self, image, prompt, sampling=None):
            self.seen[prompt] = sampling
            return super().prepare(image, prompt)

    sim = SamplingSim(n_slots=2, chunk=3)
    cb = ContinuousBatcher(sim)
    s = SamplingParams(temperature=0.9, top_p=0.5, seed=3)
    torch.manual_seed(5)
    futs = [cb.submit("a", "n=4", sampling=s), cb.submit("b", "n=2"), cb.submit("c", "n=3", sampling=SamplingParams())]
    assert [f.result(timeout=30) for f in futs] == [_want(4), _want(2), _want(3)]
    cb.close()
    torch.manual_seed(5)
    assert sim.seen["n=4"] == s and sim.seen["n=2"] is None
    assert sim.seen["n=3"] == SamplingParams().with_seed()        # drawn at submission, from torch's generator


def test_multigpu_runner_forwards_params_to_the_worker():
    from dots_ocr_b200.multigpu import MultiGpuRunner, echo_worker
    r = MultiGpuRunner(1, factory=echo_worker, factory_args=(0.0,), start_timeout=120)
    try:
        s = SamplingParams(temperature=0.3, top_k=9, seed=77)
        assert r.infer("img", "p", 5, sampling=s) == f"rank0|img|p|5|{s!r}"
        assert r.infer("img", "q", 6) == "rank0|img|q|6"
    finally:
        r.close()


def test_in_process_client_and_parser_follow_the_policy(monkeypatch, tmp_path):
    from dots_ocr_b200 import DotsOCRParser
    from dots_ocr_b200.model import inference
    rec = _Recorder()
    old = inference._state["runner"]
    monkeypatch.setenv("DOTS_B200_TRANSPORT", "inprocess")
    inference.set_default_runner(rec)
    img = Image.new("RGB", (30, 30))
    try:
        monkeypatch.delenv("DOTS_B200_SAMPLING", raising=False)
        inference.inference_with_vllm(img, "g", temperature=0.4, top_p=0.6, max_completion_tokens=3)
        DotsOCRParser(runner=rec, temperature=0.4, top_p=0.6)._inference_with_vllm(img, "h")
        assert [c[2] for c in rec.calls] == [{}, {}]
        monkeypatch.setenv("DOTS_B200_SAMPLING", "request")
        inference.inference_with_vllm(img, "g", temperature=0.4, top_p=0.6, max_completion_tokens=3)
        DotsOCRParser(runner=rec, temperature=0.1, top_p=1.0)._inference_with_vllm(img, "h")
        got = [c[2]["sampling"] for c in rec.calls[2:]]
        assert (got[0].temperature, got[0].top_p, got[0].top_k) == (0.4, 0.6, 0)
        assert (got[1].temperature, got[1].top_p) == (0.1, 1.0)
    finally:
        inference.set_default_runner(old)
