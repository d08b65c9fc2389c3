"""dots_sample_advance on the device (csrc/sampling.cu) against the fp64 oracle (oracle/sampling.py), and sampling through
the engine, the continuous batcher and the HTTP endpoint."""
import json
import threading
import urllib.request

import numpy as np
import pytest
import torch

from dots_ocr_b200 import ops
from dots_ocr_b200.sampling import GREEDY, SamplingParams, host_arrays
from oracle import sampling as osamp

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
V = 151936
MIXES = [GREEDY, SamplingParams(0.1, 1.0, 0), SamplingParams(0.1, 0.9, 0), SamplingParams(1.0, 1.0, 50), SamplingParams(0.7, 0.8, 20)]
TOL = 1e-5


def _state(B, steps=None, cols=64):
    z = lambda: torch.zeros(B, dtype=torch.int32, device=DEV)           # noqa: E731
    st = dict(nxt=torch.zeros(B, dtype=torch.int64, device=DEV), out=torch.full((B, cols), -1, dtype=torch.int64, device=DEV),
              step=z() if steps is None else torch.tensor(steps, dtype=torch.int32, device=DEV), pos=z(), ctx=z(), fin=z())
    return st


def _sample(logits, rows, st, stops=(), pad=0, forced=None):
    arrs = [a.to(DEV) for a in host_arrays(rows)]
    ops.sample_advance(logits, st["nxt"], *arrs, st["out"], st["step"], st["pos"], st["ctx"], st["fin"], stops, pad, forced)


def _rows_with_seeds(n, seed0=1000):
    return [SamplingParams(m.temperature, m.top_p, m.top_k, seed0 + 7919 * i) for i, m in enumerate(MIXES[i % len(MIXES)] for i in range(n))]


def _logits(B, seed, scale=3.0):
    g = torch.Generator(device=DEV).manual_seed(seed)
    return (torch.randn(B, V, device=DEV, generator=g) * scale).to(torch.bfloat16)


def test_kernel_replays_the_oracle_exactly():
    B = 64
    logits = _logits(B, 0)
    rows = _rows_with_seeds(B)
    steps = [(37 * b) % 50 for b in range(B)]
    st = _state(B, steps)
    _sample(logits, rows, st)
    got = st["nxt"].cpu().tolist()
    lf = logits.float().cpu().numpy()
    excused, bad = 0, []
    for b, r in enumerate(rows):
        want, info = osamp.replay(lf[b], r.temperature, r.top_p, r.top_k, r.seed, steps[b], return_info=True)
        if got[b] != want:
            if info["gap"] < TOL or info["p_margin"] < TOL:
                excused += 1
            else:
                bad.append((b, r, got[b], want, info["gap"], info["p_margin"]))
    print(f"exact replay: {B - excused - len(bad)}/{B} rows equal, {excused} excused (near-tie within {TOL})")
    assert not bad, bad
    assert st["step"].cpu().tolist() == [s + 1 for s in steps]
    assert [st["out"][b, steps[b]].item() for b in range(B)] == got


def _both(logits, steps, stops, pad, forced, fin0, rows):
    a, s = _state(logits.shape[0], steps), _state(logits.shape[0], steps)
    a["fin"].copy_(fin0)
    s["fin"].copy_(fin0)
    ops.argmax_advance(logits, a["nxt"], a["out"], a["step"], a["pos"], a["ctx"], a["fin"], stops, pad, forced)
    _sample(logits, rows, s, stops, pad, forced)
    return a, s


def test_greedy_rows_are_bit_identical_to_argmax_advance():
    B = 16
    logits = _logits(B, 1)
    logits[2, 100] = logits[2, 5000] = 50.0                                     # tied maximum: lowest index wins
    eos = int(logits[3].float().argmax())
    fin0 = torch.zeros(B, dtype=torch.int32, device=DEV)
    fin0[4] = 1                                                                  # pad after a stop
    steps = list(range(B))
    forced = torch.randint(0, V, (B, 64), device=DEV)
    for fc in (None, forced):
        a, s = _both(logits, steps, (eos, 151935), 11, fc, fin0, [GREEDY] * B)
        for k in a:
            assert torch.equal(a[k], s[k]), k
    # mixed batch: greedy rows are untouched by sampled neighbours
    rows = [GREEDY if b % 2 == 0 else SamplingParams(1.0, 0.9, 30, b) for b in range(B)]
    a, s = _both(logits, steps, (eos,), 11, None, fin0, rows)
    even = torch.arange(0, B, 2, device=DEV)
    for k in a:
        assert torch.equal(a[k][even], s[k][even]), k
    assert a["nxt"][2].item() == 100 and s["nxt"][4].item() == 11


@pytest.mark.parametrize("mix", range(1, len(MIXES)))
def test_a_rows_token_does_not_depend_on_the_batch(mix):
    m = MIXES[mix]
    r = SamplingParams(m.temperature, m.top_p, m.top_k, 424242)
    row = _logits(1, 50 + mix)[0]
    toks = []
    for B, at in ((1, 0), (64, 0), (64, 37), (256, 200)):
        logits = _logits(B, 7)
        logits[at] = row
        rows = _rows_with_seeds(B, seed0=99)
        rows[at] = r
        steps = [(s * 13) % 40 for s in range(B)]
        steps[at] = 17
        st = _state(B, steps)
        _sample(logits, rows, st)
        toks.append(st["nxt"][at].item())
    assert len(set(toks)) == 1, toks


def _chi2_draws(row, params, n_rows=256, n_steps=128):
    """n_rows x n_steps draws of one logits row: distinct seeds, step advanced by the kernel itself."""
    logits = torch.tensor(row, dtype=torch.float32, device=DEV).to(torch.bfloat16).unsqueeze(0).expand(n_rows, -1).contiguous()
    rows = [SamplingParams(params.temperature, params.top_p, params.top_k, 5000 + i) for i in range(n_rows)]
    st = _state(n_rows, cols=n_steps)
    arrs = [a.to(DEV) for a in host_arrays(rows)]
    for _ in range(n_steps):
        ops.sample_advance(logits, st["nxt"], *arrs, st["out"], st["step"], st["pos"], st["ctx"], st["fin"], (), 0, None)
    return st["out"].reshape(-1).cpu().numpy(), logits[0].float().cpu().numpy()


@pytest.mark.parametrize("case", ["tail_T1", "top_p_tied_tail", "top_k_ties", "k_and_p"])
def test_draws_follow_the_exact_distribution(case):
    from scipy.stats import chisquare
    Vd = 4096
    row = np.full(Vd, -30.0)
    cand = np.arange(0, 8 * 97, 97)                                             # 8 candidates spread over the row
    row[cand] = [2.0, 1.5, 1.5, 1.0, 0.5, 0.0, -0.5, -1.0]
    if case == "tail_T1":
        row[cand.max() + 1:] = -4.0                                             # a tail of ~3.3k tokens with a known mass
        params = SamplingParams(1.0, 1.0, 0)
    elif case == "top_p_tied_tail":
        row[cand[3:]] = 1.0                                                      # the cut-off lands inside a run of 5 ties
        params = SamplingParams(1.0, 0.7, 0)
    elif case == "top_k_ties":
        params = SamplingParams(0.8, 1.0, 2)                                     # 2nd largest is tied: 3 tokens kept
    else:
        row[cand.max() + 1:] = -3.0
        params = SamplingParams(0.7, 0.9, 6)
    toks, lrow = _chi2_draws(row, params)
    prob = osamp.distribution(lrow, params.temperature, params.top_p, params.top_k)
    kept = prob > 0
    assert kept[toks].all(), "a token outside the kept set was drawn"
    if case == "top_p_tied_tail":
        assert kept.sum() == 8                                                   # every tied token kept
    if case == "top_k_ties":
        assert kept.sum() == 3
    # bins: each candidate, plus the rest of the kept set pooled
    labels = np.full(Vd, 8)
    labels[cand] = np.arange(8)
    obs = np.bincount(labels[toks], minlength=9).astype(float)
    exp = np.bincount(labels, weights=prob, minlength=9) * len(toks)
    use = exp > 0
    assert obs[~use].sum() == 0
    stat, pval = chisquare(obs[use], exp[use])
    print(f"{case}: {len(toks)} draws, chi2 {stat:.2f}, p-value {pval:.3f}")
    assert pval > 1e-3, (obs, exp)


# ---------------------------------------------------------------------------------------------------------------- engine
def _engine(flavour):
    from dots_ocr_b200 import config, weights
    from dots_ocr_b200.engine import Engine
    cfg = config.tiny()
    return cfg, Engine(cfg, weights.make_synthetic_checkpoint(cfg, 0, flavour), DEV)


def _inputs(cfg, B=3):
    g = torch.Generator().manual_seed(11)
    gh, gw = 8, 12
    pv = torch.randn(B * gh * gw, cfg.vision.patch_dim, generator=g)
    grid = torch.tensor([[1, gh, gw]] * B)
    ids = torch.stack([torch.cat([torch.randint(0, 2000, (6,), generator=g), torch.full((gh * gw // 4,), cfg.image_token_id),
                                  torch.randint(0, 2000, (5,), generator=g)]) for _ in range(B)])
    return dict(input_ids=ids, pixel_values=pv.to(DEV), image_grid_thw=grid)


@pytest.mark.parametrize("flavour", ["random", "peaked"])
def test_engine_generate_with_sampling(flavour):
    cfg, eng = _engine(flavour)
    inp = _inputs(cfg)
    N = 12
    greedy = eng.generate(**inp, max_new_tokens=N).sequences
    assert torch.equal(eng.generate(**inp, max_new_tokens=N, sampling=SamplingParams(temperature=0.0)).sequences, greedy)
    assert torch.equal(eng.generate(**inp, max_new_tokens=N).sequences, greedy)       # the greedy graph is still the greedy one
    s1 = [SamplingParams(1.0, 1.0, 0, 100 + i) for i in range(3)]
    a = eng.generate(**inp, max_new_tokens=N, sampling=s1).sequences
    b = eng.generate(**inp, max_new_tokens=N, sampling=s1).sequences
    c = eng.generate(**inp, max_new_tokens=N, sampling=s1, use_graph=False).sequences
    assert torch.equal(a, b) and torch.equal(a, c)
    if flavour == "random":
        d = eng.generate(**inp, max_new_tokens=N, sampling=[SamplingParams(1.0, 1.0, 0, 900 + i) for i in range(3)]).sequences
        assert not torch.equal(a, d)
    # every sampled token is the oracle's draw on the logits the engine returns
    mix = [SamplingParams(1.0, 0.9, 0, 5), SamplingParams(0.7, 0.8, 20, 6), SamplingParams(1.0, 1.0, 50, 7)]
    out = eng.generate(**inp, max_new_tokens=N, sampling=mix, return_logits=True)
    T0 = inp["input_ids"].shape[1]
    lg = out.logits.float().cpu().numpy()
    excused = 0
    for r in range(3):
        for s in range(N):
            want, info = osamp.replay(lg[r, s], mix[r].temperature, mix[r].top_p, mix[r].top_k, mix[r].seed, s, return_info=True)
            got = int(out.sequences[r, T0 + s])
            if got != want:
                assert info["gap"] < TOL or info["p_margin"] < TOL, (r, s, got, want, info["gap"], info["p_margin"])
                excused += 1
    print(f"{flavour}: {3 * N - excused}/{3 * N} sampled tokens equal to the oracle replay, {excused} excused")
    if flavour == "peaked":
        low = eng.generate(**inp, max_new_tokens=N, sampling=SamplingParams(0.1, 1.0, 0, 1)).sequences
        assert torch.equal(low, greedy)
    # HF-style kwargs
    hf = eng.generate(**inp, max_new_tokens=N, do_sample=True, temperature=1.0, top_k=0, sampling=None)
    assert hf.sequences.shape == greedy.shape


def _id_tokenizer(cfg):
    from dots_ocr_b200.processing import SyntheticTokenizer

    class IdTokenizer(SyntheticTokenizer):
        def decode(self, ids):
            ids = [int(i) for i in ids]
            if self.eos_token_id is not None and self.eos_token_id in ids:
                ids = ids[: ids.index(self.eos_token_id) + 1]
            return ",".join(str(i) for i in ids)
    return IdTokenizer(cfg)


def _pages(n, seed=0):
    from PIL import Image
    rng = np.random.default_rng(seed)
    sizes = [(100, 80), (60, 120), (90, 90), (140, 70), (56, 56), (120, 120), (84, 168)]
    return [Image.fromarray(rng.integers(0, 256, (sizes[i % len(sizes)][1], sizes[i % len(sizes)][0], 3), dtype=np.uint8))
            for i in range(n)]


def test_continuous_batching_gives_sampled_pages_what_one_page_gives_them():
    from dots_ocr_b200.continuous import ContinuousBatcher, EngineSlots
    from dots_ocr_b200.runner import PageRunner
    cfg, eng = _engine("random")
    tk = _id_tokenizer(cfg)
    imgs = _pages(7)
    prompts = [f"page {i}: layout" for i in range(7)]
    budgets = [5, 20, 9, 13, 1, 24, 7]
    params = [None if i % 3 == 1 else SamplingParams(1.0, 1.0 if i % 2 else 0.9, 0, 31 + i) for i in range(7)]
    single = PageRunner(eng, tk)
    want = [single.infer(im, pr, b, sampling=s) for im, pr, b, s in zip(imgs, prompts, budgets, params)]
    backend = EngineSlots(eng, tk, n_slots=3, max_prompt=256, max_new=24, chunk=4)
    cb = ContinuousBatcher(backend)
    futs = [cb.submit(im, pr, b, sampling=s) for im, pr, b, s in zip(imgs, prompts, budgets, params)]
    got = [f.result(timeout=120) for f in futs]
    cb.close()
    assert got == want
    greedy_want = [single.infer(im, pr, b) for im, pr, b, s in zip(imgs, prompts, budgets, params) if s is None]
    assert [g for g, s in zip(got, params) if s is None] == greedy_want


def test_server_request_mode_same_seed_same_text():
    from dots_ocr_b200.continuous import serving_front
    from dots_ocr_b200.runner import PageRunner
    from dots_ocr_b200.server import IMAGE_PREFIX, serve_in_thread
    from dots_ocr_b200.utils.image_utils import PILimage_to_base64
    cfg, eng = _engine("random")
    front = serving_front(PageRunner(eng, _id_tokenizer(cfg)), max_batch=4, max_prompt=256, max_new=32, chunk=4)
    srv, _ = serve_in_thread(front, sampling="request")
    base = f"http://127.0.0.1:{srv.server_address[1]}/v1/chat/completions"
    img = _pages(1, seed=3)[0]

    def ask(seed, out, i):
        body = {"messages": [{"role": "user", "content": [{"type": "image_url", "image_url": {"url": PILimage_to_base64(img)}},
                                                          {"type": "text", "text": IMAGE_PREFIX + "layout"}]}],
                "max_tokens": 24, "temperature": 1.0, "seed": seed}
        req = urllib.request.Request(base, data=json.dumps(body).encode(), headers={"Content-Type": "application/json"}, method="POST")
        with urllib.request.urlopen(req, timeout=120) as resp:
            out[i] = json.loads(resp.read())["choices"][0]["message"]["content"]

    try:
        out = {}
        ths = [threading.Thread(target=ask, args=(s, out, i)) for i, s in enumerate((17, 17, 18))]
        [t.start() for t in ths]
        [t.join(180) for t in ths]
    finally:
        srv.shutdown()
        srv.server_close()
        front.close()
    assert out[0] == out[1] and out[0] != out[2], out
