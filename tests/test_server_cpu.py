"""The OpenAI-compatible endpoint (dots_ocr_b200/server.py) against the client library the reference uses
(``openai.OpenAI(...).chat.completions.create``, dots_ocr/model/inference.py:20-45).  The runner is a recording stand-in:
no kernels run here; the engine side is covered by the GPU tests."""
import json
import threading
import urllib.error
import urllib.request

import pytest
from PIL import Image

from dots_ocr_b200.server import BadRequest, IMAGE_PREFIX, parse_chat_request, serve_in_thread
from dots_ocr_b200.utils.image_utils import PILimage_to_base64


class _Runner:
    def __init__(self):
        self.calls = []
        self.lock = threading.Lock()
        self.fail = None

    def infer(self, image, prompt, max_new_tokens=512):
        if self.fail:
            raise self.fail
        with self.lock:
            self.calls.append((image.size, image.getpixel((0, 0)), prompt, max_new_tokens))
        return f'[{{"bbox": [0, 0, {image.size[0]}, {image.size[1]}], "category": "Text", "text": "{prompt[:8]}"}}]'


@pytest.fixture()
def endpoint():
    r = _Runner()
    srv, th = serve_in_thread(r, model_name="rednote-hilab/dots.mocr")
    yield r, f"http://127.0.0.1:{srv.server_address[1]}"
    srv.shutdown()
    srv.server_close()


def _messages(img, prompt, system=None):
    m = [{"role": "system", "content": system}] if system else []
    m.append({"role": "user", "content": [{"type": "image_url", "image_url": {"url": PILimage_to_base64(img)}},
                                          {"type": "text", "text": f"{IMAGE_PREFIX}{prompt}"}]})
    return m


def test_openai_client_round_trip(endpoint):
    from openai import OpenAI
    r, base = endpoint
    client = OpenAI(api_key="0", base_url=base + "/v1")
    img = Image.new("RGB", (90, 60), (12, 34, 56))
    resp = client.chat.completions.create(messages=_messages(img, "Please output the layout"), model="rednote-hilab/dots.mocr",
                                          max_completion_tokens=777, temperature=0.1, top_p=0.9)
    assert resp.choices[0].message.content == '[{"bbox": [0, 0, 90, 60], "category": "Text", "text": "Please o"}]'
    assert resp.choices[0].finish_reason == "stop" and resp.model == "rednote-hilab/dots.mocr"
    assert r.calls == [((90, 60), (12, 34, 56), "Please output the layout", 777)]      # PNG is lossless; prefix stripped
    # system prompt folded in front of the user prompt, max_tokens spelling, default budget
    client.chat.completions.create(messages=_messages(img, "p", system="be terse"), model="m", max_tokens=5)
    client.chat.completions.create(messages=_messages(img, "q"), model="m")
    assert r.calls[1][2:] == ("be terse\np", 5) and r.calls[2][2:] == ("q", 16384)
    assert [m.id for m in client.models.list().data] == ["rednote-hilab/dots.mocr"]


def test_concurrent_requests_are_all_answered(endpoint):
    from openai import OpenAI
    r, base = endpoint
    out = {}

    def one(i):
        c = OpenAI(api_key="0", base_url=base + "/v1")
        img = Image.new("RGB", (30 + i, 40), (i, i, i))
        out[i] = c.chat.completions.create(messages=_messages(img, f"page{i:03d}"), model="m").choices[0].message.content

    ths = [threading.Thread(target=one, args=(i,)) for i in range(16)]
    [t.start() for t in ths]
    [t.join() for t in ths]
    assert len(r.calls) == 16
    for i in range(16):
        assert json.loads(out[i])[0]["bbox"][2] == 30 + i and json.loads(out[i])[0]["text"] == f"page{i:03d}"[:8]


def _post(base, path, obj, raw=None):
    req = urllib.request.Request(base + path, data=raw if raw is not None else json.dumps(obj).encode(),
                                 headers={"Content-Type": "application/json"}, method="POST")
    try:
        with urllib.request.urlopen(req, timeout=10) as resp:
            return resp.status, json.loads(resp.read())
    except urllib.error.HTTPError as e:
        return e.code, json.loads(e.read())


def test_errors_are_openai_shaped(endpoint):
    r, base = endpoint
    img = Image.new("RGB", (20, 20))
    code, body = _post(base, "/v1/chat/completions", None, raw=b"{not json")
    assert code == 400 and body["error"]["type"] == "invalid_request_error"
    code, body = _post(base, "/v1/chat/completions", {"messages": [{"role": "user", "content": "no image"}]})
    assert code == 400 and "exactly one image" in body["error"]["message"]
    code, body = _post(base, "/v1/chat/completions", {"messages": _messages(img, "p"), "stream": True})
    assert code == 400 and "stream" in body["error"]["message"]
    bad = _messages(img, "p")
    bad[0]["content"][0]["image_url"]["url"] = "https://example.com/x.png"
    code, body = _post(base, "/v1/chat/completions", {"messages": bad})
    assert code == 400 and "data:" in body["error"]["message"]
    bad[0]["content"][0]["image_url"]["url"] = "data:image/png;base64,AAAA"
    code, body = _post(base, "/v1/chat/completions", {"messages": bad})
    assert code == 400 and "decode" in body["error"]["message"]
    code, body = _post(base, "/v1/embeddings", {})
    assert code == 404
    r.fail = RuntimeError("dots_gemm_bf16: invalid pitch")
    code, body = _post(base, "/v1/chat/completions", {"messages": _messages(img, "p")})
    assert code == 500 and "invalid pitch" in body["error"]["message"] and body["error"]["type"] == "server_error"
    with urllib.request.urlopen(base + "/health", timeout=10) as resp:
        assert resp.status == 200
    assert r.calls == []


def test_parse_chat_request_units():
    img = Image.new("RGB", (8, 8))
    im, p, n = parse_chat_request({"messages": _messages(img, "x"), "max_completion_tokens": "12"})
    assert im.size == (8, 8) and p == "x" and n == 12
    two = _messages(img, "x")
    two[0]["content"].insert(0, two[0]["content"][0])
    for body in ({"messages": two}, {"messages": []}, {"messages": _messages(img, "x"), "n": 2},
                 {"messages": _messages(img, "x"), "max_completion_tokens": 0},
                 {"messages": _messages(img, "x") + [{"role": "assistant", "content": "hi"}]}, []):
        with pytest.raises(BadRequest):
            parse_chat_request(body)


def test_unmodified_reference_client_talks_to_the_endpoint(endpoint):
    """The request the reference's own ``inference_with_vllm`` sends (recorded from an unmodified dots.ocr checkout by
    tests/golden/make_reference_client_golden.py), replayed against this endpoint: the reply parses as the OpenAI client the
    reference uses parses it, and its content is the runner's text."""
    import os
    from openai.types.chat import ChatCompletion
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_client_request.json")) as f:
        rec = json.load(f)
    assert rec["method"] == "POST" and rec["content_type"] == "application/json"
    r, base = endpoint
    code, body = _post(base, rec["path"], rec["body"])
    assert code == 200, body
    text = ChatCompletion.model_validate(body).choices[0].message.content
    assert text == '[{"bbox": [0, 0, 64, 48], "category": "Text", "text": "Parse th"}]'
    assert r.calls == [((64, 48), (200, 100, 50), "Parse this page", 99)]


def test_the_mirror_client_uses_http_on_a_machine_without_a_gpu(endpoint, monkeypatch, capsys):
    """dots_ocr_b200.model.inference.inference_with_vllm: no runner installed and no CUDA device here -> the reference's
    request shape over HTTP; a dead endpoint prints the error and returns None (inference.py:46-48)."""
    import torch
    from dots_ocr_b200.model import inference
    if torch.cuda.is_available():
        monkeypatch.setenv("DOTS_B200_TRANSPORT", "http")
    r, base = endpoint
    port = int(base.rsplit(":", 1)[1])
    old = inference._state["runner"]
    inference.set_default_runner(None)
    try:
        img = Image.new("RGB", (48, 32), (1, 2, 3))
        text = inference.inference_with_vllm(img, "Parse it", ip="127.0.0.1", port=port, max_completion_tokens=55, system_prompt="sys")
        assert text == '[{"bbox": [0, 0, 48, 32], "category": "Text", "text": "sys\nPars"}]'
        assert r.calls == [((48, 32), (1, 2, 3), "sys\nParse it", 55)]
        srv2_port = port + 1 if port < 65000 else port - 1
        assert inference.inference_with_vllm(img, "x", ip="127.0.0.1", port=srv2_port) is None
        assert "request error" in capsys.readouterr().out
        # the parser's default path goes the same way
        from dots_ocr_b200 import DotsOCRParser
        p = DotsOCRParser(ip="127.0.0.1", port=port, max_completion_tokens=9)
        assert p._inference_with_vllm(img, "q").startswith('[{"bbox": [0, 0, 48, 32]') and r.calls[-1][2:] == ("q", 9)
        # in the default transport mode an installed runner wins over the transport arguments
        monkeypatch.delenv("DOTS_B200_TRANSPORT", raising=False)
        class Local:
            def infer(self, image, prompt, max_new_tokens=0):
                return "local"
        inference.set_default_runner(Local())
        assert inference.inference_with_vllm(img, "x", ip="127.0.0.1", port=srv2_port) == "local"
    finally:
        inference.set_default_runner(old)
