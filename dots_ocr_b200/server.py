"""OpenAI-compatible endpoint in front of the in-process B200 engine.

The reference's default path (``DotsOCRParser(use_hf=False)``) sends every page to a vLLM server
(``dots_ocr/model/inference.py:20-45``: ``OpenAI(base_url=f"{protocol}://{ip}:{port}/v1").chat.completions.create(
messages=[image_url + text], model=..., max_completion_tokens=..., temperature=..., top_p=...)``; the server is started by
``demo/launch_model_vllm.sh``).  This module answers that one request shape, so an UNMODIFIED reference checkout can
point ``--ip/--port`` at a B200 box:

    python -m dots_ocr_b200.server --port 8000 --model-name rednote-hilab/dots.mocr

Only what that client needs is here: ``POST /v1/chat/completions`` (non-streaming), ``GET /v1/models``, ``GET /health``.
Request threads block on the process-wide request front (``dots_ocr_b200/continuous.py:serving_front``: continuous batching by
default, ``DOTS_B200_BATCHER=batching`` for arrival-time batches), which groups concurrent pages
into one ``generate`` call -- the role continuous batching plays inside the vLLM server.

Sampling (``--sampling``, default: environment ``DOTS_B200_SAMPLING``, else ``greedy``):
  * ``greedy``   every page decodes greedily (BASELINE.json); ``temperature`` / ``top_p`` / ``top_k`` / ``seed`` are accepted
                 and ignored;
  * ``request``  each request's ``temperature``, ``top_p``, ``seed`` (OpenAI fields) and ``top_k`` (vLLM's ``extra_body``
                 field; -1 or 0 = off) are honoured, missing ones taking OpenAI's defaults (1.0, 1.0, off, a random seed);
                 malformed or out-of-range values are a 400.
Standard library only: no web framework.
"""
from __future__ import annotations

import argparse
import base64
import io
import itertools
import json
import threading
import time
from http.server import BaseHTTPRequestHandler, ThreadingHTTPServer
from typing import Optional, Tuple

IMAGE_PREFIX = "<|img|><|imgpad|><|endofimg|>"      # inference.py:34; the runner inserts the image tokens itself
DEFAULT_MAX_TOKENS = 16384                           # DotsOCRParser's max_completion_tokens default (parser.py:29)
MAX_BODY_BYTES = 256 << 20


class BadRequest(ValueError):
    pass


def _image_from_url(url: str):
    from PIL import Image
    if not isinstance(url, str) or not url.startswith("data:"):
        raise BadRequest("image_url must be a data: URL (base64 image bytes, as PILimage_to_base64 produces)")
    head, _, payload = url.partition(",")
    if ";base64" not in head or not payload:
        raise BadRequest("image_url data: URL must be base64 encoded")
    try:
        img = Image.open(io.BytesIO(base64.b64decode(payload, validate=False)))
        img.load()
    except Exception as e:          # PIL raises several unrelated types for broken bytes
        raise BadRequest(f"cannot decode the image: {e}") from None
    return img


def parse_chat_request(body: dict) -> Tuple[object, str, int]:
    """(PIL image, prompt text, max_new_tokens) out of a chat.completions request, or BadRequest."""
    if not isinstance(body, dict):
        raise BadRequest("request body must be a JSON object")
    if body.get("stream"):
        raise BadRequest("stream=true is not supported (the reference client does not stream)")
    if int(body.get("n") or 1) != 1:
        raise BadRequest("n != 1 is not supported")
    messages = body.get("messages")
    if not isinstance(messages, list) or not messages:
        raise BadRequest("messages must be a non-empty list")
    system, images, texts = [], [], []
    for m in messages:
        role, content = (m or {}).get("role"), (m or {}).get("content")
        if role == "system":
            system.append(content if isinstance(content, str) else
                          "".join(p.get("text", "") for p in content or [] if isinstance(p, dict)))
        elif role == "user":
            if isinstance(content, str):
                texts.append(content)
                continue
            for part in content or []:
                kind = (part or {}).get("type")
                if kind == "image_url":
                    u = part.get("image_url")
                    images.append(_image_from_url(u.get("url") if isinstance(u, dict) else u))
                elif kind == "text":
                    texts.append(part.get("text", ""))
                else:
                    raise BadRequest(f"unsupported content part type {kind!r}")
        elif role == "assistant":
            raise BadRequest("multi-turn requests are not supported: one user turn per page")
        else:
            raise BadRequest(f"unsupported role {role!r}")
    if len(images) != 1:
        raise BadRequest(f"exactly one image per request is required, got {len(images)}")
    prompt = "".join(texts)
    if prompt.startswith(IMAGE_PREFIX):
        prompt = prompt[len(IMAGE_PREFIX):]
    if system:
        prompt = "\n".join(system) + "\n" + prompt        # same folding as model/inference.py of this package
    n = body.get("max_completion_tokens")
    if n is None:
        n = body.get("max_tokens")
    if n is None:
        n = DEFAULT_MAX_TOKENS
    try:
        n = int(n)
    except (TypeError, ValueError):
        raise BadRequest("max_completion_tokens must be an integer") from None
    if n < 1:
        raise BadRequest("max_completion_tokens must be >= 1")
    return images[0], prompt, n


def parse_sampling(body: dict):
    """``SamplingParams`` out of a chat.completions request (``request`` policy), or BadRequest.  A missing seed is drawn
    here, when the request arrives."""
    from .sampling import SamplingParams

    def num(name, default, kind):
        v = body.get(name)
        if v is None:
            return default
        if isinstance(v, bool) or not isinstance(v, (int, float)) or (kind is int and not float(v).is_integer()):
            raise BadRequest(f"{name} must be {'an integer' if kind is int else 'a number'}, got {v!r}")
        return kind(v)

    top_k = num("top_k", 0, int)
    try:
        return SamplingParams(temperature=num("temperature", 1.0, float), top_p=num("top_p", 1.0, float),
                              top_k=0 if top_k == -1 else top_k, seed=num("seed", None, int)).with_seed()
    except ValueError as e:
        raise BadRequest(str(e)) from None


class _Handler(BaseHTTPRequestHandler):
    protocol_version = "HTTP/1.1"
    server_version = "dots_ocr_b200"

    # set by make_server
    runner = None
    model_name = "rednote-hilab/dots.mocr"
    sampling = "greedy"
    _ids = itertools.count(1)
    quiet = True

    def log_message(self, fmt, *args):          # noqa: D401 - BaseHTTPRequestHandler hook
        if not self.quiet:
            super().log_message(fmt, *args)

    def _send(self, code: int, obj: dict):
        data = json.dumps(obj, ensure_ascii=False).encode("utf-8")
        self.send_response(code)
        self.send_header("Content-Type", "application/json")
        self.send_header("Content-Length", str(len(data)))
        self.end_headers()
        self.wfile.write(data)

    def _error(self, code: int, msg: str, kind: str):
        self._send(code, {"error": {"message": msg, "type": kind, "param": None, "code": None}})

    def do_GET(self):
        path = self.path.split("?", 1)[0].rstrip("/")
        if path in ("/health", "/ping"):
            self._send(200, {"status": "ok"})
        elif path == "/v1/models":
            self._send(200, {"object": "list", "data": [{"id": self.model_name, "object": "model", "created": 0,
                                                         "owned_by": "dots_ocr_b200"}]})
        else:
            self._error(404, f"no route {self.path}", "not_found_error")

    def do_POST(self):
        path = self.path.split("?", 1)[0].rstrip("/")
        try:
            length = int(self.headers.get("Content-Length") or 0)
        except ValueError:
            length = -1
        if length < 0 or length > MAX_BODY_BYTES:
            self.close_connection = True
            return self._error(413 if length > 0 else 400, "bad Content-Length", "invalid_request_error")
        raw = self.rfile.read(length)
        if path != "/v1/chat/completions":
            return self._error(404, f"no route {self.path}", "not_found_error")
        kw = {}
        try:
            body = json.loads(raw.decode("utf-8"))
            image, prompt, n_new = parse_chat_request(body)
            if self.sampling == "request":
                kw["sampling"] = parse_sampling(body)
        except BadRequest as e:
            return self._error(400, str(e), "invalid_request_error")
        except (UnicodeDecodeError, json.JSONDecodeError) as e:
            return self._error(400, f"body is not JSON: {e}", "invalid_request_error")
        try:
            text = self.runner.infer(image, prompt, max_new_tokens=n_new, **kw)
        except Exception as e:          # engine / kernel errors: the client sees a 500 with the message
            return self._error(500, f"{type(e).__name__}: {e}", "server_error")
        self._send(200, {
            "id": f"chatcmpl-{next(self._ids)}", "object": "chat.completion", "created": int(time.time()),
            "model": self.model_name,
            "choices": [{"index": 0, "message": {"role": "assistant", "content": text}, "logprobs": None,
                         "finish_reason": "stop"}],
        })


def make_server(runner, host: str = "127.0.0.1", port: int = 8000, model_name: str = "rednote-hilab/dots.mocr",
                quiet: bool = True, sampling: Optional[str] = None) -> ThreadingHTTPServer:
    """A ready (not yet serving) HTTP server around ``runner`` (anything with ``infer(image, prompt, max_new_tokens)``;
    under ``sampling="request"`` also taking ``sampling=``).  ``port=0`` picks a free port (``server.server_address[1]``).
    ``sampling``: ``greedy`` or ``request`` (default: ``dots_ocr_b200.sampling.sampling_policy()``)."""
    from .sampling import POLICIES, sampling_policy
    sampling = sampling or sampling_policy()
    if sampling not in POLICIES:
        raise ValueError(f"sampling must be one of {POLICIES}, got {sampling!r}")
    handler = type("DotsHandler", (_Handler,), dict(runner=runner, model_name=model_name, quiet=quiet, sampling=sampling))
    srv = ThreadingHTTPServer((host, port), handler)
    srv.daemon_threads = True
    return srv


def serve_in_thread(runner, host: str = "127.0.0.1", port: int = 0, **kw) -> Tuple[ThreadingHTTPServer, threading.Thread]:
    srv = make_server(runner, host, port, **kw)
    th = threading.Thread(target=srv.serve_forever, name="dots-http", daemon=True)
    th.start()
    return srv, th


def main(argv: Optional[list] = None) -> None:
    ap = argparse.ArgumentParser(description="OpenAI-compatible dots.ocr page endpoint on one B200")
    ap.add_argument("--host", default="0.0.0.0")
    ap.add_argument("--port", type=int, default=8000)
    ap.add_argument("--model-name", default="rednote-hilab/dots.mocr")
    ap.add_argument("--device", default="cuda:0")
    ap.add_argument("--weights-dir", default="./weights/DotsOCR")
    ap.add_argument("--max-batch", type=int, default=64)
    ap.add_argument("--gpus", type=int, default=1, help="worker processes, one per GPU (cuda:0..N-1); pages go to the least-loaded")
    ap.add_argument("--sampling", choices=["greedy", "request"], default=None,
                    help="greedy: ignore the requests' sampling fields; request: honour temperature / top_p / top_k / seed "
                         "(default: $DOTS_B200_SAMPLING, else greedy)")
    ap.add_argument("--verbose", action="store_true")
    a = ap.parse_args(argv)
    from .sampling import sampling_policy
    sampling = a.sampling or sampling_policy()
    if a.gpus > 1:
        from .multigpu import MultiGpuRunner, b200_worker
        runner = MultiGpuRunner(a.gpus, factory=b200_worker, factory_args=(a.weights_dir, None, a.max_batch))
    else:
        from .continuous import serving_front
        from .runner import PageRunner
        runner = serving_front(PageRunner.from_default(device=a.device, weights_dir=a.weights_dir), max_batch=a.max_batch)
    srv = make_server(runner, a.host, a.port, a.model_name, quiet=not a.verbose, sampling=sampling)
    print(f"dots_ocr_b200 serving {a.model_name} on http://{a.host}:{srv.server_address[1]}/v1 ({sampling} decoding)", flush=True)
    try:
        srv.serve_forever()
    except KeyboardInterrupt:
        pass
    finally:
        srv.server_close()
        runner.close()


if __name__ == "__main__":
    main()
