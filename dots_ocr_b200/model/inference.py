"""Page -> text through the in-process B200 engine, behind the reference's model-adapter seam.

``inference_with_vllm`` keeps the reference signature (``dots_ocr/model/inference.py:7-18``) so that
``from dots_ocr_b200.model.inference import inference_with_vllm`` is a drop-in for callers such as
``DotsOCRParser._inference_with_vllm`` (``dots_ocr/parser.py:119-131``) and ``demo/demo_vllm.py:35``.
Where the page is served (``DOTS_B200_TRANSPORT`` = ``auto`` | ``inprocess`` | ``http``, default ``auto``):

* in process, by the engine living in this process (one per GPU) -- whenever a runner has been installed with
  ``set_default_runner`` or this process can see a CUDA device; the transport arguments are then ignored;
* over HTTP, like the reference -- on a machine without a GPU: the same ``chat.completions`` request the reference sends
  (``inference.py:20-45``) goes to ``{protocol}://{ip}:{port}/v1``, where ``python -m dots_ocr_b200.server`` (or a vLLM server)
  answers it.  Standard library only.

Like the reference, a transport-level failure prints the error and returns ``None``; engine errors propagate as Python
exceptions (the reference's OpenAI client raises too, SURVEY.md §5).
"""
from __future__ import annotations

import json
import os
import threading
import urllib.error
import urllib.request
from typing import Optional

_state = {"runner": None}
_lock = threading.Lock()


def set_default_runner(runner) -> None:
    """Install the process-wide page runner (see ``dots_ocr_b200.runner.PageRunner``)."""
    with _lock:
        _state["runner"] = runner


def get_default_runner():
    """Process-wide runner: the engine behind a continuous batcher, so that the parser's thread fan-out (one page per call,
    parser.py:282-290) shares decode steps the way requests share a vLLM server's batches: a page that finishes frees its slot
    for the next queued page while the others keep decoding."""
    with _lock:
        if _state["runner"] is None:
            from ..continuous import serving_front
            from ..runner import PageRunner
            _state["runner"] = serving_front(PageRunner.from_default())       # continuous batching by default (DOTS_B200_BATCHER)
        return _state["runner"]


def _serve_in_process() -> bool:
    mode = os.environ.get("DOTS_B200_TRANSPORT", "auto").lower()
    if mode in ("inprocess", "http"):
        return mode == "inprocess"
    with _lock:
        if _state["runner"] is not None:
            return True
    import torch
    return torch.cuda.is_available()


def _http_chat(image, prompt, protocol, ip, port, temperature, top_p, max_completion_tokens, model_name, system_prompt,
               timeout: float = 3600.0) -> Optional[str]:
    from ..utils.image_utils import PILimage_to_base64
    messages = [{"role": "system", "content": system_prompt}] if system_prompt else []
    messages.append({"role": "user", "content": [
        {"type": "image_url", "image_url": {"url": PILimage_to_base64(image)}},
        {"type": "text", "text": f"<|img|><|imgpad|><|endofimg|>{prompt}"}]})
    body = json.dumps({"model": model_name, "messages": messages, "max_completion_tokens": max_completion_tokens,
                       "temperature": temperature, "top_p": top_p}).encode("utf-8")
    req = urllib.request.Request(f"{protocol}://{ip}:{port}/v1/chat/completions", data=body, method="POST",
                                 headers={"Content-Type": "application/json",
                                          "Authorization": "Bearer " + os.environ.get("API_KEY", "0")})
    try:
        with urllib.request.urlopen(req, timeout=timeout) as resp:
            return json.loads(resp.read().decode("utf-8"))["choices"][0]["message"]["content"]
    except (urllib.error.URLError, OSError, KeyError, IndexError, ValueError) as e:
        detail = ""
        if isinstance(e, urllib.error.HTTPError):
            try:
                detail = " " + e.read().decode("utf-8", "replace")[:300]
            except OSError:
                pass
        print(f"request error: {e}{detail}")
        return None


def inference_with_vllm(
        image,
        prompt,
        protocol="http",
        ip="localhost",
        port=8000,
        temperature=0.1,
        top_p=0.9,
        max_completion_tokens=32768,
        model_name="rednote-hilab/dots.mocr",
        system_prompt=None,
        ) -> Optional[str]:
    """Page inference.  Over HTTP, ``temperature`` / ``top_p`` go to the server as the reference sends them.  In process
    they are honoured under the sampling policy ``request`` (``DOTS_B200_SAMPLING=request``, dots_ocr_b200/sampling.py);
    under the default ``greedy`` the engine decodes greedily (BASELINE.json fixes greedy), the temperature -> 0 limit."""
    if not _serve_in_process():
        return _http_chat(image, prompt, protocol, ip, port, temperature, top_p, max_completion_tokens, model_name, system_prompt)
    from ..sampling import SamplingParams, sampling_policy
    runner = get_default_runner()
    text = prompt if system_prompt is None else f"{system_prompt}\n{prompt}"
    if sampling_policy() == "request":
        return runner.infer(image, text, max_new_tokens=max_completion_tokens,
                            sampling=SamplingParams(temperature=float(temperature), top_p=float(top_p)))
    return runner.infer(image, text, max_new_tokens=max_completion_tokens)


# explicit alias under the engine's own name
inference_with_b200 = inference_with_vllm
