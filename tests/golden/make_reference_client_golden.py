"""The HTTP request the reference's own client sends (dots_ocr/model/inference.py:7-48, ``inference_with_vllm``), recorded
from an unmodified dots.ocr checkout by a stand-in server, for tests/test_server_cpu.py to replay against this project's endpoint.

    python tests/golden/make_reference_client_golden.py <dots.ocr checkout>   # -> tests/golden/reference_client_request.json

The stand-in answers with an OpenAI-shaped completion; the text the client returns from it is recorded too.
"""
import http.server
import json
import os
import sys
import threading
import types

from PIL import Image

IMAGE_SIZE, IMAGE_COLOR = (64, 48), (200, 100, 50)
PROMPT, MAX_COMPLETION_TOKENS, MODEL = "Parse this page", 99, "rednote-hilab/dots.mocr"
REPLY = "recorded reply"


class _Recorder(http.server.BaseHTTPRequestHandler):
    seen = []

    def do_POST(self):
        body = json.loads(self.rfile.read(int(self.headers["Content-Length"])))
        self.seen.append({"method": "POST", "path": self.path, "content_type": self.headers["Content-Type"], "body": body})
        out = json.dumps({"id": "chatcmpl-0", "object": "chat.completion", "created": 0, "model": body["model"],
                          "choices": [{"index": 0, "finish_reason": "stop", "message": {"role": "assistant", "content": REPLY}}],
                          "usage": {"prompt_tokens": 0, "completion_tokens": 0, "total_tokens": 0}}).encode()
        self.send_response(200)
        self.send_header("Content-Type", "application/json")
        self.send_header("Content-Length", str(len(out)))
        self.end_headers()
        self.wfile.write(out)

    def log_message(self, *a):
        pass


def main(checkout):
    sys.path.insert(0, checkout)
    sys.modules.setdefault("fitz", types.ModuleType("fitz"))        # PyMuPDF: imported by the module, unused on this path
    from dots_ocr.model.inference import inference_with_vllm
    srv = http.server.ThreadingHTTPServer(("127.0.0.1", 0), _Recorder)
    threading.Thread(target=srv.serve_forever, daemon=True).start()
    try:
        text = inference_with_vllm(Image.new("RGB", IMAGE_SIZE, IMAGE_COLOR), PROMPT, protocol="http", ip="127.0.0.1",
                                   port=srv.server_address[1], max_completion_tokens=MAX_COMPLETION_TOKENS, model_name=MODEL)
    finally:
        srv.shutdown()
    assert len(_Recorder.seen) == 1 and text == REPLY, (_Recorder.seen, text)
    rec = dict(_Recorder.seen[0], client_returned=text)
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "reference_client_request.json")
    with open(path, "w") as f:
        json.dump(rec, f, indent=1)
        f.write("\n")
    print(path, os.path.getsize(path))


if __name__ == "__main__":
    main(sys.argv[1])
