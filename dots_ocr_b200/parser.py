"""``DotsOCRParser`` with the reference's constructor and public methods
(``dots_ocr/parser.py:22-36, 255-322``), its model call served by the B200 engine.

The hot-path seam is re-implemented here (``_load_hf_model`` / ``_inference_with_hf`` / ``_inference_with_vllm`` /
``get_prompt`` / ``parse_image`` / ``parse_file``) together with the post-decode CPU pipeline of
``_parse_single_image`` (``parser.py:143-253``): the decoded layout JSON is mapped back to page coordinates and
rendered to Markdown by ``utils/layout_utils.py`` / ``utils/format_transformer.py``, whose behaviour is pinned against
the reference functions, JSON repair of cut-off responses included (``tests/test_postprocess.py``).  Multi-page inputs fan
out over ``num_thread`` threads like the reference's ``parse_pdf`` (``parser.py:261-297``); the threads meet in the request
batcher, so the pages of one document share ``generate`` calls.  PDF rasterisation needs PyMuPDF (``utils/doc_utils.py``;
not in this image -- ``parse_pages`` takes pre-rasterised page images).
See INTEGRATION.md for patching the reference's own parser instead.
"""
from __future__ import annotations

import json
import os
from typing import Optional  # noqa: F401

from .model.inference import inference_with_vllm
from .utils.consts import MIN_PIXELS, MAX_PIXELS, image_extensions
from .utils.image_utils import smart_resize
from .utils.prompts import dict_promptmode_to_prompt


class DotsOCRParser:
    """parse image or pdf file"""

    def __init__(self,
                 protocol='http',
                 ip='localhost',
                 port=8000,
                 model_name='model',
                 temperature=0.1,
                 top_p=1.0,
                 max_completion_tokens=16384,
                 num_thread=64,
                 dpi=200,
                 output_dir="./output",
                 min_pixels=None,
                 max_pixels=None,
                 use_hf=False,
                 runner=None,
                 ):
        self.dpi = dpi
        self.protocol, self.ip, self.port, self.model_name = protocol, ip, port, model_name
        self.temperature, self.top_p = temperature, top_p
        self.max_completion_tokens = max_completion_tokens
        self.num_thread = num_thread
        self.output_dir = output_dir
        self.min_pixels, self.max_pixels = min_pixels, max_pixels
        self.use_hf = use_hf
        self._runner = runner
        if self.use_hf:
            self._load_hf_model()
        assert self.min_pixels is None or self.min_pixels >= MIN_PIXELS
        assert self.max_pixels is None or self.max_pixels <= MAX_PIXELS

    # -- model adapter ------------------------------------------------------------------------
    def _load_hf_model(self):
        """Reference: AutoModelForCausalLM + AutoProcessor from ./weights/DotsOCR (parser.py:62-76).
        Here: the in-process B200 engine (real checkpoint directory if present, else synthetic)."""
        if self._runner is None:
            from .model.inference import get_default_runner
            self._runner = get_default_runner()
        self.model = getattr(self._runner, "engine", None)
        self.processor = getattr(self._runner, "tokenizer", None)

    def _inference_with_hf(self, image, prompt):
        if self._runner is None:
            self._load_hf_model()
        return self._runner.infer(image, prompt, max_new_tokens=min(24000, self.max_completion_tokens))

    def _inference_with_vllm(self, image, prompt):
        if self._runner is not None:
            from .sampling import SamplingParams, sampling_policy
            if sampling_policy() == "request":         # the parser's temperature / top_p, as the reference sends them to its server
                return self._runner.infer(image, prompt, max_new_tokens=self.max_completion_tokens,
                                          sampling=SamplingParams(temperature=float(self.temperature), top_p=float(self.top_p)))
            return self._runner.infer(image, prompt, max_new_tokens=self.max_completion_tokens)
        return inference_with_vllm(image, prompt, model_name=self.model_name, protocol=self.protocol, ip=self.ip,
                                   port=self.port, temperature=self.temperature, top_p=self.top_p,
                                   max_completion_tokens=self.max_completion_tokens)

    def get_prompt(self, prompt_mode, bbox=None, origin_image=None, image=None, min_pixels=None, max_pixels=None):
        prompt = dict_promptmode_to_prompt[prompt_mode]
        if prompt_mode == 'prompt_grounding_ocr':
            assert bbox is not None
            # bbox is given in origin_image pixels; the model sees the smart_resize'd image.  Same call as the reference
            # (parser.py:135-139 -> layout_utils.py:115-144): its int(x / (origin_w / w)) differs from int(x * (w / origin_w))
            # by one pixel in ~0.06 % of cases, and the prompt string must be identical.
            from .utils.layout_utils import pre_process_bboxes
            bboxes = pre_process_bboxes(origin_image, [bbox], input_width=image.width, input_height=image.height,
                                        min_pixels=min_pixels or MIN_PIXELS, max_pixels=max_pixels or MAX_PIXELS)
            prompt = prompt + str(bboxes[0])
        return prompt

    # -- pages --------------------------------------------------------------------------------
    def _fetch_image(self, origin_image, min_pixels, max_pixels):
        """RGB conversion + the resize ``fetch_image`` applies when a pixel budget is given (image_utils.py:116-138)."""
        from .utils.image_utils import fetch_image
        return fetch_image(origin_image, min_pixels=min_pixels, max_pixels=max_pixels)

    def _parse_single_image(self, origin_image, prompt_mode, save_dir, save_name, source="image", page_idx=0, bbox=None,
                            fitz_preprocess=False):
        """One page: prompt -> model -> layout cells in page coordinates (.json) + Markdown (.md, _nohf.md), as the reference
        writes them (parser.py:143-253).  <name>.jpg is the page with the layout cells drawn on it (PIL overlay instead of the
        reference's PyMuPDF page), or the plain page when the response could not be parsed."""
        from .utils.layout_utils import draw_layout_on_image, post_process_output
        from .utils.format_transformer import layoutjson2md
        min_pixels, max_pixels = self.min_pixels, self.max_pixels
        if prompt_mode == "prompt_grounding_ocr":
            min_pixels = min_pixels or MIN_PIXELS
            max_pixels = max_pixels or MAX_PIXELS
        if min_pixels is not None:
            assert min_pixels >= MIN_PIXELS, f"min_pixels should >= {MIN_PIXELS}"
        if max_pixels is not None:
            assert max_pixels <= MAX_PIXELS, f"max_pixels should <= {MAX_PIXELS}"
        if source == 'image' and fitz_preprocess:
            from .utils.doc_utils import get_image_by_fitz_doc          # re-render at self.dpi (parser.py:161-163)
            image = self._fetch_image(get_image_by_fitz_doc(origin_image, target_dpi=self.dpi), min_pixels, max_pixels)
        else:
            image = self._fetch_image(origin_image, min_pixels, max_pixels)
        input_height, input_width = smart_resize(image.height, image.width)
        prompt = self.get_prompt(prompt_mode, bbox, origin_image, image, min_pixels=min_pixels, max_pixels=max_pixels)
        response = self._inference_with_hf(image, prompt) if self.use_hf else self._inference_with_vllm(image, prompt)
        result = {'page_no': page_idx, 'input_height': input_height, 'input_width': input_width}
        if source == 'pdf':
            save_name = f"{save_name}_page_{page_idx}"
        os.makedirs(save_dir, exist_ok=True)

        def write(path, text):
            with open(path, 'w', encoding='utf-8') as w:
                w.write(text if text is not None else "")

        image_path = os.path.join(save_dir, f"{save_name}.jpg")
        origin_rgb = origin_image if getattr(origin_image, "mode", "RGB") == "RGB" else origin_image.convert("RGB")
        origin_rgb.save(image_path)
        result['layout_image_path'] = image_path
        md_path = os.path.join(save_dir, f"{save_name}.md")
        if prompt_mode in ('prompt_layout_all_en', 'prompt_layout_only_en', 'prompt_grounding_ocr'):
            cells, filtered = post_process_output(response, prompt_mode, origin_image, image, min_pixels=min_pixels, max_pixels=max_pixels)
            json_path = os.path.join(save_dir, f"{save_name}.json")
            result['layout_info_path'] = json_path
            if filtered and prompt_mode != 'prompt_layout_only_en':
                with open(json_path, 'w', encoding='utf-8') as w:
                    json.dump(response, w, ensure_ascii=False)
                write(md_path, cells)
                result.update({'md_content_path': md_path, 'filtered': True})
            else:
                with open(json_path, 'w', encoding='utf-8') as w:
                    json.dump(cells, w, ensure_ascii=False)
                try:                                                    # the page with its layout drawn on it (parser.py:209-220)
                    draw_layout_on_image(origin_rgb, cells).save(image_path)
                except Exception as e:
                    print(f"Error drawing layout on image: {e}")
                if prompt_mode != 'prompt_layout_only_en' and not filtered:
                    nohf_path = os.path.join(save_dir, f"{save_name}_nohf.md")
                    write(md_path, layoutjson2md(origin_rgb, cells, text_key='text'))
                    write(nohf_path, layoutjson2md(origin_rgb, cells, text_key='text', no_page_hf=True))
                    result.update({'md_content_path': md_path, 'md_content_nohf_path': nohf_path})
        else:
            write(md_path, response)
            result['md_content_path'] = md_path
        return result

    def parse_image(self, input_path, filename, prompt_mode, save_dir, bbox=None, fitz_preprocess=False):
        from .utils.image_utils import fetch_image
        origin_image = fetch_image(input_path)          # path, file://, http(s)://, data: URL or PIL image -> RGB (parser.py:256)
        result = self._parse_single_image(origin_image, prompt_mode, save_dir, filename, source="image", bbox=bbox,
                                          fitz_preprocess=fitz_preprocess)
        result['file_path'] = input_path if isinstance(input_path, str) else filename
        return [result]

    def parse_pages(self, images, filename, prompt_mode, save_dir, file_path=None):
        """The pages of one document (PIL images, in order) -> one result per page, sorted by ``page_no``; outputs are named
        ``<filename>_page_<i>.*`` as for a PDF (parser.py:261-297).  Up to ``num_thread`` pages are in flight at once, in
        both modes: the threads block in the request batcher, which is what turns a document into batched ``generate``
        calls (the reference drops to one thread under ``use_hf`` because the HF model object is not re-entrant)."""
        from multiprocessing.pool import ThreadPool
        images = list(images)
        if not images:
            return []
        tasks = [dict(origin_image=im, prompt_mode=prompt_mode, save_dir=save_dir, save_name=filename, source="pdf", page_idx=i)
                 for i, im in enumerate(images)]
        with ThreadPool(max(1, min(len(tasks), int(self.num_thread)))) as pool:
            results = list(pool.imap_unordered(lambda kw: self._parse_single_image(**kw), tasks))
        results.sort(key=lambda r: r["page_no"])
        for r in results:
            r['file_path'] = file_path if file_path is not None else filename
        return results

    def parse_pdf(self, input_path, filename, prompt_mode, save_dir):
        from .utils.doc_utils import load_images_from_pdf
        return self.parse_pages(load_images_from_pdf(input_path, dpi=self.dpi), filename, prompt_mode, save_dir, file_path=input_path)

    def parse_file(self, input_path, output_dir="", prompt_mode="prompt_layout_all_en", bbox=None, fitz_preprocess=False):
        output_dir = os.path.abspath(output_dir or self.output_dir)
        filename, file_ext = os.path.splitext(os.path.basename(input_path))
        save_dir = os.path.join(output_dir, filename)
        os.makedirs(save_dir, exist_ok=True)
        if file_ext == '.pdf':
            results = self.parse_pdf(input_path, filename, prompt_mode, save_dir)
        elif file_ext in image_extensions:
            results = self.parse_image(input_path, filename, prompt_mode, save_dir, bbox=bbox, fitz_preprocess=fitz_preprocess)
        else:
            raise ValueError(f"file extension {file_ext} not supported, supported extensions are {image_extensions} and pdf")
        with open(os.path.join(output_dir, os.path.basename(filename) + '.jsonl'), 'w', encoding='utf-8') as w:
            for result in results:
                w.write(json.dumps(result, ensure_ascii=False) + '\n')
        return results


_CLI_OPTIONS = (
    # (flag, type, default): the reference CLI's options (dots_ocr/parser.py:325-407), same names and defaults
    ("--output", str, "./output"), ("--protocol", str, "http"), ("--ip", str, "localhost"), ("--port", int, 8000),
    ("--model_name", str, "model"), ("--temperature", float, 0.1), ("--top_p", float, 1.0), ("--dpi", int, 200),
    ("--max_completion_tokens", int, 16384), ("--num_thread", int, 16), ("--min_pixels", int, None), ("--max_pixels", int, None),
)


def main(argv=None):
    """``python -m dots_ocr_b200.parser page.jpg [--use_hf true] ...``: the reference's command line on the B200 engine.
    Pages are served in process when this process can see a GPU (or a runner was installed with ``set_default_runner``);
    on a machine without one, and without ``--use_hf``, requests go to ``--ip/--port`` over HTTP like the reference
    (``python -m dots_ocr_b200.server`` answers them).  See ``model/inference.py``."""
    import argparse
    ap = argparse.ArgumentParser(description="dots.ocr document layout parser on the B200 engine")
    ap.add_argument("input_path", type=str, help="input PDF / image file")
    ap.add_argument("--prompt", choices=list(dict_promptmode_to_prompt), default="prompt_layout_all_en")
    ap.add_argument("--bbox", type=int, nargs=4, metavar=("x1", "y1", "x2", "y2"), help="required by prompt_grounding_ocr")
    for flag, typ, default in _CLI_OPTIONS:
        ap.add_argument(flag, type=typ, default=default)
    ap.add_argument("--no_fitz_preprocess", action="store_true", help="skip the PyMuPDF re-render of image inputs at --dpi")
    ap.add_argument("--use_hf", type=lambda v: str(v).lower() in ("1", "true", "yes"), default=False,
                    help="serve pages with the in-process engine instead of an HTTP endpoint")
    a = ap.parse_args(argv)
    fitz_preprocess = not a.no_fitz_preprocess
    if fitz_preprocess:
        try:
            from .utils.doc_utils import _fitz
            _fitz()
        except ImportError:
            print("PyMuPDF is not installed: image inputs are used as they are (--no_fitz_preprocess)")
            fitz_preprocess = False
    p = DotsOCRParser(protocol=a.protocol, ip=a.ip, port=a.port, model_name=a.model_name, temperature=a.temperature, top_p=a.top_p,
                      max_completion_tokens=a.max_completion_tokens, num_thread=a.num_thread, dpi=a.dpi, output_dir=a.output,
                      min_pixels=a.min_pixels, max_pixels=a.max_pixels, use_hf=a.use_hf)
    results = p.parse_file(a.input_path, prompt_mode=a.prompt, bbox=a.bbox, fitz_preprocess=fitz_preprocess)
    print(f"{len(results)} page(s) written under {os.path.abspath(a.output)}")
    return results


if __name__ == "__main__":
    main()
