"""In-process engine for the dots.ocr page-parsing hot path on one B200.

Replaces what ``self.model.generate(**inputs, max_new_tokens=N)`` does in the reference
(``dots_ocr/parser.py:110``): DotsVisionTransformer forward -> embed + masked_scatter ->
Qwen2 prefill -> greedy decode with a KV cache.  Host code is Python; every device operation
is a call into libdots_ocr_b200.so (``ops``).  torch is used for tensor storage, streams and a
handful of index-array constructions on the host side.

Layout in HBM (all bf16 unless noted):
  * weights: nn.Linear layout [out, in]; fused qkv; gate|up (fc1|fc3) interleaved per 256 rows
    as [64 gate | 64 up] per 128 rows so both SwiGLU epilogues (prefill: 256-wide accumulator tile; decode swap-AB:
    128-row tile) find matching gate/up features in one tile.
  * activations: token-major packed [sum_tokens, width] (no padding between sequences).
  * KV cache: [layers, batch, kv_heads, ctx_max, 128], appended in place.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Dict, List, Optional

import torch

from . import ops
from .config import DotsConfig


def _interleave_gate_up(gate: torch.Tensor, up: torch.Tensor) -> torch.Tensor:
    I, H = gate.shape
    assert I % 128 == 0, "intermediate size must be a multiple of 128"
    g = gate.view(I // 64, 64, H)
    u = up.view(I // 64, 64, H)
    return torch.stack([g, u], dim=1).reshape(2 * I, H).contiguous()


def _round_up(x: int, m: int) -> int:
    return (x + m - 1) // m * m


def _on_device(fn):
    """Run an Engine method with the engine's GPU as the calling thread's current device.  CUDA's current device is
    per thread and new threads start on device 0, while the C-ABI launches go to the current device's stream: a request
    batcher or parser thread driving an engine on cuda:3 would otherwise launch on the wrong GPU."""
    import functools

    @functools.wraps(fn)
    def wrapper(self, *args, **kwargs):
        with torch.cuda.device(self.device):
            return fn(self, *args, **kwargs)
    return wrapper


def stop_list(eos_token_id) -> List[int]:
    """``eos_token_id`` as HF accepts it (None, an int, or a list of ints) -> ordered, de-duplicated list."""
    if eos_token_id is None:
        return []
    if isinstance(eos_token_id, (list, tuple)):
        return list(dict.fromkeys(int(e) for e in eos_token_id))
    if isinstance(eos_token_id, torch.Tensor):
        return list(dict.fromkeys(int(e) for e in eos_token_id.reshape(-1).tolist()))
    return [int(eos_token_id)]


def finalize_new_tokens(out_new: torch.Tensor, stops: List[int], pad: int) -> torch.Tensor:
    """The generated block [B, N] the way HF's greedy loop leaves it: everything after a row's first stop id is
    ``pad``, and the block ends at the step where the last row stopped (``GenerationMixin._sample``: finished rows
    keep emitting pad, the loop ends once every row has finished).  The decode kernels already stop a row on any of the
    first ``ops.MAX_STOP_IDS`` ids and pad behind it on the device; this pass is what makes longer lists correct too."""
    if not stops:
        return out_new
    hit = out_new == stops[0]
    for s in stops[1:]:
        hit |= out_new == s
    has = hit.any(dim=1)
    fin_step = hit.int().argmax(dim=1)
    if len(stops) > 1:
        col = torch.arange(out_new.shape[1], device=out_new.device).unsqueeze(0)
        after = has.unsqueeze(1) & (col > fin_step.unsqueeze(1))
        out_new = torch.where(after, torch.full_like(out_new, int(pad)), out_new)
    if bool(has.all()):
        out_new = out_new[:, : int(fin_step.max().item()) + 1]      # HF stops once every row has finished
    return out_new


def replay_steps(launch, n: int, every: int, all_finished) -> int:
    """Run ``launch()`` up to ``n`` times; after every ``every`` launches (0 = never) ask ``all_finished()`` (one
    device->host read of the finished flags) and stop early when it says so.  Returns the launches made."""
    done = 0
    while done < n:
        launch()
        done += 1
        if every and done % every == 0 and done < n and all_finished():
            break
    return done


@dataclass
class GenerateOutput:
    sequences: torch.Tensor                 # [B, T + N] int64 (prompt included, HF layout)
    logits: Optional[torch.Tensor] = None   # [B, N, V] bf16 pre-sampling logits (when requested)
    image_embeds: Optional[torch.Tensor] = None


class Engine:
    def __init__(self, cfg: DotsConfig, ckpt: Dict[str, torch.Tensor], device: str | torch.device = "cuda:0"):
        self.cfg = cfg
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("dots_ocr_b200.Engine needs a CUDA device (there is no CPU fallback)")
        from . import _lib
        _lib.load()
        torch.cuda.set_device(self.device)
        v, t = cfg.vision, cfg.text
        assert v.head_dim == 128 and t.head_dim == 128, "kernels are specialised for head_dim 128"
        dev = self.device

        def W(name):
            return ckpt[name].to(device=dev, dtype=torch.bfloat16).contiguous()

        # ---- vision tower ---------------------------------------------------------------
        self.patch_k = _round_up(v.patch_dim, 64)                   # 588 -> 640 (TMA row pitch % 16 B)
        pw = W("vision_tower.patch_embed.patchifier.proj.weight").reshape(v.embed_dim, v.patch_dim)
        self.v_patch_w = torch.zeros((v.embed_dim, self.patch_k), device=dev, dtype=torch.bfloat16)
        self.v_patch_w[:, : v.patch_dim] = pw
        self.v_patch_b = W("vision_tower.patch_embed.patchifier.proj.bias")
        self.v_patch_norm = W("vision_tower.patch_embed.patchifier.norm.weight")
        self.v_layers: List[dict] = []
        for i in range(v.num_hidden_layers):
            p = f"vision_tower.blocks.{i}."
            self.v_layers.append(dict(
                norm1=W(p + "norm1.weight"), qkv=W(p + "attn.qkv.weight"), proj=W(p + "attn.proj.weight"),
                norm2=W(p + "norm2.weight"),
                fc13=_interleave_gate_up(W(p + "mlp.fc1.weight"), W(p + "mlp.fc3.weight")),
                fc2=W(p + "mlp.fc2.weight")))
        self.v_post_norm = W("vision_tower.post_trunk_norm.weight")
        self.v_ln_w = W("vision_tower.merger.ln_q.weight")
        self.v_ln_b = W("vision_tower.merger.ln_q.bias")
        self.v_m0_w = W("vision_tower.merger.mlp.0.weight")
        self.v_m0_b = W("vision_tower.merger.mlp.0.bias")
        self.v_m2_w = W("vision_tower.merger.mlp.2.weight")
        self.v_m2_b = W("vision_tower.merger.mlp.2.bias")
        half = v.head_dim // 4                                      # 32 frequencies per axis
        dim = v.head_dim // 2
        self.v_inv_freq = (1.0 / (v.rope_theta ** (torch.arange(0, dim, 2, dtype=torch.float) / dim))).to(dev)
        assert self.v_inv_freq.numel() == half

        # ---- decoder --------------------------------------------------------------------
        self.embed = W("model.embed_tokens.weight")
        self.t_layers: List[dict] = []
        for i in range(t.num_hidden_layers):
            p = f"model.layers.{i}."
            qkv_w = torch.cat([W(p + "self_attn.q_proj.weight"), W(p + "self_attn.k_proj.weight"),
                               W(p + "self_attn.v_proj.weight")], dim=0).contiguous()
            qkv_b = torch.cat([W(p + "self_attn.q_proj.bias"), W(p + "self_attn.k_proj.bias"),
                               W(p + "self_attn.v_proj.bias")], dim=0).contiguous()
            L = dict(
                ln1=W(p + "input_layernorm.weight"), qkv_w=qkv_w, qkv_b=qkv_b, o=W(p + "self_attn.o_proj.weight"),
                ln2=W(p + "post_attention_layernorm.weight"),
                gu=_interleave_gate_up(W(p + "mlp.gate_proj.weight"), W(p + "mlp.up_proj.weight")),
                down=W(p + "mlp.down_proj.weight"))
            # second copy for the decode step: 128 x 64 tiles stored as contiguous 16 KB blobs in the tensor cores' shared-memory
            # image, so that a ring stage is one bulk copy (ops.tile_weight; +3.1 GB at full size)
            for k in ("qkv_w", "o", "gu", "down"):
                L[k + "_t"] = ops.tile_weight(L[k])
            self.t_layers.append(L)
        self.final_norm = W("model.norm.weight")
        self.lm_head = W("lm_head.weight")
        self.lm_head_t = ops.tile_weight(self.lm_head)
        hd = t.head_dim
        self.t_inv_freq = (1.0 / (t.rope_theta ** (torch.arange(0, hd, 2, dtype=torch.int64).float() / hd))).to(dev)
        self.sms = torch.cuda.get_device_properties(dev).multi_processor_count
        self.launches = 0       # C-ABI kernel launches issued (bench.py reports it)
        self.eos_check_every = 64       # decode steps between looks at the finished flags (only when a stop id is given)
        # Decode layer for batches <= 64 (DESIGN.md section 3):
        #   "tiled"  7 kernels per layer over pre-tiled operands fetched with bulk copies (split-K partials + finalize kernels)
        #   "fused"  5 kernels per layer: cluster split-K GEMMs with the reduction, residual add and RMSNorm on chip (DSMEM)
        #   "perop"  7 kernels per layer over row-major operands and tensor-map copies; the only mode for batches of 65..256
        self.decode_mode = "tiled"
        self.attn_splits = 0            # 0: planned from the batch size; n: force n key splits in decode attention (tuning runs)
        self.decode_sms = 0             # 0: plan the decode step for the whole device; n: for an SM partition of n SMs (pipeline.py)
        self._fused_ok: Dict[int, bool] = {}
        self._dec_cache: Optional[dict] = None
        self._cap_stream = torch.cuda.Stream(device=dev)
        self.decode_log: List[tuple] = []     # (algorithmic bytes, steps, start event, end event) of the last generate calls' decode loops

    # ------------------------------------------------------------------------------ vision
    @_on_device
    @torch.no_grad()
    def encode_pages_u8(self, pages, return_layers: bool = False, min_pixels: Optional[int] = None, max_pixels: Optional[int] = None):
        """ViT forward from uint8 RGB pages [H, W, 3] of ANY size.  The whole image processor runs on the GPU (SURVEY.md section
        8f N1): smart_resize picks the model size (multiples of 28 inside the pixel budget, image_utils.py:29-63), dots_resize_bicubic_u8
        resizes bit-identically to the CPU processor, dots_patchify_u8 rescales / normalises / patchifies.  A page costs 3 B per ORIGINAL
        pixel of host->device traffic instead of 12 B per resized pixel, and no host resize."""
        from .processing import CLIP_MEAN, CLIP_STD
        from .utils.consts import MIN_PIXELS, MAX_PIXELS
        from .utils.image_utils import smart_resize
        v = self.cfg.vision
        f = v.patch_size * v.spatial_merge_size
        sized = []
        for pg in pages:
            pg = pg.to(self.device)
            H, W = int(pg.shape[0]), int(pg.shape[1])
            rh, rw = smart_resize(H, W, factor=f, min_pixels=min_pixels or MIN_PIXELS, max_pixels=max_pixels or MAX_PIXELS)
            if (rh, rw) != (H, W):
                pg = ops.resize_u8(pg.contiguous(), rh, rw)
                self.launches += (1 if H != rh else 0) + (1 if W != rw else 0)
            sized.append(pg)
        pages = sized
        mean255 = (torch.tensor(CLIP_MEAN, dtype=torch.float32) * 255.0).tolist()
        std255 = (torch.tensor(CLIP_STD, dtype=torch.float32) * 255.0).tolist()
        grid = [[1, int(pg.shape[0]) // v.patch_size, int(pg.shape[1]) // v.patch_size] for pg in pages]
        S = sum(g[1] * g[2] for g in grid)
        xin = torch.empty((S, self.patch_k), device=self.device, dtype=torch.bfloat16)
        a = 0
        for pg, g in zip(pages, grid):
            n = g[1] * g[2]
            ops.patchify_u8(pg.to(self.device).contiguous(), v.patch_size, v.spatial_merge_size, mean255, std255, self.patch_k, out=xin[a:a + n])
            a += n
        self.launches += len(grid)
        return self.encode_images(None, grid, return_layers=return_layers, _xin=xin)

    @_on_device
    @torch.no_grad()
    def encode_images(self, pixel_values: Optional[torch.Tensor], image_grid_thw, return_layers: bool = False, _xin: Optional[torch.Tensor] = None):
        """DotsVisionTransformer.forward ([V] dots_ocr.py:580-611): pixel_values [sum S, 588] ->
        image embeddings [sum S / 4, hidden]."""
        v = self.cfg.vision
        dev = self.device
        grid = image_grid_thw.tolist() if torch.is_tensor(image_grid_thw) else [list(g) for g in image_grid_thw]
        seqlens, ghw = [], []
        for tt, h, w in grid:
            for _ in range(int(tt)):
                seqlens.append(int(h) * int(w))
                ghw.append([int(h), int(w)])
        S = sum(seqlens)
        if _xin is None:
            pv = pixel_values.to(dev)
            assert pv.shape == (S, v.patch_dim), (pv.shape, S, v.patch_dim)
        else:
            assert _xin.shape == (S, self.patch_k) and _xin.dtype == torch.bfloat16
        cu = torch.tensor([0] + list(torch.tensor(seqlens).cumsum(0).tolist()), dtype=torch.int32, device=dev)
        ghw_t = torch.tensor(ghw, dtype=torch.int32, device=dev)
        max_seqlen = max(seqlens)
        D, Hh = v.embed_dim, v.num_attention_heads
        scale = v.head_dim ** -0.5

        cos, sin = ops.vit_rope_table(cu, ghw_t, self.v_inv_freq, v.spatial_merge_size, S)
        xin = _xin if _xin is not None else ops.cast_pad(pv.contiguous(), self.patch_k)
        x = ops.gemm(xin, self.v_patch_w, epilogue=ops.EPI_BIAS, bias=self.v_patch_b)
        del xin
        x = ops.rmsnorm(x, self.v_patch_norm, v.rms_norm_eps, out=x)
        self.launches += 4
        normed = torch.empty_like(x)
        qkv = torch.empty((S, 3 * D), device=dev, dtype=torch.bfloat16)
        attn = torch.empty((S, D), device=dev, dtype=torch.bfloat16)
        act = torch.empty((S, v.intermediate_size), device=dev, dtype=torch.bfloat16)
        layers = [x.clone()] if return_layers else None
        for L in self.v_layers:
            ops.rmsnorm(x, L["norm1"], v.rms_norm_eps, out=normed)
            ops.gemm_rope(normed, L["qkv"], qkv, cos, sin, 2 * D)          # q|k|v projection + 2-D RoPE of q, k in the epilogue
            ops.attn_varlen(qkv[:, :D], qkv[:, D:2 * D], qkv[:, 2 * D:], attn, cu, max_seqlen, Hh, Hh, False, scale)
            ops.gemm(attn, L["proj"], out=x, epilogue=ops.EPI_RESIDUAL, residual=x)
            ops.rmsnorm(x, L["norm2"], v.rms_norm_eps, out=normed)
            ops.gemm(normed, L["fc13"], out=act, epilogue=ops.EPI_SWIGLU)
            ops.gemm(act, L["fc2"], out=x, epilogue=ops.EPI_RESIDUAL, residual=x)
            self.launches += 7
            if return_layers:
                layers.append(x.clone())
        del qkv, attn, act
        ops.rmsnorm(x, self.v_post_norm, v.rms_norm_eps, out=normed)
        ops.layernorm(normed, self.v_ln_w, self.v_ln_b, v.merger_ln_eps, out=x)
        merged = x.view(S // (v.spatial_merge_size ** 2), v.merge_dim)
        h = ops.gemm(merged, self.v_m0_w, epilogue=ops.EPI_BIAS_GELU, bias=self.v_m0_b)
        out = ops.gemm(h, self.v_m2_w, epilogue=ops.EPI_BIAS, bias=self.v_m2_b)
        self.launches += 4
        return (out, layers) if return_layers else out

    # ------------------------------------------------------------------------------ decoder
    def _alloc_cache(self, B: int, ctx_max: int):
        t = self.cfg.text
        shape = (t.num_hidden_layers, B, t.num_key_value_heads, ctx_max, t.head_dim)
        k = torch.empty(shape, device=self.device, dtype=torch.bfloat16)
        vv = torch.empty(shape, device=self.device, dtype=torch.bfloat16)
        return k, vv

    @torch.no_grad()
    def _prefill(self, ids_packed, slots, img_embeds, cu, seq_lens, positions, seq_of_tok, kc, vc, ctx_max, want_hidden=False):
        t = self.cfg.text
        dev = self.device
        T = ids_packed.numel()
        nq, nkv, hd = t.num_attention_heads, t.num_key_value_heads, t.head_dim
        scale = hd ** -0.5
        x = ops.embed_scatter(ids_packed, slots, self.embed, img_embeds)
        normed = torch.empty_like(x)
        qkv = torch.empty((T, (nq + 2 * nkv) * hd), device=dev, dtype=torch.bfloat16)
        attn = torch.empty((T, nq * hd), device=dev, dtype=torch.bfloat16)
        act = torch.empty((T, t.intermediate_size), device=dev, dtype=torch.bfloat16)
        max_len = int(max(seq_lens))
        self.launches += 1
        for li, L in enumerate(self.t_layers):
            ops.rmsnorm(x, L["ln1"], t.rms_norm_eps, out=normed)
            ops.gemm(normed, L["qkv_w"], out=qkv, epilogue=ops.EPI_BIAS, bias=L["qkv_b"])
            ops.llm_rope_kv_append(qkv, nq, nkv, positions, seq_of_tok, self.t_inv_freq, kc[li], vc[li], ctx_max)
            ops.attn_varlen(qkv[:, : nq * hd], qkv[:, nq * hd:(nq + nkv) * hd], qkv[:, (nq + nkv) * hd:], attn, cu, max_len,
                            nq, nkv, True, scale)
            ops.gemm(attn, L["o"], out=x, epilogue=ops.EPI_RESIDUAL, residual=x)
            ops.rmsnorm(x, L["ln2"], t.rms_norm_eps, out=normed)
            ops.gemm(normed, L["gu"], out=act, epilogue=ops.EPI_SWIGLU)
            ops.gemm(act, L["down"], out=x, epilogue=ops.EPI_RESIDUAL, residual=x)
            self.launches += 8
        return x

    @property
    def decode_fused(self) -> bool:
        return self.decode_mode == "fused"

    @decode_fused.setter
    def decode_fused(self, on: bool) -> None:
        self.decode_mode = "fused" if on else "perop"

    def _mode_for(self, B: int) -> str:
        """The decode-layer variant a batch of B rows runs with."""
        if B > 64 or self.decode_mode == "perop":
            return "perop"
        if self.decode_mode == "fused":
            # the cluster GEMMs rendezvous on a device-wide counter: every row-tile cluster of a launch must be resident at once
            key = 32 if B <= 32 else 64
            if key not in self._fused_ok:
                self._fused_ok[key] = ops.decode_gemm_max_clusters(key) >= -(-self.cfg.text.hidden_size // 128)
            return "fused" if self._fused_ok[key] else "tiled"
        return "tiled"

    def _decode_plan(self, B: int):
        t = self.cfg.text
        H, I = t.hidden_size, t.intermediate_size
        qkv_n = (t.num_attention_heads + 2 * t.num_key_value_heads) * t.head_dim
        kb = lambda k: -(-k // 64)
        tiles = lambda n: -(-n // 128)
        pairs = max(1, B * t.num_key_value_heads)
        mode = self._mode_for(B)
        sms = int(self.decode_sms) or self.sms
        if self.attn_splits:
            attn = int(self.attn_splits)
        else:
            # one CTA per (sequence, kv head) once that alone covers most SMs; flash-decoding splits below (<= 4 merge inside a
            # cluster, more go through the combine kernel)
            # (the attention CTA keeps a 128 KB K/V ring: one CTA per SM)
            attn = 1 if pairs >= (3 * sms) // 4 else max(1, min(16, sms // pairs))
        return dict(
            mode=mode, fused=(mode == "fused"),
            qkv=ops.pick_splits(tiles(qkv_n), kb(H), sms),
            o=ops.pick_splits(tiles(H), kb(t.num_attention_heads * t.head_dim), sms),
            gu=ops.pick_splits(tiles(2 * I), kb(H), sms),
            down=ops.pick_splits(tiles(H), kb(I), sms),
            attn=attn,
        )

    def _decode_step(self, st: dict):
        """One decode step for the whole batch; every call is a C-ABI kernel launch (graph-capturable)."""
        t = self.cfg.text
        nq, nkv, hd = t.num_attention_heads, t.num_key_value_heads, t.head_dim
        H, I = t.hidden_size, t.intermediate_size
        qkv_n = (nq + 2 * nkv) * hd
        pl = st["plan"]
        scale = hd ** -0.5
        n_layers = len(self.t_layers)
        B = st["resid"].shape[0]
        if pl["mode"] == "fused":
            R = st["tile_rows"]
            ops.decode_embed_rmsnorm(st["last"], self.embed, self.t_layers[0]["ln1"], st["resid"], st["normed_t"], t.rms_norm_eps,
                                     counters=st["counters"], tile_rows=R)
            for li, L in enumerate(self.t_layers):
                nxt = self.t_layers[li + 1]["ln1"] if li + 1 < n_layers else self.final_norm
                ops.decode_gemm_qkv(st["normed_t"], L["qkv_w_t"], L["qkv_b"], st["qkv"], H)
                ops.attn_decode_qkv(st["qkv"], st["pos"], self.t_inv_freq, st["kc"][li], st["vc"][li], st["ctx_len"], st["attn_t"], nq, nkv,
                                    st["ctx_max"], pl["attn"], scale, st["part_o"], st["part_ml"], out_tile_rows=R)
                ops.decode_gemm_resnorm(st["attn_t"], L["o_t"], st["resid"], L["ln2"], st["normed_t"], st["stats"][0],
                                        st["counters"][2 * li:2 * li + 1], t.rms_norm_eps, nq * hd)
                ops.decode_gemm_swiglu(st["normed_t"], L["gu_t"], st["act_t"], B, H)
                ops.decode_gemm_resnorm(st["act_t"], L["down_t"], st["resid"], nxt, st["normed_t"], st["stats"][1],
                                        st["counters"][2 * li + 1:2 * li + 2], t.rms_norm_eps, I)
            ops.decode_gemm_head(st["normed_t"], self.lm_head_t, st["logits"], t.vocab_size, H, tiled=True)
        elif pl["mode"] == "tiled":
            R = st["tile_rows"]
            ops.decode_embed_rmsnorm(st["last"], self.embed, self.t_layers[0]["ln1"], st["resid"], st["normed_t"], t.rms_norm_eps, tile_rows=R)
            for li, L in enumerate(self.t_layers):
                nxt = self.t_layers[li + 1]["ln1"] if li + 1 < n_layers else self.final_norm
                ops.decode_gemm_partial(st["normed_t"], L["qkv_w_t"], st["partial"], B, qkv_n, H, pl["qkv"])
                ops.attn_decode_fused(st["partial"], pl["qkv"], L["qkv_b"], st["pos"], self.t_inv_freq, st["kc"][li], st["vc"][li],
                                      st["ctx_len"], st["attn_t"], nq, nkv, st["ctx_max"], pl["attn"], scale, st["part_o"], st["part_ml"],
                                      out_tile_rows=R)
                ops.decode_gemm_partial(st["attn_t"], L["o_t"], st["partial"], B, H, nq * hd, pl["o"])
                ops.decode_residual_rmsnorm(st["partial"], pl["o"], st["resid"], L["ln2"], st["normed_t"], t.rms_norm_eps, tile_rows=R)
                ops.decode_gemm_swiglu(st["normed_t"], L["gu_t"], st["act_t"], B, H)
                ops.decode_gemm_partial(st["act_t"], L["down_t"], st["partial"], B, H, I, pl["down"])
                ops.decode_residual_rmsnorm(st["partial"], pl["down"], st["resid"], nxt, st["normed_t"], t.rms_norm_eps, tile_rows=R)
            ops.decode_gemm_head(st["normed_t"], self.lm_head_t, st["logits"], t.vocab_size, H, tiled=True)
        else:
            ops.decode_embed_rmsnorm(st["last"], self.embed, self.t_layers[0]["ln1"], st["resid"], st["normed"], t.rms_norm_eps)
            for li, L in enumerate(self.t_layers):
                ops.gemm_skinny(st["normed"], L["qkv_w"], pl["qkv"], partial=st["partial"])
                ops.attn_decode_fused(st["partial"], pl["qkv"], L["qkv_b"], st["pos"], self.t_inv_freq, st["kc"][li], st["vc"][li],
                                      st["ctx_len"], st["attn"], nq, nkv, st["ctx_max"], pl["attn"], scale, st["part_o"], st["part_ml"])
                nxt = self.t_layers[li + 1]["ln1"] if li + 1 < n_layers else self.final_norm
                ops.gemm_skinny(st["attn"], L["o"], pl["o"], partial=st["partial"])
                ops.decode_residual_rmsnorm(st["partial"], pl["o"], st["resid"], L["ln2"], st["normed"], t.rms_norm_eps)
                ops.gemm_skinny_swiglu(st["normed"], L["gu"], st["act"])
                ops.gemm_skinny(st["act"], L["down"], pl["down"], partial=st["partial"])
                ops.decode_residual_rmsnorm(st["partial"], pl["down"], st["resid"], nxt, st["normed"], t.rms_norm_eps)
            ops.gemm_skinny(st["normed"], self.lm_head, 1, out_bf16=st["logits"])
        self._select(st)

    @staticmethod
    def _select(st: dict) -> None:
        """Token selection + bookkeeping of one step: the sampling kernel when the state carries per-row sampling
        parameters, else the greedy argmax kernel."""
        if "temperature" in st:
            ops.sample_advance(st["logits"], st["last"], st["temperature"], st["top_p"], st["top_k"], st["seed"], st["out_ids"], st["step"],
                               st["pos"], st["ctx_len"], st["finished"], st["stops"], st["pad"], st["forced"])
        else:
            ops.argmax_advance(st["logits"], st["last"], st["out_ids"], st["step"], st["pos"], st["ctx_len"], st["finished"],
                               st["stops"], st["pad"], st["forced"])

    def _new_decode_state(self, B: int, lens: torch.Tensor, kc, vc, ctx_max: int, N: int, eos_token_id=None, pad_token_id: int = 0,
                          forced_ids: Optional[torch.Tensor] = None, sampling: bool = False) -> dict:
        """Every buffer one decode step touches (allocated once per generate; the CUDA graph captures their addresses).
        ``sampling``: also the per-row parameter arrays of ``dots_sample_advance`` (the values are written per call)."""
        t = self.cfg.text
        dev = self.device
        H = t.hidden_size
        stops = stop_list(eos_token_id)
        st = dict(plan=self._decode_plan(B), kc=kc, vc=vc, ctx_max=ctx_max, stops=tuple(stops[: ops.MAX_STOP_IDS]), pad=int(pad_token_id))
        pl = st["plan"]
        max_part = max(pl["qkv"] * (t.num_attention_heads + 2 * t.num_key_value_heads) * t.head_dim, pl["o"] * H, pl["down"] * H)
        st["partial"] = torch.empty(max_part * B, device=dev, dtype=torch.float32)
        st["resid"] = torch.empty((B, H), device=dev, dtype=torch.bfloat16)
        st["normed"] = torch.empty((B, H), device=dev, dtype=torch.bfloat16)
        st["attn"] = torch.empty((B, t.num_attention_heads * t.head_dim), device=dev, dtype=torch.bfloat16)
        st["act"] = torch.empty((B, t.intermediate_size), device=dev, dtype=torch.bfloat16)
        st["logits"] = torch.empty((B, t.vocab_size), device=dev, dtype=torch.bfloat16)
        st["part_o"] = torch.empty((B, t.num_attention_heads, pl["attn"], t.head_dim), device=dev, dtype=torch.float32)
        st["part_ml"] = torch.empty((B, t.num_attention_heads, pl["attn"], 2), device=dev, dtype=torch.float32)
        st["last"] = torch.zeros(B, device=dev, dtype=torch.int64)
        st["out_ids"] = torch.full((B, N), int(pad_token_id), device=dev, dtype=torch.int64)
        st["step"] = torch.zeros(B, device=dev, dtype=torch.int32)
        st["pos"] = (lens - 1).to(torch.int32)
        st["ctx_len"] = lens.to(torch.int32)
        st["finished"] = torch.zeros(B, device=dev, dtype=torch.int32)
        st["forced"] = forced_ids.to(dev).long().contiguous() if forced_ids is not None else None
        st["qkv"] = torch.empty((B, (t.num_attention_heads + 2 * t.num_key_value_heads) * t.head_dim), device=dev, dtype=torch.bfloat16)
        if pl["mode"] != "perop":
            # k-block-tiled activation buffers of the bulk-copy decode paths (rows beyond the batch stay zero)
            R = st["tile_rows"] = ops.decode_tile_rows(B)
            tiled = lambda k: torch.zeros(-(-k // 64) * R * 64, device=dev, dtype=torch.bfloat16)
            st["normed_t"], st["attn_t"], st["act_t"] = tiled(H), tiled(t.num_attention_heads * t.head_dim), tiled(t.intermediate_size)
        st["stats"] = torch.zeros((2, -(-H // 128) * 64), device=dev, dtype=torch.float32)
        st["counters"] = torch.zeros(2 * t.num_hidden_layers, device=dev, dtype=torch.int32)
        if sampling:
            st["temperature"] = torch.zeros(B, device=dev, dtype=torch.float32)
            st["top_p"] = torch.ones(B, device=dev, dtype=torch.float32)
            st["top_k"] = torch.zeros(B, device=dev, dtype=torch.int32)
            st["seed"] = torch.zeros(B, device=dev, dtype=torch.int64)
        return st

    def decode_weight_bytes(self) -> int:
        """bf16 bytes every decode step must stream: all decoder-layer weights + final norm + lm_head."""
        n = self.final_norm.numel() + self.lm_head.numel()
        for L in self.t_layers:
            n += sum(v.numel() for k, v in L.items() if not k.endswith("_t"))       # the tiled copies are the same parameters
        return 2 * n

    def decode_bytes(self, B: int, seq_lens, n_steps: int) -> float:
        """Algorithmic HBM bytes of `n_steps` decode steps: weights once per step + KV read of every visible
        key + KV write of the new token (BASELINE.md section 3: 28 672 B per token per sequence at full size)."""
        t = self.cfg.text
        per_tok = 2 * t.num_hidden_layers * t.num_key_value_heads * t.head_dim * 2
        total = float(n_steps) * self.decode_weight_bytes()
        for L in seq_lens:
            # step s (1-based) processes the token at position L + s - 1 and sees L + s keys
            total += per_tok * (n_steps * L + n_steps * (n_steps + 1) / 2.0) + per_tok * n_steps
        return total

    def launches_per_decode_step(self, B: int) -> int:
        pl = self._decode_plan(B)
        combine = 1 if pl["attn"] > 1 and not (ops.DECODE_CLUSTER and pl["attn"] <= ops.ATTN_DECODE_MAX_CLUSTER) else 0
        per_layer = (5 if pl["mode"] == "fused" else 7) + combine
        return 1 + per_layer * len(self.t_layers) + 2

    @_on_device
    @torch.no_grad()
    def generate(self, input_ids: torch.Tensor, attention_mask: Optional[torch.Tensor] = None,
                 pixel_values: Optional[torch.Tensor] = None, image_grid_thw=None, max_new_tokens: int = 16,
                 eos_token_id=None, pad_token_id: int = 0, forced_ids: Optional[torch.Tensor] = None,
                 return_logits: bool = False, use_graph: bool = True, image_embeds: Optional[torch.Tensor] = None,
                 pages_u8=None, min_pixels: Optional[int] = None, max_pixels: Optional[int] = None, sampling=None,
                 **unused) -> GenerateOutput:
        """HF-shaped generation: returns ids [B, T + N'] including the prompt (parser.py:110-113).  Greedy unless
        ``sampling`` (one ``SamplingParams`` for every row, or a sequence of B) or HF's ``do_sample=True`` (with
        ``temperature`` / ``top_p`` / ``top_k``, HF defaults 1.0 / 1.0 / 50) asks for sampling (dots_ocr_b200/sampling.py)."""
        from . import sampling as _sampling
        t = self.cfg.text
        dev = self.device
        ids = input_ids.to(dev).long()
        B, Tpad = ids.shape
        assert B <= 256, "batch > 256 pages per call is not supported; shard the pages"
        if sampling is None:
            sampling = _sampling.from_hf_kwargs(unused)
        rows = None if sampling is None else _sampling.per_row(sampling, B)
        mask = torch.ones_like(ids) if attention_mask is None else attention_mask.to(dev).long()
        lens = mask.sum(dim=1).to(torch.int64)
        seq_lens = lens.tolist()
        N = int(max_new_tokens)
        assert N >= 1
        ctx_max = _round_up(int(max(seq_lens)) + N, 64)

        # packed (un-padded) token stream; HF positions = cumsum(mask) - 1
        keep = mask.bool()
        ids_packed = ids[keep].contiguous()
        positions = (mask.cumsum(1) - 1)[keep].to(torch.int32).contiguous()
        seq_of_tok = torch.arange(B, device=dev, dtype=torch.int32).unsqueeze(1).expand(B, Tpad)[keep].contiguous()
        cu = torch.zeros(B + 1, dtype=torch.int32, device=dev)
        cu[1:] = lens.cumsum(0).to(torch.int32)

        if image_embeds is None and pages_u8 is not None:
            image_embeds = self.encode_pages_u8(pages_u8, min_pixels=min_pixels, max_pixels=max_pixels)    # the image processor on the GPU
        elif image_embeds is None and pixel_values is not None:
            image_embeds = self.encode_images(pixel_values, image_grid_thw)
        slots = None
        if image_embeds is not None:
            slots, count = ops.image_slots(ids_packed, self.cfg.image_token_id)
            self.launches += 1
            n_img = int(count.item())
            if n_img != image_embeds.shape[0]:
                raise ValueError(f"image tokens in input_ids ({n_img}) != image embedding rows ({image_embeds.shape[0]})")

        # KV cache, decode workspaces and the captured decode graph are kept from call to call when the shape key repeats
        # (a serving loop and the benchmark call generate with the same batch geometry over and over)
        stops_key = tuple(stop_list(eos_token_id)[: ops.MAX_STOP_IDS])
        key = (B, ctx_max, N, stops_key, int(pad_token_id), self.decode_mode, self.attn_splits, ops.DECODE_CLUSTER, int(self.decode_sms),
               rows is not None)
        ent = self._dec_cache if (self._dec_cache is not None and self._dec_cache["key"] == key and forced_ids is None) else None
        if ent is None:
            self._dec_cache = None                      # release the previous geometry's buffers before allocating new ones
            kc, vc = self._alloc_cache(B, ctx_max)
            st = self._new_decode_state(B, lens, kc, vc, ctx_max, N, eos_token_id, pad_token_id, forced_ids, sampling=rows is not None)
            ent = dict(key=key, st=st, graph=None)
            if forced_ids is None:
                self._dec_cache = ent
        else:
            st = ent["st"]
            kc, vc = st["kc"], st["vc"]
            st["last"].zero_()
            st["out_ids"].fill_(int(pad_token_id))
            st["step"].zero_()
            st["finished"].zero_()
            st["pos"].copy_((lens - 1).to(torch.int32))
            st["ctx_len"].copy_(lens.to(torch.int32))
        if rows is not None:
            for name, v in zip(("temperature", "top_p", "top_k", "seed"), _sampling.host_arrays(rows)):
                st[name].copy_(v)
        x = self._prefill(ids_packed, slots, image_embeds, cu, seq_lens, positions, seq_of_tok, kc, vc, ctx_max)
        pl = st["plan"]
        all_logits = torch.empty((N, B, t.vocab_size), device=dev, dtype=torch.bfloat16) if return_logits else None

        # first token: final norm + lm_head on each sequence's last prompt position
        last_rows = (cu[1:] - 1).to(torch.int32)
        hl = ops.gather_rows(x, last_rows)
        ops.rmsnorm(hl, self.final_norm, t.rms_norm_eps, out=st["normed"])
        ops.gemm_skinny(st["normed"], self.lm_head, 1, out_bf16=st["logits"])
        self._select(st)
        self.launches += 4
        del x
        if return_logits:
            all_logits[0].copy_(st["logits"])

        n_steps = N - 1
        per_step = self.launches_per_decode_step(B)
        # with a stop id, look at the finished flags every `eos_check_every` steps and leave once every page is done
        check = int(self.eos_check_every) if st["stops"] else 0

        def all_finished() -> bool:
            return bool(st["finished"].all().item())

        # two events around the decode loop (always on: they sit outside the PDL-chained kernels and cost nothing); bench.py
        # turns them into the decode-step HBM roofline
        prof_ev = None
        if n_steps > 0:
            prof_ev = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
            prof_ev[0].record()
        done = 0
        if n_steps > 0:
            if use_graph and not return_logits:
                if ent["graph"] is None:
                    self._decode_step(st)               # eager once (also warms every kernel variant)
                    done = 1
                if n_steps > done:
                    cap = self._cap_stream
                    cap.wait_stream(torch.cuda.current_stream())
                    with torch.cuda.stream(cap):
                        if ent["graph"] is None:
                            ent["graph"] = ops.capture(lambda: self._decode_step(st))      # capture does not execute
                        done += replay_steps(ent["graph"].launch, n_steps - done, check, all_finished)
                    torch.cuda.current_stream().wait_stream(cap)
                self.launches += per_step * done
            else:
                for s in range(n_steps):
                    self._decode_step(st)
                    done += 1
                    if return_logits:
                        all_logits[s + 1].copy_(st["logits"])
                    if check and done % check == 0 and done < n_steps and all_finished():
                        break
                self.launches += per_step * done

        if prof_ev is not None:
            prof_ev[1].record()
            self.decode_log.append((self.decode_bytes(B, seq_lens, done), done, prof_ev[0], prof_ev[1]))
            del self.decode_log[:-64]
        out_new = finalize_new_tokens(st["out_ids"], stop_list(eos_token_id), int(pad_token_id))
        seqs = torch.cat([ids, out_new], dim=1)
        if return_logits and out_new.shape[1] < N:
            all_logits = all_logits[: out_new.shape[1]]
        return GenerateOutput(sequences=seqs, logits=all_logits.transpose(0, 1) if return_logits else None,
                              image_embeds=image_embeds)
