"""Tensor-level wrappers over the C ABI.  PyTorch tensors are containers only: each function
checks dtype / device / alignment, then passes raw device pointers and the current CUDA stream.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional

import torch

from . import _lib

K = _lib.header_constants()
EPI_STORE, EPI_BIAS, EPI_BIAS_GELU, EPI_RESIDUAL, EPI_SWIGLU = (
    K["DOTS_EPI_STORE"], K["DOTS_EPI_BIAS"], K["DOTS_EPI_BIAS_GELU"], K["DOTS_EPI_RESIDUAL"], K["DOTS_EPI_SWIGLU"])

MAX_STOP_IDS = K["DOTS_MAX_STOP_IDS"]

_ll = C.c_longlong
_vp = C.c_void_p

# Optional profiling hook (bench.py): when a list, selected launches are bracketed by CUDA events on the
# launching stream and (kernel name, algorithmic work, start, end) is appended.
PROFILE = None


class _Prof:
    def __init__(self, name: str, work: float):
        self.on = PROFILE is not None
        if self.on:
            self.name, self.work = name, work
            self.e0 = torch.cuda.Event(enable_timing=True)
            self.e1 = torch.cuda.Event(enable_timing=True)

    def __enter__(self):
        if self.on:
            self.e0.record()
        return self

    def __exit__(self, *a):
        if self.on:
            self.e1.record()
            PROFILE.append((self.name, self.work, self.e0, self.e1))
        return False


def _stream() -> _vp:
    return _vp(torch.cuda.current_stream().cuda_stream)


def _p(t: Optional[torch.Tensor]) -> _vp:
    return _vp(0 if t is None else t.data_ptr())


def _bf16_2d(t: torch.Tensor, name: str) -> None:
    if not (t.is_cuda and t.dtype == torch.bfloat16 and t.dim() == 2 and t.stride(1) == 1):
        raise ValueError(f"{name}: need a CUDA bf16 2-D tensor with unit inner stride, got {t.dtype} {tuple(t.shape)} {t.stride()}")


def gemm(a: torch.Tensor, w: torch.Tensor, out: Optional[torch.Tensor] = None, epilogue: int = EPI_STORE,
         bias: Optional[torch.Tensor] = None, residual: Optional[torch.Tensor] = None) -> torch.Tensor:
    """out = epilogue(a @ w.T); a [M, K], w [N, K] (nn.Linear layout)."""
    _bf16_2d(a, "a"); _bf16_2d(w, "w")
    M, Kd = a.shape
    N = w.shape[0]
    assert w.shape[1] == Kd, (a.shape, w.shape)
    n_out = N // 2 if epilogue == EPI_SWIGLU else N
    if out is None:
        out = torch.empty((M, n_out), device=a.device, dtype=torch.bfloat16)
    _bf16_2d(out, "out")
    assert out.shape == (M, n_out), (out.shape, M, n_out)
    ldr = residual.stride(0) if residual is not None else 0
    with _Prof("gemm_bf16_tcgen05", 2.0 * M * N * Kd):
        rc = _lib.load().dots_gemm_bf16(_p(a), _ll(a.stride(0)), _p(w), _ll(w.stride(0)), _p(out), _ll(out.stride(0)),
                                        M, N, Kd, epilogue, _p(bias), _p(residual), _ll(ldr), _stream())
    _lib.check(rc, "dots_gemm_bf16")
    return out


def gemm_rope(a: torch.Tensor, w: torch.Tensor, out: torch.Tensor, cos: torch.Tensor, sin: torch.Tensor, rope_cols: int) -> torch.Tensor:
    """ViT q|k|v projection with the 2-D rotary embedding of q and k fused into the GEMM epilogue (out [M, N] bf16)."""
    _bf16_2d(a, "a"); _bf16_2d(w, "w"); _bf16_2d(out, "out")
    M, Kd = a.shape
    N = w.shape[0]
    assert out.shape == (M, N) and cos.dtype == torch.float32 and cos.shape == (M, 64) and sin.shape == (M, 64) and cos.is_contiguous()
    with _Prof("gemm_bf16_tcgen05", 2.0 * M * N * Kd):
        rc = _lib.load().dots_gemm_bf16_rope(_p(a), _ll(a.stride(0)), _p(w), _ll(w.stride(0)), _p(out), _ll(out.stride(0)), M, N, Kd,
                                             _p(cos), _p(sin), int(rope_cols), _stream())
    _lib.check(rc, "dots_gemm_bf16_rope")
    return out


def gemm_skinny(x: torch.Tensor, w: torch.Tensor, splits: int = 1, partial: Optional[torch.Tensor] = None,
                out_bf16: Optional[torch.Tensor] = None, bias: Optional[torch.Tensor] = None):
    """Decode GEMM (batch <= 256).  Returns fp32 partials [splits, B, N] or bf16 [B, N] when out_bf16 is given."""
    _bf16_2d(x, "x"); _bf16_2d(w, "w")
    B, Kd = x.shape
    N = w.shape[0]
    if out_bf16 is None and partial is None:
        partial = torch.empty((splits, B, N), device=x.device, dtype=torch.float32)
    if partial is not None:
        assert partial.dtype == torch.float32 and partial.is_contiguous() and partial.numel() >= splits * B * N
    ldo = out_bf16.stride(0) if out_bf16 is not None else 0
    rc = _lib.load().dots_gemm_skinny_bf16(_p(x), _ll(x.stride(0)), _p(w), _ll(w.stride(0)),
                                           _p(partial if out_bf16 is None else None), _p(out_bf16), _ll(ldo), _p(bias),
                                           B, N, Kd, splits, _stream())
    _lib.check(rc, "dots_gemm_skinny_bf16")
    return out_bf16 if out_bf16 is not None else partial


def gemm_skinny_swiglu(x: torch.Tensor, w_gu: torch.Tensor, act: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Decode gate|up projection with the SwiGLU fused into the GEMM epilogue: act [B, I] from x [B, K], w_gu [2I, K]."""
    _bf16_2d(x, "x"); _bf16_2d(w_gu, "w_gu")
    B, Kd = x.shape
    two_i = w_gu.shape[0]
    if act is None:
        act = torch.empty((B, two_i // 2), device=x.device, dtype=torch.bfloat16)
    _bf16_2d(act, "act")
    rc = _lib.load().dots_gemm_skinny_swiglu_bf16(_p(x), _ll(x.stride(0)), _p(w_gu), _ll(w_gu.stride(0)), _p(act), _ll(act.stride(0)),
                                                  B, two_i, Kd, _stream())
    _lib.check(rc, "dots_gemm_skinny_swiglu_bf16")
    return act


def pick_splits(n_tiles: int, num_kb: int, sms: int = 148) -> int:
    """Largest valid split-K factor s with n_tiles * s <= sms (every split non-empty)."""
    best = 1
    for s in range(1, num_kb + 1):
        per = -(-num_kb // s)
        if -(-num_kb // per) != s:
            continue
        if n_tiles * s <= sms:
            best = s
    return best


def _experiment(name: str):
    """Entry point of a kernel kept as a negative result (csrc/experiments/): present only in a library built with
    DOTS_BUILD_EXPERIMENTS=1."""
    lib = _lib.load()
    if not hasattr(lib, name):
        raise RuntimeError(f"{name} is an experiment kernel and is not in this build (DOTS_BUILD_EXPERIMENTS=1 python -m dots_ocr_b200.build --force)")
    fn = getattr(lib, name)
    fn.restype = C.c_int
    return fn


def has_experiments() -> bool:
    return hasattr(_lib.load(), "dots_decode_chain")


ATTN_IMPL = "tc"       # "tc": tcgen05/TMEM kernel (product path); "mma": mma.sync kernel (kept as the cross-check)


def attn_varlen(q, k, v, out, cu_seqlens, max_seqlen: int, n_q_heads: int, n_kv_heads: int, causal: bool,
                scale: float, head_dim: int = 128, impl: Optional[str] = None):
    """q/k/v/out: 2-D token-major views (may alias one fused qkv buffer)."""
    impl = impl or ATTN_IMPL
    for t in (q, k, v, out):
        assert t.is_cuda and t.dtype == torch.bfloat16 and t.stride(-1) == 1
    assert cu_seqlens.dtype == torch.int32 and cu_seqlens.is_cuda
    work = 0.0
    if PROFILE is not None:        # algorithmic FLOPs: 4 * L^2 * d per head (half that when causal)
        lens = (cu_seqlens[1:] - cu_seqlens[:-1]).double()
        work = float((lens * lens).sum().item()) * 4.0 * head_dim * n_q_heads * (0.5 if causal else 1.0)
    if impl in ("tc", "pair"):
        fn = _lib.load().dots_attn_varlen_fwd_tc if impl == "tc" else _experiment("dots_attn_varlen_fwd_pair")
        with _Prof("attn_fwd_prefill" if causal else "attn_fwd_vit", work):
            rc = fn(_p(q), _ll(q.stride(0)), _p(k), _ll(k.stride(0)), _p(v), _ll(v.stride(0)),
                                                     _p(out), _ll(out.stride(0)), _p(cu_seqlens), cu_seqlens.numel() - 1,
                                                     int(max_seqlen), _ll(q.shape[0]), n_q_heads, n_kv_heads, head_dim,
                                                     int(causal), C.c_float(scale), _stream())
        _lib.check(rc, "dots_attn_varlen_fwd_" + impl)
        return out
    with _Prof("attn_fwd_prefill" if causal else "attn_fwd_vit", work):
        rc = _lib.load().dots_attn_varlen_fwd(_p(q), _ll(q.stride(0)), _p(k), _ll(k.stride(0)), _p(v), _ll(v.stride(0)),
                                              _p(out), _ll(out.stride(0)), _p(cu_seqlens), cu_seqlens.numel() - 1,
                                              int(max_seqlen), n_q_heads, n_kv_heads, head_dim, int(causal),
                                              C.c_float(scale), _stream())
    _lib.check(rc, "dots_attn_varlen_fwd")
    return out


def attn_decode(q, k_cache, v_cache, ctx_len, out, n_q_heads: int, n_kv_heads: int, ctx_max: int, n_splits: int,
                scale: float, part_o=None, part_ml=None, head_dim: int = 128):
    B = q.shape[0]
    assert ctx_len.dtype == torch.int32
    if n_splits > 1:
        if part_o is None:
            part_o = torch.empty((B, n_q_heads, n_splits, head_dim), device=q.device, dtype=torch.float32)
        if part_ml is None:
            part_ml = torch.empty((B, n_q_heads, n_splits, 2), device=q.device, dtype=torch.float32)
    rc = _lib.load().dots_attn_decode(_p(q), _p(k_cache), _p(v_cache), _p(ctx_len), _p(out), _p(part_o), _p(part_ml),
                                      B, n_q_heads, n_kv_heads, head_dim, _ll(ctx_max), n_splits, C.c_float(scale),
                                      _stream())
    _lib.check(rc, "dots_attn_decode")
    return out


def attn_decode_fused(partial, qkv_splits: int, bias, pos, inv_freq, k_cache, v_cache, ctx_len, out, n_q_heads: int,
                      n_kv_heads: int, ctx_max: int, n_splits: int, scale: float, part_o=None, part_ml=None, head_dim: int = 128,
                      out_tile_rows: int = 0):
    """QKV finalize (split-K reduce + bias + RoPE + KV append) fused into the decode attention kernel."""
    B = ctx_len.numel()
    assert ctx_len.dtype == torch.int32 and pos.dtype == torch.int32 and partial.dtype == torch.float32
    if n_splits > 1:
        if part_o is None:
            part_o = torch.empty((B, n_q_heads, n_splits, head_dim), device=out.device, dtype=torch.float32)
        if part_ml is None:
            part_ml = torch.empty((B, n_q_heads, n_splits, 2), device=out.device, dtype=torch.float32)
    rc = _lib.load().dots_attn_decode_fused(_p(partial), qkv_splits, _p(bias), _p(pos), _p(inv_freq), _p(k_cache), _p(v_cache),
                                            _p(ctx_len), _p(out), int(out_tile_rows), _p(part_o), _p(part_ml), B, n_q_heads, n_kv_heads, head_dim,
                                            _ll(ctx_max), n_splits, C.c_float(scale), _stream())
    _lib.check(rc, "dots_attn_decode_fused")
    return out


def cast_pad(x: torch.Tensor, ldo: int, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    assert x.is_cuda and x.dim() == 2 and x.is_contiguous() and x.dtype in (torch.float32, torch.bfloat16)
    rows, cols = x.shape
    if out is None:
        out = torch.empty((rows, ldo), device=x.device, dtype=torch.bfloat16)
    rc = _lib.load().dots_cast_pad_bf16(_p(x), int(x.dtype == torch.bfloat16), _ll(rows), cols, _p(out), ldo, _stream())
    _lib.check(rc, "dots_cast_pad_bf16")
    return out


def patchify_u8(img: torch.Tensor, patch: int, merge: int, mean255, std255, ldo: int, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """uint8 HWC page on the device -> normalised, patchified, zero-padded bf16 rows [gh * gw, ldo] (merge-block token order)."""
    assert img.is_cuda and img.dtype == torch.uint8 and img.dim() == 3 and img.shape[2] == 3 and img.is_contiguous()
    H, W = int(img.shape[0]), int(img.shape[1])
    rows = (H // patch) * (W // patch)
    if out is None:
        out = torch.empty((rows, ldo), device=img.device, dtype=torch.bfloat16)
    assert out.shape == (rows, ldo) and out.is_contiguous()
    m = (C.c_float * 3)(*[float(v) for v in mean255])
    sd = (C.c_float * 3)(*[float(v) for v in std255])
    rc = _lib.load().dots_patchify_u8(_p(img), H, W, patch, merge, m, sd, _p(out), ldo, _stream())
    _lib.check(rc, "dots_patchify_u8")
    return out


_RESIZE_TABLES = {}


def _resize_tables(in_size: int, out_size: int, device):
    """Device copies of one axis's tap tables (dots_ocr_b200/resize.py), cached per (in, out, device)."""
    key = (in_size, out_size, str(device))
    t = _RESIZE_TABLES.get(key)
    if t is None:
        from .resize import axis_tables
        lo, n, w, prec = axis_tables(in_size, out_size)
        t = (torch.from_numpy(lo).to(device), torch.from_numpy(n).to(device), torch.from_numpy(w).to(device), int(w.shape[1]), int(prec))
        if len(_RESIZE_TABLES) < 512:
            _RESIZE_TABLES[key] = t
    return t


def resize_u8(img: torch.Tensor, rh: int, rw: int) -> torch.Tensor:
    """uint8 HWC page on the device -> [rh, rw, 3], bicubic + antialias, bit-identical to the CPU image processor's resize."""
    assert img.is_cuda and img.dtype == torch.uint8 and img.dim() == 3 and img.shape[2] == 3 and img.is_contiguous()
    H, W = int(img.shape[0]), int(img.shape[1])
    if (H, W) == (rh, rw):
        return img
    out = torch.empty((rh, rw, 3), device=img.device, dtype=torch.uint8)
    tmp = torch.empty((H, rw, 3), device=img.device, dtype=torch.uint8) if (H != rh and W != rw) else None
    tx = _resize_tables(W, rw, img.device) if W != rw else (None, None, None, 0, 0)
    ty = _resize_tables(H, rh, img.device) if H != rh else (None, None, None, 0, 0)
    rc = _lib.load().dots_resize_bicubic_u8(_p(img), H, W, _p(tmp), _p(out), rh, rw, _p(tx[0]), _p(tx[1]), _p(tx[2]), tx[3], tx[4],
                                            _p(ty[0]), _p(ty[1]), _p(ty[2]), ty[3], ty[4], _stream())
    _lib.check(rc, "dots_resize_bicubic_u8")
    return out


def rmsnorm(x: torch.Tensor, w: torch.Tensor, eps: float, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    _bf16_2d(x, "x")
    if out is None:
        out = torch.empty_like(x)
    rc = _lib.load().dots_rmsnorm(_p(x), _ll(x.stride(0)), _p(w), _p(out), _ll(out.stride(0)), _ll(x.shape[0]), x.shape[1],
                                  C.c_float(eps), _stream())
    _lib.check(rc, "dots_rmsnorm")
    return out


def layernorm(x, w, b, eps: float, out=None):
    _bf16_2d(x, "x")
    if out is None:
        out = torch.empty_like(x)
    rc = _lib.load().dots_layernorm(_p(x), _ll(x.stride(0)), _p(w), _p(b), _p(out), _ll(out.stride(0)), _ll(x.shape[0]),
                                    x.shape[1], C.c_float(eps), _stream())
    _lib.check(rc, "dots_layernorm")
    return out


def vit_rope_table(cu_seqlens, grid_hw, inv_freq, merge: int, total_tokens: int):
    half = inv_freq.numel()
    cos = torch.empty((total_tokens, 2 * half), device=cu_seqlens.device, dtype=torch.float32)
    sin = torch.empty_like(cos)
    rc = _lib.load().dots_vit_rope_table(_p(cu_seqlens), _p(grid_hw), grid_hw.shape[0], _p(inv_freq), half, merge, _p(cos),
                                         _p(sin), total_tokens, _stream())
    _lib.check(rc, "dots_vit_rope_table")
    return cos, sin


def vit_rope_apply(qkv: torch.Tensor, heads: int, cos, sin, head_dim: int = 128):
    _bf16_2d(qkv, "qkv")
    rc = _lib.load().dots_vit_rope_apply(_p(qkv), _ll(qkv.stride(0)), qkv.shape[0], heads, head_dim, _p(cos), _p(sin), _stream())
    _lib.check(rc, "dots_vit_rope_apply")
    return qkv


def llm_rope_kv_append(qkv, n_q_heads, n_kv_heads, positions, seq_of_tok, inv_freq, k_cache, v_cache, ctx_max, head_dim=128):
    _bf16_2d(qkv, "qkv")
    assert positions.dtype == torch.int32 and seq_of_tok.dtype == torch.int32 and inv_freq.dtype == torch.float32
    rc = _lib.load().dots_llm_rope_kv_append(_p(qkv), _ll(qkv.stride(0)), qkv.shape[0], n_q_heads, n_kv_heads, head_dim,
                                             _p(positions), _p(seq_of_tok), _p(inv_freq), _p(k_cache), _p(v_cache),
                                             _ll(ctx_max), _stream())
    _lib.check(rc, "dots_llm_rope_kv_append")


def image_slots(ids: torch.Tensor, image_token_id: int):
    assert ids.dtype == torch.int64 and ids.is_cuda and ids.is_contiguous()
    slots = torch.empty(ids.numel(), device=ids.device, dtype=torch.int32)
    count = torch.zeros(1, device=ids.device, dtype=torch.int32)
    rc = _lib.load().dots_image_slots(_p(ids), ids.numel(), _ll(image_token_id), _p(slots), _p(count), _stream())
    _lib.check(rc, "dots_image_slots")
    return slots, count


def embed_scatter(ids, slots, table, img_embeds, out=None):
    T = ids.numel()
    V, H = table.shape
    if out is None:
        out = torch.empty((T, H), device=ids.device, dtype=torch.bfloat16)
    rc = _lib.load().dots_embed_scatter(_p(ids), _p(slots), _p(table), _p(img_embeds), _p(out), T, H, _ll(V), _stream())
    _lib.check(rc, "dots_embed_scatter")
    return out


def gather_rows(src, rows, out=None):
    _bf16_2d(src, "src")
    assert rows.dtype == torch.int32
    n = rows.numel()
    if out is None:
        out = torch.empty((n, src.shape[1]), device=src.device, dtype=torch.bfloat16)
    rc = _lib.load().dots_gather_rows(_p(src), _ll(src.stride(0)), _p(rows), _p(out), _ll(out.stride(0)), n, src.shape[1], _stream())
    _lib.check(rc, "dots_gather_rows")
    return out


def argmax_advance(logits, next_ids, out_ids=None, step=None, pos=None, ctx_len=None, finished=None, stop_ids=(),
                   pad_id: int = 0, forced_ids=None):
    """``stop_ids``: an int (< 0 = none) or a sequence of up to DOTS_MAX_STOP_IDS ids; any of them finishes a row."""
    _bf16_2d(logits, "logits")
    B, V = logits.shape
    if isinstance(stop_ids, int):
        stop_ids = () if stop_ids < 0 else (stop_ids,)
    stops = [int(s) for s in stop_ids]
    if len(stops) > K["DOTS_MAX_STOP_IDS"]:
        raise ValueError(f"at most {K['DOTS_MAX_STOP_IDS']} stop ids are handled on the device, got {len(stops)}")
    arr = (_ll * max(1, len(stops)))(*stops)
    rc = _lib.load().dots_argmax_advance(_p(logits), _ll(logits.stride(0)), B, V, _p(next_ids), _p(out_ids),
                                         _ll(out_ids.stride(0) if out_ids is not None else 0), _p(step), _p(pos), _p(ctx_len),
                                         _p(finished), arr, len(stops), _ll(pad_id), _p(forced_ids),
                                         _ll(forced_ids.stride(0) if forced_ids is not None else 0), _stream())
    _lib.check(rc, "dots_argmax_advance")


def sample_advance(logits, next_ids, temperature, top_p, top_k, seed, out_ids=None, step=None, pos=None, ctx_len=None,
                   finished=None, stop_ids=(), pad_id: int = 0, forced_ids=None):
    """``argmax_advance`` with a sampled token per row (DESIGN.md section 3): ``temperature`` / ``top_p`` float32 [B],
    ``top_k`` int32 [B], ``seed`` int64 [B] (the bits of a u64) are device arrays read when the kernel runs, so a captured
    graph follows later writes to them.  Rows with temperature < 1e-5 get exactly what ``argmax_advance`` gives them."""
    _bf16_2d(logits, "logits")
    B, V = logits.shape
    for t, name, dt in ((temperature, "temperature", torch.float32), (top_p, "top_p", torch.float32),
                        (top_k, "top_k", torch.int32), (seed, "seed", torch.int64)):
        if not (t.is_cuda and t.dtype == dt and t.is_contiguous() and t.numel() == B):
            raise ValueError(f"{name}: need a contiguous CUDA {dt} tensor of {B} elements, got {t.dtype} {tuple(t.shape)}")
    if isinstance(stop_ids, int):
        stop_ids = () if stop_ids < 0 else (stop_ids,)
    stops = [int(s) for s in stop_ids]
    if len(stops) > K["DOTS_MAX_STOP_IDS"]:
        raise ValueError(f"at most {K['DOTS_MAX_STOP_IDS']} stop ids are handled on the device, got {len(stops)}")
    arr = (_ll * max(1, len(stops)))(*stops)
    rc = _lib.load().dots_sample_advance(_p(logits), _ll(logits.stride(0)), B, V, _p(next_ids), _p(out_ids),
                                         _ll(out_ids.stride(0) if out_ids is not None else 0), _p(step), _p(pos), _p(ctx_len),
                                         _p(finished), arr, len(stops), _ll(pad_id), _p(forced_ids),
                                         _ll(forced_ids.stride(0) if forced_ids is not None else 0), _p(temperature), _p(top_p),
                                         _p(top_k), _p(seed), _stream())
    _lib.check(rc, "dots_sample_advance")


def decode_embed_rmsnorm(ids, table, w, resid, normed, eps, counters=None, tile_rows: int = 0):
    """tile_rows > 0: ``normed`` is written k-block-tiled (the B operand of the cluster GEMMs), else row-major."""
    V, H = table.shape
    if counters is not None:
        assert counters.dtype == torch.int32 and counters.is_cuda
    rc = _lib.load().dots_decode_embed_rmsnorm(_p(ids), _p(table), _ll(V), _p(w), _p(resid), _p(normed), ids.numel(), H,
                                               C.c_float(eps), _p(counters), 0 if counters is None else counters.numel(), int(tile_rows), _stream())
    _lib.check(rc, "dots_decode_embed_rmsnorm")


def decode_tile_rows(batch: int) -> int:
    """Rows per tile of the k-block-tiled activation buffers of a decode step with this batch size."""
    assert 0 < batch <= 64
    return 32 if batch <= 32 else 64


def _tiled_act_ok(t: torch.Tensor, batch: int, K: int, name: str) -> None:
    need = -(-K // 64) * decode_tile_rows(batch) * 64
    if not (t.is_cuda and t.dtype == torch.bfloat16 and t.is_contiguous() and t.numel() >= need):
        raise ValueError(f"{name}: need a contiguous CUDA bf16 buffer of >= {need} elements (k-block-tiled [{batch}, {K}]), got {t.dtype} {tuple(t.shape)}")


def _tiled_w_ok(wt: torch.Tensor, N: int, K: int, name: str) -> None:
    if not (wt.is_cuda and wt.dtype == torch.bfloat16 and wt.is_contiguous() and tuple(wt.shape) == (-(-N // 128), -(-K // 64), 128 * 64)):
        raise ValueError(f"{name}: need ops.tile_weight(W) of a [{N}, {K}] weight, got {tuple(wt.shape)}")


def decode_gemm_qkv(xt: torch.Tensor, wt: torch.Tensor, bias: Optional[torch.Tensor], out: torch.Tensor, K: int) -> torch.Tensor:
    """q|k|v projection of a decode step (batch <= 64), split-K reduced inside thread-block clusters: out = bf16(x @ w.T + bias).
    xt: k-block-tiled activations [batch, K]; wt = tile_weight(w)."""
    _bf16_2d(out, "out")
    B, N = out.shape
    _tiled_act_ok(xt, B, K, "xt"); _tiled_w_ok(wt, N, K, "wt")
    rc = _lib.load().dots_decode_gemm_qkv(_p(xt), _p(wt), _p(bias), _p(out), _ll(out.stride(0)), B, N, K, _stream())
    _lib.check(rc, "dots_decode_gemm_qkv")
    return out


def decode_gemm_resnorm(xt: torch.Tensor, wt: torch.Tensor, resid: torch.Tensor, ln_w: torch.Tensor, normed_t: torch.Tensor, stats: torch.Tensor,
                        counter: torch.Tensor, eps: float, K: int) -> None:
    """o_proj / down_proj of a decode step with residual add and the next RMSNorm fused (batch <= 64):
    resid += bf16(x @ w.T) (row-major); normed_t = RMSNorm(resid) * ln_w (k-block-tiled).  ``counter``: one zeroed int32."""
    _bf16_2d(resid, "resid")
    B, N = resid.shape
    assert resid.is_contiguous()
    _tiled_act_ok(xt, B, K, "xt"); _tiled_act_ok(normed_t, B, N, "normed_t"); _tiled_w_ok(wt, N, K, "wt")
    assert stats.dtype == torch.float32 and stats.numel() >= -(-N // 128) * 64 and counter.dtype == torch.int32
    rc = _lib.load().dots_decode_gemm_resnorm(_p(xt), _p(wt), _p(resid), _p(ln_w), _p(normed_t), _p(stats), _p(counter), B, N, K, C.c_float(eps),
                                              _stream())
    _lib.check(rc, "dots_decode_gemm_resnorm")


def decode_gemm_partial(xt: torch.Tensor, wt: torch.Tensor, partial: torch.Tensor, batch: int, N: int, K: int, splits: int) -> torch.Tensor:
    """Split-K partials [splits, batch, N] fp32 over tiled operands (gemm_skinny with bulk-copied operands)."""
    _tiled_act_ok(xt, batch, K, "xt"); _tiled_w_ok(wt, N, K, "wt")
    assert partial.dtype == torch.float32 and partial.is_contiguous() and partial.numel() >= splits * batch * N
    rc = _lib.load().dots_decode_gemm_partial(_p(xt), _p(wt), _p(partial), batch, N, K, splits, _stream())
    _lib.check(rc, "dots_decode_gemm_partial")
    return partial


def decode_gemm_swiglu(xt: torch.Tensor, wt: torch.Tensor, act_t: torch.Tensor, batch: int, K: int) -> torch.Tensor:
    """gate|up + SwiGLU of a decode step over tiled operands; act_t (k-block-tiled [batch, I]) is the B operand of down_proj."""
    two_i = wt.shape[0] * 128
    _tiled_act_ok(xt, batch, K, "xt"); _tiled_act_ok(act_t, batch, two_i // 2, "act_t"); _tiled_w_ok(wt, two_i, K, "wt")
    rc = _lib.load().dots_decode_gemm_swiglu(_p(xt), _p(wt), _p(act_t), batch, two_i, K, _stream())
    _lib.check(rc, "dots_decode_gemm_swiglu")
    return act_t


def decode_gemm_head(x: torch.Tensor, wt: torch.Tensor, out: torch.Tensor, N: int, K: int, tiled: bool) -> torch.Tensor:
    """lm_head of a decode step: out [batch, N] = bf16(x @ w.T); x k-block-tiled (tiled=True) or row-major [batch, K]."""
    _bf16_2d(out, "out")
    B = out.shape[0]
    _tiled_w_ok(wt, N, K, "wt")
    if tiled:
        _tiled_act_ok(x, B, K, "x")
        ldx, rows = 0, decode_tile_rows(B)
    else:
        _bf16_2d(x, "x")
        assert x.shape == (B, K)
        ldx, rows = x.stride(0), 0
    rc = _lib.load().dots_decode_gemm_head(_p(x), _ll(ldx), rows, _p(wt), _p(out), _ll(out.stride(0)), B, N, K, _stream())
    _lib.check(rc, "dots_decode_gemm_head")
    return out


def decode_gemm_max_clusters(batch: int) -> int:
    n = C.c_int(0)
    _lib.check(_lib.load().dots_decode_gemm_max_clusters(int(batch), C.byref(n)), "dots_decode_gemm_max_clusters")
    return int(n.value)


def attn_decode_qkv(qkv, pos, inv_freq, k_cache, v_cache, ctx_len, out, n_q_heads: int, n_kv_heads: int, ctx_max: int, n_splits: int,
                    scale: float, part_o=None, part_ml=None, head_dim: int = 128, out_tile_rows: int = 0):
    """RoPE + KV append + decode attention from the bf16 q|k|v row of decode_gemm_qkv.  out_tile_rows > 0: ``out`` is a k-block-tiled
    activation buffer (B operand of o_proj), else row-major [B, n_q_heads * 128]."""
    _bf16_2d(qkv, "qkv")
    B = qkv.shape[0]
    assert qkv.is_contiguous() and ctx_len.dtype == torch.int32 and pos.dtype == torch.int32
    if out_tile_rows:
        _tiled_act_ok(out, B, n_q_heads * head_dim, "out")
    rc = _lib.load().dots_attn_decode_qkv(_p(qkv), _p(pos), _p(inv_freq), _p(k_cache), _p(v_cache), _p(ctx_len), _p(out), int(out_tile_rows),
                                          _p(part_o), _p(part_ml), B, n_q_heads, n_kv_heads, head_dim, _ll(ctx_max), n_splits, C.c_float(scale),
                                          _stream())
    _lib.check(rc, "dots_attn_decode_qkv")
    return out


ATTN_DECODE_MAX_CLUSTER = 4      # key splits the decode attention merges on chip (DEC_MAX_CLUSTER in attn_decode.cu)
DECODE_CLUSTER = True


def set_decode_cluster(enable: bool) -> None:
    global DECODE_CLUSTER
    DECODE_CLUSTER = bool(enable)
    _lib.check(_lib.load().dots_set_decode_cluster(int(bool(enable))), "dots_set_decode_cluster")


_PARTITIONS = {}      # device index -> (sms_first, stream_first, stream_rest, n_first, n_rest)


def partition(sms_first: int):
    """Split the current device's SMs into a first group of ``sms_first`` (multiple of 8) and the rest (CUDA green contexts).
    Returns ``(stream_first, stream_rest, n_first, n_rest)``: torch streams whose kernels run on their own SMs only.

    The partition lives as long as the process: torch's allocators remember every stream a tensor was used on (a pinned host
    buffer copied on a partition stream gets an event recorded on that stream when it is freed), so the streams must not die
    before the tensors do.  Asking again for the same split returns the same streams; a different split needs an explicit
    ``partition_destroy()`` first (only safe once nothing that touched the old streams is alive)."""
    dev = torch.cuda.current_device()
    have = _PARTITIONS.get(dev)
    if have is not None:
        if have[0] != int(sms_first):
            raise RuntimeError(f"device {dev} is already split {have[3]} + {have[4]} SMs; partition_destroy() before asking for {sms_first}")
        return have[1:]
    s0, s1 = _vp(0), _vp(0)
    n0, n1 = C.c_int(0), C.c_int(0)
    _lib.check(_lib.load().dots_partition_create(int(sms_first), C.byref(s0), C.byref(s1), C.byref(n0), C.byref(n1)), "dots_partition_create")
    ent = (int(sms_first), torch.cuda.ExternalStream(s0.value, device=dev), torch.cuda.ExternalStream(s1.value, device=dev), int(n0.value), int(n1.value))
    _PARTITIONS[dev] = ent
    return ent[1:]


def partition_destroy() -> None:
    _PARTITIONS.pop(torch.cuda.current_device(), None)
    _lib.check(_lib.load().dots_partition_destroy(), "dots_partition_destroy")


def set_sm_count(n: int) -> None:
    """Persistent kernels launched next size their grids for ``n`` SMs (an SM partition); 0 = the whole device."""
    _lib.check(_lib.load().dots_set_sm_count(int(n)), "dots_set_sm_count")


class on_partition:
    """``with on_partition(stream, n_sms):`` -- C-ABI launches and torch ops inside go to that partition's stream, grids sized for it."""

    def __init__(self, stream, n_sms: int):
        self.stream, self.n = stream, int(n_sms)
        self._ctx = None

    def __enter__(self):
        self._ctx = torch.cuda.stream(self.stream)
        self._ctx.__enter__()
        set_sm_count(self.n)
        return self

    def __exit__(self, *exc):
        set_sm_count(0)
        return self._ctx.__exit__(*exc)


def debug_set_trace(buf: Optional[torch.Tensor]) -> None:
    """Arm (int64 CUDA tensor: [0] = 0, [1] = capacity in records, 3 words per record after that) or disarm (None) the kernel timeline."""
    if buf is not None:
        assert buf.is_cuda and buf.dtype == torch.int64 and buf.is_contiguous()
    _lib.check(_lib.load().dots_debug_set_trace(_p(buf)), "dots_debug_set_trace")


def debug_set_fault(code: int) -> None:
    """Test-only fault injection (0 = off); see dots_debug_set_fault."""
    _lib.check(_lib.load().dots_debug_set_fault(int(code)), "dots_debug_set_fault")


def decode_residual_rmsnorm(partial, splits, resid, w, normed, eps, tile_rows: int = 0):
    B, H = resid.shape
    rc = _lib.load().dots_decode_residual_rmsnorm(_p(partial), splits, _p(resid), _p(w), _p(normed), B, H, C.c_float(eps), int(tile_rows), _stream())
    _lib.check(rc, "dots_decode_residual_rmsnorm")


def decode_qkv_rope_append(partial, splits, bias, pos, inv_freq, q_out, k_cache, v_cache, ctx_max, n_q_heads, n_kv_heads,
                           head_dim=128):
    B = q_out.shape[0]
    rc = _lib.load().dots_decode_qkv_rope_append(_p(partial), splits, _p(bias), _p(pos), _p(inv_freq), _p(q_out), _p(k_cache),
                                                 _p(v_cache), _ll(ctx_max), B, n_q_heads, n_kv_heads, head_dim, _stream())
    _lib.check(rc, "dots_decode_qkv_rope_append")


def decode_swiglu(partial, splits, act):
    B, I = act.shape
    rc = _lib.load().dots_decode_swiglu(_p(partial), splits, _p(act), B, I, _stream())
    _lib.check(rc, "dots_decode_swiglu")


def decode_chain(attn, w_o, w_gu, w_down, w_qkv_next, partial, resid, normed, act, ln_mid, ln_next, counters, splits_o: int,
                 splits_down: int, splits_qkv: int, eps: float):
    """Persistent per-layer decode kernel: o_proj -> norm -> gate|up+SwiGLU -> down_proj -> norm -> [next layer's qkv]."""
    B, H = resid.shape
    inter = act.shape[1]
    assert counters.dtype == torch.int32 and counters.numel() >= 8 and partial.dtype == torch.float32
    qkv_n = w_qkv_next.shape[0] if w_qkv_next is not None else 0
    rc = _experiment("dots_decode_chain")(_p(attn), _p(w_o), _p(w_gu), _p(w_down), _p(w_qkv_next), _p(partial), _p(resid), _p(normed),
                                       _p(act), _p(ln_mid), _p(ln_next), _p(counters), B, H, inter, qkv_n, attn.shape[1], splits_o,
                                       splits_down, splits_qkv, C.c_float(eps), _stream())
    _lib.check(rc, "dots_decode_chain")


def set_decode_stages(partial: int = 6, swiglu: int = 5, head: int = 4) -> None:
    """Ring depths of the decode GEMM families (tuning; see dots_set_decode_stages)."""
    _lib.check(_lib.load().dots_set_decode_stages(int(partial), int(swiglu), int(head)), "dots_set_decode_stages")


def set_gemm_pair(enable: bool) -> None:
    """CTA-pair (cta_group::2) kernel for large prefill GEMMs."""
    _lib.check(_lib.load().dots_set_gemm_pair(int(bool(enable))), "dots_set_gemm_pair")


def set_pdl(enable: bool) -> None:
    """Programmatic dependent launch between consecutive kernels (default on)."""
    _lib.check(_lib.load().dots_set_pdl(int(bool(enable))), "dots_set_pdl")


class Graph:
    """Capture the C-ABI launches issued inside the ``with`` block on the current stream."""

    def __init__(self):
        self.exec = _vp(0)

    def __enter__(self):
        _lib.check(_lib.load().dots_graph_begin(_stream()), "dots_graph_begin")
        return self

    def __exit__(self, et, ev, tb):
        ex = _vp(0)
        rc = _lib.load().dots_graph_end(_stream(), C.byref(ex))
        if et is None:
            _lib.check(rc, "dots_graph_end")
            self.exec = ex
        return False

    def launch(self):
        _lib.check(_lib.load().dots_graph_launch(self.exec, _stream()), "dots_graph_launch")

    def __del__(self):
        try:
            if self.exec:
                _lib.load().dots_graph_destroy(self.exec)
        except Exception:
            pass


def capture(fn) -> Graph:
    """Capture ``fn()`` (C-ABI launches on the current stream) into a replayable graph.  A driver that cannot record
    programmatic-dependent-launch edges fails the capture with a stream-capture error: only then is PDL switched off
    (for the process, with a warning) and the capture retried; any other failure propagates unchanged."""
    try:
        g = Graph()
        with g:
            fn()
        return g
    except RuntimeError as e:
        msg = str(e).lower()
        if not any(k in msg for k in ("capture", "not permitted", "not supported", "unsupported")):
            raise
        import warnings
        warnings.warn(f"CUDA graph capture with programmatic dependent launch failed ({e}); retrying with PDL off")
        set_pdl(False)
        g = Graph()
        with g:
            fn()
        return g


# ---------------------------------------------------------------------------------------------------------------------
# Pre-tiled HBM layouts of the decode step.  A 2-D tensor-map copy of a [rows x 128 B] box costs one L2 request per row
# and tops out near 40 GB/s per SM on B200, a 1-D bulk copy of the same bytes streams at > 100 GB/s per SM
# (profiles/microbench_r2.md).  Everything a decode step streams is therefore stored as contiguous blobs that already
# have the shared-memory image the tensor cores / ldmatrix expect (128-byte rows, 16-byte chunks XOR-swizzled by row & 7,
# i.e. what a SWIZZLE_128B tensor-map copy would have produced) and is fetched with cp.async.bulk.
# ---------------------------------------------------------------------------------------------------------------------
def _swizzle_chunks(t: torch.Tensor) -> torch.Tensor:
    """t [..., rows, 8 chunks, 8 elems]: chunk p of row r receives source chunk p ^ (r & 7)."""
    rows = t.shape[-3]
    r7 = (torch.arange(rows, device=t.device) & 7).view(rows, 1)
    src = (torch.arange(8, device=t.device).view(1, 8) ^ r7)                     # [rows, 8]
    idx = src.view(*([1] * (t.dim() - 3)), rows, 8, 1).expand(*t.shape)
    return t.gather(-2, idx)


def tile_weight(w: torch.Tensor) -> torch.Tensor:
    """[N, K] bf16 nn.Linear weight -> [ceil(N/128), ceil(K/64), 128 x 64] blobs of 16 KB (zero padded), each the K-major
    SWIZZLE_128B image of that 128-row x 64-column tile: the A operand of a swap-AB decode GEMM stage in ONE bulk copy."""
    assert w.dim() == 2 and w.dtype == torch.bfloat16
    N, K = w.shape
    Np, Kp = -(-N // 128) * 128, -(-K // 64) * 64
    if (Np, Kp) != (N, K):
        wp = torch.zeros((Np, Kp), device=w.device, dtype=w.dtype)
        wp[:N, :K] = w
        w = wp
    t = w.view(Np // 128, 128, Kp // 64, 8, 8).permute(0, 2, 1, 3, 4)            # [tile, kb, r, c, e]
    return _swizzle_chunks(t).contiguous().view(Np // 128, Kp // 64, 128 * 64)


def tile_rows(x: torch.Tensor, rows_per_tile: int) -> torch.Tensor:
    """[B <= rows_per_tile, K] bf16 activations -> [ceil(K/64), rows_per_tile x 64] blobs (the B operand of one k-block)."""
    assert x.dim() == 2 and x.dtype == torch.bfloat16 and x.shape[0] <= rows_per_tile and rows_per_tile % 8 == 0
    B, K = x.shape
    Kp = -(-K // 64) * 64
    xp = torch.zeros((rows_per_tile, Kp), device=x.device, dtype=x.dtype)
    xp[:B, :K] = x
    t = xp.view(rows_per_tile, Kp // 64, 8, 8).permute(1, 0, 2, 3)               # [kb, r, c, e]
    return _swizzle_chunks(t).contiguous().view(Kp // 64, rows_per_tile * 64)


def untile_rows(t: torch.Tensor, B: int, K: int) -> torch.Tensor:
    """Inverse of tile_rows: [ceil(K/64), rows x 64] -> [B, K]."""
    kb, n = t.shape
    rows = n // 64
    u = _swizzle_chunks(t.view(kb, rows, 8, 8))                                   # the XOR swizzle is its own inverse
    return u.permute(1, 0, 2, 3).reshape(rows, kb * 64)[:B, :K].contiguous()


def kv_tile(x: torch.Tensor) -> torch.Tensor:
    """[..., ctx, 128] (ctx % 64 == 0) row-major keys or values -> the cache layout: per 64-key tile a 16 KB blob
    [dims 0-63 | dims 64-127][64 keys][8 chunks swizzled by key & 7] (same shape, different element order)."""
    assert x.shape[-1] == 128 and x.shape[-2] % 64 == 0
    lead, ctx = x.shape[:-2], x.shape[-2]
    t = x.reshape(*lead, ctx // 64, 64, 2, 8, 8).transpose(-4, -3)               # [..., tile, half, key, c, e]
    return _swizzle_chunks(t).contiguous().view(*lead, ctx, 128)


def kv_untile(x: torch.Tensor) -> torch.Tensor:
    """Inverse of kv_tile (tests / debugging): cache layout -> [..., ctx, 128] row-major."""
    lead, ctx = x.shape[:-2], x.shape[-2]
    t = _swizzle_chunks(x.reshape(*lead, ctx // 64, 2, 64, 8, 8))
    return t.transpose(-4, -3).reshape(*lead, ctx, 128).contiguous()
