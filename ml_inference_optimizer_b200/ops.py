"""Torch-facing wrappers over the C-ABI (``include/b200_attn_mlp.h``).

PyTorch is plumbing here: it owns device memory and streams; the arithmetic happens in the hand-written sm_100a
kernels behind ``libb200_attn_mlp.so``. Every function raises (``B200Error`` / ``ValueError``) instead of falling
back to eager PyTorch.

Function ↔ reference map (paths under the reference tree):
  flash_attn_fwd      ↔ kernels/triton/flash_attention_kernels.py:1150 ``triton_flash_attention``
  decode_attention    ↔ kernels/triton/attention_kernels.py:1206 ``triton_paged_attention_forward``
  kv_append           ↔ kernels/triton/attention_kernels.py:1314 ``triton_reshape_and_cache``
  fused_mlp           ↔ kernels/triton/mlp_kernels.py:648 ``triton_fused_mlp``
  lse_merge           ↔ kernels/triton/attention_kernels.py:1567-1585 (online-softmax merge algebra)
"""
from __future__ import annotations

import ctypes
import math
from typing import Optional, Tuple

import torch

from . import _lib
from ._lib import (ACT_GELU_ERF, ACT_GELU_TANH, ACT_NONE, ACT_RELU, ACT_SWIGLU, DTYPE_BF16, DTYPE_FP16, KV_CONTIGUOUS,
                   KV_PAGED, check, strides3)

_ACTIVATIONS = {
    None: ACT_NONE, "none": ACT_NONE, "identity": ACT_NONE,
    "gelu_tanh": ACT_GELU_TANH, "gelu_new": ACT_GELU_TANH, "gelu_pytorch_tanh": ACT_GELU_TANH,
    "gelu": ACT_GELU_ERF, "gelu_erf": ACT_GELU_ERF,
    "relu": ACT_RELU,
    "swiglu": ACT_SWIGLU, "silu": ACT_SWIGLU,
}


def _dtype_code(t: torch.Tensor) -> int:
    if t.dtype == torch.bfloat16:
        return DTYPE_BF16
    if t.dtype == torch.float16:
        return DTYPE_FP16
    raise ValueError(f"b200 kernels compute on bf16/fp16 tensors, got {t.dtype}")


def _require_cuda(*tensors: Optional[torch.Tensor]) -> torch.device:
    dev = None
    for t in tensors:
        if t is None:
            continue
        if not t.is_cuda:
            raise RuntimeError("b200 kernels need CUDA tensors: there is no CPU fallback for this path")
        if dev is None:
            dev = t.device
        elif t.device != dev:
            raise ValueError("all tensors must be on the same CUDA device")
    return dev


def _stream_ptr(dev: torch.device) -> int:
    return torch.cuda.current_stream(dev).cuda_stream


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _last_dim_contiguous(t: torch.Tensor) -> torch.Tensor:
    return t if t.stride(-1) == 1 else t.contiguous()


def cache_head_dim(head_dim: int) -> int:
    """Head width a KV cache is allocated with: the decode kernels and ``kv_append`` are built for 64 and 128 columns, so a
    narrower head (any multiple of 8) is stored in the next wider cache with zero columns behind it — exact, the zeros add
    nothing to a score and produce zero outputs. q / k / v narrower than the cache are padded on the fly by the ops below."""
    if head_dim <= 0 or head_dim % 8 != 0 or head_dim > 128:
        raise ValueError(f"head_dim {head_dim} unsupported (a multiple of 8, at most 128)")
    return 64 if head_dim <= 64 else 128


def _pad_head(t: torch.Tensor, width: int) -> torch.Tensor:
    return t if t.shape[-1] == width else torch.nn.functional.pad(t, (0, width - t.shape[-1]))


#: element type of an FP8 KV cache (e4m3, max finite 448); the format is defined in include/b200_attn_mlp.h
FP8 = torch.float8_e4m3fn


def _fp8_cache(k_cache: torch.Tensor, v_cache: torch.Tensor, block_tables: Optional[torch.Tensor], k_scale: float,
               v_scale: float) -> bool:
    """True for an FP8 cache pair. Scales other than 1.0 belong to an FP8 cache; an FP8 cache is paged."""
    fp8 = k_cache.dtype == FP8
    if fp8 != (v_cache.dtype == FP8):
        raise ValueError("k_cache and v_cache must both be FP8 or both 16-bit")
    if not fp8:
        if float(k_scale) != 1.0 or float(v_scale) != 1.0:
            raise ValueError("k_scale / v_scale apply to an FP8 (torch.float8_e4m3fn) cache only")
        return False
    if block_tables is None:
        raise NotImplementedError("an FP8 KV cache exists in the paged layout only: pass block_tables")
    return True


# --------------------------------------------------------------------------------------------------------
# K1 prefill attention
# --------------------------------------------------------------------------------------------------------
def flash_attn_fwd(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, causal: bool = False,
                   softmax_scale: Optional[float] = None, causal_offset: int = 0,
                   kv_lens: Optional[torch.Tensor] = None, return_lse: bool = False,
                   out: Optional[torch.Tensor] = None):
    """Attention forward. q ``[B,Sq,Hq,D]``, k/v ``[B,Sk,Hkv,D]`` (any batch/seq/head strides, D contiguous).

    Returns ``o [B,Sq,Hq,D]`` (same dtype as q) and, if ``return_lse``, ``lse [B,Hq,Sq]`` fp32 (natural log).
    ``causal_offset`` = global position of query row 0 minus global position of key row 0. Keys at or past
    ``kv_lens[b]`` never affect the result, whatever they hold (NaN and Inf included).
    """
    if q.dim() != 4 or k.dim() != 4 or v.dim() != 4:
        raise ValueError(f"expected 4-D [B,S,H,D] tensors, got {tuple(q.shape)}, {tuple(k.shape)}, {tuple(v.shape)}")
    dev = _require_cuda(q, k, v, kv_lens, out)
    B, Sq, Hq, D = q.shape
    Bk, Sk, Hkv, Dk = k.shape
    if (Bk, Dk) != (B, D) or tuple(v.shape) != tuple(k.shape):
        raise ValueError(f"q/k/v shapes do not match: {tuple(q.shape)}, {tuple(k.shape)}, {tuple(v.shape)}")
    if k.dtype != q.dtype or v.dtype != q.dtype:
        raise ValueError("q, k, v must share a dtype")
    dt = _dtype_code(q)
    q, k, v = _last_dim_contiguous(q), _last_dim_contiguous(k), _last_dim_contiguous(v)
    if out is None:
        out = torch.empty((B, Sq, Hq, D), dtype=q.dtype, device=dev)
    elif tuple(out.shape) != (B, Sq, Hq, D) or out.dtype != q.dtype or out.stride(-1) != 1:
        raise ValueError("out must be [B,Sq,Hq,D], same dtype as q, D contiguous")
    lse = torch.empty((B, Hq, Sq), dtype=torch.float32, device=dev) if return_lse else None
    if kv_lens is not None:
        if kv_lens.dtype != torch.int32 or kv_lens.numel() != B or not kv_lens.is_contiguous():
            raise ValueError("kv_lens must be a contiguous int32 tensor of shape [B]")
    scale = float(softmax_scale) if softmax_scale is not None else 1.0 / math.sqrt(D)
    lib = _lib.load()
    with torch.cuda.device(dev):
        rc = lib.b200_fa_fwd(q.data_ptr(), k.data_ptr(), v.data_ptr(), out.data_ptr(), _ptr(lse), B, Sq, Sk, Hq, Hkv, D,
                             strides3(q.stride()[:3]), strides3(k.stride()[:3]), strides3(v.stride()[:3]),
                             strides3(out.stride()[:3]), scale, int(bool(causal)), int(causal_offset), _ptr(kv_lens), dt,
                             _stream_ptr(dev))
    check("b200_fa_fwd", rc)
    return (out, lse) if return_lse else out


def flash_attn_fwd_accum(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, o_acc: torch.Tensor, lse_acc: torch.Tensor,
                         init: bool, causal: bool = False, softmax_scale: Optional[float] = None, causal_offset: int = 0,
                         kv_lens: Optional[torch.Tensor] = None) -> None:
    """One ring step: attention of q over this key block, merged in the kernel epilogue into the running fp32
    ``o_acc [B,Sq,Hq,D]`` (any batch/seq/head strides, D contiguous) and ``lse_acc [B,Hq,Sq]`` (rows contiguous).
    ``init=True`` overwrites the accumulator (first step), otherwise the block is log-sum-exp merged into it."""
    if q.dim() != 4 or k.dim() != 4 or v.dim() != 4:
        raise ValueError(f"expected 4-D [B,S,H,D] tensors, got {tuple(q.shape)}, {tuple(k.shape)}, {tuple(v.shape)}")
    dev = _require_cuda(q, k, v, o_acc, lse_acc, kv_lens)
    B, Sq, Hq, D = q.shape
    Bk, Sk, Hkv, Dk = k.shape
    if (Bk, Dk) != (B, D) or tuple(v.shape) != tuple(k.shape):
        raise ValueError(f"q/k/v shapes do not match: {tuple(q.shape)}, {tuple(k.shape)}, {tuple(v.shape)}")
    if k.dtype != q.dtype or v.dtype != q.dtype:
        raise ValueError("q, k, v must share a dtype")
    if o_acc.dtype != torch.float32 or tuple(o_acc.shape) != (B, Sq, Hq, D) or o_acc.stride(-1) != 1:
        raise ValueError("o_acc must be fp32 [B,Sq,Hq,D] with a contiguous head dimension")
    if lse_acc.dtype != torch.float32 or tuple(lse_acc.shape) != (B, Hq, Sq) or lse_acc.stride(-1) != 1:
        raise ValueError("lse_acc must be fp32 [B,Hq,Sq] with contiguous rows")
    dt = _dtype_code(q)
    q, k, v = _last_dim_contiguous(q), _last_dim_contiguous(k), _last_dim_contiguous(v)
    if kv_lens is not None:
        if kv_lens.dtype != torch.int32 or kv_lens.numel() != B or not kv_lens.is_contiguous():
            raise ValueError("kv_lens must be a contiguous int32 tensor of shape [B]")
    scale = float(softmax_scale) if softmax_scale is not None else 1.0 / math.sqrt(D)
    lse_strides = (ctypes.c_int64 * 2)(int(lse_acc.stride(0)), int(lse_acc.stride(1)))
    lib = _lib.load()
    with torch.cuda.device(dev):
        rc = lib.b200_fa_fwd_accum(q.data_ptr(), k.data_ptr(), v.data_ptr(), o_acc.data_ptr(), lse_acc.data_ptr(), B, Sq, Sk,
                                   Hq, Hkv, D, strides3(q.stride()[:3]), strides3(k.stride()[:3]), strides3(v.stride()[:3]),
                                   strides3(o_acc.stride()[:3]), lse_strides, scale, int(bool(causal)), int(causal_offset),
                                   _ptr(kv_lens), int(bool(init)), dt, _stream_ptr(dev))
    check("b200_fa_fwd_accum", rc)


def paged_prefill_attention(q: torch.Tensor, k_cache: torch.Tensor, v_cache: torch.Tensor, block_tables: torch.Tensor,
                            context_lens: torch.Tensor, layer_idx: int = 0, causal: bool = True,
                            softmax_scale: Optional[float] = None, return_lse: bool = False,
                            out: Optional[torch.Tensor] = None):
    """Short-q / chunked-prefill attention against the paged cache: q ``[B,Sq,Hq,D]`` are the LAST ``Sq`` tokens of every
    sequence (their K/V already appended), cache ``[num_blocks, L, block_size, Hkv, D]``, ``context_lens`` int32 ``[B]``
    counts all keys. ``causal``: query i sees keys up to ``context_lens[b] - Sq + i``. Cache slots at or past
    ``context_lens[b]``, blocks the table does not name for the sequence and the other layers never affect the result,
    whatever they hold (NaN and Inf included)."""
    dev = _require_cuda(q, k_cache, v_cache, block_tables, context_lens, out)
    if q.dim() != 4 or k_cache.dim() != 5 or v_cache.shape != k_cache.shape:
        raise ValueError("expected q [B,Sq,Hq,D] and caches [num_blocks, L, block_size, Hkv, D]")
    B, Sq, Hq, D = q.shape
    num_blocks, num_layers, block_size, Hkv, Dk = k_cache.shape
    if k_cache.dtype == FP8 or v_cache.dtype == FP8:
        raise NotImplementedError("paged_prefill_attention reads 16-bit caches only: an FP8 cache is read by decode_attention")
    if Dk < D or k_cache.dtype != q.dtype or v_cache.dtype != q.dtype:
        raise ValueError("cache head_dim / dtype must match q")
    if Dk != D:   # a narrower head stored in a wider cache (cache_head_dim): zero columns behind q, the caller's scale
        scale = float(softmax_scale) if softmax_scale is not None else 1.0 / math.sqrt(D)
        res = paged_prefill_attention(_pad_head(q, Dk), k_cache, v_cache, block_tables, context_lens, layer_idx, causal, scale,
                                      return_lse)
        o = (res[0] if return_lse else res)[..., :D]
        if out is not None:
            out.copy_(o)
            o = out
        return (o, res[1]) if return_lse else o
    if not k_cache.is_contiguous() or not v_cache.is_contiguous():
        raise ValueError("paged cache must be contiguous")
    if block_tables.dtype != torch.int32 or block_tables.dim() != 2 or block_tables.shape[0] != B or not block_tables.is_contiguous():
        raise ValueError("block_tables must be a contiguous int32 [B, max_blocks] tensor")
    if context_lens.dtype != torch.int32 or context_lens.numel() != B or not context_lens.is_contiguous():
        raise ValueError("context_lens must be a contiguous int32 [B] tensor")
    dt = _dtype_code(q)
    q = _last_dim_contiguous(q)
    if out is None:
        out = torch.empty((B, Sq, Hq, D), dtype=q.dtype, device=dev)
    elif tuple(out.shape) != (B, Sq, Hq, D) or out.dtype != q.dtype or out.stride(-1) != 1:
        raise ValueError("out must be [B,Sq,Hq,D], same dtype as q, D contiguous")
    lse = torch.empty((B, Hq, Sq), dtype=torch.float32, device=dev) if return_lse else None
    scale = float(softmax_scale) if softmax_scale is not None else 1.0 / math.sqrt(D)
    lib = _lib.load()
    with torch.cuda.device(dev):
        rc = lib.b200_fa_fwd_paged(q.data_ptr(), k_cache.data_ptr(), v_cache.data_ptr(), out.data_ptr(), _ptr(lse), B, Sq, Hq,
                                   Hkv, D, strides3(q.stride()[:3]), strides3(out.stride()[:3]), block_tables.data_ptr(),
                                   block_tables.shape[1], block_size, num_blocks, num_layers, int(layer_idx),
                                   context_lens.data_ptr(), scale, int(bool(causal)), dt, _stream_ptr(dev))
    check("b200_fa_fwd_paged", rc)
    return (out, lse) if return_lse else out


def lse_merge(o_acc: torch.Tensor, lse_acc: torch.Tensor, o_b: torch.Tensor, lse_b: torch.Tensor) -> None:
    """In place: merge the partial result ``(o_b [B,Sq,Hq,D] 16-bit, lse_b [B,Hq,Sq])`` into the fp32 accumulator."""
    dev = _require_cuda(o_acc, lse_acc, o_b, lse_b)
    B, Sq, Hq, D = o_b.shape
    if o_acc.dtype != torch.float32 or not o_acc.is_contiguous() or tuple(o_acc.shape) != (B, Sq, Hq, D):
        raise ValueError("o_acc must be a contiguous fp32 [B,Sq,Hq,D] tensor")
    for name, t in (("lse_acc", lse_acc), ("lse_b", lse_b)):
        if t.dtype != torch.float32 or not t.is_contiguous() or tuple(t.shape) != (B, Hq, Sq):
            raise ValueError(f"{name} must be a contiguous fp32 [B,Hq,Sq] tensor")
    o_b = _last_dim_contiguous(o_b)
    lib = _lib.load()
    with torch.cuda.device(dev):
        rc = lib.b200_lse_merge(o_acc.data_ptr(), lse_acc.data_ptr(), o_b.data_ptr(), lse_b.data_ptr(), B, Sq, Hq, D,
                                strides3(o_b.stride()[:3]), _dtype_code(o_b), _stream_ptr(dev))
    check("b200_lse_merge", rc)


def cast_out(o_acc: torch.Tensor, dtype: torch.dtype, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    dev = _require_cuda(o_acc, out)
    B, Sq, Hq, D = o_acc.shape
    if o_acc.dtype != torch.float32 or not o_acc.is_contiguous():
        raise ValueError("o_acc must be a contiguous fp32 tensor")
    if out is None:
        out = torch.empty((B, Sq, Hq, D), dtype=dtype, device=dev)
    elif tuple(out.shape) != (B, Sq, Hq, D) or out.dtype != dtype or out.stride(-1) != 1:
        raise ValueError(f"out must be {dtype} of shape {(B, Sq, Hq, D)} with a contiguous last dimension")
    lib = _lib.load()
    with torch.cuda.device(dev):
        rc = lib.b200_cast_out(o_acc.data_ptr(), out.data_ptr(), B, Sq, Hq, D, strides3(out.stride()[:3]),
                               _dtype_code(out), _stream_ptr(dev))
    check("b200_cast_out", rc)
    return out


# --------------------------------------------------------------------------------------------------------
# K2 decode attention
# --------------------------------------------------------------------------------------------------------
_workspaces: dict = {}


def _workspace(dev: torch.device, nbytes: int) -> Optional[torch.Tensor]:
    """Per-(device, stream) grow-only scratch buffer (the C-ABI never allocates)."""
    if nbytes <= 0:
        return None
    key = (dev.index, torch.cuda.current_stream(dev).cuda_stream)
    buf = _workspaces.get(key)
    if buf is None or buf.numel() < nbytes:
        buf = torch.empty(max(nbytes, 1 << 20), dtype=torch.uint8, device=dev)
        _workspaces[key] = buf
    return buf


def decode_attention(q: torch.Tensor, k_cache: torch.Tensor, v_cache: torch.Tensor, context_lens: torch.Tensor,
                     softmax_scale: Optional[float] = None, block_tables: Optional[torch.Tensor] = None,
                     layer_idx: int = 0, max_context_len: Optional[int] = None, num_splits: int = 0,
                     return_lse: bool = False, out: Optional[torch.Tensor] = None, k_scale: float = 1.0,
                     v_scale: float = 1.0):
    """Single-token attention against a KV cache.

    q ``[B,Hq,D]``. Contiguous cache: k/v ``[B,S_max,Hkv,D]`` (``block_tables is None``). Paged cache: k/v
    ``[num_blocks, L, block_size, Hkv, D]`` + ``block_tables`` int32 ``[B,max_blocks]`` + ``layer_idx``.
    ``context_lens`` int32 ``[B]`` counts the valid keys (the appended token included).
    A ``torch.float8_e4m3fn`` cache (paged only) holds K / ``k_scale`` and V / ``v_scale`` (``b200_fa_decode_fp8``).
    """
    dev = _require_cuda(q, k_cache, v_cache, context_lens, block_tables, out)
    if q.dim() != 3:
        raise ValueError(f"q must be [B,Hq,D], got {tuple(q.shape)}")
    B, Hq, D = q.shape
    dt = _dtype_code(q)
    fp8 = _fp8_cache(k_cache, v_cache, block_tables, k_scale, v_scale)
    if not fp8 and (k_cache.dtype != q.dtype or v_cache.dtype != q.dtype):
        raise ValueError("cache dtype must match q")
    if context_lens.dtype != torch.int32 or not context_lens.is_contiguous() or context_lens.numel() != B:
        raise ValueError("context_lens must be a contiguous int32 [B] tensor")
    if out is not None and (tuple(out.shape) != (B, Hq, D) or out.dtype != q.dtype or not out.is_contiguous()):
        raise ValueError(f"out must be a contiguous {q.dtype} tensor of shape {(B, Hq, D)} (the kernels write it densely)")
    q = q.contiguous()
    paged = block_tables is not None
    if paged:
        if k_cache.dim() != 5 or not k_cache.is_contiguous() or not v_cache.is_contiguous():
            raise ValueError("paged cache must be contiguous [num_blocks, L, block_size, Hkv, D]")
        _, num_layers, block_size, Hkv, Dk = k_cache.shape
        if block_tables.dtype != torch.int32 or block_tables.dim() != 2 or not block_tables.is_contiguous():
            raise ValueError("block_tables must be a contiguous int32 [B, max_blocks] tensor")
        max_blocks = block_tables.shape[1]
        cap = max_blocks * block_size
        kv_bs = kv_ts = 0
        layout = KV_PAGED
    else:
        if k_cache.dim() != 4 or k_cache.stride(-1) != 1 or k_cache.stride(2) != k_cache.shape[3]:
            raise ValueError("contiguous cache must be [B,S_max,Hkv,D] with (Hkv, D) dense")
        if v_cache.stride() != k_cache.stride() or v_cache.shape != k_cache.shape:
            raise ValueError("k_cache and v_cache must share shape and strides")
        _, cap, Hkv, Dk = k_cache.shape
        kv_bs, kv_ts = k_cache.stride(0), k_cache.stride(1)
        num_layers, block_size, max_blocks = 1, 0, 0
        layout = KV_CONTIGUOUS
    if Dk < D:
        raise ValueError("head_dim of q and cache differ")
    if Dk != D:   # a narrower head stored in a wider cache (cache_head_dim)
        scale = float(softmax_scale) if softmax_scale is not None else 1.0 / math.sqrt(D)
        res = decode_attention(_pad_head(q, Dk), k_cache, v_cache, context_lens, scale, block_tables, layer_idx, max_context_len,
                               num_splits, return_lse, k_scale=k_scale, v_scale=v_scale)
        o = (res[0] if return_lse else res)[..., :D]
        if out is not None:
            out.copy_(o)
            o = out
        return (o, res[1]) if return_lse else o
    if max_context_len is None:
        max_context_len = cap
    max_context_len = int(min(max_context_len, cap))
    if out is None:
        out = torch.empty((B, Hq, D), dtype=q.dtype, device=dev)
    lse = torch.empty((B, Hq), dtype=torch.float32, device=dev) if return_lse else None
    scale = float(softmax_scale) if softmax_scale is not None else 1.0 / math.sqrt(D)
    lib = _lib.load()
    with torch.cuda.device(dev):
        splits = num_splits if num_splits > 0 else lib.b200_fa_decode_num_splits(B, Hq, Hkv, D, max_context_len)
        ws_bytes = lib.b200_fa_decode_workspace_bytes(B, Hq, Hkv, D, max_context_len, splits)
        ws = _workspace(dev, ws_bytes)
        if fp8:
            rc = lib.b200_fa_decode_fp8(q.data_ptr(), k_cache.data_ptr(), v_cache.data_ptr(), out.data_ptr(), _ptr(lse), B,
                                        Hq, Hkv, D, context_lens.data_ptr(), max_context_len, scale, layout,
                                        _ptr(block_tables), max_blocks, block_size, num_layers, int(layer_idx), splits,
                                        _ptr(ws), ws_bytes, float(k_scale), float(v_scale), dt, _stream_ptr(dev))
            check("b200_fa_decode_fp8", rc)
            return (out, lse) if return_lse else out
        rc = lib.b200_fa_decode(q.data_ptr(), k_cache.data_ptr(), v_cache.data_ptr(), out.data_ptr(), _ptr(lse), B, Hq,
                                Hkv, D, context_lens.data_ptr(), max_context_len, scale, layout, kv_bs, kv_ts,
                                _ptr(block_tables), max_blocks, block_size, num_layers, int(layer_idx), splits,
                                _ptr(ws), ws_bytes, dt, _stream_ptr(dev))
    check("b200_fa_decode", rc)
    return (out, lse) if return_lse else out


def kv_append(key: torch.Tensor, value: torch.Tensor, k_cache: torch.Tensor, v_cache: torch.Tensor,
              context_lens: torch.Tensor, block_tables: Optional[torch.Tensor] = None, layer_idx: int = 0,
              k_scale: float = 1.0, v_scale: float = 1.0) -> None:
    """Write the new token's K,V ``[B,Hkv,D]`` into the cache at position ``context_lens[b]-1``.

    A ``torch.float8_e4m3fn`` cache (paged only) stores e4m3(K / ``k_scale``) and e4m3(V / ``v_scale``)
    (``b200_kv_append_fp8``); it also takes ``[B,n,Hkv,D]`` rows, written to positions ``[context_lens[b]-n,
    context_lens[b])`` (the prompt of a prefill)."""
    dev = _require_cuda(key, value, k_cache, v_cache, context_lens, block_tables)
    fp8 = _fp8_cache(k_cache, v_cache, block_tables, k_scale, v_scale)
    if fp8 and key.dim() == 4 and value.shape == key.shape:
        B, n_tokens, Hkv, D = key.shape
    elif key.dim() != 3 or value.shape != key.shape:
        raise ValueError(f"key / value must be [B,Hkv,D], got {tuple(key.shape)}, {tuple(value.shape)}")
    else:
        (B, Hkv, D), n_tokens = key.shape, 1
    _dtype_code(key)
    if value.dtype != key.dtype or (not fp8 and (k_cache.dtype != key.dtype or v_cache.dtype != key.dtype)):
        raise ValueError("key, value and both caches must share a dtype")
    if context_lens.dtype != torch.int32 or not context_lens.is_contiguous() or context_lens.numel() != B:
        raise ValueError("context_lens must be a contiguous int32 [B] tensor")
    key, value = key.contiguous(), value.contiguous()
    paged = block_tables is not None
    if paged:
        if not k_cache.is_contiguous() or not v_cache.is_contiguous() or k_cache.dim() != 5 or v_cache.shape != k_cache.shape:
            raise ValueError("paged cache must be contiguous [num_blocks, L, block_size, Hkv, D]")
        _, num_layers, block_size, Hc, Dc = k_cache.shape
        if block_tables.dtype != torch.int32 or block_tables.dim() != 2 or block_tables.shape[0] != B or \
                not block_tables.is_contiguous():
            raise ValueError("block_tables must be a contiguous int32 [B, max_blocks] tensor")
        if not 0 <= int(layer_idx) < num_layers:
            raise ValueError(f"layer_idx {layer_idx} outside the cache's {num_layers} layers")
        max_blocks = block_tables.shape[1]
        kv_bs = kv_ts = 0
    else:
        if k_cache.dim() != 4 or k_cache.stride(-1) != 1 or k_cache.stride(2) != D or v_cache.shape != k_cache.shape or \
                v_cache.stride() != k_cache.stride() or k_cache.shape[0] < B:
            raise ValueError("contiguous cache must be [B,S_max,Hkv,D] with (Hkv, D) dense, k and v alike")
        Hc, Dc = k_cache.shape[2], k_cache.shape[3]
        kv_bs, kv_ts = k_cache.stride(0), k_cache.stride(1)
        num_layers, block_size, max_blocks = 1, 0, k_cache.shape[1]  # contiguous: the capacity S_max travels in max_blocks
    if Hc != Hkv or Dc < D:
        raise ValueError(f"cache heads / head_dim {(Hc, Dc)} do not match key {(Hkv, D)}")
    if Dc != D:   # a narrower head stored in a wider cache (cache_head_dim): zero columns behind the new token's K, V
        key, value, D = _pad_head(key, Dc), _pad_head(value, Dc), Dc
    lib = _lib.load()
    if fp8:
        with torch.cuda.device(dev):
            rc = lib.b200_kv_append_fp8(key.data_ptr(), value.data_ptr(), k_cache.data_ptr(), v_cache.data_ptr(), B, n_tokens,
                                        Hkv, D, context_lens.data_ptr(), block_tables.data_ptr(), max_blocks, block_size,
                                        num_layers, int(layer_idx), float(k_scale), float(v_scale), _dtype_code(key),
                                        _stream_ptr(dev))
        check("b200_kv_append_fp8", rc)
        return
    with torch.cuda.device(dev):
        rc = lib.b200_kv_append(key.data_ptr(), value.data_ptr(), k_cache.data_ptr(), v_cache.data_ptr(), B, Hkv, D,
                                context_lens.data_ptr(), KV_PAGED if paged else KV_CONTIGUOUS, kv_bs, kv_ts,
                                _ptr(block_tables), max_blocks, block_size, num_layers, int(layer_idx),
                                _dtype_code(key), _stream_ptr(dev))
    check("b200_kv_append", rc)


# --------------------------------------------------------------------------------------------------------
# K3 fused MLP
# --------------------------------------------------------------------------------------------------------
def activation_code(name) -> int:
    try:
        return _ACTIVATIONS[name]
    except KeyError:
        raise ValueError(f"unsupported activation {name!r}; supported: {sorted(k for k in _ACTIVATIONS if k)}") from None


def _out_rows(out: torch.Tensor, lead: Tuple[int, ...], width: int, dtype: torch.dtype) -> torch.Tensor:
    """``out`` seen as ``[rows, width]`` without a copy: the kernels write through its pointer and one row stride, so an
    ``out`` they cannot address that way is refused rather than written into a temporary the caller never sees."""
    if tuple(out.shape) != (*lead, width) or out.dtype != dtype:
        raise ValueError(f"out must be {dtype} of shape {(*lead, width)}, got {out.dtype} {tuple(out.shape)}")
    if out.stride(-1) != 1:
        raise ValueError("out must have a contiguous last dimension")
    try:
        return out.view(-1, width)
    except RuntimeError:
        raise ValueError(f"out (strides {out.stride()}) cannot be addressed as rows of one stride") from None


def _as_rows(x: torch.Tensor) -> Tuple[torch.Tensor, Tuple[int, ...]]:
    lead = tuple(x.shape[:-1])
    x2 = x.reshape(-1, x.shape[-1])
    if x2.stride(-1) != 1 or (x2.shape[0] > 1 and x2.stride(0) % 8 != 0):
        x2 = x2.contiguous()
    return x2, lead


def linear_act(x: torch.Tensor, weight: torch.Tensor, bias: Optional[torch.Tensor] = None, activation=None,
               gate_weight: Optional[torch.Tensor] = None, gate_bias: Optional[torch.Tensor] = None,
               out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """``act(x @ weight.T + bias)`` or, for SwiGLU, ``silu(x @ gate_weight.T + gate_bias) * (x @ weight.T + bias)``."""
    dev = _require_cuda(x, weight, bias, gate_weight, gate_bias, out)
    act = activation_code(activation)
    dt = _dtype_code(x)
    x2, lead = _as_rows(x)
    T, K = x2.shape
    N, Kw = weight.shape
    if Kw != K:
        raise ValueError(f"weight {tuple(weight.shape)} does not match input width {K}")
    for t in (weight, bias, gate_weight, gate_bias):
        if t is not None and t.dtype != x.dtype:
            raise ValueError("weights and biases must have the dtype of x")
    weight = weight.contiguous()
    bias = None if bias is None else bias.contiguous()
    if act == ACT_SWIGLU:
        if gate_weight is None:
            raise ValueError("SwiGLU needs gate_weight")
        gate_weight = gate_weight.contiguous()
        gate_bias = None if gate_bias is None else gate_bias.contiguous()
    y = _out_rows(out, lead, N, x.dtype) if out is not None else torch.empty((T, N), dtype=x.dtype, device=dev)
    lib = _lib.load()
    with torch.cuda.device(dev):
        ws_bytes = lib.b200_linear_act_workspace_bytes(T, K, N, act)
        ws = _workspace(dev, ws_bytes)
        rc = lib.b200_linear_act(x2.data_ptr(), x2.stride(0) if T > 1 else K, weight.data_ptr(), _ptr(bias),
                                 _ptr(gate_weight), _ptr(gate_bias), y.data_ptr(), y.stride(0) if T > 1 else N, T, K, N,
                                 act, _ptr(ws), ws_bytes, dt, _stream_ptr(dev))
    check("b200_linear_act", rc)
    return out if out is not None else y.reshape(*lead, N)


def fused_mlp(x: torch.Tensor, w_up: torch.Tensor, b_up: Optional[torch.Tensor], w_down: torch.Tensor,
              b_down: Optional[torch.Tensor], activation: str = "gelu_tanh", w_gate: Optional[torch.Tensor] = None,
              b_gate: Optional[torch.Tensor] = None, out: Optional[torch.Tensor] = None,
              timing_events=None) -> torch.Tensor:
    """FusedMLP forward: ``act(x W_up^T + b_up) W_down^T + b_down`` (SwiGLU: ``silu(x W_gate^T + b_gate) * up``).

    ``timing_events`` (three ``torch.cuda.Event``) is a measurement hook for bench.py: the same two kernel launches
    ``b200_fused_mlp`` makes are issued one by one with an event recorded before, between and after them."""
    dev = _require_cuda(x, w_up, b_up, w_down, b_down, w_gate, b_gate, out)
    act = activation_code(activation)
    if act == ACT_NONE:
        raise ValueError("fused_mlp needs an activation")
    dt = _dtype_code(x)
    x2, lead = _as_rows(x)
    T, h = x2.shape
    i, hw = w_up.shape
    h_out, iw = w_down.shape
    if hw != h or iw != i:
        raise ValueError(f"weight shapes {tuple(w_up.shape)} / {tuple(w_down.shape)} do not match input width {h}")
    for t in (w_up, b_up, w_down, b_down, w_gate, b_gate):
        if t is not None and t.dtype != x.dtype:
            raise ValueError("weights and biases must have the dtype of x")
    w_up, w_down = w_up.contiguous(), w_down.contiguous()
    if act == ACT_SWIGLU:
        if w_gate is None or tuple(w_gate.shape) != (i, h):
            raise ValueError("SwiGLU needs w_gate of shape [intermediate, hidden]")
        w_gate = w_gate.contiguous()
    else:
        w_gate = b_gate = None
    b_up = None if b_up is None else b_up.contiguous()
    b_down = None if b_down is None else b_down.contiguous()
    b_gate = None if b_gate is None else b_gate.contiguous()
    y = _out_rows(out, lead, h_out, x.dtype) if out is not None else torch.empty((T, h_out), dtype=x.dtype, device=dev)
    lib = _lib.load()
    with torch.cuda.device(dev):
        ws_bytes = lib.b200_fused_mlp_workspace_bytes(T, h, i)
        ws = _workspace(dev, ws_bytes)
        if timing_events is not None:
            e0, e1, e2 = timing_events
            stream = torch.cuda.current_stream(dev)
            e0.record(stream)
            inter = (T * i * 2 + 255) & ~255
            sk_ptr, sk_bytes = ws.data_ptr() + inter, ws_bytes - inter
            rc = lib.b200_linear_act(x2.data_ptr(), x2.stride(0) if T > 1 else h, w_up.data_ptr(), _ptr(b_up), _ptr(w_gate),
                                     _ptr(b_gate), ws.data_ptr(), i, T, h, i, act, sk_ptr, sk_bytes, dt, _stream_ptr(dev))
            check("b200_linear_act", rc)
            e1.record(stream)
            rc = lib.b200_linear_act(ws.data_ptr(), i, w_down.data_ptr(), _ptr(b_down), None, None, y.data_ptr(),
                                     y.stride(0) if T > 1 else h_out, T, i, h_out, ACT_NONE, sk_ptr, sk_bytes, dt,
                                     _stream_ptr(dev))
            check("b200_linear_act", rc)
            e2.record(stream)
            return out if out is not None else y.reshape(*lead, h_out)
        rc = lib.b200_fused_mlp(x2.data_ptr(), x2.stride(0) if T > 1 else h, w_up.data_ptr(), _ptr(b_up), _ptr(w_gate),
                                _ptr(b_gate), w_down.data_ptr(), _ptr(b_down), y.data_ptr(),
                                y.stride(0) if T > 1 else h_out, T, h, i, h_out, act, _ptr(ws), ws_bytes, dt,
                                _stream_ptr(dev))
    check("b200_fused_mlp", rc)
    return out if out is not None else y.reshape(*lead, h_out)


def layernorm(x: torch.Tensor, weight: torch.Tensor, bias: Optional[torch.Tensor] = None, eps: float = 1e-5,
              residual: Optional[torch.Tensor] = None, residual_alpha: float = 1.0,
              out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """``LayerNorm(x + residual_alpha * residual) * weight + bias`` over the last dimension (fp32 statistics)."""
    dev = _require_cuda(x, weight, bias, residual, out)
    dt = _dtype_code(x)
    cols = x.shape[-1]
    x2, lead = _as_rows(x)
    r2 = None
    if residual is not None:
        if residual.shape != x.shape or residual.dtype != x.dtype:
            raise ValueError("residual must match x in shape and dtype")
        r2, _ = _as_rows(residual)
    for t in (weight, bias):
        if t is not None and (t.dtype != x.dtype or t.numel() != cols):
            raise ValueError("weight / bias must be [hidden] tensors of the dtype of x")
    weight = weight.contiguous()
    bias = None if bias is None else bias.contiguous()
    rows = x2.shape[0]
    y = _out_rows(out, lead, cols, x.dtype) if out is not None else torch.empty((rows, cols), dtype=x.dtype, device=dev)
    ld = lambda t: t.stride(0) if t.shape[0] > 1 else cols
    lib = _lib.load()
    with torch.cuda.device(dev):
        rc = lib.b200_layernorm(x2.data_ptr(), _ptr(r2), weight.data_ptr(), _ptr(bias), y.data_ptr(), rows, cols, ld(x2),
                                ld(r2) if r2 is not None else 0, ld(y), float(eps), float(residual_alpha), dt, _stream_ptr(dev))
    check("b200_layernorm", rc)
    return out if out is not None else y.reshape(*lead, cols)


def set_sm_limit(max_ctas: int) -> None:
    """Cap the CTAs of the persistent GEMM kernels (0 = no cap); see ``b200_set_sm_limit``."""
    check("b200_set_sm_limit", _lib.load().b200_set_sm_limit(int(max_ctas)))


def set_gemm_group_rows(rows: int) -> None:
    """Rows of the activation panel one L2 raster group of the persistent GEMMs covers; see ``b200_set_gemm_group_rows``."""
    check("b200_set_gemm_group_rows", _lib.load().b200_set_gemm_group_rows(int(rows)))


def launch_count() -> int:
    """Kernel launches issued by the library in this process so far (``b200_launch_count``)."""
    return int(_lib.load().b200_launch_count())


def last_kernel() -> str:
    """Name of the kernel the library launched last (``b200_last_kernel``)."""
    return (_lib.load().b200_last_kernel() or b"").decode()


def last_gemm_kernel() -> str:
    """Name of the GEMM kernel the last linear / FusedMLP call dispatched to."""
    return (_lib.load().b200_last_gemm_kernel() or b"").decode()


def sm_count(device=None) -> int:
    return torch.cuda.get_device_properties(device if device is not None else torch.cuda.current_device()).multi_processor_count


def arch_ok() -> bool:
    return _lib.load().b200_arch_ok() == 1


def version() -> str:
    return _lib.load().b200_version().decode()
