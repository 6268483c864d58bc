"""Host-side mirror of the reference's ``kernels/attention/flash_attention.py`` (module API + model surgery).

Same class names, constructor arguments, attribute names (``q_proj/k_proj/v_proj/o_proj/qkv_proj``) and forward
signatures as the reference (file:line citations on each class); the arithmetic runs in the sm_100a kernels behind
the C-ABI (K1 ``b200_fa_fwd`` for prefill, K2 ``b200_fa_decode`` for the paged/decode branch). Differences from the
reference are the defects listed in SURVEY.md Appendix B, fixed here: the result is exact softmax attention (the
reference's fallbacks return zeros), GQA is handled, non-contiguous views are accepted, and a kernel failure raises
instead of silently falling back.
"""
from __future__ import annotations

import logging
import math
from dataclasses import dataclass
from typing import Any, Dict, Optional, Set, Tuple, Union

import torch
import torch.nn as nn
import torch.nn.functional as F

from ... import ops

logger = logging.getLogger(__name__)

__all__ = ["FlashAttentionConfig", "FlashAttention3", "FlashAttentionLayer", "FlashSelfAttention", "ModelConverter",
           "benchmark_flash_attention_speed", "benchmark_memory_usage", "key_padding_mask_to_lengths"]


@dataclass
class FlashAttentionConfig:
    """reference: kernels/attention/flash_attention.py:53-104. ``use_triton``, ``block_size`` and
    ``memory_efficient`` are accepted for compatibility and ignored (the tile shape is fixed by the tcgen05 kernel)."""
    block_size: int = 128
    causal: bool = False
    softmax_scale: Optional[float] = None
    dropout_p: float = 0.0
    return_softmax: bool = False
    use_triton: bool = True
    memory_efficient: bool = True
    precision: str = "fp16"
    normalize_query: bool = False
    fp8_ortho_matrix: Optional[torch.Tensor] = None

    @property
    def allowed_precisions(self) -> Set[str]:
        return {"fp16", "bf16", "fp32", "fp8"}

    def __post_init__(self):
        if self.precision not in self.allowed_precisions:
            raise ValueError(f"Unsupported precision mode: {self.precision}. Allowed: {self.allowed_precisions}")


def key_padding_mask_to_lengths(mask: torch.Tensor, seq_len: int) -> torch.Tensor:
    """Lower a key-padding mask ([B,S] or [B,1,S], nonzero = keep — flash_attention.py:359) to per-batch key counts.
    Only right-padding masks are representable; anything else raises (no slow fallback, SURVEY.md §8 a2)."""
    if mask.dim() == 3 and mask.shape[1] == 1:
        mask = mask[:, 0]
    if mask.dim() != 2 or mask.shape[-1] != seq_len:
        raise NotImplementedError(
            f"attention mask of shape {tuple(mask.shape)} is not supported by the B200 attention kernel: only causal "
            "masking and [B,S] / [B,1,S] right-padding key masks are (dense [B,S,S] masks would need a slow path)")
    keep = mask != 0
    lens = keep.sum(dim=-1).to(torch.int32)
    expect = torch.arange(seq_len, device=mask.device).unsqueeze(0) < lens.unsqueeze(1)
    if not torch.equal(keep, expect):
        raise NotImplementedError("only right-padding key masks are supported (kept keys must form a prefix)")
    return lens.contiguous()


class FlashAttention3(nn.Module):
    """reference: kernels/attention/flash_attention.py:107-472. ``forward(q,k,v,mask)`` with q ``[B,S,Hq,D]`` and
    k/v ``[B,S,Hkv,D]`` (Hkv may divide Hq: GQA by head group, :894-903)."""

    def __init__(self, config: Optional[FlashAttentionConfig] = None):
        super().__init__()
        self.config = config or FlashAttentionConfig()

    def _compute_dtype(self, orig: torch.dtype) -> torch.dtype:
        p = self.config.precision
        if p == "fp16":
            return torch.float16
        if p == "bf16":
            return torch.bfloat16
        if p == "fp8":
            raise NotImplementedError("precision='fp8' (incoherent-processing FP8 attention) is not implemented on the B200 path")
        # "fp32": there is no fp32 tensor-core path; keep 16-bit inputs as they are, compute fp32 inputs in bf16 storage
        # with fp32 accumulation/softmax
        return orig if orig in (torch.float16, torch.bfloat16) else torch.bfloat16

    def forward(self, q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, mask: Optional[torch.Tensor] = None
                ) -> Union[torch.Tensor, Tuple[torch.Tensor, torch.Tensor]]:
        if q.dim() != 4 or k.dim() != 4 or v.dim() != 4:
            raise ValueError(f"Expected 4D tensors for q, k, v but got shapes: q={q.shape}, k={k.shape}, v={v.shape}")
        if not q.is_cuda:
            raise ValueError("The B200 attention kernels require input tensors on a CUDA device (there is no CPU fallback).")
        if self.config.dropout_p > 0.0 and self.training:
            raise NotImplementedError("attention dropout is not implemented (inference path; reference :270 disables it in eval)")
        if self.config.return_softmax:
            raise NotImplementedError("return_softmax=True would materialise the S x S matrix; use return_lse via ops.flash_attn_fwd")
        orig_dtype = q.dtype
        dt = self._compute_dtype(orig_dtype)
        if q.dtype != dt:
            q, k, v = q.to(dt), k.to(dt), v.to(dt)
        if self.config.normalize_query:
            q = F.normalize(q, dim=-1)
        kv_lens = None
        if mask is not None:
            kv_lens = key_padding_mask_to_lengths(mask, k.shape[1])
        out = ops.flash_attn_fwd(q, k, v, causal=self.config.causal, softmax_scale=self.config.softmax_scale,
                                 kv_lens=kv_lens)
        return out.to(orig_dtype)

    def get_theoretical_memory_usage(self, seq_len: int, batch_size: int, num_heads: int, head_dim: int) -> Dict[str, float]:
        """reference :409-460 — bytes (as MB) of standard attention (S x S scores materialised) vs the tiled kernel."""
        elt = 2 if self.config.precision in ("fp16", "bf16") else 4
        qkv = 3 * batch_size * seq_len * num_heads * head_dim * elt
        out = batch_size * seq_len * num_heads * head_dim * elt
        scores = batch_size * num_heads * seq_len * seq_len * elt
        standard = qkv + out + 2 * scores
        flash = qkv + out + batch_size * num_heads * seq_len * 4  # + LSE
        mb = 1024.0 * 1024.0
        return {"standard_attention_mb": standard / mb, "flash_attention_mb": flash / mb,
                "memory_reduction_factor": standard / flash, "attention_matrix_mb": scores / mb}

    def use_vllm_compatible_kernels(self) -> bool:
        """reference :462-471 — the paged layout [num_blocks, L, block_size, Hkv, D] is what the decode kernel reads."""
        return True


def _paged_kwargs(kwargs: Dict[str, Any]):
    names = ("physical_kv_cache_k", "physical_kv_cache_v", "block_tables", "context_lengths", "kv_cache_block_size",
             "max_seq_len", "layer_idx")
    vals = [kwargs.get(n) for n in names]
    if any(v is None for v in vals):
        raise ValueError("Missing required arguments for PagedAttention in FlashAttentionLayer forward pass.")
    return vals


class _AttentionBase(nn.Module):
    def _paged_decode(self, q: torch.Tensor, kwargs: Dict[str, Any]) -> torch.Tensor:
        """q [B, q_len, Hq, D] against the paged cache (reference flash_attention.py:572-621 -> attention_kernels.py:1206):
        q_len == 1 runs the decode kernel K2, q_len > 1 the prefill kernel K1 over the block table."""
        k_cache, v_cache, block_tables, context_lengths, block_size, max_seq_len, layer_idx = _paged_kwargs(kwargs)
        B, q_len, Hq, D = q.shape
        if k_cache.shape[2] != block_size:
            raise ValueError("kv_cache_block_size does not match the cache tensor")
        dt = self.flash_attention._compute_dtype(q.dtype)
        orig = q.dtype
        lens = context_lengths.to(torch.int32).contiguous()
        tables = block_tables.to(torch.int32).contiguous()
        if q_len != 1:
            # short-q / chunked prefill against the cache (reference attention_kernels.py:1251 picks BLOCK_SIZE_M = 64 for
            # it): K1 gathers the KV tiles through the block table; the q_len new tokens are the last keys of each sequence
            out = ops.paged_prefill_attention(q.to(dt), k_cache, v_cache, tables, lens, layer_idx=int(layer_idx), causal=True,
                                              softmax_scale=self.config.softmax_scale)
            return out.reshape(B, q_len, Hq * D).to(orig)
        qd = q.reshape(B, Hq, D).to(dt)
        out = ops.decode_attention(qd, k_cache, v_cache, lens, softmax_scale=self.config.softmax_scale, block_tables=tables,
                                   layer_idx=int(layer_idx), max_context_len=int(max_seq_len))
        return out.view(B, 1, Hq * D).to(orig)


class FlashAttentionLayer(_AttentionBase):
    """reference: kernels/attention/flash_attention.py:474-659 (separate q/k/v projections, bias=True)."""

    def __init__(self, hidden_size: int, num_attention_heads: int, config: Optional[FlashAttentionConfig] = None,
                 num_kv_heads: Optional[int] = None):
        super().__init__()
        self.hidden_size = hidden_size
        self.num_attention_heads = num_attention_heads
        self.num_kv_heads = num_kv_heads if num_kv_heads is not None else num_attention_heads
        if hidden_size % num_attention_heads != 0:
            raise ValueError(f"hidden_size {hidden_size} must be divisible by num_attention_heads {num_attention_heads}")
        if num_attention_heads % self.num_kv_heads != 0:
            raise ValueError(f"num_attention_heads {num_attention_heads} must be divisible by num_kv_heads {self.num_kv_heads}")
        self.head_dim = hidden_size // num_attention_heads
        self.config = config or FlashAttentionConfig()
        self.q_proj = nn.Linear(hidden_size, hidden_size)
        self.k_proj = nn.Linear(hidden_size, self.num_kv_heads * self.head_dim)
        self.v_proj = nn.Linear(hidden_size, self.num_kv_heads * self.head_dim)
        self.o_proj = nn.Linear(hidden_size, hidden_size)
        self.flash_attention = FlashAttention3(self.config)
        self._init_weights()

    def _init_weights(self):
        for lin in (self.q_proj, self.k_proj, self.v_proj, self.o_proj):
            nn.init.normal_(lin.weight, mean=0.0, std=0.02)  # reference :531-542
            if lin.bias is not None:
                nn.init.zeros_(lin.bias)

    def forward(self, hidden_states: torch.Tensor, attention_mask: Optional[torch.Tensor] = None, **kwargs: Any) -> torch.Tensor:
        B, S, _ = hidden_states.shape
        if "block_tables" in kwargs:
            q = self.q_proj(hidden_states).view(B, S, self.num_attention_heads, self.head_dim)
            return self.o_proj(self._paged_decode(q, kwargs))
        q = self.q_proj(hidden_states).view(B, S, self.num_attention_heads, self.head_dim)
        k = self.k_proj(hidden_states).view(B, S, self.num_kv_heads, self.head_dim)
        v = self.v_proj(hidden_states).view(B, S, self.num_kv_heads, self.head_dim)
        ctx = self.flash_attention(q, k, v, attention_mask)
        return self.o_proj(ctx.reshape(B, S, self.hidden_size))


class FlashSelfAttention(_AttentionBase):
    """reference: kernels/attention/flash_attention.py:662-949 (fused qkv projection, out = h + 2*Hkv*D)."""

    def __init__(self, hidden_size: int, num_attention_heads: int, config: Optional[FlashAttentionConfig] = None,
                 num_kv_heads: Optional[int] = None):
        super().__init__()
        self.hidden_size = hidden_size
        self.num_attention_heads = num_attention_heads
        self.num_kv_heads = num_kv_heads if num_kv_heads is not None else num_attention_heads
        if hidden_size % num_attention_heads != 0:
            raise ValueError(f"hidden_size {hidden_size} must be divisible by num_attention_heads {num_attention_heads}")
        if num_attention_heads % self.num_kv_heads != 0:
            raise ValueError(f"num_attention_heads {num_attention_heads} must be divisible by num_kv_heads {self.num_kv_heads}")
        self.head_dim = hidden_size // num_attention_heads
        self.config = config or FlashAttentionConfig()
        kv_dim = self.num_kv_heads * self.head_dim
        self.qkv_proj = nn.Linear(hidden_size, hidden_size + 2 * kv_dim)
        self.o_proj = nn.Linear(hidden_size, hidden_size)
        self.flash_attention = FlashAttention3(self.config)
        self._init_weights()

    def _init_weights(self):
        for lin in (self.qkv_proj, self.o_proj):
            nn.init.normal_(lin.weight, mean=0.0, std=0.02)
            if lin.bias is not None:
                nn.init.zeros_(lin.bias)

    def _prepare_qkv(self, hidden_states: torch.Tensor):
        """reference :829-860 — one GEMM, then strided views (the kernel takes the strides; no copies)."""
        B, S, _ = hidden_states.shape
        qkv = self.qkv_proj(hidden_states)
        kv_dim = self.num_kv_heads * self.head_dim
        q, k, v = qkv.split([self.hidden_size, kv_dim, kv_dim], dim=-1)
        return (q.view(B, S, self.num_attention_heads, self.head_dim), k.view(B, S, self.num_kv_heads, self.head_dim),
                v.view(B, S, self.num_kv_heads, self.head_dim))

    def forward(self, hidden_states: torch.Tensor, attention_mask: Optional[torch.Tensor] = None, **kwargs: Any) -> torch.Tensor:
        B, S, _ = hidden_states.shape
        q, k, v = self._prepare_qkv(hidden_states)
        if "block_tables" in kwargs:
            return self.o_proj(self._paged_decode(q, kwargs))
        ctx = self.flash_attention(q, k, v, attention_mask)
        return self.o_proj(ctx.reshape(B, S, self.hidden_size))


# Paged-generation context (baseline.inference.generate_paged): HF model forwards do not carry custom keyword arguments
# down to the attention blocks, so the adapters read the paged cache / block tables of the current step from here.
_PAGED_CONTEXT: Optional[Dict[str, Any]] = None


def set_paged_context(ctx: Optional[Dict[str, Any]]) -> None:
    global _PAGED_CONTEXT
    _PAGED_CONTEXT = ctx


class _HFAttentionAdapter(nn.Module):
    """Stands in for a HuggingFace attention block: accepts HF's keyword arguments, returns HF's tuple, and keeps the HF
    KV cache protocol (``past_key_values.update``) so ``model.generate`` works unchanged. Prefill and cached decode
    both run K1; the causal diagonal is aligned bottom-right (``causal_offset = Sk - Sq``) when a cache is present."""

    def __init__(self, inner: nn.Module, layer_idx: Optional[int] = None, returns_tuple_len: int = 2, rotary: bool = False):
        super().__init__()
        self.inner = inner
        self.layer_idx = layer_idx
        self.returns_tuple_len = returns_tuple_len
        self.rotary = rotary  # Llama family: q/k are rotated with the (cos, sin) HF passes as ``position_embeddings``

    @staticmethod
    def _apply_rotary(q, k, position_embeddings):
        """HF ``apply_rotary_pos_emb`` for the [B,S,H,D] layout (modeling_llama.py: q*cos + rotate_half(q)*sin; the
        reference's converter (flash_attention.py:1063-1142) replaces these modules without rotating at all)."""
        if position_embeddings is None:
            raise NotImplementedError("this attention module needs rotary position embeddings: the caller must pass "
                                      "position_embeddings=(cos, sin) as HuggingFace decoder layers do")
        cos, sin = position_embeddings
        cos, sin = cos.unsqueeze(2).to(q.dtype), sin.unsqueeze(2).to(q.dtype)  # [B,S,1,D]

        def rot(x):
            half = x.shape[-1] // 2
            return torch.cat((-x[..., half:], x[..., :half]), dim=-1)
        return q * cos + rot(q) * sin, k * cos + rot(k) * sin

    @staticmethod
    def _mask_to_kv_lens(attention_mask, B: int, Sq: int, Sk: int, causal: bool):
        """Lower HF's ``attention_mask`` to per-sequence key counts (right padding), or raise.

        HF passes None (no padding, causal handled by the kernel), a 2-D ``[B,Sk]`` keep-mask, or a 4-D ``[B,1,Sq,Sk]``
        additive / boolean mask that already contains the causal triangle. Supported: (causal +) RIGHT padding, i.e. the
        keys a sequence keeps form a prefix. Anything else (left padding, sliding windows, prefix-LM, arbitrary masks)
        raises NotImplementedError — never a silent unmasked run (reference convert_mask, flash_attention.py:1145-1168,
        passes masks through to a kernel that ignores them)."""
        if attention_mask is None:
            return None
        m = attention_mask
        if m.dim() == 2:
            keep_last = m != 0
            keep_first = None
        elif m.dim() == 4 and m.shape[1] == 1 and m.shape[-1] == Sk and m.shape[2] in (1, Sq):
            vis = m if m.dtype == torch.bool else (m == 0)
            keep_last = vis[:, 0, -1, :]   # the last query sees every kept key (causal or not)
            keep_first = vis[:, 0, 0, :] if m.shape[2] == Sq and Sq > 1 else None
        else:
            raise NotImplementedError(f"attention_mask of shape {tuple(m.shape)} is not supported by the B200 attention path")
        if keep_last.shape != (B, Sk):
            raise NotImplementedError(f"attention_mask of shape {tuple(m.shape)} does not match keys [{B},{Sk}]")
        lens = keep_last.sum(dim=-1).to(torch.int32)
        idx = torch.arange(Sk, device=m.device).unsqueeze(0)
        ok = torch.equal(keep_last, idx < lens.unsqueeze(1))
        if ok and keep_first is not None:
            # the first query (global position Sk - Sq) sees keys [0, Sk - Sq] under a causal mask, all kept keys otherwise
            want = (idx <= (Sk - Sq)) & keep_last if causal else keep_last
            ok = torch.equal(keep_first & keep_last, want)
        if not ok:
            raise NotImplementedError("only causal masks with RIGHT padding are supported on the B200 attention path (kept keys "
                                      "must form a prefix; left padding / windows / arbitrary masks would need a dense-mask kernel)")
        if bool((lens == Sk).all()):
            return None
        return lens.contiguous()

    def _qkv(self, hidden_states):
        inner = self.inner
        if isinstance(inner, FlashSelfAttention):
            return inner._prepare_qkv(hidden_states)
        B, S, _ = hidden_states.shape
        return (inner.q_proj(hidden_states).view(B, S, inner.num_attention_heads, inner.head_dim),
                inner.k_proj(hidden_states).view(B, S, inner.num_kv_heads, inner.head_dim),
                inner.v_proj(hidden_states).view(B, S, inner.num_kv_heads, inner.head_dim))

    def forward(self, hidden_states, *args, attention_mask=None, **kwargs):
        inner = self.inner
        if "block_tables" in kwargs:
            passthrough = {k: v for k, v in kwargs.items() if k in ("physical_kv_cache_k", "physical_kv_cache_v", "block_tables",
                                                                     "context_lengths", "kv_cache_block_size", "max_seq_len",
                                                                     "layer_idx")}
            return (inner(hidden_states, None, **passthrough),) + (None,) * (self.returns_tuple_len - 1)
        cache = kwargs.get("past_key_values", kwargs.get("past_key_value", kwargs.get("layer_past")))
        if cache is None and args and hasattr(args[0], "update"):
            cache = args[0]
        B, S, _ = hidden_states.shape
        q, k, v = self._qkv(hidden_states)
        if self.rotary:
            pe = kwargs.get("position_embeddings")
            if pe is None and args and isinstance(args[0], (tuple, list)) and len(args[0]) == 2:
                pe = args[0]  # LlamaDecoderLayer passes it as a keyword; positional callers use slot 1
            q, k = self._apply_rotary(q, k, pe)
        fa = inner.flash_attention
        orig = q.dtype
        dt = fa._compute_dtype(orig)
        if _PAGED_CONTEXT is not None:
            ctx_ = _PAGED_CONTEXT
            paged = ctx_["cache"]
            # (the check reads the mask back to the host: skipped while the decode step is being captured into a CUDA graph —
            # the eager warm-up steps before the capture have already validated the same mask pattern)
            if attention_mask is not None and not torch.cuda.is_current_stream_capturing() and \
                    self._mask_to_kv_lens(attention_mask, B, S, attention_mask.shape[-1], True) is not None:
                raise NotImplementedError("the paged prefill / decode path serves equal-length, unpadded prompts")
            if q.dtype != dt:
                q, k, v = q.to(dt), k.to(dt), v.to(dt)
            if ctx_["mode"] == "prefill":
                paged.write_prefill(self.layer_idx, ctx_["seq_ids"], k, v)
                attn = ops.flash_attn_fwd(q, k, v, causal=True, softmax_scale=inner.config.softmax_scale)
            else:
                kc, vc = paged.get_physical_caches()
                ks, vs = paged.layer_scales(self.layer_idx)
                ops.kv_append(k[:, 0], v[:, 0], kc, vc, ctx_["context_lengths"], ctx_["block_tables"], self.layer_idx,
                              k_scale=ks, v_scale=vs)
                attn = ops.decode_attention(q[:, 0].contiguous(), kc, vc, ctx_["context_lengths"],
                                            softmax_scale=inner.config.softmax_scale, block_tables=ctx_["block_tables"],
                                            layer_idx=self.layer_idx, max_context_len=ctx_.get("max_context_len"),
                                            k_scale=ks, v_scale=vs).unsqueeze(1)
            out = inner.o_proj(attn.reshape(B, S, inner.hidden_size).to(orig))
            return (out,) + (None,) * (self.returns_tuple_len - 1)
        if cache is not None and hasattr(cache, "update"):
            k_all, v_all = cache.update(k.transpose(1, 2), v.transpose(1, 2), self.layer_idx)  # [B,Hkv,Sk,D]
            k, v = k_all.transpose(1, 2), v_all.transpose(1, 2)
        if q.dtype != dt:
            q, k, v = q.to(dt), k.to(dt), v.to(dt)
        # HF passes an additive 4-D mask: causal triangle (the kernel does that itself) + padding (lowered to kv_lens)
        kv_lens = self._mask_to_kv_lens(attention_mask, B, S, k.shape[1], inner.config.causal)
        ctx = ops.flash_attn_fwd(q, k, v, causal=inner.config.causal, softmax_scale=inner.config.softmax_scale,
                                 causal_offset=k.shape[1] - S, kv_lens=kv_lens)
        out = inner.o_proj(ctx.reshape(B, S, inner.hidden_size).to(orig))
        return (out,) + (None,) * (self.returns_tuple_len - 1)


class ModelConverter:
    """reference: kernels/attention/flash_attention.py:952-1168 — walks a model and swaps attention modules. Unlike
    the reference (which builds fresh random modules for most architectures, Appendix B) the projection weights
    are copied, including GPT-2's fused ``c_attn`` Conv1D (weight stored [in, out])."""

    def __init__(self, config: Optional[FlashAttentionConfig] = None):
        self.config = config or FlashAttentionConfig()

    def convert_model(self, model: nn.Module) -> nn.Module:
        return self._find_and_replace_attention(model)

    def _find_and_replace_attention(self, module: nn.Module) -> nn.Module:
        for name, sub in list(module.named_children()):
            if self._is_attention_module(sub):
                setattr(module, name, self._create_flash_replacement(sub))
            else:
                self._find_and_replace_attention(sub)
        return module

    @staticmethod
    def _is_attention_module(m: nn.Module) -> bool:
        if isinstance(m, (FlashAttentionLayer, FlashSelfAttention, _HFAttentionAdapter)):
            return False
        cls = type(m).__name__
        if cls in ("GPT2Attention", "GPT2SdpaAttention", "GPT2FlashAttention2"):
            return hasattr(m, "c_attn") and hasattr(m, "c_proj")
        has_sep = all(hasattr(m, a) for a in ("q_proj", "k_proj", "v_proj")) and (hasattr(m, "o_proj") or hasattr(m, "out_proj"))
        has_fused = (hasattr(m, "qkv_proj") or hasattr(m, "qkv")) and (hasattr(m, "o_proj") or hasattr(m, "out_proj"))
        return ("attention" in cls.lower() or "attn" in cls.lower()) and (has_sep or has_fused)

    @staticmethod
    def _copy_linear(dst: nn.Linear, weight: torch.Tensor, bias: Optional[torch.Tensor]):
        with torch.no_grad():
            dst.weight.copy_(weight.to(dst.weight.dtype))
            if bias is not None:
                dst.bias.copy_(bias.to(dst.bias.dtype))
            else:
                dst.bias.zero_()

    def _create_flash_replacement(self, m: nn.Module) -> nn.Module:
        cfg = self.config
        ref_param = next(m.parameters())
        cls = type(m).__name__
        if cls.startswith("GPT2"):
            hidden = m.embed_dim
            heads = m.num_heads
            new = FlashSelfAttention(hidden, heads, FlashAttentionConfig(**{**cfg.__dict__, "causal": True}))
            # HF Conv1D computes x @ W + b with W [in, out]; nn.Linear wants [out, in]
            self._copy_linear(new.qkv_proj, m.c_attn.weight.t(), m.c_attn.bias)
            self._copy_linear(new.o_proj, m.c_proj.weight.t(), m.c_proj.bias)
            new.to(device=ref_param.device, dtype=ref_param.dtype)
            return _HFAttentionAdapter(new, layer_idx=getattr(m, "layer_idx", None), returns_tuple_len=2)
        o_src = m.o_proj if hasattr(m, "o_proj") else m.out_proj
        hidden = o_src.out_features
        heads = getattr(m, "num_heads", None) or getattr(m, "num_attention_heads", None) or \
            getattr(getattr(m, "config", None), "num_attention_heads", None)
        if heads is None:
            raise ValueError(f"cannot infer the number of heads of {cls}")
        if hasattr(m, "q_proj"):
            head_dim = m.q_proj.out_features // heads
            kv_heads = m.k_proj.out_features // head_dim
            causal = bool(getattr(m, "is_causal", cfg.causal))
            new = FlashAttentionLayer(hidden, heads, FlashAttentionConfig(**{**cfg.__dict__, "causal": causal}), num_kv_heads=kv_heads)
            for dst, src in ((new.q_proj, m.q_proj), (new.k_proj, m.k_proj), (new.v_proj, m.v_proj), (new.o_proj, o_src)):
                self._copy_linear(dst, src.weight, src.bias)
            if hasattr(m, "layer_idx") and type(m).__module__.startswith("transformers."):
                for extra in ("q_norm", "k_norm", "sliding_window"):
                    if getattr(m, extra, None) is not None:
                        raise NotImplementedError(f"{cls}.{extra} is not supported by the B200 attention replacement")
                scaling = getattr(m, "scaling", None)
                if scaling is not None and abs(float(scaling) - head_dim ** -0.5) > 1e-9:
                    new.config.softmax_scale = float(scaling)
                rotary = hasattr(m, "rotary_emb") or any(t in cls for t in ("Llama", "Mistral", "Qwen2"))
                new.to(device=ref_param.device, dtype=ref_param.dtype)
                return _HFAttentionAdapter(new, layer_idx=m.layer_idx, returns_tuple_len=2, rotary=rotary)
        else:
            src = m.qkv_proj if hasattr(m, "qkv_proj") else m.qkv
            head_dim = hidden // heads
            kv_heads = (src.out_features - hidden) // (2 * head_dim)
            new = FlashSelfAttention(hidden, heads, cfg, num_kv_heads=kv_heads)
            self._copy_linear(new.qkv_proj, src.weight, src.bias)
            self._copy_linear(new.o_proj, o_src.weight, o_src.bias)
        new.to(device=ref_param.device, dtype=ref_param.dtype)
        return new

    @staticmethod
    def convert_mask(attention_mask: Optional[torch.Tensor]) -> Optional[torch.Tensor]:
        """reference :1145-1168."""
        if attention_mask is None:
            return None
        if attention_mask.dim() == 2:
            attention_mask = attention_mask.unsqueeze(1).unsqueeze(2)
        elif attention_mask.dim() == 3 and attention_mask.shape[1] == 1:
            attention_mask = attention_mask.unsqueeze(2)
        return attention_mask.bool()


def _cuda_time_ms(fn, iters: int, warmup: int) -> float:
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(iters):
        fn()
    e.record()
    torch.cuda.synchronize()
    return s.elapsed_time(e) / iters


def benchmark_flash_attention_speed(batch_size: int = 32, seq_len: int = 512, num_heads: int = 8, head_dim: int = 64,
                                    device: str = "cuda", causal: bool = False, num_iters: int = 100,
                                    warmup_iters: int = 10) -> Dict[str, float]:
    """reference :1171-1279 — FlashAttention3 vs eager ``standard_attention`` (einsum / softmax / einsum)."""
    q, k, v = (torch.randn(batch_size, seq_len, num_heads, head_dim, device=device, dtype=torch.bfloat16) for _ in range(3))
    fa = FlashAttention3(FlashAttentionConfig(causal=causal, precision="bf16"))

    def standard_attention():
        scores = torch.einsum("bshd,bthd->bhst", q, k) / math.sqrt(head_dim)
        if causal:
            scores = scores.masked_fill(torch.triu(torch.ones(seq_len, seq_len, device=device, dtype=torch.bool), 1), float("-inf"))
        return torch.einsum("bhst,bthd->bshd", torch.softmax(scores.float(), dim=-1).to(q.dtype), v)

    flash_ms = _cuda_time_ms(lambda: fa(q, k, v), num_iters, warmup_iters)
    std_ms = _cuda_time_ms(standard_attention, max(1, num_iters // 10), max(1, warmup_iters // 5))
    max_diff = (fa(q, k, v).float() - standard_attention().float()).abs().max().item()
    return {"flash_attention_ms": flash_ms, "standard_attention_ms": std_ms, "speedup": std_ms / flash_ms, "max_diff": max_diff}


def benchmark_memory_usage(batch_size: int = 8, seq_len: int = 2048, num_heads: int = 8, head_dim: int = 64,
                           device: str = "cuda", causal: bool = False) -> Dict[str, float]:
    """reference :1282-1375 — peak allocator bytes of one forward."""
    q, k, v = (torch.randn(batch_size, seq_len, num_heads, head_dim, device=device, dtype=torch.bfloat16) for _ in range(3))
    fa = FlashAttention3(FlashAttentionConfig(causal=causal, precision="bf16"))
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    fa(q, k, v)
    torch.cuda.synchronize()
    flash_peak = torch.cuda.max_memory_allocated() - base
    theory = fa.get_theoretical_memory_usage(seq_len, batch_size, num_heads, head_dim)
    return {"flash_attention_peak_mb": flash_peak / 2 ** 20, **theory}
