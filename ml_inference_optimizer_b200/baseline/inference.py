"""Mirror of the hot-path slice of the reference's ``baseline/inference.py`` (SURVEY.md §8 f1).

* ``BlockManager`` / ``SequenceMetadata`` / ``PagedKVCache`` — same classes, constructor arguments and method names as
  the reference (:1045-1302); the physical cache is ``[num_blocks, num_layers, block_size, num_kv_heads, head_dim]``
  (:1077-1084), the layout K2 (``b200_fa_decode``) and ``b200_kv_append`` read and write.
* ``InferenceRunner.run_inference`` — the reference's timing / memory harness with its metric keys (:653-713);
  ``create_inference_runner`` (:1779-1838) returns a runner whose ``_forward`` actually exists (the reference's
  ``TransformerInferenceRunner`` is abstract, SURVEY.md F10).
* ``generate_paged`` — a greedy decode loop that drives prefill (K1), KV append and paged decode attention (K2) through
  the attention modules installed by ``kernels.attention.flash_attention.ModelConverter``. Nothing in the reference
  drives its paged kernel (SURVEY.md §3B); this is that missing loop.
"""
from __future__ import annotations

import logging
import math
import time
from copy import deepcopy
from typing import Any, Callable, Dict, List, Optional, Sequence, Tuple, Union

import torch
import torch.nn as nn

from ..kernels.attention import flash_attention as _fa

__all__ = ["BlockManager", "SequenceMetadata", "PagedKVCache", "KVCache", "InferenceRunner", "BasicInferenceRunner",
           "TransformerInferenceRunner", "create_inference_runner", "generate_paged", "FusionPattern", "FusionRegistry",
           "fusion_registry", "convert_to_flash_attention"]


class BlockManager:
    """reference :1045-1127 — free-list allocator with reference counts over the physical blocks."""

    def __init__(self, num_blocks: int, block_size: int, num_layers: int, num_heads: int, head_dim: int, dtype: torch.dtype,
                 device: str):
        self.num_blocks, self.block_size, self.num_layers = num_blocks, block_size, num_layers
        self.num_heads, self.head_dim, self.dtype, self.device = num_heads, head_dim, dtype, device
        self.free_blocks = list(range(num_blocks))
        self.ref_counts = [0] * num_blocks  # host-side (the reference keeps them on the device and syncs on every access)
        from .. import ops
        # physical width: 64 or 128 columns (what K2 / kv_append are built for); a narrower head leaves zero columns behind it
        self.physical_head_dim = ops.cache_head_dim(head_dim)
        shape = (num_blocks, num_layers, block_size, num_heads, self.physical_head_dim)
        self.gpu_cache_k = torch.zeros(shape, dtype=dtype, device=device)
        self.gpu_cache_v = torch.zeros(shape, dtype=dtype, device=device)
        self.is_initialized = True

    def allocate_block(self) -> int:
        if not self.free_blocks:
            raise MemoryError("Out of memory: No free blocks available in KV cache.")
        idx = self.free_blocks.pop()
        self.ref_counts[idx] = 1
        return idx

    def free_block(self, block_idx: int) -> None:
        if self.ref_counts[block_idx] <= 0:
            logging.warning(f"Attempting to free block {block_idx} with ref count {self.ref_counts[block_idx]}.")
            return
        self.ref_counts[block_idx] -= 1
        if self.ref_counts[block_idx] == 0:
            self.free_blocks.append(block_idx)

    def increase_ref_count(self, block_idx: int) -> None:
        if self.ref_counts[block_idx] <= 0:
            raise ValueError(f"Cannot increase ref count for unallocated block {block_idx}.")
        self.ref_counts[block_idx] += 1

    def get_num_free_blocks(self) -> int:
        return len(self.free_blocks)

    def get_physical_block(self, block_idx: int, layer_idx: int) -> Tuple[torch.Tensor, torch.Tensor]:
        return self.gpu_cache_k[block_idx, layer_idx], self.gpu_cache_v[block_idx, layer_idx]

    def get_physical_caches(self) -> Tuple[torch.Tensor, torch.Tensor]:
        return self.gpu_cache_k, self.gpu_cache_v


class SequenceMetadata:
    """reference :1129-1147."""

    def __init__(self, seq_id: int):
        self.seq_id = seq_id
        self.block_table: List[int] = []
        self.logical_len = 0

    def append_block(self, block_idx: int):
        self.block_table.append(block_idx)

    def get_last_block_physical_idx(self) -> Optional[int]:
        return self.block_table[-1] if self.block_table else None

    def __len__(self) -> int:
        return len(self.block_table)


def _per_layer_scales(name: str, scale: Union[float, Sequence[float]], num_layers: int) -> List[float]:
    vals = [float(scale)] * num_layers if isinstance(scale, (int, float)) else [float(x) for x in scale]
    if len(vals) != num_layers:
        raise ValueError(f"{name} has {len(vals)} values for {num_layers} layers")
    if not all(math.isfinite(x) and x > 0 for x in vals):
        raise ValueError(f"{name} values must be positive and finite, got {vals}")
    return vals


class PagedKVCache:
    """reference :1150-1302.

    ``dtype=torch.float8_e4m3fn`` stores K and V as e4m3 bytes: half the memory of a 16-bit cache, read by the FP8 decode
    kernels. ``k_scale`` / ``v_scale`` (a float, or one value per layer) are what a stored byte is multiplied by when it is
    read (K is stored as e4m3(K / k_scale)); a 16-bit cache takes only 1.0."""

    def __init__(self, num_blocks: int, block_size: int, num_layers: int, num_heads: int, head_dim: int,
                 dtype: torch.dtype = torch.float16, device: str = "cuda", k_scale: Union[float, Sequence[float]] = 1.0,
                 v_scale: Union[float, Sequence[float]] = 1.0):
        self.k_scales = _per_layer_scales("k_scale", k_scale, num_layers)
        self.v_scales = _per_layer_scales("v_scale", v_scale, num_layers)
        if dtype != torch.float8_e4m3fn and any(x != 1.0 for x in self.k_scales + self.v_scales):
            raise ValueError("k_scale / v_scale apply to an FP8 (torch.float8_e4m3fn) cache only")
        self.block_manager = BlockManager(num_blocks, block_size, num_layers, num_heads, head_dim, dtype, device)
        self.block_size, self.num_layers, self.num_heads, self.head_dim = block_size, num_layers, num_heads, head_dim
        self.dtype, self.device = dtype, device
        self.sequences: Dict[int, SequenceMetadata] = {}

    def layer_scales(self, layer_idx: int) -> Tuple[float, float]:
        """``(k_scale, v_scale)`` of one layer: a stored K / V byte is worth ``byte * scale``."""
        return self.k_scales[layer_idx], self.v_scales[layer_idx]

    def _ensure_sequence_exists(self, seq_id: int):
        if seq_id not in self.sequences:
            self.sequences[seq_id] = SequenceMetadata(seq_id)

    def _get_logical_block_idx(self, token_pos: int) -> int:
        return token_pos // self.block_size

    def _get_block_offset(self, token_pos: int) -> int:
        return token_pos % self.block_size

    def allocate_blocks_for_sequence(self, seq_id: int, num_tokens: int):
        self._ensure_sequence_exists(seq_id)
        meta = self.sequences[seq_id]
        for _ in range(math.ceil(num_tokens / self.block_size) - len(meta)):
            meta.append_block(self.block_manager.allocate_block())
        meta.logical_len = max(meta.logical_len, num_tokens)

    def reserve_blocks(self, seq_id: int, num_tokens: int) -> None:
        """Allocate the blocks that ``num_tokens`` tokens will need without changing the sequence length, so the block
        table stays fixed while the tokens are appended (what a captured decode graph needs)."""
        self._ensure_sequence_exists(seq_id)
        meta = self.sequences[seq_id]
        for _ in range(math.ceil(num_tokens / self.block_size) - len(meta)):
            meta.append_block(self.block_manager.allocate_block())

    def append_token(self, seq_id: int) -> None:
        self._ensure_sequence_exists(seq_id)
        meta = self.sequences[seq_id]
        new_len = meta.logical_len + 1
        if math.ceil(new_len / self.block_size) > len(meta):
            try:
                meta.append_block(self.block_manager.allocate_block())
            except MemoryError:
                self.free_sequence(seq_id)
                raise
        meta.logical_len = new_len

    def get_block_table(self, seq_id: int) -> List[int]:
        if seq_id not in self.sequences:
            raise ValueError(f"Sequence {seq_id} not found in cache.")
        return self.sequences[seq_id].block_table

    def get_sequence_length(self, seq_id: int) -> int:
        return self.sequences[seq_id].logical_len if seq_id in self.sequences else 0

    def free_sequence(self, seq_id: int) -> None:
        meta = self.sequences.pop(seq_id, None)
        if meta is not None:
            for blk in meta.block_table:
                self.block_manager.free_block(blk)

    def get_physical_caches(self) -> Tuple[torch.Tensor, torch.Tensor]:
        return self.block_manager.get_physical_caches()

    def get_memory_usage(self) -> Dict[str, float]:
        k, v = self.get_physical_caches()
        total = (k.numel() + v.numel()) * k.element_size() / 2 ** 20
        used = self.block_manager.num_blocks - self.block_manager.get_num_free_blocks()
        return {"total_mb": total, "used_blocks": used, "free_blocks": self.block_manager.get_num_free_blocks(),
                "used_mb": total * used / max(1, self.block_manager.num_blocks)}

    # ---- device-side views the kernels consume ----
    def device_tables(self, seq_ids: List[int]) -> Tuple[torch.Tensor, torch.Tensor]:
        """int32 ``block_tables [B, max_blocks]`` and ``context_lengths [B]`` for a batch of sequences."""
        tables = [self.get_block_table(s) for s in seq_ids]
        width = max(1, max(len(t) for t in tables))
        bt = torch.zeros(len(seq_ids), width, dtype=torch.int32)
        for i, t in enumerate(tables):
            bt[i, :len(t)] = torch.tensor(t, dtype=torch.int32)
        lens = torch.tensor([self.get_sequence_length(s) for s in seq_ids], dtype=torch.int32)
        return bt.to(self.device), lens.to(self.device)

    def write_prefill(self, layer_idx: int, seq_ids: List[int], k: torch.Tensor, v: torch.Tensor) -> None:
        """Scatter the prompt's K,V ``[B,S,Hkv,D]`` into the blocks (prefill; the per-token path is ``b200_kv_append``).
        An FP8 cache is written by ``b200_kv_append_fp8`` with all S rows at once, so prefill and decode quantize alike."""
        kc, vc = self.get_physical_caches()
        B, S = k.shape[:2]
        if self.dtype == torch.float8_e4m3fn:
            from .. import ops
            bt, _ = self.device_tables(seq_ids)
            lens = torch.full((B,), S, dtype=torch.int32, device=bt.device)
            ks, vs = self.layer_scales(layer_idx)
            ops.kv_append(k, v, kc, vc, lens, bt, layer_idx, k_scale=ks, v_scale=vs)
            return
        pos = torch.arange(S)
        for b, sid in enumerate(seq_ids):
            table = torch.tensor(self.get_block_table(sid), dtype=torch.long)
            blk = table[pos // self.block_size].to(k.device)
            off = (pos % self.block_size).to(k.device)
            kc[blk, layer_idx, off, :, :k.shape[-1]] = k[b].to(kc.dtype)   # (columns past head_dim stay zero)
            vc[blk, layer_idx, off, :, :v.shape[-1]] = v[b].to(vc.dtype)


# ------------------------------------------------------------------------------------------------------------------
# runners
# ------------------------------------------------------------------------------------------------------------------
class InferenceRunner:
    """reference :377-789 reduced to its measurement harness: ``run_inference(inputs, **kw) -> (outputs, metrics)`` with
    the reference's metric keys (:653-713)."""

    def __init__(self, model: nn.Module, device: str = "cuda", precision: str = "fp16"):
        self.model, self.device, self.precision = model, device, precision

    def _forward(self, inputs: Any, **kwargs) -> Any:
        raise NotImplementedError

    def run_inference(self, inputs: Any, **kwargs) -> Tuple[Any, Dict[str, float]]:
        metrics: Dict[str, float] = {}
        cuda = torch.cuda.is_available() and str(self.device).startswith("cuda")
        if cuda:
            torch.cuda.synchronize()
            torch.cuda.reset_peak_memory_stats()
            metrics["memory_before_mb"] = torch.cuda.memory_allocated() / 2 ** 20
            start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            start.record()
        t0 = time.perf_counter()
        with torch.no_grad():
            outputs = self._forward(inputs, **kwargs)
        if cuda:
            end.record()
            torch.cuda.synchronize()
            metrics["cuda_time_ms"] = start.elapsed_time(end)
        metrics["total_time_ms"] = (time.perf_counter() - t0) * 1e3
        if cuda:
            metrics["memory_after_mb"] = torch.cuda.memory_allocated() / 2 ** 20
            metrics["peak_memory_mb"] = torch.cuda.max_memory_allocated() / 2 ** 20
            metrics["memory_change_mb"] = metrics["memory_after_mb"] - metrics["memory_before_mb"]
        return outputs, metrics


    def warmup(self, inputs: Any, iterations: int = 10) -> None:
        """reference :616-639."""
        self.model.eval()
        with torch.no_grad():
            for _ in range(iterations):
                self._forward(inputs)
        if torch.cuda.is_available() and str(self.device).startswith("cuda"):
            torch.cuda.synchronize()

    def run_batch_inference(self, batch_inputs: List[Any], **kwargs) -> List[Tuple[Any, Dict[str, float]]]:
        """reference :715-746 — ``run_inference`` per element; the batch totals (``total_batch_time_ms``,
        ``avg_inference_time_ms`` and the per-key sums) are kept on ``self.last_batch_metrics`` (the reference computes and
        drops them)."""
        results, totals = [], {}
        t0 = time.perf_counter()
        for inputs in batch_inputs:
            outputs, metrics = self.run_inference(inputs, **kwargs)
            results.append((outputs, metrics))
            for k, v in metrics.items():
                totals[k] = totals.get(k, 0.0) + v
        totals["total_batch_time_ms"] = (time.perf_counter() - t0) * 1e3
        totals["avg_inference_time_ms"] = totals["total_batch_time_ms"] / max(1, len(batch_inputs))
        self.last_batch_metrics = totals
        return results

    def profile_model(self, inputs: Any, use_cuda: bool = True) -> Dict[str, Any]:
        """reference :748-784 — one forward under ``torch.profiler``; returns the table, the events and the key averages."""
        from torch.profiler import ProfilerActivity, profile, record_function

        cuda = use_cuda and torch.cuda.is_available() and str(self.device).startswith("cuda")
        acts = [ProfilerActivity.CPU] + ([ProfilerActivity.CUDA] if cuda else [])
        self.model.eval()
        with profile(activities=acts, record_shapes=True) as prof:
            with record_function("model_inference"), torch.no_grad():
                self._forward(inputs)
        avg = prof.key_averages()
        return {"table": avg.table(sort_by="cuda_time_total" if cuda else "cpu_time_total", row_limit=20), "events": prof.events(),
                "key_averages": avg}


class BasicInferenceRunner(InferenceRunner):
    """reference :1834-1838 plus the generation branch ``verify_baseline.py:277-288`` expects."""

    def _forward(self, inputs: Any, **kwargs) -> Any:
        gen_keys = {"max_new_tokens", "max_length", "do_sample", "num_beams", "temperature", "top_k", "top_p"}
        if isinstance(inputs, dict):
            if gen_keys & set(kwargs) and hasattr(self.model, "generate"):
                return self.model.generate(**inputs, **kwargs)
            return self.model(**inputs, **kwargs)
        if gen_keys & set(kwargs) and hasattr(self.model, "generate"):
            return self.model.generate(inputs, **kwargs)
        return self.model(inputs, **kwargs)


def create_inference_runner(model: nn.Module, device: str = "cuda", precision: str = "fp16", model_type: str = "transformer",
                            use_flash_attention: bool = False, use_kernel_fusion: bool = False, use_kv_cache: bool = True,
                            use_cuda_graph: bool = False) -> InferenceRunner:
    """reference :1779-1838. ``use_flash_attention`` / ``use_kernel_fusion`` swap in the B200 attention / FusedMLP modules
    (weights copied) before the runner is built."""
    if use_flash_attention or use_kernel_fusion:
        from ..optimizer import Optimizer
        model = Optimizer(model).optimize(use_flash_attention=use_flash_attention, use_fused_mlp=use_kernel_fusion)
    # (the reference builds a TransformerInferenceRunner here, :1806-1822; that runner sizes a paged cache from the free
    #  device memory, so it is constructed explicitly by callers that want it, with ``kv_cache_num_gpu_blocks``)
    del model_type, use_kv_cache, use_cuda_graph
    return BasicInferenceRunner(model, device, precision)


class KVCache:
    """reference :791-1043 — the plain (non-paged) per-layer cache with the reference's constructor, methods and statistics.

    Storage is ``[max_batch_size, max_seq_len, num_heads, head_dim]`` per layer: exactly the contiguous layout K2
    (``ops.decode_attention`` without block tables) reads, so ``decode_views`` hands a layer to the decode kernel without a
    gather. ``use_block_storage`` / ``block_size`` are accepted; they only change how ``memory_efficiency`` is reported
    (blocks touched / blocks held), the values returned are identical. The reference advances one shared length per
    ``append`` call, so appending the same tokens to two layers counts them twice; here lengths are kept per layer and
    ``current_seq_lengths[b]`` is the longest layer."""

    def __init__(self, max_batch_size: int = 1, max_seq_len: int = 2048, use_block_storage: bool = True, block_size: int = 64):
        self.max_batch_size, self.max_seq_len = max_batch_size, max_seq_len
        self.use_block_storage, self.block_size = use_block_storage, block_size
        self.num_layers = self.num_heads = self.head_dim = 0
        self.k_caches: Dict[int, torch.Tensor] = {}
        self.v_caches: Dict[int, torch.Tensor] = {}
        self._lengths: List[List[int]] = []
        self.is_initialized = False

    @property
    def current_seq_lengths(self) -> List[int]:
        if not self._lengths:
            return [0] * self.max_batch_size
        return [max(layer[b] for layer in self._lengths) for b in range(self.max_batch_size)]

    def initialize(self, num_layers: int, num_heads: int, head_dim: int, dtype: torch.dtype = torch.float16,
                   device: str = "cuda") -> None:
        self.num_layers, self.num_heads, self.head_dim = num_layers, num_heads, head_dim
        from .. import ops
        shape = (self.max_batch_size, self.max_seq_len, num_heads, ops.cache_head_dim(head_dim))   # zero columns past head_dim
        self.k_caches = {l: torch.zeros(shape, dtype=dtype, device=device) for l in range(num_layers)}
        self.v_caches = {l: torch.zeros(shape, dtype=dtype, device=device) for l in range(num_layers)}
        self._lengths = [[0] * self.max_batch_size for _ in range(num_layers)]
        self.is_initialized = True

    def reset(self) -> None:
        """Empty the cache, keep the allocation."""
        self._lengths = [[0] * self.max_batch_size for _ in range(self.num_layers)] if self.is_initialized else []

    def clear(self) -> None:
        """Free the tensors."""
        self.k_caches, self.v_caches, self._lengths, self.is_initialized = {}, {}, [], False

    def _check(self, layer_idx: int, batch_idx: int) -> None:
        if not self.is_initialized:
            raise RuntimeError("Cache not initialized. Call initialize() first.")
        if not (0 <= layer_idx < self.num_layers and 0 <= batch_idx < self.max_batch_size):
            raise IndexError(f"layer {layer_idx} / batch {batch_idx} outside the cache ({self.num_layers} layers, "
                             f"{self.max_batch_size} sequences)")

    def get_kv_cache(self, layer_idx: int, batch_idx: int = 0) -> Tuple[Optional[torch.Tensor], Optional[torch.Tensor]]:
        """``(k, v)`` of shape ``[seq_len, num_heads, head_dim]`` (views), or ``(None, None)`` for an empty sequence in block
        mode, as the reference returns (:917-918)."""
        self._check(layer_idx, batch_idx)
        n = self._lengths[layer_idx][batch_idx]
        if n == 0 and self.use_block_storage:
            return None, None
        return self.k_caches[layer_idx][batch_idx, :n, :, :self.head_dim], self.v_caches[layer_idx][batch_idx, :n, :, :self.head_dim]

    def append(self, layer_idx: int, batch_idx: int, k: torch.Tensor, v: torch.Tensor) -> None:
        """k, v ``[seq_len, num_heads, head_dim]`` appended behind what the layer already holds."""
        self._check(layer_idx, batch_idx)
        cur = self._lengths[layer_idx][batch_idx]
        new = cur + k.size(0)
        if new > self.max_seq_len:
            raise ValueError(f"Sequence length {new} exceeds maximum {self.max_seq_len}")
        self.k_caches[layer_idx][batch_idx, cur:new, :, :self.head_dim] = k
        self.v_caches[layer_idx][batch_idx, cur:new, :, :self.head_dim] = v
        self._lengths[layer_idx][batch_idx] = new

    def decode_views(self, layer_idx: int) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
        """``(k_cache, v_cache, context_lens int32)`` of one layer in the form ``ops.decode_attention`` takes."""
        self._check(layer_idx, 0)
        k = self.k_caches[layer_idx]
        return k, self.v_caches[layer_idx], torch.tensor(self._lengths[layer_idx], dtype=torch.int32, device=k.device)

    def get_memory_usage(self) -> Dict[str, float]:
        if not self.is_initialized:
            return {"total_memory_mb": 0}
        kb = sum(t.element_size() * t.nelement() for t in self.k_caches.values())
        vb = sum(t.element_size() * t.nelement() for t in self.v_caches.values())
        if self.use_block_storage:
            per_seq = math.ceil(self.max_seq_len / self.block_size)
            used = sum(math.ceil(n / self.block_size) for layer in self._lengths for n in layer)
            total = per_seq * self.max_batch_size * self.num_layers
        else:
            used = sum(n for layer in self._lengths for n in layer)
            total = self.max_batch_size * self.max_seq_len * self.num_layers
        return {"k_cache_memory_mb": kb / 2 ** 20, "v_cache_memory_mb": vb / 2 ** 20, "total_memory_mb": (kb + vb) / 2 ** 20,
                "memory_efficiency": used / total if total else 1.0}


class TransformerInferenceRunner(InferenceRunner):
    """reference :1306-1592 — the runner that owns the KV cache. With ``use_paged_attention`` (CUDA only) the model's
    attention layers are converted (``add_paged_attention_to_model``), a ``PagedKVCache`` is sized from the model
    (``kv_cache_num_gpu_blocks`` or the reference's free-memory rule) and generation requests (``max_new_tokens=``) run through
    ``generate_paged`` (K1 prefill, ``b200_kv_append`` + K2 per step, optionally one CUDA graph per step). Other calls are a
    plain forward. The reference's class is abstract (no ``_forward``, SURVEY.md F10)."""

    def __init__(self, model: nn.Module, device: str, precision: str = "fp16", is_encoder_decoder: bool = False,
                 use_kv_cache: bool = True, use_cuda_graph: bool = False, use_paged_attention: bool = True,
                 kv_cache_num_gpu_blocks: Optional[int] = None, kv_cache_block_size: int = 16,
                 kv_cache_dtype: Optional[torch.dtype] = None):
        super().__init__(model, device, precision)
        self.kv_cache_dtype = kv_cache_dtype   # None: the model's dtype; torch.float8_e4m3fn: the FP8 paged cache
        cuda = str(device).startswith("cuda")
        self.is_encoder_decoder = is_encoder_decoder
        self.use_kv_cache = use_kv_cache and cuda
        self.use_cuda_graph = use_cuda_graph and cuda
        self.use_paged_attention = use_paged_attention and self.use_kv_cache
        self.kv_cache_block_size = kv_cache_block_size
        self.kv_cache_num_gpu_blocks = kv_cache_num_gpu_blocks
        self.triton_available = True   # (the reference's flag for "the paged kernels exist")
        self.kv_cache: Optional[KVCache] = None
        self.paged_kv_cache: Optional[PagedKVCache] = None
        if self.use_kv_cache:
            if self.use_paged_attention:
                from .model_utils import add_paged_attention_to_model
                self.model = add_paged_attention_to_model(self.model)
            else:
                self.kv_cache = KVCache(max_batch_size=1, max_seq_len=2048)
            self._detect_model_params()
            self._initialize_kv_cache()

    def _detect_model_params(self) -> None:
        """reference :1373-1446 — layer / KV-head / head-dim counts, from the converted attention layers when there are
        any, else from the HuggingFace config."""
        adapters = [m for m in self.model.modules() if isinstance(m, _fa._HFAttentionAdapter)]
        if adapters:
            inner = adapters[0].inner
            self.num_layers, self.num_heads, self.head_dim = len(adapters), inner.num_kv_heads, inner.head_dim
            return
        cfg = getattr(self.model, "config", None)
        layers = getattr(cfg, "num_hidden_layers", getattr(cfg, "n_layer", None))
        heads = getattr(cfg, "num_attention_heads", getattr(cfg, "n_head", None))
        hidden = getattr(cfg, "hidden_size", getattr(cfg, "n_embd", None))
        if layers and heads and hidden:
            self.num_layers = layers
            self.num_heads = getattr(cfg, "num_key_value_heads", None) or heads
            self.head_dim = getattr(cfg, "head_dim", None) or hidden // heads

    def _calculate_num_gpu_blocks(self) -> int:
        """reference :1448-1500 — free memory minus 4x the 16-bit weights (activations) minus 10 % headroom, at most 80 % of
        the device, divided by the bytes of one block across all layers."""
        if not torch.cuda.is_available():
            return 0
        dev = torch.device(self.device if ":" in str(self.device) else "cuda")
        total = torch.cuda.get_device_properties(dev).total_memory
        weights = sum(p.numel() for p in self.model.parameters()) * 2
        avail = total - torch.cuda.memory_allocated(dev) - 4 * weights - 0.10 * total
        elem = 1 if self.kv_cache_dtype == torch.float8_e4m3fn else 2
        per_block = 2 * self.num_layers * self.kv_cache_block_size * self.num_heads * self.head_dim * elem
        if per_block == 0 or avail <= 0:
            return 0
        return int(min(avail, 0.8 * total) // per_block)

    def _initialize_kv_cache(self) -> None:
        if not self.use_kv_cache:
            return
        if not all(hasattr(self, a) for a in ("num_layers", "num_heads", "head_dim")):
            logging.warning("Model parameters not detected. Cannot initialize KV cache.")
            self.use_kv_cache = False
            return
        dtype = self.kv_cache_dtype or next(self.model.parameters()).dtype
        if self.use_paged_attention:
            if self.kv_cache_num_gpu_blocks is None:
                self.kv_cache_num_gpu_blocks = self._calculate_num_gpu_blocks()
            if self.kv_cache_num_gpu_blocks <= 0:
                raise MemoryError("Insufficient GPU memory for PagedKVCache.")   # (the reference falls back silently)
            self.paged_kv_cache = PagedKVCache(self.kv_cache_num_gpu_blocks, self.kv_cache_block_size, self.num_layers,
                                               self.num_heads, self.head_dim, dtype=dtype, device=str(self.device))
            if hasattr(self.model, "set_paged_kv_cache"):
                self.model.set_paged_kv_cache(self.paged_kv_cache)
        elif self.kv_cache is not None and not self.kv_cache.is_initialized:
            self.kv_cache.initialize(self.num_layers, self.num_heads, self.head_dim, dtype, str(self.device))

    def _forward(self, inputs: Any, **kwargs) -> Any:
        ids = inputs["input_ids"] if isinstance(inputs, dict) else inputs
        new_tokens = kwargs.pop("max_new_tokens", None)
        if new_tokens is not None and self.paged_kv_cache is not None:
            if set(kwargs) - {"do_sample"} or kwargs.get("do_sample"):
                raise NotImplementedError("the paged generation loop is greedy: unsupported arguments " + ", ".join(sorted(kwargs)))
            mask = inputs.get("attention_mask") if isinstance(inputs, dict) else None
            if mask is not None and bool((mask == 0).any()):
                raise NotImplementedError("the paged generation loop serves equal-length, unpadded prompts (attention_mask has zeros)")
            cache = self.paged_kv_cache
            try:
                return generate_paged(self.model, ids, new_tokens, cache=cache, block_size=self.kv_cache_block_size,
                                      use_cuda_graph=self.use_cuda_graph)
            finally:
                for sid in range(ids.shape[0]):   # the runner's cache outlives the request
                    cache.free_sequence(sid)
        if new_tokens is not None:
            kwargs["max_new_tokens"] = new_tokens
            return self.model.generate(**inputs, **kwargs) if isinstance(inputs, dict) else self.model.generate(inputs, **kwargs)
        return self.model(**inputs, **kwargs) if isinstance(inputs, dict) else self.model(inputs, **kwargs)

    def get_kv_cache_stats(self) -> Dict[str, Any]:
        """reference :1558-1592."""
        if not self.use_kv_cache:
            return {"kv_cache_enabled": False}
        if self.paged_kv_cache is not None:
            return {"kv_cache_enabled": True, "kv_cache_type": "PagedAttention", **self.paged_kv_cache.get_memory_usage()}
        if self.kv_cache is not None and self.kv_cache.is_initialized:
            return {"kv_cache_enabled": True, "kv_cache_type": "Standard", **self.kv_cache.get_memory_usage(),
                    "current_seq_lengths": self.kv_cache.current_seq_lengths}
        return {"kv_cache_enabled": False, "kv_cache_type": "None"}


# ------------------------------------------------------------------------------------------------------------------
# kernel fusion by module pattern (reference :26-281) and the attention conversion entry point (:283-375)
# ------------------------------------------------------------------------------------------------------------------
class FusionPattern:
    """reference :26-73 — a run of consecutive child modules (by type) and the function that replaces it."""

    def __init__(self, name: str, pattern: List[Union[type, Tuple[type, ...]]], fusion_fn: Callable[[List[nn.Module]], nn.Module],
                 description: Optional[str] = None):
        self.name, self.pattern, self.fusion_fn = name, list(pattern), fusion_fn
        self.description = description or "Fuses " + " + ".join(getattr(p, "__name__", str(p)) for p in self.pattern)

    def match(self, modules: Sequence[nn.Module]) -> bool:
        return len(modules) == len(self.pattern) and all(isinstance(m, t) for m, t in zip(modules, self.pattern))

    def fuse(self, modules: List[nn.Module]) -> nn.Module:
        return self.fusion_fn(modules)


class FusionRegistry:
    """reference :76-215 — scans every container for runs of children that match a registered pattern and swaps each run
    for the fused module (first child's slot; the other slots are removed, a ``Sequential`` is renumbered)."""

    def __init__(self):
        self.patterns: List[FusionPattern] = []

    def register_pattern(self, pattern: FusionPattern) -> None:
        self.patterns.append(pattern)

    def find_matching_pattern(self, modules: Sequence[nn.Module]) -> Optional[FusionPattern]:
        return next((p for p in self.patterns if p.match(modules)), None)

    def fuse_modules(self, model: nn.Module, inplace: bool = False) -> nn.Module:
        if not inplace:
            model = deepcopy(model)
        if not self.patterns:
            return model
        longest = max(len(p.pattern) for p in self.patterns)
        for parent in list(model.modules()):
            names = list(parent._modules)
            i = 0
            while i < len(names):
                hit = None
                for n in range(min(longest, len(names) - i), 1, -1):
                    run = [parent._modules[k] for k in names[i:i + n]]
                    pat = self.find_matching_pattern(run) if all(m is not None for m in run) else None
                    if pat is not None:
                        hit = (n, pat.fuse(run))
                        break
                if hit is None:
                    i += 1
                    continue
                n, fused = hit
                parent._modules[names[i]] = fused
                for k in names[i + 1:i + n]:
                    del parent._modules[k]
                names = names[:i + 1] + names[i + n:]
                i += 1
            if isinstance(parent, nn.Sequential) and list(parent._modules) != [str(j) for j in range(len(parent._modules))]:
                mods = list(parent._modules.values())
                parent._modules.clear()
                for j, m in enumerate(mods):
                    parent._modules[str(j)] = m
        return model


def _fuse_linear_act_linear(cls_name: str) -> Callable[[List[nn.Module]], nn.Module]:
    def fuse(modules: List[nn.Module]) -> nn.Module:
        from ..kernels.mlp import fused_mlp as _fm

        fc1, act, fc2 = modules
        if fc2.in_features != fc1.out_features:
            raise ValueError(f"cannot fuse Linear({fc1.in_features}->{fc1.out_features}) with Linear({fc2.in_features}->...)")
        if fc2.out_features != fc1.in_features:
            raise ValueError("the fused MLP maps hidden -> intermediate -> hidden; the two Linears do not")
        if isinstance(act, nn.GELU):   # erf GELU unless the module asks for the tanh form
            new = _fm.FusedMLPGeluTanh(fc1.in_features, fc1.out_features) if getattr(act, "approximate", "none") == "tanh" \
                else _fm.FusedMLP(fc1.in_features, fc1.out_features, _fm.FusedMLPConfig(activation_fn="gelu"))
        else:
            new = getattr(_fm, cls_name)(fc1.in_features, fc1.out_features)
        new = new.to(device=fc1.weight.device, dtype=fc1.weight.dtype)
        with torch.no_grad():
            for dst, src in ((new.fc1, fc1), (new.fc2, fc2)):
                dst.weight.copy_(src.weight)
                dst.bias.zero_() if src.bias is None else dst.bias.copy_(src.bias)
        return new
    return fuse


fusion_registry = FusionRegistry()
fusion_registry.register_pattern(FusionPattern("linear_gelu_linear", [nn.Linear, nn.GELU, nn.Linear], _fuse_linear_act_linear("FusedMLPGeluTanh"),
                                               "Fuses Linear + GELU + Linear into one FusedMLP (K3), weights copied"))
fusion_registry.register_pattern(FusionPattern("linear_relu_linear", [nn.Linear, nn.ReLU, nn.Linear], _fuse_linear_act_linear("FusedMLPReLU"),
                                               "Fuses Linear + ReLU + Linear into one FusedMLPReLU (K3), weights copied"))


def convert_to_flash_attention(model: nn.Module) -> nn.Module:
    """reference :283-375 — swap the model's attention layers for the K1 / K2 modules (``ModelConverter``, weights copied).
    Raises when nothing was converted (the reference returns the model untouched)."""
    dtype = next(model.parameters()).dtype
    prec = {torch.bfloat16: "bf16", torch.float16: "fp16"}.get(dtype, "bf16")
    converted = _fa.ModelConverter(_fa.FlashAttentionConfig(causal=True, precision=prec)).convert_model(model)
    if not any(isinstance(m, (_fa._HFAttentionAdapter, _fa.FlashAttentionLayer, _fa.FlashSelfAttention)) for m in converted.modules()):
        raise ValueError("convert_to_flash_attention: no convertible attention layer found in the model")
    return converted


# ------------------------------------------------------------------------------------------------------------------
# greedy generation over the paged cache
# ------------------------------------------------------------------------------------------------------------------
def _adapters(model: nn.Module) -> List[_fa._HFAttentionAdapter]:
    mods = [m for m in model.modules() if isinstance(m, _fa._HFAttentionAdapter)]
    if not mods:
        raise ValueError("generate_paged needs a model converted by kernels.attention.flash_attention.ModelConverter")
    return mods


def generate_paged(model: nn.Module, input_ids: torch.Tensor, max_new_tokens: int, cache: Optional[PagedKVCache] = None,
                   block_size: int = 16, use_cuda_graph: bool = False,
                   kv_cache_dtype: Optional[torch.dtype] = None) -> torch.Tensor:
    """Greedy generation with the paged KV cache: prefill runs K1 and scatters the prompt's K,V into blocks; every decode
    step appends the new token's K,V (``b200_kv_append``) and attends through the block tables (K2). Returns
    ``[B, S + max_new_tokens]`` token ids.

    ``use_cuda_graph=True`` captures one decode step (all layers: projections, KV append, K2, MLP, LM head, argmax) in a
    CUDA graph and replays it: block tables are reserved up front, lengths / positions / the token are advanced on the
    device, so a step has no host work besides the replay (the loop is launch-bound otherwise).

    ``kv_cache_dtype=torch.float8_e4m3fn`` allocates an FP8 cache (scales 1.0) when no ``cache`` is passed."""
    adapters = _adapters(model)
    first = adapters[0].inner
    B, S = input_ids.shape
    dev = input_ids.device
    compute = first.flash_attention._compute_dtype(next(model.parameters()).dtype)
    if kv_cache_dtype not in (None, compute, torch.float8_e4m3fn):
        raise ValueError(f"kv_cache_dtype must be None, {compute} or torch.float8_e4m3fn, got {kv_cache_dtype}")
    if cache is None:
        blocks = B * math.ceil((S + max_new_tokens) / block_size) + 1
        cache = PagedKVCache(blocks, block_size, len(adapters), first.num_kv_heads, first.head_dim,
                             dtype=kv_cache_dtype or compute, device=str(dev))
    elif kv_cache_dtype is not None and cache.dtype != kv_cache_dtype:
        raise ValueError(f"kv_cache_dtype {kv_cache_dtype} differs from the dtype of the cache passed ({cache.dtype})")
    seq_ids = list(range(B))
    for sid in seq_ids:
        cache.allocate_blocks_for_sequence(sid, S)
    out = input_ids
    try:
        with torch.no_grad():
            _fa.set_paged_context({"mode": "prefill", "cache": cache, "seq_ids": seq_ids})
            logits = model(input_ids, use_cache=False).logits
            nxt = logits[:, -1].argmax(-1, keepdim=True)
            out = torch.cat([out, nxt], dim=1)
            if use_cuda_graph and max_new_tokens > 1:
                return torch.cat([out, _decode_with_graph(model, cache, seq_ids, nxt, S, max_new_tokens - 1)], dim=1)
            for step in range(1, max_new_tokens):
                for sid in seq_ids:
                    cache.append_token(sid)
                bt, lens = cache.device_tables(seq_ids)
                _fa.set_paged_context({"mode": "decode", "cache": cache, "seq_ids": seq_ids, "block_tables": bt,
                                       "context_lengths": lens})
                pos = torch.full((B, 1), S + step - 1, dtype=torch.long, device=dev)
                logits = model(nxt, position_ids=pos, use_cache=False).logits
                nxt = logits[:, -1].argmax(-1, keepdim=True)
                out = torch.cat([out, nxt], dim=1)
    finally:
        _fa.set_paged_context(None)
    return out


def _decode_with_graph(model: nn.Module, cache: PagedKVCache, seq_ids: List[int], first_token: torch.Tensor, prompt_len: int,
                       steps: int, eager_steps: int = 2) -> torch.Tensor:
    """``steps`` greedy decode steps after the prefill; returns the generated ids ``[B, steps]``. The first
    ``eager_steps`` run eagerly (they also size the kernel workspaces), then one step is captured and replayed."""
    B = first_token.shape[0]
    dev = first_token.device
    total = prompt_len + steps + 1
    for sid in seq_ids:
        cache.reserve_blocks(sid, total)
    bt, lens = cache.device_tables(seq_ids)            # fixed block tables; lens = prompt length
    tok = first_token.clone()
    pos = torch.full((B, 1), prompt_len, dtype=torch.long, device=dev)
    out_buf = torch.zeros(B, steps, dtype=torch.long, device=dev)
    idx = torch.zeros(1, 1, dtype=torch.long, device=dev)
    _fa.set_paged_context({"mode": "decode", "cache": cache, "seq_ids": seq_ids, "block_tables": bt, "context_lengths": lens,
                           "max_context_len": total})

    def step():
        lens.add_(1)                                   # the token appended in this step counts (attention_kernels.py:862-866)
        logits = model(tok, position_ids=pos, use_cache=False).logits
        n = logits[:, -1].argmax(-1, keepdim=True)
        tok.copy_(n)
        pos.add_(1)
        out_buf.scatter_(1, idx.expand(B, 1), n)
        idx.add_(1)

    # The attention blocks of a converted model mask inside the kernels; HF's "eager" mask builder would still create a
    # dense additive mask per step (with a host scalar -> device copy, which a capture forbids). The "sdpa" mask interface
    # returns None for a single un-padded query token, so it is selected for the duration of the decode loop.
    configs = {id(m.config): m.config for m in model.modules() if hasattr(getattr(m, "config", None), "_attn_implementation")}
    saved_impl = {k: c._attn_implementation for k, c in configs.items()}
    for c in configs.values():
        c._attn_implementation = "sdpa"
    try:
        return _decode_with_graph_body(step, steps, eager_steps, dev, cache, seq_ids, out_buf)
    finally:
        for k, c in configs.items():
            c._attn_implementation = saved_impl[k]


#: timing of the last captured decode loop (device time): {"replay_steps", "replay_ms", "capture_s"}
LAST_DECODE_STATS: Dict[str, float] = {}


def _decode_with_graph_body(step, steps, eager_steps, dev, cache, seq_ids, out_buf):
    done = 0
    side = torch.cuda.Stream(dev)
    side.wait_stream(torch.cuda.current_stream(dev))
    with torch.cuda.stream(side):                      # warm-up on the stream the capture will use
        for _ in range(min(eager_steps, steps)):
            step()
            done += 1
    torch.cuda.current_stream(dev).wait_stream(side)
    if done < steps:
        t0 = time.perf_counter()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=side):
            step()
        capture_s = time.perf_counter() - t0
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps - done):
            graph.replay()
        e1.record()
        e1.synchronize()
        LAST_DECODE_STATS.update(replay_steps=steps - done, replay_ms=e0.elapsed_time(e1), capture_s=capture_s)
    for sid in seq_ids:                                # host bookkeeping of the lengths (blocks are already there)
        for _ in range(steps):
            cache.append_token(sid)
    return out_buf
