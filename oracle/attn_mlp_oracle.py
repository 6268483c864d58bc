"""CPU restatement (fp32, torch on CPU) of the reference's attention + FusedMLP arithmetic.

THIS IS TEST INFRASTRUCTURE. Only ``tests/``, ``__graft_entry__.smoke()`` and the ``cpu_baseline`` /
``--impl reference`` legs of ``bench.py`` may import it, and only as the checker or the timed CPU baseline.
Nothing under ``ml_inference_optimizer_b200/`` imports it; the product path has no CPU fallback.

Parity pinning. The reference ships no golden vectors (SURVEY.md §4, F12) and its attention modules cannot be
imported (F1-F3), so the oracle is pinned against OUTPUTS OF THE REFERENCE ITSELF RUN IN THE AUTHORING CONTAINER,
committed under ``tests/golden/`` by ``tests/golden/make_golden.py``:
  * kernels/mlp/fused_mlp.py ``FusedTransformerMLP`` / ``FusedMLPSwiGLU`` / ``FusedMLPGeluTanh`` / ``FusedMLPReLU``
    forward (the reference's only runnable MLP path, fused_mlp.py:159-178, :223-237, :262-275);
  * kernels/triton/attention_kernels.py:1520-1591, the PyTorch body of ``triton_ring_attention_forward`` — the one
    correct online-softmax implementation in the reference (F8) — for non-causal attention and the LSE-merge
    algebra;
  * parallelism/tensor_parallel.py:569-586 / parallelism/sequence_parallel.py:498-517 eager softmax attention.
Causal masking, GQA and decode follow the reference's stated semantics (citations on each function); they have
no runnable reference implementation, which DESIGN.md records as "pinned by construction, not by fixture".
"""
from __future__ import annotations

import math
from typing import Optional, Tuple

import torch

__all__ = [
    "attention_ref", "decode_attention_ref", "paged_gather", "kv_append_ref", "lse_merge_ref", "mlp_ref",
    "linear_act_ref", "layernorm_ref", "gelu_tanh", "rel_err_percent", "max_abs_err", "tile_errors", "ring_attention_ref",
    "tp_mlp_ref",
]


# --------------------------------------------------------------------------------------------------------------
# error metrics — benchmarks/metrics.py:211-238 (mean relative error, %) and :241-262 (max abs error)
# --------------------------------------------------------------------------------------------------------------
def rel_err_percent(a: torch.Tensor, b: torch.Tensor) -> float:
    a, b = a.double(), b.double()
    return float(((a - b).abs() / (b.abs() + 1e-8)).mean() * 100.0)


def max_abs_err(a: torch.Tensor, b: torch.Tensor) -> float:
    return float((a.double() - b.double()).abs().max())


def _tiles(t: torch.Tensor, tiling: str, hkv: Optional[int], tile: int) -> torch.Tensor:
    """``t`` regrouped as [num_tiles, elements]; ragged edges are zero-padded (zeros add nothing to either sum or max)."""
    if tiling == "attn":                                   # [B,S,H,D]: one tile per (b, h, `tile` query rows)
        B, S, H, D = t.shape
        t = torch.nn.functional.pad(t, (0, 0, 0, 0, 0, (-S) % tile))
        return t.view(B, -1, tile, H, D).permute(0, 3, 1, 2, 4).reshape(-1, tile * D)
    if tiling == "decode":                                 # [B,Hq,D]: one tile per (b, kv head) = the G query heads it serves
        B, Hq, D = t.shape
        return t.reshape(B * hkv, (Hq // hkv) * D)
    if tiling == "2d":                                     # [T,N]: one tile per `tile` x `tile` block
        t = t.reshape(-1, t.shape[-1])
        T, N = t.shape
        t = torch.nn.functional.pad(t, (0, (-N) % tile, 0, (-T) % tile))
        return t.view(t.shape[0] // tile, tile, t.shape[1] // tile, tile).permute(0, 2, 1, 3).reshape(-1, tile * tile)
    raise ValueError(f"unknown tiling {tiling!r}")


def tile_errors(got: torch.Tensor, ref: torch.Tensor, tiling: str, hkv: Optional[int] = None, tile: int = 128) -> dict:
    """Error of ``got`` against the fp32 / fp64 ``ref``, tile by tile, so that an error confined to one head, one row block
    or one GEMM tile is not averaged away by the rest of the tensor.

    ``tiling``: ``"attn"`` ([B,S,H,D], one tile per (batch, head, 128 query rows)), ``"decode"`` ([B,Hq,D], one tile per
    (batch, kv head); ``hkv`` = number of KV heads) or ``"2d"`` (a [T,N] output, one tile per 128 x 128 block).
    Returns, over the tiles whose reference is not all zero, ``mean_rel`` = mean|err| / mean|ref| and ``max_rel`` =
    max|err| / max|ref| (fp64 tensors, one value per tile), and ``empty_max`` = max|got| over the tiles whose reference is
    all zero (they carry no relative error, so a value written there is reported as it is)."""
    got, ref = got.double().cpu(), ref.double().cpu()
    if got.shape != ref.shape:
        raise ValueError(f"shapes differ: {tuple(got.shape)} vs {tuple(ref.shape)}")
    err = _tiles((got - ref).abs(), tiling, hkv, tile)
    mag = _tiles(ref.abs(), tiling, hkv, tile)
    live = mag.amax(dim=1) > 0
    dead = _tiles(got.abs(), tiling, hkv, tile)[~live]
    return {
        "mean_rel": err[live].sum(dim=1) / mag[live].sum(dim=1),
        "max_rel": err[live].amax(dim=1) / mag[live].amax(dim=1),
        "empty_max": float(dead.max()) if dead.numel() else 0.0,
    }


# --------------------------------------------------------------------------------------------------------------
# attention
# --------------------------------------------------------------------------------------------------------------
def attention_ref(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, causal: bool = False,
                  softmax_scale: Optional[float] = None, causal_offset: int = 0,
                  kv_lens: Optional[torch.Tensor] = None) -> Tuple[torch.Tensor, torch.Tensor]:
    """Exact softmax attention in fp32. q [B,Sq,Hq,D], k/v [B,Sk,Hkv,D] -> (O [B,Sq,Hq,D], LSE [B,Hq,Sq]).

    Follows the reference's own correctness closures ``standard_attention``
    (kernels/attention/flash_attention.py:1216-1229, kernels/triton/flash_attention_kernels.py:1913-1918):
    scores = einsum(q,k) * scale; causal = strict upper triangle masked (``triu(diagonal=1)``, :1221-1225);
    softmax over keys; einsum with v. Scale default 1/sqrt(D) (flash_attention.py:247). GQA by
    ``repeat_interleave`` of KV heads: q head h uses kv head h // (Hq/Hkv) (flash_attention.py:894-903).
    Fully masked rows give O = 0 and LSE = -inf (SURVEY.md §8c item 4). ``causal_offset`` shifts the diagonal:
    key j is visible to query i iff j <= i + causal_offset (ring steps / chunked prefill).
    """
    q, k, v = q.float(), k.float(), v.float()
    B, Sq, Hq, D = q.shape
    _, Sk, Hkv, _ = k.shape
    g = Hq // Hkv
    if g > 1:
        k = k.repeat_interleave(g, dim=2)
        v = v.repeat_interleave(g, dim=2)
    scale = softmax_scale if softmax_scale is not None else 1.0 / math.sqrt(D)
    scores = torch.einsum("bqhd,bkhd->bhqk", q, k) * scale
    neg = torch.finfo(torch.float32).min
    mask = torch.zeros(B, 1, Sq, Sk, dtype=torch.bool)
    if causal:
        qi = torch.arange(Sq).view(Sq, 1)
        kj = torch.arange(Sk).view(1, Sk)
        mask = mask | (kj > qi + causal_offset).view(1, 1, Sq, Sk)
    if kv_lens is not None:
        kj = torch.arange(Sk).view(1, 1, 1, Sk)
        mask = mask | (kj >= kv_lens.view(B, 1, 1, 1).long())
    scores = scores.masked_fill(mask, float("-inf"))
    lse = torch.logsumexp(scores, dim=-1)  # -inf where every key is masked
    probs = torch.exp(scores - torch.where(torch.isinf(lse), torch.zeros_like(lse), lse).unsqueeze(-1))
    probs = torch.where(mask.expand_as(probs), torch.zeros_like(probs), probs)
    out = torch.einsum("bhqk,bkhd->bqhd", probs, v)
    del neg
    return out, lse


def paged_gather(cache: torch.Tensor, block_table: torch.Tensor, layer_idx: int, length: int) -> torch.Tensor:
    """Gather ``length`` tokens of one sequence from a paged cache [num_blocks, L, block_size, Hkv, D]
    (layout: baseline/inference.py:1077-1084; addressing: kernels/triton/attention_kernels.py:736-751)."""
    block_size = cache.shape[2]
    rows = []
    for t in range(length):
        blk = int(block_table[t // block_size])
        rows.append(cache[blk, layer_idx, t % block_size])
    if not rows:
        return cache.new_zeros((0,) + tuple(cache.shape[3:]))
    return torch.stack(rows, dim=0)


def decode_attention_ref(q: torch.Tensor, k_cache: torch.Tensor, v_cache: torch.Tensor, context_lens: torch.Tensor,
                         softmax_scale: Optional[float] = None, block_tables: Optional[torch.Tensor] = None,
                         layer_idx: int = 0) -> Tuple[torch.Tensor, torch.Tensor]:
    """Single-token attention vs a KV cache, fp32. q [B,Hq,D] -> (O [B,Hq,D], LSE [B,Hq]).

    Semantics of _paged_attention_fwd_kernel (kernels/triton/attention_kernels.py:628-808): no causal mask, key
    position < context_len only (:771-777); context_len counts the token just appended (:862-866). GQA by
    head-group as in ``attention_ref`` (the reference's paged kernel ignores GQA, Appendix B — fixed here).
    """
    B, Hq, D = q.shape
    outs, lses = [], []
    for b in range(B):
        n = int(context_lens[b])
        if block_tables is not None:
            kb = paged_gather(k_cache, block_tables[b], layer_idx, n)
            vb = paged_gather(v_cache, block_tables[b], layer_idx, n)
        else:
            kb, vb = k_cache[b, :n], v_cache[b, :n]
        if n == 0:
            outs.append(torch.zeros(Hq, D))
            lses.append(torch.full((Hq,), float("-inf")))
            continue
        o, l = attention_ref(q[b].view(1, 1, Hq, D), kb.unsqueeze(0), vb.unsqueeze(0), causal=False,
                             softmax_scale=softmax_scale)
        outs.append(o.view(Hq, D))
        lses.append(l.view(Hq))
    return torch.stack(outs), torch.stack(lses)


def paged_prefill_attention_ref(q: torch.Tensor, k_cache: torch.Tensor, v_cache: torch.Tensor, block_tables: torch.Tensor,
                                context_lens: torch.Tensor, layer_idx: int = 0, causal: bool = True,
                                softmax_scale: Optional[float] = None) -> Tuple[torch.Tensor, torch.Tensor]:
    """Short-q attention vs the paged cache, fp32: q [B,Sq,Hq,D] are the last Sq tokens of each sequence (their K/V are in
    the cache), keys = the ``context_lens[b]`` gathered tokens (addressing of _paged_attention_fwd_kernel,
    kernels/triton/attention_kernels.py:722-760; q_len > 1 is its BLOCK_SIZE_M = 64 case, :1251). ``causal``: query i sees
    keys <= context_len - Sq + i — the mask the reference kernel carries commented out (:774-777); ``causal=False`` is the
    kernel as written (every query sees all context_len keys). Returns (O [B,Sq,Hq,D], LSE [B,Hq,Sq])."""
    B, Sq, Hq, D = q.shape
    outs, lses = [], []
    for b in range(B):
        n = int(context_lens[b])
        kb = paged_gather(k_cache, block_tables[b], layer_idx, n)
        vb = paged_gather(v_cache, block_tables[b], layer_idx, n)
        if n == 0:
            outs.append(torch.zeros(Sq, Hq, D))
            lses.append(torch.full((Hq, Sq), float("-inf")))
            continue
        o, l = attention_ref(q[b:b + 1], kb.unsqueeze(0), vb.unsqueeze(0), causal=causal, softmax_scale=softmax_scale,
                             causal_offset=n - Sq)
        outs.append(o[0])
        lses.append(l[0])
    return torch.stack(outs), torch.stack(lses)


def kv_append_ref(key: torch.Tensor, value: torch.Tensor, k_cache: torch.Tensor, v_cache: torch.Tensor,
                  context_lens: torch.Tensor, block_tables: Optional[torch.Tensor] = None, layer_idx: int = 0) -> None:
    """In place: store the new token's K,V [B,Hkv,D] at position context_len-1
    (_reshape_and_cache_kernel, kernels/triton/attention_kernels.py:811-905, position rule :862-866)."""
    B = key.shape[0]
    for b in range(B):
        pos = int(context_lens[b]) - 1
        if pos < 0:
            continue
        if block_tables is not None:
            bs = k_cache.shape[2]
            blk = int(block_tables[b, pos // bs])
            k_cache[blk, layer_idx, pos % bs] = key[b]
            v_cache[blk, layer_idx, pos % bs] = value[b]
        else:
            k_cache[b, pos] = key[b]
            v_cache[b, pos] = value[b]


def lse_merge_ref(o_a: torch.Tensor, lse_a: torch.Tensor, o_b: torch.Tensor, lse_b: torch.Tensor):
    """Merge two partial attention results over disjoint key sets (o [B,Sq,Hq,D], lse [B,Hq,Sq]).

    The running (m, l, acc) update of kernels/triton/attention_kernels.py:1567-1585 written in LSE form:
    lse = logaddexp(lse_a, lse_b); o = o_a e^{lse_a-lse} + o_b e^{lse_b-lse}."""
    o_a, o_b, lse_a, lse_b = o_a.float(), o_b.float(), lse_a.float(), lse_b.float()
    lse = torch.logaddexp(lse_a, lse_b)
    safe = torch.where(torch.isinf(lse) & (lse < 0), torch.zeros_like(lse), lse)
    wa = torch.exp(lse_a - safe).transpose(1, 2).unsqueeze(-1)
    wb = torch.exp(lse_b - safe).transpose(1, 2).unsqueeze(-1)
    return o_a * wa + o_b * wb, lse


def ring_attention_ref(q_chunks, k_chunks, v_chunks, causal: bool, positions, softmax_scale=None):
    """Serial emulation of exact ring attention. ``q_chunks[r]`` etc. are rank r's [B,S_r,H,D] shards and
    ``positions[r]`` the global token index of each of its rows (LongTensor [S_r]); every rank's queries visit
    every rank's keys (parallelism/sequence_parallel.py:555-580 loop) with the merge of ``lse_merge_ref``.
    Returns the per-rank outputs. Used to check the distributed driver's bookkeeping on CPU."""
    n = len(q_chunks)
    outs = []
    for r in range(n):
        q = q_chunks[r].float()
        B, Sq, H, D = q.shape
        o_acc = torch.zeros(B, Sq, H, D)
        lse_acc = torch.full((B, H, Sq), float("-inf"))
        for step in range(n):
            src = (r - step) % n
            k, v = k_chunks[src].float(), v_chunks[src].float()
            scale = softmax_scale if softmax_scale is not None else 1.0 / math.sqrt(D)
            kk = k.repeat_interleave(H // k.shape[2], dim=2)
            vv = v.repeat_interleave(H // v.shape[2], dim=2)
            scores = torch.einsum("bqhd,bkhd->bhqk", q, kk) * scale
            if causal:
                vis = positions[src].view(1, -1) <= positions[r].view(-1, 1)
                scores = scores.masked_fill(~vis.view(1, 1, Sq, -1), float("-inf"))
            lse = torch.logsumexp(scores, dim=-1)
            safe = torch.where(torch.isinf(lse), torch.zeros_like(lse), lse)
            probs = torch.exp(scores - safe.unsqueeze(-1))
            probs = torch.where(torch.isinf(scores) & (scores < 0), torch.zeros_like(probs), probs)
            o = torch.einsum("bhqk,bkhd->bqhd", probs, vv)
            o_acc, lse_acc = lse_merge_ref(o_acc, lse_acc, o, lse)
        outs.append(o_acc)
    return outs


# --------------------------------------------------------------------------------------------------------------
# MLP
# --------------------------------------------------------------------------------------------------------------
def gelu_tanh(x: torch.Tensor) -> torch.Tensor:
    """0.5 x (1 + tanh(sqrt(2/pi) (x + 0.044715 x^3))) — kernels/mlp/fused_mlp.py:223-237,
    kernels/triton/mlp_kernels.py:144-161 (== HF ``gelu_new``)."""
    return 0.5 * x * (1.0 + torch.tanh(math.sqrt(2.0 / math.pi) * (x + 0.044715 * x.pow(3))))


def _act(name: str, x: torch.Tensor) -> torch.Tensor:
    if name in ("gelu_tanh", "gelu_new"):
        return gelu_tanh(x)
    if name in ("gelu", "gelu_erf"):
        return torch.nn.functional.gelu(x)  # exact erf GELU: fused_mlp.py:162-163, mlp_kernels.py:783
    if name == "relu":
        return torch.relu(x)  # fused_mlp.py:299-315
    if name in (None, "none"):
        return x
    raise ValueError(f"unknown activation {name}")


def linear_act_ref(x, w, b=None, activation=None, w_gate=None, b_gate=None) -> torch.Tensor:
    x = x.float()
    up = torch.nn.functional.linear(x, w.float(), None if b is None else b.float())
    if activation == "swiglu":
        gate = torch.nn.functional.linear(x, w_gate.float(), None if b_gate is None else b_gate.float())
        return torch.nn.functional.silu(gate) * up
    return _act(activation, up)


def mlp_ref(x, w_up, b_up, w_down, b_down, activation: str = "gelu_tanh", w_gate=None, b_gate=None) -> torch.Tensor:
    """fp32 FusedMLP: ``fc2(act(fc1 x))``; SwiGLU: ``fc2(silu(fc1_gate x) * fc1 x)``
    (kernels/mlp/fused_mlp.py:159-178, :262-275; kernels/triton/mlp_kernels.py:759-803)."""
    h = linear_act_ref(x, w_up, b_up, activation, w_gate, b_gate)
    return torch.nn.functional.linear(h, w_down.float(), None if b_down is None else b_down.float())


def layernorm_ref(x, weight, bias=None, eps: float = 1e-5, residual=None, residual_alpha: float = 1.0) -> torch.Tensor:
    """fp32 LayerNorm(x + alpha * residual) — the arithmetic of ``pytorch_layernorm``
    (kernels/triton/layernorm_kernels.py:279-311): mean, biased variance as mean((x-u)^2), eps inside the sqrt."""
    x = x.float()
    if residual is not None:
        x = x + residual_alpha * residual.float()
    u = x.mean(dim=-1, keepdim=True)
    s = (x - u).pow(2).mean(dim=-1, keepdim=True)
    x = (x - u) / torch.sqrt(s + eps)
    return weight.float() * x + (bias.float() if bias is not None else 0.0)


def tp_mlp_ref(x, w_up, b_up, w_down, b_down, activation, tp: int, w_gate=None, b_gate=None, return_partial_abs_sum: bool = False):
    """Column/row tensor-parallel MLP emulated serially: rank r holds rows [r*i/tp, (r+1)*i/tp) of W_up / W_gate
    and the matching columns of W_down (parallelism/tensor_parallel.py:130-135, :249-254); partial outputs are
    summed (the all-reduce, :302) and the down bias is added once after the reduction (:304-308).

    ``return_partial_abs_sum``: also return max over elements of sum_r |partial_r| — the quantity that bounds what
    rounding every rank's partial output to 16 bits before the all-reduce (as the reference does: the partials are in the
    activation dtype) can cost: at most 2^-9 of it for bf16."""
    i = w_up.shape[0]
    assert i % tp == 0
    s = i // tp
    total, abs_sum = None, None
    for r in range(tp):
        sl = slice(r * s, (r + 1) * s)
        h = linear_act_ref(x, w_up[sl], None if b_up is None else b_up[sl], activation,
                           None if w_gate is None else w_gate[sl], None if b_gate is None else b_gate[sl])
        part = torch.nn.functional.linear(h, w_down[:, sl].float())
        total = part if total is None else total + part
        abs_sum = part.abs() if abs_sum is None else abs_sum + part.abs()
    if b_down is not None:
        total = total + b_down.float()
    if return_partial_abs_sum:
        return total, abs_sum.max().item()
    return total


def tp_mlp_tolerance(ref: torch.Tensor, partial_abs_sum: float, tp: int, multicast: bool = True) -> float:
    """Max-abs bound for the tensor-parallel MLP in bf16, term by term (no factor fitted to the rank count):
      2e-2 * max(1, |ref|max / 4)   the single-GPU bound (GEMM arithmetic + one bf16 rounding of the result)
      2^-9 * max sum_r |partial_r|  every rank rounds its partial output to bf16 before the reduction (tp > 1)
      2^-8 * |ref|max               the NVSwitch's fp32 -> bf16 conversion of the reduced value is not round-to-nearest:
                                    up to one ulp instead of half (measured, tests/symm_probe.py)"""
    m = ref.abs().max().item()
    tol = 2e-2 * max(1.0, m / 4)
    if tp > 1:
        tol += 2.0 ** -9 * partial_abs_sum
        if multicast:
            tol += 2.0 ** -8 * m
    return tol
