"""Generate golden input/output vectors by RUNNING THE REFERENCE (the original project) on CPU.

    B200_REFERENCE_DIR=<checkout of the reference> python tests/golden/make_golden.py   # writes tests/golden/*.pt

The reference is not part of this repository, so the vectors are committed. What is runnable in the reference
(SURVEY.md §0):
  * kernels/mlp/fused_mlp.py — FusedTransformerMLP / FusedMLP* forward (always the eager path, F5)
  * kernels/triton/mlp_kernels.py:759 pytorch_fused_mlp
  * kernels/triton/attention_kernels.py:1520-1591 — the PyTorch body of triton_ring_attention_forward, defined
    only when ``import triton`` fails (F8); we mask triton in sys.modules to reach it. Causal vectors use the
    finite -1e9 additive mask the reference's FA kernels use (flash_attention_kernels.py:253).
  * parallelism/sequence_parallel.py:480-517 SequenceParallelAttention._local_attention (eager softmax attention)
Everything is seeded; tensors are small (fp32) so every fixture file stays under 1 MB.
"""
from __future__ import annotations

import math
import os
import sys
import types

import torch

REF = os.environ.get("B200_REFERENCE_DIR", "")
OUT = os.path.dirname(os.path.abspath(__file__))


def mlp_vectors():
    from kernels.mlp import fused_mlp as fm
    from kernels.triton import mlp_kernels as mk

    out = {}
    torch.manual_seed(1234)
    h, i, B, S = 64, 192, 2, 12
    x = torch.randn(B, S, h)
    for act in ("gelu", "relu", "swiglu"):
        torch.manual_seed(100 + len(out))
        mod = fm.FusedTransformerMLP(h, i, activation_fn=act)
        mod.eval()
        for prm in mod.parameters():  # biases are zero-initialised in the reference; make them non-trivial
            if prm.dim() == 1:
                torch.nn.init.normal_(prm, std=0.1)
        with torch.no_grad():
            y = mod(x)
        sd = {k: v.clone() for k, v in mod.state_dict().items()}
        out[f"FusedTransformerMLP_{act}"] = {"x": x.clone(), "state_dict": sd, "y": y.clone(), "hidden": h,
                                              "intermediate": i, "activation_fn": act}
    # bare FusedMLP(activation_fn="gelu") = exact erf GELU (fused_mlp.py:162-163)
    torch.manual_seed(7)
    cfg = fm.FusedMLPConfig(activation_fn="gelu")
    mod = fm.FusedMLP(h, i, cfg)
    mod.eval()
    with torch.no_grad():
        y = mod(x)
    out["FusedMLP_gelu_erf"] = {"x": x.clone(), "state_dict": {k: v.clone() for k, v in mod.state_dict().items()},
                                "y": y.clone(), "hidden": h, "intermediate": i, "activation_fn": "gelu"}
    # functional form
    torch.manual_seed(8)
    w1, b1 = torch.randn(i, h) * 0.1, torch.randn(i) * 0.1
    w2, b2 = torch.randn(h, i) * 0.1, torch.randn(h) * 0.1
    wg, bg = torch.randn(i, h) * 0.1, torch.randn(i) * 0.1
    for act in ("gelu", "relu", "swiglu"):
        y = mk.pytorch_fused_mlp(x, w1, b1, w2, b2, act, wg if act == "swiglu" else None, bg if act == "swiglu" else None)
        out[f"pytorch_fused_mlp_{act}"] = {"x": x.clone(), "w1": w1, "b1": b1, "w2": w2, "b2": b2, "wg": wg, "bg": bg,
                                           "y": y.clone(), "activation": act}
    return out


def layernorm_vectors():
    from kernels.triton import layernorm_kernels as lk

    torch.manual_seed(99)
    x, r = torch.randn(2, 7, 96), torch.randn(2, 7, 96)
    w, b = torch.randn(96), torch.randn(96)
    return {
        "pytorch_layernorm": {"x": x, "w": w, "b": b, "eps": 1e-5, "y": lk.pytorch_layernorm(x, w, b, 1e-5)},
        "pytorch_layernorm_residual": {"x": x, "r": r, "w": w, "b": b, "eps": 1e-5, "alpha": 0.5,
                                       "y": lk.pytorch_layernorm(x, w, b, 1e-5, r, 0.5)},
        "pytorch_layernorm_nobias": {"x": x, "w": w, "eps": 1e-6, "y": lk.pytorch_layernorm(x, w, None, 1e-6)},
    }


def attention_vectors():
    # reach the PyTorch fallback of triton_ring_attention_forward: it is defined only when triton is missing
    saved = {k: sys.modules.get(k) for k in ("triton", "triton.language")}
    sys.modules["triton"] = None
    sys.modules["triton.language"] = None
    for k in list(sys.modules):
        if k.startswith("kernels.triton.attention_kernels"):
            del sys.modules[k]
    try:
        from kernels.triton import attention_kernels as ak
        assert not ak.TRITON_AVAILABLE
        out = {}
        torch.manual_seed(4321)
        B, H, S, D = 2, 4, 200, 64  # 200 keys -> two chunks of 128 in the reference loop, ragged tail
        q, k, v = torch.randn(B, H, S, D), torch.randn(B, H, S, D), torch.randn(B, H, S, D)
        y = ak.triton_ring_attention_forward(q, k, v, None)  # [B, S, H*D]
        out["ring_fallback_noncausal"] = {"q": q, "k": k, "v": v, "y": y.clone()}
        mask = torch.triu(torch.full((S, S), -1e9), diagonal=1).view(1, 1, S, S)
        y = ak.triton_ring_attention_forward(q, k, v, mask)
        out["ring_fallback_causal_finite_mask"] = {"q": q, "k": k, "v": v, "y": y.clone()}
        # cross lengths (Sq != Sk)
        q2 = torch.randn(B, H, 70, D)
        y = ak.triton_ring_attention_forward(q2, k, v, None)
        out["ring_fallback_cross"] = {"q": q2, "k": k, "v": v, "y": y.clone()}
    finally:
        for k_, v_ in saved.items():
            if v_ is None:
                sys.modules.pop(k_, None)
            else:
                sys.modules[k_] = v_
    # eager softmax attention of the sequence-parallel module (additive mask form)
    from parallelism import sequence_parallel as sp
    stub = types.SimpleNamespace(head_dim=D, dropout=torch.nn.Identity())
    y = sp.SequenceParallelAttention._local_attention(stub, q, k, v, None)  # [B,H,S,D]
    out["sp_local_attention"] = {"q": q, "k": k, "v": v, "y": y.clone()}
    pad = torch.zeros(B, 1, 1, S)
    pad[1, :, :, 150:] = -1e9  # right padding of batch 1
    y = sp.SequenceParallelAttention._local_attention(stub, q, k, v, pad)
    out["sp_local_attention_padmask"] = {"q": q, "k": k, "v": v, "mask": pad, "kv_lens": torch.tensor([S, 150]),
                                         "y": y.clone()}
    return keep_heads(out, ATTN_KEPT_HEADS)


# Attention is independent per (batch, head): the vectors are generated at H=4 (so the seeded inputs stay the ones first
# generated) and only these heads are stored, which keeps the file under 1 MB.
ATTN_KEPT_HEADS = [0]


def keep_heads(vecs, heads):
    """The attention vectors restricted to ``heads``: q/k/v/y [B,H,S,D] (ring fallback y [B,S,H*D]) sliced on the head
    axis into compact storage; tensors shared between entries stay shared so that torch.save writes them once."""
    idx = torch.tensor(heads)
    sliced = {}

    def head_slice(t):
        if id(t) not in sliced:
            sliced[id(t)] = t.index_select(1, idx).contiguous()
        return sliced[id(t)]

    out = {}
    for name, d in vecs.items():
        e = dict(d)
        for n in ("q", "k", "v"):
            e[n] = head_slice(d[n])
        y = d["y"]
        if name.startswith("ring_fallback"):  # [B, S, H*D] -> [B, S, len(heads)*D]
            B, S, _ = y.shape
            D = d["q"].shape[-1]
            e["y"] = y.view(B, S, -1, D).index_select(2, idx).reshape(B, S, len(heads) * D).contiguous()
        else:
            e["y"] = y.index_select(1, idx).contiguous()
        out[name] = e
    return out


def main():
    if not os.path.isdir(REF):
        raise SystemExit(f"B200_REFERENCE_DIR={REF!r} is not a directory: golden vectors can only be regenerated from a "
                         "checkout of the reference")
    sys.path.insert(0, REF)
    torch.set_num_threads(1)
    torch.use_deterministic_algorithms(True)
    mlp = mlp_vectors()
    attn = attention_vectors()
    torch.save(mlp, os.path.join(OUT, "mlp_reference_vectors.pt"))
    torch.save(attn, os.path.join(OUT, "attention_reference_vectors.pt"))
    ln = layernorm_vectors()
    torch.save(ln, os.path.join(OUT, "layernorm_reference_vectors.pt"))
    for name, d in {**mlp, **attn, **ln}.items():
        print(f"{name}: y{tuple(d['y'].shape)} |y|max={d['y'].abs().max():.4f}")


if __name__ == "__main__":
    main()
