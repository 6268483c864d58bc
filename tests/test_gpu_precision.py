"""fp16 is the default compute type of the modules (FlashAttentionConfig / FusedMLPConfig precision="fp16"), so every kernel
is built for __half as well as __nv_bfloat16. This file pins what the parity tests alone would not:

  (a) on inputs that are exact in both formats, the fp16 build's error is well below the bf16 build's — a 16-bit rounding
      that goes through bf16 on the fp16 path (P, the MLP intermediate, an output pack) shows up here;
  (b) the dispatch matrix: which kernel each shape / knob launches, in both dtypes, checked against the oracle;
  (c) non-default softmax scales (folded into scale_log2 by K1 and K2);
  (d) fp16 operations that must be byte-exact (kv_append, cast_out) and lse_merge with an fp16 block;
  (e) the modules with their default (fp16) configuration;
  (f) CPU: the tile-local checker accepts an emulated correct kernel and rejects emulated defects;
  (g) CPU: every __global__ instantiation in the built library is listed below with the test that launches it.

GPU tests are marked one by one; (f) and (g) run without a GPU.
"""
import math
import os
import re
import shutil
import subprocess

import pytest
import torch

from oracle import attn_mlp_oracle as orc
from test_gpu_parity import BF16, DTYPES, FP16, check_lse, check_out, make_mlp, rand_qkv

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
gpu = pytest.mark.gpu
DT_IDS = {BF16: "bf16", FP16: "fp16"}
# fp16 keeps 3 more mantissa bits than bf16: a kernel that rounds only to fp16 has ~1/8 of the bf16 error on the same
# inputs (0.12-0.13 in a CPU emulation of the kernels' rounding); one 16-bit step that goes through bf16 gives ~0.7.
# Measured on a B200 (1000 W): 0.125-0.129 on every case, gelu_tanh included (its tanh.approx.f32 error stays below the
# fp16 rounding of the intermediate, so the fp16 epilogue keeps the fast tanh).
FP16_OVER_BF16 = 0.35


@pytest.fixture(scope="module")
def ops(built_lib):
    assert torch.cuda.is_available(), "gpu tests need CUDA"
    from ml_inference_optimizer_b200 import ops as _ops

    assert _ops.arch_ok(), "gpu tests need an sm_100 device"
    return _ops


def exact_in_both(*shape, scale=1.0, seed=0, device="cuda"):
    """bf16 values that fp16 represents exactly (no magnitude below fp16's normal range): the same numbers in both types."""
    g = torch.Generator(device=device).manual_seed(seed)
    x = (torch.randn(*shape, device=device, generator=g) * scale).to(BF16)
    x[x.abs() < 2.0 ** -14] = 0
    assert torch.equal(x.to(FP16).float(), x.float())
    return x


def mean_abs_err(got, ref):
    return (got.double().cpu() - ref.double().cpu()).abs().mean().item()


# ------------------------------------------------------------------------------------------------- (a) fp16 vs bf16
def _attn_case(ops, dt, pair, monkeypatch):
    monkeypatch.setenv("B200_FA_PAIR", "1" if pair else "0")
    q, k, v = (exact_in_both(1, 640, 4, 128, seed=s) for s in (1, 2, 3))
    k, v = k[:, :, :2], v[:, :, :2]
    o = ops.flash_attn_fwd(q.to(dt), k.to(dt), v.to(dt), causal=True)
    assert ops.last_kernel() == ("fa_fwd_pair_kernel" if pair else "fa_fwd_kernel")
    return o, orc.attention_ref(q.cpu(), k.cpu(), v.cpu(), causal=True)[0]


def _decode_case(ops, dt, G, monkeypatch):
    B, Hkv, S = 3, 2, 700
    q, kc, vc = exact_in_both(B, Hkv * G, 128, seed=4), exact_in_both(B, S, Hkv, 128, seed=5), exact_in_both(B, S, Hkv, 128, seed=6)
    lens = torch.tensor([700, 333, 64], device="cuda", dtype=torch.int32)
    o = ops.decode_attention(q.to(dt), kc.to(dt), vc.to(dt), lens, num_splits=1)
    assert ops.last_kernel() == ("decode_kernel" if G <= 2 else "decode_gqa_mma_kernel")
    return o, orc.decode_attention_ref(q.cpu(), kc.cpu(), vc.cpu(), lens.cpu())[0]


MLP_PATHS = {   # GEMM path -> (T, environment)
    "gemm_act": (300, {"B200_GEMM_K_SPLITS": "1"}),
    "split_k": (300, {"B200_GEMM_K_SPLITS": "5"}),
    "pair": (1024, {"B200_GEMM_K_SPLITS": "1", "B200_MLP_FUSED": "0"}),
    "fused": (1024, {"B200_MLP_FUSED": "1"}),
}


def _mlp_case(ops, dt, act, path, monkeypatch):
    T, env = MLP_PATHS[path]
    for key, val in env.items():
        monkeypatch.setenv(key, val)
    h, i = 512, 1032
    x, wu, wd = exact_in_both(T, h, seed=7), exact_in_both(i, h, scale=0.05, seed=8), exact_in_both(h, i, scale=0.05, seed=9)
    bu, bd = exact_in_both(i, scale=0.1, seed=10), exact_in_both(h, scale=0.1, seed=11)
    wg = exact_in_both(i, h, scale=0.05, seed=12) if act == "swiglu" else None
    bg = exact_in_both(i, scale=0.1, seed=13) if act == "swiglu" else None
    c = lambda t, to: None if t is None else t.to(to)
    y = ops.fused_mlp(x.to(dt), c(wu, dt), c(bu, dt), c(wd, dt), c(bd, dt), act, c(wg, dt), c(bg, dt))
    name = ops.last_gemm_kernel()
    assert name.startswith("fused_mlp_pair_kernel" if path == "fused" else "gemm_act_pair_kernel<NONE" if path == "pair"
                           else "gemm_act_kernel<NONE>"), name
    cpu = lambda t: c(t, "cpu")
    return y, orc.mlp_ref(cpu(x), cpu(wu), cpu(bu), cpu(wd), cpu(bd), act, cpu(wg), cpu(bg))


def _ln_case(ops, dt, cols, monkeypatch):
    rows = 700
    x, r = exact_in_both(rows, cols, scale=2.0, seed=14), exact_in_both(rows, cols, seed=15)
    w, b = exact_in_both(cols, seed=16), exact_in_both(cols, seed=17)
    y = ops.layernorm(x.to(dt), w.to(dt), b.to(dt), 1e-5, r.to(dt), 0.5)
    return y, orc.layernorm_ref(x.cpu(), w.cpu(), b.cpu(), 1e-5, r.cpu(), 0.5)


RATIO_CASES = (["attn-default", "attn-pair", "decode-mha", "decode-mma", "layernorm-warp", "layernorm-cta"]
               + [f"mlp-{a}-{p}" for a in ("gelu_tanh", "gelu", "relu", "swiglu") for p in MLP_PATHS])


@gpu
@pytest.mark.parametrize("case", RATIO_CASES)
def test_fp16_error_well_below_bf16_error(ops, monkeypatch, case):
    """Same inputs in both formats: mean|err_fp16| <= 0.35 mean|err_bf16| against the fp32 oracle. Every 16-bit rounding of
    the fp16 path (Q K^T operands, P, the MLP intermediate, the output) must be an fp16 rounding."""
    kind, _, rest = case.partition("-")
    errs = {}
    for dt in DTYPES:
        if kind == "attn":
            got, ref = _attn_case(ops, dt, rest == "pair", monkeypatch)
        elif kind == "decode":
            got, ref = _decode_case(ops, dt, 1 if rest == "mha" else 4, monkeypatch)
        elif kind == "layernorm":
            got, ref = _ln_case(ops, dt, 768 if rest == "warp" else 4096, monkeypatch)
        else:
            act, path = rest.rsplit("-", 1)
            got, ref = _mlp_case(ops, dt, act, path, monkeypatch)
        assert got.dtype == dt
        errs[dt] = mean_abs_err(got, ref)
    ratio = errs[FP16] / errs[BF16]
    print(f"[fp16/bf16] {case} {ratio:.3f} (bf16 {errs[BF16]:.3e}, fp16 {errs[FP16]:.3e})")
    assert ratio <= FP16_OVER_BF16, f"{case}: fp16 error is {ratio:.2f} of the bf16 error"


# ------------------------------------------------------------------------------------------------- (b) dispatch matrix
@gpu
@pytest.mark.parametrize("D", [64, 128, 80])
@pytest.mark.parametrize("pair", [False, True])
@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS.get)
def test_dispatch_prefill(ops, monkeypatch, dtype, pair, D):
    """K1 default / CTA-pair kernel (D 64 and 128 builds; 80 runs in the 128 build), plain and accumulate output, and the
    paged gather (always the default kernel: the pair kernel does not read the paged cache)."""
    monkeypatch.setenv("B200_FA_PAIR", "1" if pair else "0")
    name = "fa_fwd_pair_kernel" if pair else "fa_fwd_kernel"
    B, Sq, Sk, Hq, Hkv = 2, 300, 420, 4, 2
    q, k, v = rand_qkv(B, Sq, Sk, Hq, Hkv, D, dtype, seed=D)
    o, lse = ops.flash_attn_fwd(q, k, v, causal=True, causal_offset=Sk - Sq - 150, return_lse=True)   # some rows see nothing
    assert ops.last_kernel() == name
    ro, rl = orc.attention_ref(q.cpu(), k.cpu(), v.cpu(), causal=True, causal_offset=Sk - Sq - 150)
    check_out(o, ro, dtype, lse=lse, ref_lse=rl)
    o_acc = torch.full((B, Sq, Hq, D), float("nan"), device="cuda")
    l_acc = torch.full((B, Hq, Sq), float("nan"), device="cuda")
    for i, (a, b) in enumerate(((0, 128), (128, Sk))):
        ops.flash_attn_fwd_accum(q, k[:, a:b], v[:, a:b], o_acc, l_acc, init=(i == 0), causal=True,
                                 causal_offset=Sk - Sq - 150 - a)
        assert ops.last_kernel() == name
    check_out(o_acc, ro, dtype, lse=l_acc, ref_lse=rl)
    if D in (64, 128):
        bs, L, nblk = 16, 2, 64
        kc = torch.randn(nblk, L, bs, Hkv, D, device="cuda", dtype=dtype)
        vc = torch.randn_like(kc)
        bt = torch.randperm(nblk, device="cuda")[:B * 24].view(B, 24).to(torch.int32).contiguous()
        ctx = torch.tensor([Sq + 50, Sq], dtype=torch.int32)
        o, lse = ops.paged_prefill_attention(q, kc, vc, bt, ctx.cuda(), layer_idx=1, causal=True, return_lse=True)
        assert ops.last_kernel() == "fa_fwd_kernel"
        ro, rl = orc.paged_prefill_attention_ref(q.cpu(), kc.cpu(), vc.cpu(), bt.cpu(), ctx, layer_idx=1, causal=True)
        check_out(o, ro, dtype, lse=lse, ref_lse=rl)


@gpu
@pytest.mark.parametrize("paged", [False, True])
@pytest.mark.parametrize("D", [64, 128])
@pytest.mark.parametrize("G", [1, 2, 3, 8, 16])
@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS.get)
def test_dispatch_decode(ops, monkeypatch, dtype, G, D, paged):
    """K2: G = Hq/Hkv of 1 and 2 run decode_kernel, 3..16 the tensor-core GQA kernel (register- or ring-staged); one split
    (the kernel writes O itself) and a forced 3 splits (decode_reduce_kernel merges them)."""
    g = torch.Generator(device="cuda").manual_seed(G * D)
    B, Hkv, S = 3, 2, 520
    q = torch.randn(B, Hkv * G, D, device="cuda", dtype=dtype, generator=g)
    lens = torch.tensor([S, 1, 333], device="cuda", dtype=torch.int32)
    if paged:
        bs, nblk = 16, 120
        kc = torch.randn(nblk, 2, bs, Hkv, D, device="cuda", dtype=dtype, generator=g)
        vc = torch.randn_like(kc)
        bt = torch.randperm(nblk, device="cuda")[:B * 40].view(B, 40).to(torch.int32).contiguous()
        kw = dict(block_tables=bt, layer_idx=1)
        ro, rl = orc.decode_attention_ref(q.cpu(), kc.cpu(), vc.cpu(), lens.cpu(), block_tables=bt.cpu(), layer_idx=1)
    else:
        kc = torch.randn(B, S, Hkv, D, device="cuda", dtype=dtype, generator=g)
        vc = torch.randn_like(kc)
        kw = {}
        ro, rl = orc.decode_attention_ref(q.cpu(), kc.cpu(), vc.cpu(), lens.cpu())
    for ring in ((False, True) if G >= 3 else (False,)):
        monkeypatch.setenv("B200_GQA_RING", "1" if ring else "0")
        for splits in (1, 3):
            o, lse = ops.decode_attention(q, kc, vc, lens, num_splits=splits, return_lse=True, **kw)
            want = "decode_kernel" if G <= 2 else "decode_gqa_ring_kernel" if ring else "decode_gqa_mma_kernel"
            assert ops.last_kernel() == (want if splits == 1 else "decode_reduce_kernel")
            check_out(o, ro, dtype, "decode", Hkv, lse=lse, ref_lse=rl)


ACTS = {None: "NONE", "gelu_tanh": "GELU_TANH", "gelu": "GELU_ERF", "relu": "RELU", "swiglu": "SWIGLU"}


@gpu
@pytest.mark.parametrize("act", list(ACTS), ids=str)
@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS.get)
def test_dispatch_gemm(ops, monkeypatch, dtype, act):
    """K3: gemm_act_kernel (T < 1024), forced split-K at a ragged K (584 = 10 k-blocks, the last 8 wide) with 2 and 5
    splits, with and without bias (splitk_reduce_kernel applies bias and activation), the CTA-pair kernel with one and two
    epilogue warpgroups, and the single-launch fused MLP."""
    c = lambda t: None if t is None else t.cpu()
    for T, K, N, splits in ((300, 512, 1032, "1"), (200, 584, 520, "2"), (200, 584, 520, "5")):
        monkeypatch.setenv("B200_GEMM_K_SPLITS", splits)
        for bias in (True, False):
            x, w, b, _, _, wg, bg = make_mlp(T, K, N, act or "relu", seed=T + K, bias=bias, std=0.05, dtype=dtype)
            y = ops.linear_act(x, w, b, act, wg, bg)
            assert ops.last_gemm_kernel() == f"gemm_act_kernel<{ACTS[act]}>"
            assert (ops.last_kernel() == "splitk_reduce_kernel") == (splits != "1")
            check_out(y, orc.linear_act_ref(c(x), c(w), c(b), act, c(wg), c(bg)), dtype, "2d")
    monkeypatch.setenv("B200_GEMM_K_SPLITS", "1")
    x, w, b, _, _, wg, bg = make_mlp(1100, 512, 1032, act or "relu", seed=5, std=0.05, dtype=dtype)
    ref = orc.linear_act_ref(c(x), c(w), c(b), act, c(wg), c(bg))
    for epi in (("1",) if act == "swiglu" else ("1", "2")):
        monkeypatch.setenv("B200_GEMM_EPI_WGS", epi)
        y = ops.linear_act(x, w, b, act, wg, bg)
        assert ops.last_gemm_kernel() == f"gemm_act_pair_kernel<{ACTS[act]}{',2wg' if epi == '2' else ''}>"
        check_out(y, ref, dtype, "2d")
    if act is not None:
        monkeypatch.setenv("B200_MLP_FUSED", "1")
        x, wu, bu, wd, bd, wg, bg = make_mlp(1100, 512, 1032, act, seed=6, dtype=dtype)
        y = ops.fused_mlp(x, wu, bu, wd, bd, act, wg, bg)
        assert ops.last_gemm_kernel() == f"fused_mlp_pair_kernel<{ACTS[act]}>"
        check_out(y, orc.mlp_ref(c(x), c(wu), c(bu), c(wd), c(bd), act, c(wg), c(bg)), dtype, "2d")


@gpu
@pytest.mark.parametrize("res", [False, True])
@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS.get)
def test_dispatch_layernorm(ops, monkeypatch, dtype, res):
    """LayerNorm: the warp-per-row kernel for every row width it is built for (1..8 x 256 columns, with and without the
    next-row prefetch) and the CTA-per-row kernel for 1..4 x 2048 columns, each width ragged by 8 columns."""
    g = torch.Generator(device="cuda").manual_seed(int(res))
    r = lambda *s: torch.randn(*s, device="cuda", generator=g).to(dtype)
    c = lambda t: None if t is None else t.cpu()
    cases = [("2048", pf, 256 * it - 8) for pf in ("0", "1") for it in range(1, 9)] + [("8", "1", 2048 * it - 8) for it in range(1, 5)]
    for narrow_max, prefetch, cols in cases:
        monkeypatch.setenv("B200_LN_NARROW_MAX", narrow_max)
        monkeypatch.setenv("B200_LN_PREFETCH", prefetch)
        x, w, b = r(301, cols) * 2 + 0.5, r(cols), r(cols)
        rs = r(301, cols) if res else None
        y = ops.layernorm(x, w, b, 1e-5, rs, 0.7)
        assert ops.last_kernel() == "layernorm_kernel"
        check_out(y, orc.layernorm_ref(c(x), c(w), c(b), 1e-5, c(rs), 0.7), dtype, "2d")


# ------------------------------------------------------------------------------------------------- (c) softmax_scale
@gpu
@pytest.mark.parametrize("scale", [1.0, 0.03])
@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS.get)
def test_softmax_scale(ops, monkeypatch, dtype, scale):
    """A scale other than 1/sqrt(D): 1.0 gives near one-hot rows and many lazy rescales, 0.03 near-uniform rows. Output and
    the natural-log LSE must match the oracle at the same scale through K1 (default, pair, accumulate, paged) and K2."""
    B, S, Hq, Hkv, D = 2, 384, 4, 2, 128
    q, k, v = rand_qkv(B, S, S, Hq, Hkv, D, dtype, seed=21)
    ro, rl = orc.attention_ref(q.cpu(), k.cpu(), v.cpu(), causal=True, softmax_scale=scale)
    for pair in ("0", "1"):
        monkeypatch.setenv("B200_FA_PAIR", pair)
        o, lse = ops.flash_attn_fwd(q, k, v, causal=True, softmax_scale=scale, return_lse=True)
        check_out(o, ro, dtype, lse=lse, ref_lse=rl)
        o_acc, l_acc = torch.empty(B, S, Hq, D, device="cuda"), torch.empty(B, Hq, S, device="cuda")
        for i, (a, b) in enumerate(((0, 256), (256, S))):
            ops.flash_attn_fwd_accum(q, k[:, a:b], v[:, a:b], o_acc, l_acc, init=(i == 0), causal=True, softmax_scale=scale,
                                     causal_offset=-a)
        check_out(o_acc, ro, dtype, lse=l_acc, ref_lse=rl)
    bs, nblk = 32, 40
    kc = torch.zeros(nblk, 1, bs, Hkv, D, device="cuda", dtype=dtype)
    vc = torch.zeros_like(kc)
    bt = torch.randperm(nblk, device="cuda")[:B * 12].view(B, 12).to(torch.int32).contiguous()
    for b in range(B):   # the same keys, stored through the block table
        idx = torch.arange(S, device="cuda")
        kc[bt[b, idx // bs].long(), 0, idx % bs] = k[b]
        vc[bt[b, idx // bs].long(), 0, idx % bs] = v[b]
    ctx = torch.full((B,), S, device="cuda", dtype=torch.int32)
    o, lse = ops.paged_prefill_attention(q[:, -64:], kc, vc, bt, ctx, causal=True, softmax_scale=scale, return_lse=True)
    check_out(o, ro[:, -64:], dtype, lse=lse, ref_lse=rl[:, :, -64:])
    for G in (1, 4):
        qd = torch.randn(B, Hkv * G, D, device="cuda", dtype=dtype)
        lens = torch.tensor([S, 100], device="cuda", dtype=torch.int32)
        o, lse = ops.decode_attention(qd, k, v, lens, softmax_scale=scale, return_lse=True)
        assert ops.last_kernel() in ("decode_kernel", "decode_gqa_mma_kernel", "decode_reduce_kernel")
        rd, rdl = orc.decode_attention_ref(qd.cpu(), k.cpu(), v.cpu(), lens.cpu(), softmax_scale=scale)
        check_out(o, rd, dtype, "decode", Hkv, lse=lse, ref_lse=rdl)


# ------------------------------------------------------------------------------------------------- (d) byte-exact fp16
@gpu
def test_fp16_byte_exact_ops(ops):
    """kv_append moves fp16 bits unchanged (contiguous and paged cache), cast_out(fp16) is round-to-nearest of the fp32
    accumulator (== Tensor.half()), and lse_merge reads an fp16 partial output."""
    g = torch.Generator(device="cuda").manual_seed(31)
    r = lambda *s: torch.randn(*s, device="cuda", generator=g).to(FP16)
    B, Hkv, D = 3, 2, 128
    key, val = r(B, Hkv, D), r(B, Hkv, D)
    lens = torch.tensor([37, 256, 129], device="cuda", dtype=torch.int32)
    kc, vc = r(B, 300, Hkv, D), r(B, 300, Hkv, D)
    rk, rv = kc.cpu().clone(), vc.cpu().clone()
    ops.kv_append(key, val, kc, vc, lens)
    assert ops.last_kernel() == "kv_append_kernel"
    orc.kv_append_ref(key.cpu(), val.cpu(), rk, rv, lens.cpu())
    assert torch.equal(kc.cpu().view(torch.int16), rk.view(torch.int16)) and torch.equal(vc.cpu().view(torch.int16), rv.view(torch.int16))
    kp, vp = r(60, 2, 16, Hkv, D), r(60, 2, 16, Hkv, D)
    bt = torch.randperm(60, device="cuda")[:B * 17].view(B, 17).to(torch.int32).contiguous()
    rk, rv = kp.cpu().clone(), vp.cpu().clone()
    ops.kv_append(key, val, kp, vp, lens, block_tables=bt, layer_idx=1)
    orc.kv_append_ref(key.cpu(), val.cpu(), rk, rv, lens.cpu(), bt.cpu(), 1)
    assert torch.equal(kp.cpu().view(torch.int16), rk.view(torch.int16)) and torch.equal(vp.cpu().view(torch.int16), rv.view(torch.int16))
    o_acc = torch.randn(2, 200, 4, 128, device="cuda", generator=g) * 3
    o_acc[0, 0, 0, :4] = torch.tensor([65504.0, 1e-6, -2.0 ** -20, 70000.0])   # largest finite, fp16 subnormals, overflow
    out = ops.cast_out(o_acc, FP16)
    assert ops.last_kernel() == "cast_out_kernel"
    assert torch.equal(out.cpu().view(torch.int16), o_acc.cpu().half().view(torch.int16))
    oa, la = torch.randn(2, 200, 4, 128, device="cuda", generator=g), torch.randn(2, 4, 200, device="cuda", generator=g)
    ob, lb = r(2, 200, 4, 128), torch.randn(2, 4, 200, device="cuda", generator=g)
    la[0, 0, :5] = float("-inf")
    lb[0, 1, :5] = float("-inf")
    la[1, 2, :3] = lb[1, 2, :3] = float("-inf")
    ro, rl = orc.lse_merge_ref(oa.cpu(), la.cpu(), ob.cpu(), lb.cpu())
    ops.lse_merge(oa, la, ob, lb)
    assert ops.last_kernel() == "lse_merge_kernel"
    assert (oa.cpu() - ro).abs().max().item() <= 1e-5
    check_lse(la, rl)


# ------------------------------------------------------------------------------------------------- (e) module defaults
@gpu
def test_modules_default_config_runs_fp16(ops, golden_dir):
    """fp32 activations into the modules with their default configuration run the fp16 kernels: the result meets the fp16
    tolerance against the oracle on fp16-rounded inputs (a bf16 run would not), and stays next to the reference's own
    fp32 outputs."""
    from kernels.attention.flash_attention import FlashAttention3
    from kernels.mlp.fused_mlp import FusedMLP, FusedTransformerMLP

    vecs = torch.load(os.path.join(golden_dir, "mlp_reference_vectors.pt"))
    h16 = lambda t: None if t is None else t.half().float()
    for name in ("FusedTransformerMLP_gelu", "FusedTransformerMLP_relu", "FusedTransformerMLP_swiglu", "FusedMLP_gelu_erf"):
        d = vecs[name]
        if name.startswith("FusedMLP_"):
            mod, act = FusedMLP(d["hidden"], d["intermediate"]), "gelu"
        else:
            mod = FusedTransformerMLP(d["hidden"], d["intermediate"], d["activation_fn"])
            act = {"gelu": "gelu_tanh"}.get(d["activation_fn"], d["activation_fn"])
        mod.load_state_dict(d["state_dict"])
        y = mod.to("cuda")(d["x"].to("cuda"))
        assert y.dtype == torch.float32
        sd = {k: h16(v) for k, v in d["state_dict"].items()}
        p = "mlp." if name.startswith("FusedTransformerMLP") else ""
        ref = orc.mlp_ref(h16(d["x"]), sd[p + "fc1.weight"], sd[p + "fc1.bias"], sd[p + "fc2.weight"], sd[p + "fc2.bias"], act,
                          sd.get(p + "fc1_gate.weight"), sd.get(p + "fc1_gate.bias"))
        check_out(y, ref, FP16, "2d")
        check_out(y, d["y"], FP16, "2d", mean_rel=2e-3, max_rel=3e-3)
    g = torch.Generator(device="cuda").manual_seed(41)
    q = torch.randn(2, 300, 8, 128, device="cuda", generator=g)
    k, v = (torch.randn(2, 300, 2, 128, device="cuda", generator=g) for _ in range(2))
    o = FlashAttention3()(q, k, v)
    assert o.dtype == torch.float32 and ops.last_kernel() in ("fa_fwd_kernel", "fa_fwd_pair_kernel")
    ro, _ = orc.attention_ref(q.half().cpu(), k.half().cpu(), v.half().cpu())
    check_out(o, ro, FP16)


# ------------------------------------------------------------------------------------------------- (f) checker self-test
def _emulate_attention(q, k, v, dt, p_dt=None, hide=None):
    """The rounding of the attention kernels, on the CPU: fp32 scores, P rounded to 16 bit (``p_dt``, default the compute
    type), fp32 row sum, output rounded to ``dt``. ``hide`` = (b, h, rows, keys) masks those keys for those rows only."""
    qf, kf, vf = q.float(), k.float(), v.float()
    B, S, H, D = q.shape
    s = torch.einsum("bqhd,bkhd->bhqk", qf, kf) / math.sqrt(D)
    mask = torch.ones(S, S, dtype=torch.bool).triu(1).expand(B, H, S, S).clone()
    if hide is not None:
        b, h, rows, keys = hide
        mask[b, h, rows.unsqueeze(1), keys.unsqueeze(0)] = True
    s = s.masked_fill(mask, float("-inf"))
    p = torch.exp(s - s.amax(-1, keepdim=True))
    o = torch.einsum("bhqk,bkhd->bqhd", p.to(p_dt or dt).float(), vf) / p.sum(-1).transpose(1, 2).unsqueeze(-1)
    return o.to(dt)


def _emulate_mlp(x, wu, bu, wd, bd, dt, mid_dt=None):
    h = torch.nn.functional.gelu(x.float() @ wu.float().t() + bu.float(), approximate="tanh")
    return (h.to(mid_dt or dt).float() @ wd.float().t() + bd.float()).to(dt)


def _rejects(fn):
    try:
        fn()
    except AssertionError:
        return True
    return False


def test_tile_checker_accepts_correct_rounding_and_rejects_defects():
    """The thresholds must pass the rounding a correct kernel does and fail each of these defects, which the old whole-tensor
    max-abs / mean-rel check let through: one key dropped in one head for 512 rows, one 128-row tile missing a KV block,
    an fp16 path that rounds P (attention) or the intermediate (MLP) through bf16."""
    B, S, H, D = 1, 1024, 4, 128
    qkv = [exact_in_both(B, S, H, D, seed=s, device="cpu") for s in (1, 2)] + [exact_in_both(B, S, H, D, scale=0.25, seed=3, device="cpu")]
    ref = orc.attention_ref(*qkv, causal=True)[0]
    T, h, i = 512, 256, 768
    x, wu, wd = (exact_in_both(*s, scale=sc, seed=n, device="cpu") for n, (s, sc) in enumerate((((T, h), 1.0), ((i, h), 0.06), ((h, i), 0.04))))
    bu, bd = exact_in_both(i, scale=0.1, seed=7, device="cpu"), exact_in_both(h, scale=0.1, seed=8, device="cpu")
    mref = orc.mlp_ref(x, wu, bu, wd, bd, "gelu_tanh")
    for dt in DTYPES:
        q, k, v = (t.to(dt) for t in qkv)
        check_out(_emulate_attention(q, k, v, dt), ref, dt)
        check_out(_emulate_mlp(*(t.to(dt) for t in (x, wu, bu, wd, bd)), dt), mref, dt, "2d")
        dropped_key = (0, 1, torch.arange(512, 1024), torch.tensor([300]))
        assert _rejects(lambda: check_out(_emulate_attention(q, k, v, dt, hide=dropped_key), ref, dt))
        missing_block = (0, 2, torch.arange(640, 768), torch.arange(256, 384))
        assert _rejects(lambda: check_out(_emulate_attention(q, k, v, dt, hide=missing_block), ref, dt))
    q, k, v = (t.to(FP16) for t in qkv)
    assert _rejects(lambda: check_out(_emulate_attention(q, k, v, FP16, p_dt=BF16), ref, FP16))
    args = [t.to(FP16) for t in (x, wu, bu, wd, bd)]
    assert _rejects(lambda: check_out(_emulate_mlp(*args, FP16, mid_dt=BF16), mref, FP16, "2d"))


def test_tile_errors_tilings():
    """Tiles are where they are said to be: an error in one (b, h, 128-row) block, one kv head of a decode batch or one
    128 x 128 block of a 2-D output lands in exactly one tile; an all-zero reference tile is reported through empty_max."""
    ref = torch.ones(2, 300, 3, 16)
    got = ref.clone()
    got[1, 260, 2, 5] += 0.5
    e = orc.tile_errors(got, ref, "attn")
    assert e["mean_rel"].numel() == 2 * 3 * 3 and (e["max_rel"] > 0).sum() == 1
    assert e["max_rel"].argmax().item() == (1 * 3 + 2) * 3 + 2
    ref = torch.ones(2, 8, 4)
    got = ref.clone()
    got[1, 5] += 1.0                                   # kv head 1 of batch 1 when Hkv = 2 (G = 4)
    e = orc.tile_errors(got, ref, "decode", hkv=2)
    assert e["mean_rel"].tolist() == [0, 0, 0, 4 / 16]
    ref = torch.ones(300, 260)
    ref[256:, 256:] = 0
    got = ref.clone()
    got[299, 259] = 1.0
    e = orc.tile_errors(got, ref, "2d")
    assert e["mean_rel"].numel() == 3 * 3 - 1 and e["empty_max"] == 1.0 and e["max_rel"].max() == 0


# ------------------------------------------------------------------------------------------------- (g) kernel inventory
def _instantiations():
    """Every __global__ instantiation in the library -> the test that launches it."""
    p = "tests/test_gpu_precision.py::"
    t = {"kv_append_kernel<unsignedshort>": p + "test_fp16_byte_exact_ops"}
    for dt in ("__nv_bfloat16", "__half"):
        for D in (64, 128):
            for acc in (0, 1):
                t[f"fa_fwd_kernel<{D},{dt},{acc}>"] = p + "test_dispatch_prefill"
                t[f"fa_fwd_pair_kernel<{D},{dt},{acc}>"] = p + "test_dispatch_prefill"
            for paged in (0, 1):
                for G in (1, 2):
                    t[f"decode_kernel<{D},{G},{dt},{paged}>"] = p + "test_dispatch_decode"
                for ring in (0, 1):
                    t[f"decode_gqa_mma_kernel<{D},{dt},{paged},{ring}>"] = p + "test_dispatch_decode"
            t[f"decode_reduce_kernel<{D},{dt}>"] = p + "test_dispatch_decode"
        for act in range(5):
            t[f"gemm_act_kernel<{act},{dt}>"] = p + "test_dispatch_gemm"
            t[f"splitk_reduce_kernel<{act},{dt}>"] = p + "test_dispatch_gemm"
            t[f"gemm_act_pair_kernel<{act},{dt},1>"] = p + "test_dispatch_gemm"
            if act != 4:                                    # SwiGLU has one epilogue warpgroup only
                t[f"gemm_act_pair_kernel<{act},{dt},2>"] = p + "test_dispatch_gemm"
                t[f"fused_mlp_pair_kernel<{act + 1},{dt}>"] = p + "test_dispatch_gemm"
        for res in (0, 1):
            for it in range(1, 9):
                for pf in (0, 1):
                    t[f"layernorm_warp_kernel<{dt},{res},{it},{pf}>"] = p + "test_dispatch_layernorm"
            for it in range(1, 5):
                t[f"layernorm_kernel<{dt},{res},{it}>"] = p + "test_dispatch_layernorm"
        t[f"lse_merge_kernel<{dt}>"] = p + "test_fp16_byte_exact_ops"
        t[f"cast_out_kernel<{dt}>"] = p + "test_fp16_byte_exact_ops"
        for mc in (0, 1):
            t[f"tp_allreduce_kernel<{dt},{mc}>"] = "tests/multi_gpu_check.py"
    return t


def test_every_compiled_kernel_has_a_test(built_lib):
    """The set of __global__ instantiations in the built library equals the table above: a new instantiation (or a dispatch
    branch that is compiled but unreachable) without a test that launches it fails here."""
    from ml_inference_optimizer_b200 import build as b

    cuda_bin = os.path.dirname(shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc")
    tools = [shutil.which(n) or os.path.join(cuda_bin, n) for n in ("cuobjdump", "cu++filt")]
    for tool in tools:
        if not os.path.exists(tool):
            pytest.skip(f"{tool} not available")
    syms = subprocess.run([tools[0], "-symbols", str(b.LIB_PATH)], capture_output=True, text=True, check=True).stdout
    mangled = sorted({ln.split()[-1] for ln in syms.splitlines() if "STT_FUNC" in ln and "STB_GLOBAL" in ln})
    names = subprocess.run([tools[1]], input="\n".join(mangled), capture_output=True, text=True, check=True).stdout
    found = set()
    for ln in names.splitlines():
        m = re.match(r"void b200::\w+::(\w+<.*?>)\(", ln)
        if m:
            found.add(re.sub(r"\((?:int|bool)\)|\s", "", m.group(1)))
    table = _instantiations()
    assert found - set(table) == set(), "compiled kernels no test launches"
    assert set(table) - found == set(), "listed kernels that are not compiled"
    assert not any(re.match(r"decode_kernel<\d+,(4|8),", k) for k in found)
    for target in set(table.values()):
        path, _, fn = target.partition("::")
        assert os.path.exists(os.path.join(ROOT, path)) and (not fn or fn in globals()), target
