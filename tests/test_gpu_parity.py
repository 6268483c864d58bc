"""Parity of the CUDA path (through the C-ABI) against the fp32 oracle — the parity tests proper. Need a B200.

Every kernel is built for bf16 and for fp16 and every case here runs in both. Outputs are compared tile by tile
(oracle.tile_errors): one tile per (batch, head, 128 query rows) for attention, per (batch, kv head) for decode, per 128 x 128
block for GEMM / MLP / LayerNorm outputs, each against its own reference magnitude — an error confined to one head, one KV
block or one GEMM tile is not averaged away by the rest of the tensor. Rows without a visible key must be exactly 0 with an
LSE of exactly -inf.
"""
import math
import os

import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import attn_mlp_oracle as orc  # noqa: E402

BF16, FP16 = torch.bfloat16, torch.float16
DTYPES = (BF16, FP16)
# Tolerances, relative to each tile's own reference (16-bit storage, fp32 accumulate / softmax). The worst value measured on
# a B200 (1000 W) over this file and tests/test_gpu_precision.py is noted beside each (bf16 / fp16).
TILE_MEAN_REL = {BF16: 5e-3, FP16: 1e-3}     # attention, GEMM, MLP, LayerNorm tiles: mean|err| / mean|ref|   2.7e-3 / 3.1e-4
ROW_MEAN_REL = {BF16: 6e-3, FP16: 1.2e-3}    # decode tiles (the 1..16 query heads of one kv head)           2.2e-3 / 2.7e-4
TILE_MAX_REL = {BF16: 1.6e-2, FP16: 2.5e-3}  # max|err| / max|ref| of a tile                                 6.3e-3 / 6.8e-4
LSE_MAX_ABS = 1e-3                           # natural-log LSE, absolute                                      9.9e-5 (both)
WORST: dict = {}                            # worst value of each metric seen in this session, printed per module


@pytest.fixture(scope="module")
def ops(built_lib):
    assert torch.cuda.is_available(), "gpu tests need CUDA"
    from ml_inference_optimizer_b200 import ops as _ops

    assert _ops.arch_ok(), "gpu tests need an sm_100 device"
    return _ops


@pytest.fixture(scope="module", autouse=True)
def _report_worst():
    yield
    for (metric, dt), val in sorted(WORST.items()):
        print(f"[worst] {metric} {dt} {val:.3e}")


def _note(metric, dtype, val):
    key = (metric, str(dtype).replace("torch.", ""))
    WORST[key] = max(WORST.get(key, 0.0), float(val))


def with_dtypes(argnames, cases):
    """parametrize() arguments running every case in bf16 and fp16: a bf16 case keeps the id pytest gives the bare case,
    the fp16 one is prefixed with ``fp16-``."""
    names = [n.strip() for n in argnames.split(",")]
    plain = lambda v: v is None or isinstance(v, (bool, int, float, str))
    params = []
    for dt, prefix in ((BF16, ""), (FP16, "fp16-")):
        for i, c in enumerate(cases):
            c = c if isinstance(c, tuple) else (c,)
            cid = "-".join(str(v) if plain(v) else f"{n}{i}" for n, v in zip(names, c))
            params.append(pytest.param(*c, dt, id=prefix + cid))
    return ",".join(names + ["dtype"]), params


def check_lse(got, ref):
    """-inf exactly where the oracle has no visible key, |err| <= LSE_MAX_ABS elsewhere (natural log)."""
    got, ref = got.float().cpu(), ref.float().cpu()
    ninf = torch.isinf(ref) & (ref < 0)
    assert torch.equal(torch.isinf(got) & (got < 0), ninf), "-inf pattern of LSE differs"
    if (~ninf).any():
        err = (got[~ninf] - ref[~ninf]).abs().max().item()
        _note("lse_abs", "any", err)
        assert err <= LSE_MAX_ABS, f"LSE max abs err {err:.3e}"


def check_out(got, ref, dtype, tiling="attn", hkv=None, lse=None, ref_lse=None, mean_rel=None, max_rel=None):
    """Tile-local comparison of a kernel output with the oracle (see the module docstring). ``dtype`` is the compute type
    that selects the thresholds; ``lse`` / ``ref_lse`` also check the LSE and that rows without a visible key are exactly 0."""
    got, ref = got.float().cpu(), ref.float().cpu()
    assert torch.isfinite(got).all()
    if ref_lse is not None:
        check_lse(lse, ref_lse)
        dead = torch.isinf(ref_lse) & (ref_lse < 0)
        if tiling == "attn":
            dead = dead.transpose(1, 2)                  # [B,H,S] -> rows of [B,S,H,D]
        assert (got[dead] == 0).all(), "a row without a visible key is not exactly 0"
    e = orc.tile_errors(got, ref, tiling, hkv)
    assert e["empty_max"] == 0, f"non-zero output {e['empty_max']:.3e} in a tile whose reference is all zero"
    if e["mean_rel"].numel() == 0:
        return
    mean_tol = mean_rel if mean_rel is not None else (ROW_MEAN_REL if tiling == "decode" else TILE_MEAN_REL)[dtype]
    max_tol = max_rel if max_rel is not None else TILE_MAX_REL[dtype]
    worst_mean, worst_max = e["mean_rel"].max().item(), e["max_rel"].max().item()
    if mean_rel is None and max_rel is None:
        _note("row_mean_rel" if tiling == "decode" else "tile_mean_rel", dtype, worst_mean)
        _note("tile_max_rel", dtype, worst_max)
    assert worst_mean <= mean_tol, f"worst tile mean rel err {worst_mean:.3e} (tile {int(e['mean_rel'].argmax())})"
    assert worst_max <= max_tol, f"worst tile max rel err {worst_max:.3e} (tile {int(e['max_rel'].argmax())})"


def rand_qkv(B, Sq, Sk, Hq, Hkv, D, dtype=BF16, seed=0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    q = torch.randn(B, Sq, Hq, D, device="cuda", dtype=dtype, generator=g)
    k = torch.randn(B, Sk, Hkv, D, device="cuda", dtype=dtype, generator=g)
    v = torch.randn(B, Sk, Hkv, D, device="cuda", dtype=dtype, generator=g)
    return q, k, v


# ------------------------------------------------------------------------------------------ K1 prefill
FA_CASES = [
    # B, Sq, Sk, Hq, Hkv, D, causal, offset, kv_lens
    (1, 128, 128, 1, 1, 128, False, 0, None),
    (1, 256, 256, 2, 2, 128, True, 0, None),
    (2, 1024, 1024, 4, 4, 128, True, 0, None),
    (2, 1024, 1024, 8, 2, 128, True, 0, None),       # GQA 4:1 (Llama-3 style)
    (2, 512, 512, 12, 12, 64, True, 0, None),        # GPT-2 head shape
    (1, 300, 300, 2, 2, 128, True, 0, None),         # ragged tail
    (1, 1, 1, 1, 1, 64, False, 0, None),             # minimum size
    (1, 77, 333, 2, 1, 64, False, 0, None),          # Sq != Sk, MQA
    (2, 512, 512, 2, 2, 128, False, 0, [512, 100]),  # right-padding mask
    (2, 384, 384, 2, 2, 64, True, 0, [1, 384]),      # one visible key
    (1, 256, 512, 2, 2, 128, True, 256, None),       # later ring chunk / bottom-right alignment
    (1, 256, 256, 2, 2, 128, True, -128, None),      # rows with no visible key -> O = 0, LSE = -inf
    (1, 256, 256, 2, 2, 128, True, -1000, None),     # nothing visible at all
    (1, 2048, 2048, 2, 2, 128, True, 0, None),
]


@pytest.mark.parametrize(*with_dtypes("B,Sq,Sk,Hq,Hkv,D,causal,offset,kv_lens", FA_CASES))
def test_fa_fwd_vs_oracle(ops, B, Sq, Sk, Hq, Hkv, D, causal, offset, kv_lens, dtype):
    q, k, v = rand_qkv(B, Sq, Sk, Hq, Hkv, D, dtype)
    lens = None if kv_lens is None else torch.tensor(kv_lens, device="cuda", dtype=torch.int32)
    o, lse = ops.flash_attn_fwd(q, k, v, causal=causal, causal_offset=offset, kv_lens=lens, return_lse=True)
    assert ops.last_kernel() == "fa_fwd_kernel"
    ro, rl = orc.attention_ref(q.cpu(), k.cpu(), v.cpu(), causal=causal, causal_offset=offset,
                               kv_lens=None if lens is None else lens.cpu())
    check_out(o, ro, dtype, lse=lse, ref_lse=rl)


@pytest.mark.parametrize("pair", [False, True])
@pytest.mark.parametrize("D", [8, 32, 40, 80, 96, 120])
def test_fa_fwd_any_head_dim(ops, monkeypatch, D, pair):
    """head_dim = any multiple of 8 up to 128 (the reference takes hidden_size // num_heads as it comes,
    flash_attention.py:176): the 64- / 128-column builds run it with the missing columns zero-filled by the TMA loads, which is
    exact, and the epilogue must not store past column D (guard columns next to every output row stay untouched). Both output
    modes (16-bit and the fp32 accumulate of a ring step)."""
    monkeypatch.setenv("B200_FA_PAIR", "1" if pair else "0")
    B, Sq, Sk, Hq, Hkv = 2, 300, 520, 4, 2
    q, k, v = rand_qkv(B, Sq, Sk, Hq, Hkv, D, seed=D)
    big = torch.full((B, Sq, Hq, D + 8), -7.0, device="cuda", dtype=torch.bfloat16)
    o, lse = ops.flash_attn_fwd(q, k, v, causal=True, causal_offset=Sk - Sq, return_lse=True, out=big[..., :D])
    assert ops.last_kernel() == ("fa_fwd_pair_kernel" if pair else "fa_fwd_kernel")
    ro, rl = orc.attention_ref(q.cpu(), k.cpu(), v.cpu(), causal=True, causal_offset=Sk - Sq)
    check_out(o, ro, BF16, lse=lse, ref_lse=rl)
    assert (big[..., D:] == -7.0).all(), "columns past head_dim were written"
    acc_big = torch.full((B, Sq, Hq, D + 8), -7.0, device="cuda", dtype=torch.float32)
    lse_acc = torch.empty((B, Hq, Sq), device="cuda", dtype=torch.float32)
    for i, (a, b) in enumerate(((0, 256), (256, Sk))):
        ops.flash_attn_fwd_accum(q, k[:, a:b], v[:, a:b], acc_big[..., :D], lse_acc, init=(i == 0), causal=True,
                                 causal_offset=Sk - Sq - a)
    check_out(acc_big[..., :D], ro, BF16, lse=lse_acc, ref_lse=rl)
    assert (acc_big[..., D:] == -7.0).all()
    with pytest.raises(RuntimeError, match="head_dim"):
        ops.flash_attn_fwd(*rand_qkv(1, 128, 128, 1, 1, 136))


PAIR_CASES = FA_CASES + [
    (2, 640, 640, 4, 2, 128, True, 0, None),         # odd number of 128-row tiles: the second CTA of the last cluster has no rows
    (1, 1536, 1536, 2, 2, 64, True, 0, [1000]),      # padding + causal, D = 64
    (1, 384, 2048, 2, 1, 128, False, 0, [1500]),     # 12-16 KV blocks per tile: both softmax groups take several blocks
    (3, 768, 768, 6, 6, 128, True, 0, None),
]


@pytest.mark.parametrize(*with_dtypes("B,Sq,Sk,Hq,Hkv,D,causal,offset,kv_lens", PAIR_CASES))
def test_fa_pair_kernel_vs_oracle(ops, monkeypatch, B, Sq, Sk, Hq, Hkv, D, causal, offset, kv_lens, dtype):
    """The CTA-pair kernel (one 128-row tile per CTA, S and P double-buffered in TMEM, two softmax warpgroups on alternate KV
    blocks sharing the running reference maximum, K/V halves TMA-multicast across the cluster) is opt-in
    (B200_FA_PAIR=1, read per call); it must agree with the oracle on every case of the default kernel, including tiles
    whose two CTAs need different numbers of KV blocks and rows without a visible key."""
    monkeypatch.setenv("B200_FA_PAIR", "1")
    q, k, v = rand_qkv(B, Sq, Sk, Hq, Hkv, D, dtype)
    lens = None if kv_lens is None else torch.tensor(kv_lens, device="cuda", dtype=torch.int32)
    o, lse = ops.flash_attn_fwd(q, k, v, causal=causal, causal_offset=offset, kv_lens=lens, return_lse=True)
    assert ops.last_kernel() == "fa_fwd_pair_kernel"
    ro, rl = orc.attention_ref(q.cpu(), k.cpu(), v.cpu(), causal=causal, causal_offset=offset,
                               kv_lens=None if lens is None else lens.cpu())
    check_out(o, ro, dtype, lse=lse, ref_lse=rl)
    o2, lse2 = ops.flash_attn_fwd(q, k, v, causal=causal, causal_offset=offset, kv_lens=lens, return_lse=True)
    assert torch.equal(o, o2) and torch.equal(lse, lse2)   # run-to-run bit equality (no atomics, fixed reduction order)


def test_fa_pair_kernel_large_scores_and_accumulate(ops, monkeypatch):
    """Lazy rescaling across the two softmax groups (the reference maximum moves by far more than 2^8 between blocks that
    different warpgroups own) and the accumulate (ring-step) epilogue of the pair kernel."""
    monkeypatch.setenv("B200_FA_PAIR", "1")
    B, S, H, D = 1, 1024, 2, 128
    q, k, v = rand_qkv(B, S, S, H, H, D, seed=5)
    k = k.clone()
    for blk, gain in ((1, 6.0), (2, 0.1), (3, 12.0), (6, 25.0)):   # block maxima jump up and down between the groups
        k[:, blk * 128:(blk + 1) * 128] *= gain
    o, lse = ops.flash_attn_fwd(q, k, v, causal=False, return_lse=True)
    ro, rl = orc.attention_ref(q.cpu(), k.cpu(), v.cpu(), causal=False)
    check_out(o, ro, BF16, lse=lse, ref_lse=rl)
    o_acc = torch.full((B, S, H, D), float("nan"), device="cuda", dtype=torch.float32)
    lse_acc = torch.full((B, H, S), float("nan"), device="cuda", dtype=torch.float32)
    for i, (a, b) in enumerate(((0, 384), (384, 512), (512, 1024))):
        ops.flash_attn_fwd_accum(q, k[:, a:b], v[:, a:b], o_acc, lse_acc, init=(i == 0), causal=True, causal_offset=-a)
        assert ops.last_kernel() == "fa_fwd_pair_kernel"
    ro, rl = orc.attention_ref(q.cpu(), k.cpu(), v.cpu(), causal=True)
    check_out(ops.cast_out(o_acc, q.dtype), ro, BF16, lse=lse_acc, ref_lse=rl)


@pytest.mark.parametrize("B,S,H,Hkv,D,causal,kv_lens", [
    (6, 256, 64, 64, 64, True, None),                     # 384 one/two-iteration items: > 2 per SM, every CTA steals blocks
    (3, 768, 80, 16, 128, True, None),                    # 720 items, GQA 5:1, mixed item lengths (heavy-first order)
    (5, 512, 40, 40, 128, False, [512, 0, 37, 300, 1]),   # items with no key at all between normal ones
])
def test_fa_fwd_work_stealing_many_items(ops, B, S, H, Hkv, D, causal, kv_lens):
    """The kernel is persistent: a CTA that finished its block takes over blocks that have not started (cluster launch
    control), carrying barrier phases, the KV ring and TMEM from item to item. Grids with several items per SM, item
    lengths that differ by up to 6x and empty items exercise every carry-over; results must match the oracle exactly as
    for a single item per CTA."""
    q, k, v = rand_qkv(B, S, S, H, Hkv, D, seed=11)
    lens = None if kv_lens is None else torch.tensor(kv_lens, device="cuda", dtype=torch.int32)
    o, lse = ops.flash_attn_fwd(q, k, v, causal=causal, kv_lens=lens, return_lse=True)
    o2, lse2 = ops.flash_attn_fwd(q, k, v, causal=causal, kv_lens=lens, return_lse=True)
    assert torch.equal(o, o2) and torch.equal(lse, lse2), "result depends on which CTA picked up which block"
    ro, rl = orc.attention_ref(q.cpu(), k.cpu(), v.cpu(), causal=causal, kv_lens=None if lens is None else lens.cpu())
    check_out(o, ro, BF16, lse=lse, ref_lse=rl)


@pytest.mark.parametrize(*with_dtypes("B,Sq,Sk,Hq,Hkv,D,causal", [
    (2, 512, 1024, 4, 2, 128, False),
    (1, 384, 768, 2, 2, 64, False),
    (2, 512, 512, 4, 4, 128, True),      # causal: second key block partly / fully invisible for early rows
]))
def test_fa_fwd_accum_key_blocks_equal_full_attention(ops, B, Sq, Sk, Hq, Hkv, D, causal, dtype):
    """Accumulate mode (one ring step per call): attending to the key blocks one after the other, each merged into the
    fp32 accumulator in the kernel epilogue, equals attention over all keys — including rows for which a later block
    is fully masked (accumulator untouched) and views of the accumulator for a subset of the rows."""
    q, k, v = rand_qkv(B, Sq, Sk, Hq, Hkv, D, dtype, seed=3)
    off = Sk - Sq if causal else 0      # bottom-right aligned causal mask over the concatenated keys
    o_acc = torch.full((B, Sq, Hq, D), float("nan"), device="cuda", dtype=torch.float32)
    lse_acc = torch.full((B, Hq, Sq), float("nan"), device="cuda", dtype=torch.float32)
    cuts = [0, Sk // 4, Sk // 4 + 128, Sk]
    for i, (a, b) in enumerate(zip(cuts, cuts[1:])):
        ops.flash_attn_fwd_accum(q, k[:, a:b], v[:, a:b], o_acc, lse_acc, init=(i == 0), causal=causal, causal_offset=off - a)
    ro, rl = orc.attention_ref(q.cpu(), k.cpu(), v.cpu(), causal=causal, causal_offset=off)
    check_out(ops.cast_out(o_acc, q.dtype), ro, dtype, lse=lse_acc, ref_lse=rl)
    # a step that only concerns the second half of the rows, through views (zigzag ring, src > r)
    h = Sq // 2
    o2 = torch.zeros_like(o_acc)
    l2 = torch.full_like(lse_acc, float("-inf"))
    ops.flash_attn_fwd_accum(q[:, h:], k, v, o2[:, h:], l2[:, :, h:], init=True, causal=False)
    ops.flash_attn_fwd_accum(q[:, h:], k, v, o2[:, h:], l2[:, :, h:], init=False, causal=False)  # same block twice
    ro2, rl2 = orc.attention_ref(q[:, h:].cpu(), k.cpu(), v.cpu())
    check_out(o2[:, h:], ro2, dtype)                             # merging a block with itself leaves O unchanged
    assert (l2[:, :, h:].cpu() - (rl2 + math.log(2.0))).abs().max().item() <= LSE_MAX_ABS   # and adds ln 2 to the LSE
    assert torch.all(o2[:, :h] == 0) and torch.all(torch.isinf(l2[:, :, :h]))               # other rows untouched


def test_fa_fwd_strided_bhsd_views(ops):
    # the ring / TP internals hold [B,H,S,D]; the kernel takes any (batch, seq, head) strides
    B, H, S, D = 2, 4, 256, 128
    g = torch.Generator(device="cuda").manual_seed(5)
    q, k, v = (torch.randn(B, H, S, D, device="cuda", dtype=torch.bfloat16, generator=g) for _ in range(3))
    o = ops.flash_attn_fwd(q.transpose(1, 2), k.transpose(1, 2), v.transpose(1, 2), causal=True)
    ro, _ = orc.attention_ref(q.transpose(1, 2).cpu(), k.transpose(1, 2).cpu(), v.transpose(1, 2).cpu(), causal=True)
    check_out(o, ro, BF16)
    # fused qkv projection output [B,S,3*H*D] sliced into heads
    qkv = torch.randn(B, S, 3 * H * D, device="cuda", dtype=torch.bfloat16, generator=g)
    q2, k2, v2 = (t.view(B, S, H, D) for t in qkv.split(H * D, dim=-1))
    o2 = ops.flash_attn_fwd(q2, k2, v2, causal=False)
    ro2, _ = orc.attention_ref(q2.cpu(), k2.cpu(), v2.cpu())
    check_out(o2, ro2, BF16)


def test_fa_large_scores_and_lazy_rescale(ops):
    # growing scores along the key axis force many running-max updates (exercise the O rescale path)
    B, S, H, D = 1, 1024, 2, 128
    q, k, v = rand_qkv(B, S, S, H, H, D, seed=7)
    ramp = torch.linspace(0.2, 3.0, S, device="cuda").view(1, S, 1, 1)
    k = (k * ramp).to(torch.bfloat16)
    o, lse = ops.flash_attn_fwd(q, k, v, causal=False, return_lse=True)
    ro, rl = orc.attention_ref(q.cpu(), k.cpu(), v.cpu())
    check_out(o, ro, BF16, lse=lse, ref_lse=rl)


def test_fa_full_size_properties(ops):
    """BASELINE config shapes (C3: B4 S8192 H32 D128 causal) through size-independent properties: (1) a row's output
    only depends on keys <= its position, (2) splitting the keys and LSE-merging reproduces the full result,
    (3) the first 128 rows equal the small problem the oracle can check."""
    B, S, H, D = 1, 8192, 4, 128
    q, k, v = rand_qkv(B, S, S, H, H, D, seed=11)
    o, lse = ops.flash_attn_fwd(q, k, v, causal=True, return_lse=True)
    # (3) prefix equals oracle
    ro, rl = orc.attention_ref(q[:, :256].cpu(), k[:, :256].cpu(), v[:, :256].cpu(), causal=True)
    check_out(o[:, :256], ro, BF16, lse=lse[:, :, :256], ref_lse=rl)
    # (1) causality: perturbing late keys leaves early rows bit-identical
    k2, v2 = k.clone(), v.clone()
    k2[:, 4096:] = 0
    v2[:, 4096:] = 1
    o2 = ops.flash_attn_fwd(q, k2, v2, causal=True)
    assert torch.equal(o2[:, :4096], o[:, :4096])
    # (2) two key halves merged by LSE == full (rows of the last quarter, non-causal over all keys)
    qs = q[:, -512:]
    oa, la = ops.flash_attn_fwd(qs, k[:, :5000], v[:, :5000], return_lse=True)
    ob, lb = ops.flash_attn_fwd(qs, k[:, 5000:], v[:, 5000:], return_lse=True)
    of, lf = ops.flash_attn_fwd(qs, k, v, return_lse=True)
    acc = oa.float().contiguous()
    lacc = la.clone()
    ops.lse_merge(acc, lacc, ob, lb)
    check_out(acc, of.float(), BF16)
    assert (lacc - lf).abs().max().item() <= 1e-3


def test_lse_merge_and_cast(ops):
    torch.manual_seed(0)
    B, S, H, D = 2, 200, 4, 128
    oa, la = torch.randn(B, S, H, D, device="cuda"), torch.randn(B, H, S, device="cuda")
    ob, lb = torch.randn(B, S, H, D, device="cuda", dtype=torch.bfloat16), torch.randn(B, H, S, device="cuda")
    la[0, 0, :5] = float("-inf")
    lb[0, 1, :5] = float("-inf")
    la[1, 2, :3] = float("-inf")
    lb[1, 2, :3] = float("-inf")
    ro, rl = orc.lse_merge_ref(oa.cpu(), la.cpu(), ob.cpu(), lb.cpu())
    ops.lse_merge(oa, la, ob, lb)
    assert (oa.cpu() - ro).abs().max().item() <= 1e-5
    check_lse(la, rl)
    out = ops.cast_out(oa, torch.bfloat16)
    assert torch.equal(out.cpu(), oa.cpu().to(torch.bfloat16))


# ------------------------------------------------------------------------------------------ K2 decode
DECODE_CASES = [
    # B, Hq, Hkv, D, S, splits
    (2, 4, 4, 128, 300, 1),
    (3, 8, 2, 128, 1000, 0),
    (2, 4, 4, 64, 517, 3),
    (4, 8, 8, 128, 2048, 0),
    (2, 8, 1, 64, 700, 2),
    (1, 32, 8, 128, 8192, 0),   # Llama-3 GQA, long context, small batch -> many splits
    (2, 12, 12, 64, 129, 4),    # GPT-2 heads, more splits than 64-key tiles in some batches
    (2, 12, 4, 128, 500, 0),    # G = 3 (tensor-core GQA path, rows padded to 16)
    (2, 40, 8, 128, 700, 3),    # G = 5
    (1, 16, 1, 64, 333, 2),     # MQA with 16 query heads: all 16 MMA rows live
    (3, 16, 2, 128, 17, 1),     # G = 8, context shorter than two tiles
]


@pytest.mark.parametrize(*with_dtypes("B,Hq,Hkv,D,S,splits", DECODE_CASES))
def test_decode_contiguous_vs_oracle(ops, B, Hq, Hkv, D, S, splits, dtype):
    g = torch.Generator(device="cuda").manual_seed(1)
    q = torch.randn(B, Hq, D, device="cuda", dtype=dtype, generator=g)
    kc = torch.randn(B, S, Hkv, D, device="cuda", dtype=dtype, generator=g)
    vc = torch.randn(B, S, Hkv, D, device="cuda", dtype=dtype, generator=g)
    lens = torch.randint(1, S + 1, (B,), device="cuda", dtype=torch.int32, generator=g)
    lens[0] = S
    o, lse = ops.decode_attention(q, kc, vc, lens, num_splits=splits, return_lse=True)
    ro, rl = orc.decode_attention_ref(q.cpu(), kc.cpu(), vc.cpu(), lens.cpu())
    check_out(o, ro, dtype, "decode", Hkv, lse=lse, ref_lse=rl)


@pytest.mark.parametrize(*with_dtypes("B,Hq,Hkv,D,S,splits", [c for c in DECODE_CASES if c[1] // c[2] >= 3]))
def test_decode_gqa_ring_variant_vs_oracle(ops, monkeypatch, B, Hq, Hkv, D, S, splits, dtype):
    """The shared-memory-ring variant of the GQA decode kernel (B200_GQA_RING=1: per-lane cp.async staging, fragments read
    back with 128-bit shared loads; measured slower than the register-staged default, kept as an option) — same results,
    including tiles whose last rows are zero-filled."""
    monkeypatch.setenv("B200_GQA_RING", "1")
    g = torch.Generator(device="cuda").manual_seed(1)
    q = torch.randn(B, Hq, D, device="cuda", dtype=dtype, generator=g)
    kc = torch.randn(B, S, Hkv, D, device="cuda", dtype=dtype, generator=g)
    vc = torch.randn(B, S, Hkv, D, device="cuda", dtype=dtype, generator=g)
    lens = torch.randint(1, S + 1, (B,), device="cuda", dtype=torch.int32, generator=g)
    lens[0] = S
    o, lse = ops.decode_attention(q, kc, vc, lens, num_splits=splits, return_lse=True)
    ro, rl = orc.decode_attention_ref(q.cpu(), kc.cpu(), vc.cpu(), lens.cpu())
    check_out(o, ro, dtype, "decode", Hkv, lse=lse, ref_lse=rl)
    monkeypatch.setenv("B200_GQA_RING", "0")
    o0, lse0 = ops.decode_attention(q, kc, vc, lens, num_splits=splits, return_lse=True)
    assert (o.float() - o0.float()).abs().max().item() <= 2e-2


def test_decode_paged_and_kv_append(ops):
    g = torch.Generator(device="cuda").manual_seed(2)
    B, Hq, Hkv, D, bs, L, nblk = 3, 8, 4, 128, 16, 2, 64
    kc = torch.randn(nblk, L, bs, Hkv, D, device="cuda", dtype=torch.bfloat16, generator=g)
    vc = torch.randn(nblk, L, bs, Hkv, D, device="cuda", dtype=torch.bfloat16, generator=g)
    lens = torch.tensor([37, 256, 129], device="cuda", dtype=torch.int32)
    tables = torch.randperm(nblk)[:B * 16].view(B, 16).to(device="cuda", dtype=torch.int32)
    q = torch.randn(B, Hq, D, device="cuda", dtype=torch.bfloat16, generator=g)
    # append the new token first (the reference order: reshape_and_cache, then attention)
    key = torch.randn(B, Hkv, D, device="cuda", dtype=torch.bfloat16, generator=g)
    val = torch.randn(B, Hkv, D, device="cuda", dtype=torch.bfloat16, generator=g)
    rk, rv = kc.cpu().clone(), vc.cpu().clone()
    ops.kv_append(key, val, kc, vc, lens, block_tables=tables, layer_idx=1)
    orc.kv_append_ref(key.cpu(), val.cpu(), rk, rv, lens.cpu(), tables.cpu(), 1)
    assert torch.equal(kc.cpu(), rk) and torch.equal(vc.cpu(), rv)  # bit-exact byte movement
    o, lse = ops.decode_attention(q, kc, vc, lens, block_tables=tables, layer_idx=1, return_lse=True)
    ro, rl = orc.decode_attention_ref(q.cpu(), rk, rv, lens.cpu(), block_tables=tables.cpu(), layer_idx=1)
    check_out(o, ro, BF16, "decode", Hkv, lse=lse, ref_lse=rl)


@pytest.mark.parametrize("D", [32, 80, 96])
def test_paged_cache_with_narrow_heads(ops, D):
    """Head dims the decode kernels are not built for live in the next wider cache (ops.cache_head_dim) with zero columns
    behind them: kv_append writes the padded token bit-exactly, decode and short-q attention on the narrow q equal the oracle
    on the narrow tensors, with the softmax scale of the REAL head_dim."""
    g = torch.Generator(device="cuda").manual_seed(D)
    Dp = ops.cache_head_dim(D)
    assert Dp == (64 if D <= 64 else 128)
    B, Hq, Hkv, bs, L, nblk = 2, 8, 2, 16, 2, 40
    r = lambda *shape: torch.randn(*shape, device="cuda", dtype=torch.bfloat16, generator=g)
    kc, vc = torch.zeros(nblk, L, bs, Hkv, Dp, device="cuda", dtype=torch.bfloat16), torch.zeros(nblk, L, bs, Hkv, Dp, device="cuda", dtype=torch.bfloat16)
    kc[..., :D], vc[..., :D] = r(nblk, L, bs, Hkv, D), r(nblk, L, bs, Hkv, D)
    lens = torch.tensor([37, 250], device="cuda", dtype=torch.int32)
    tables = torch.randperm(nblk)[:B * 16].view(B, 16).to(device="cuda", dtype=torch.int32)
    key, val = r(B, Hkv, D), r(B, Hkv, D)
    ops.kv_append(key, val, kc, vc, lens, block_tables=tables, layer_idx=1)
    rk, rv = kc[..., :D].cpu().clone(), vc[..., :D].cpu().clone()        # narrow reference cache, after the append
    for b in range(B):
        pos = int(lens[b]) - 1
        blk = int(tables[b, pos // bs])
        assert torch.equal(kc[blk, 1, pos % bs, :, :D], key[b]) and kc[blk, 1, pos % bs, :, D:].abs().sum() == 0
        assert torch.equal(vc[blk, 1, pos % bs, :, :D], val[b])
    q = r(B, Hq, D)
    o, lse = ops.decode_attention(q, kc, vc, lens, block_tables=tables, layer_idx=1, return_lse=True)
    assert o.shape == (B, Hq, D)
    ro, rl = orc.decode_attention_ref(q.cpu(), rk, rv, lens.cpu(), block_tables=tables.cpu(), layer_idx=1)
    check_out(o, ro, BF16, "decode", Hkv, lse=lse, ref_lse=rl)
    Sq = 24
    q4 = r(B, Sq, Hq, D)
    o4 = ops.paged_prefill_attention(q4, kc, vc, tables, lens, layer_idx=1, causal=True)
    assert o4.shape == (B, Sq, Hq, D)
    for b in range(B):
        n = int(lens[b])
        idx = torch.arange(n)
        kb = rk[tables[b].cpu().long()[idx // bs], 1, idx % bs][None]
        vb = rv[tables[b].cpu().long()[idx // bs], 1, idx % bs][None]
        ref, _ = orc.attention_ref(q4[b:b + 1].cpu(), kb, vb, causal=True, causal_offset=n - Sq)
        check_out(o4[b:b + 1], ref, BF16)
    # contiguous cache, same rule
    kcc, vcc = torch.zeros(B, 300, Hkv, Dp, device="cuda", dtype=torch.bfloat16), torch.zeros(B, 300, Hkv, Dp, device="cuda", dtype=torch.bfloat16)
    kn, vn = r(B, 300, Hkv, D), r(B, 300, Hkv, D)
    kcc[..., :D], vcc[..., :D] = kn, vn
    oc = ops.decode_attention(q, kcc, vcc, lens)
    roc, _ = orc.decode_attention_ref(q.cpu(), kn.cpu(), vn.cpu(), lens.cpu())
    check_out(oc, roc, BF16, "decode", Hkv)


@pytest.mark.parametrize(*with_dtypes("Sq,Hq,Hkv,D,block_size,causal", [
    (64, 8, 8, 128, 16, True),      # the reference's BLOCK_SIZE_M = 64 case
    (200, 8, 2, 128, 16, True),     # GQA, q tile pair partly empty, ragged context lengths
    (300, 4, 4, 64, 32, True),      # D = 64, two q tiles + a third partial
    (48, 4, 1, 128, 8, False),      # MQA, smallest block; the reference kernel as written (no causal mask)
    (128, 4, 4, 128, 128, True),    # one physical block per KV tile
]))
def test_paged_short_q_attention_vs_oracle(ops, Sq, Hq, Hkv, D, block_size, causal, dtype):
    """VERDICT r1 missing #4: q_len > 1 against the paged cache (chunked prefill) — K1 gathering K/V through the block
    table, vs the oracle's gather + exact attention with the diagonal ending at each sequence's last key."""
    B, L, layer = 3, 2, 1
    g = torch.Generator(device="cuda").manual_seed(11)
    ctx = torch.tensor([Sq + 517, Sq, Sq + 130], dtype=torch.int32)       # includes a sequence with no history at all
    max_blocks = (int(ctx.max()) + block_size - 1) // block_size + 1
    num_blocks = B * max_blocks + 3
    kc = torch.randn(num_blocks, L, block_size, Hkv, D, device="cuda", dtype=dtype, generator=g)
    vc = torch.randn(num_blocks, L, block_size, Hkv, D, device="cuda", dtype=dtype, generator=g)
    perm = torch.randperm(num_blocks, generator=torch.Generator().manual_seed(5))[:B * max_blocks]
    bt = perm.view(B, max_blocks).to(torch.int32)                           # scattered, non-monotonic physical blocks
    q = torch.randn(B, Sq, Hq, D, device="cuda", dtype=dtype, generator=g)
    o, lse = ops.paged_prefill_attention(q, kc, vc, bt.cuda(), ctx.cuda(), layer_idx=layer, causal=causal, return_lse=True)
    assert ops.last_kernel() == "fa_fwd_kernel"
    ro, rl = orc.paged_prefill_attention_ref(q.cpu(), kc.cpu(), vc.cpu(), bt, ctx, layer_idx=layer, causal=causal)
    check_out(o, ro, dtype, lse=lse, ref_lse=rl)
    # the functional shim of the reference signature ([B,H,q,D] in and out) goes the same way
    from ml_inference_optimizer_b200.kernels.triton.attention_kernels import triton_paged_attention_forward
    out = torch.empty(B, Hq, Sq, D, device="cuda", dtype=dtype)
    triton_paged_attention_forward(q.transpose(1, 2).contiguous(), out, kc, vc, bt.cuda(), ctx.cuda(), block_size, max_blocks * block_size,
                                   layer, causal=causal)
    assert torch.equal(out.transpose(1, 2), o)
    if causal:  # the last query row is exactly a decode step over the same cache
        od = ops.decode_attention(q[:, -1].contiguous(), kc, vc, ctx.cuda(), block_tables=bt.cuda(), layer_idx=layer)
        assert (od.float() - o[:, -1].float()).abs().max().item() <= 2e-2


def test_kv_append_and_decode_clamp_overlong_lengths(ops):
    """ADVICE r1: device-side lengths past the cache capacity (e.g. advanced under a CUDA graph) must neither write into
    another sequence's block nor read past the block table."""
    B, Hkv, D, bs, nblk = 2, 2, 64, 16, 3
    kc = torch.zeros(B * nblk, 1, bs, Hkv, D, device="cuda", dtype=torch.bfloat16)
    vc = torch.zeros_like(kc)
    bt = torch.arange(B * nblk, dtype=torch.int32, device="cuda").view(B, nblk)
    k = torch.ones(B, Hkv, D, device="cuda", dtype=torch.bfloat16)
    lens = torch.tensor([nblk * bs + 5, 7], device="cuda", dtype=torch.int32)   # sequence 0 ran past its 48 slots
    ops.kv_append(k, k, kc, vc, lens, bt, 0)
    assert kc[:nblk].abs().sum().item() == 0 and kc[nblk:].abs().sum().item() == Hkv * D   # only sequence 1's token landed
    assert kc[nblk, 0, 6].abs().sum().item() == Hkv * D
    q = torch.randn(B, 4, D, device="cuda", dtype=torch.bfloat16)
    o = ops.decode_attention(q, kc, vc, lens, block_tables=bt)                 # clamped to 48 keys: finite, no fault
    torch.cuda.synchronize()
    assert torch.isfinite(o.float()).all()
    kcc = torch.zeros(B, 8, Hkv, D, device="cuda", dtype=torch.bfloat16)
    lens2 = torch.tensor([9, 8], device="cuda", dtype=torch.int32)             # contiguous cache of 8 slots
    ops.kv_append(k, k, kcc, kcc.clone(), lens2)
    assert kcc[0].abs().sum().item() == 0 and kcc[1, 7].abs().sum().item() == Hkv * D
    with pytest.raises(ValueError):
        ops.kv_append(k, k, kc, vc, lens.long(), bt, 0)
    with pytest.raises(ValueError):
        ops.kv_append(k, k, kc, vc, lens, bt[:1], 0)


def test_decode_equals_last_prefill_row(ops):
    B, S, Hq, Hkv, D = 2, 1024, 8, 2, 128
    q, k, v = rand_qkv(B, S, S, Hq, Hkv, D, seed=3)
    o_pre, lse_pre = ops.flash_attn_fwd(q, k, v, causal=True, return_lse=True)
    lens = torch.full((B,), S, device="cuda", dtype=torch.int32)
    o_dec, lse_dec = ops.decode_attention(q[:, -1].contiguous(), k, v, lens, return_lse=True)
    assert (o_dec.float() - o_pre[:, -1].float()).abs().max().item() <= 1e-2
    assert (lse_dec - lse_pre[:, :, -1]).abs().max().item() <= 1e-3


def test_decode_full_size_property(ops):
    """C3 decode shape (B64, 8K context, 32 heads, D128 — 8.6 GB of KV) checked by a size-independent property:
    constant V rows give exactly that constant back, and LSE equals log(context_len) for zero queries."""
    B, S, H, D = 64, 8192, 32, 128
    kc = torch.randn(B, S, H, D, device="cuda", dtype=torch.bfloat16)
    vc = torch.empty(B, S, H, D, device="cuda", dtype=torch.bfloat16)
    vc[:] = torch.arange(D, device="cuda", dtype=torch.float32).mul(1 / 64).to(torch.bfloat16)
    q = torch.zeros(B, H, D, device="cuda", dtype=torch.bfloat16)
    lens = torch.randint(4096, S + 1, (B,), device="cuda", dtype=torch.int32)
    o, lse = ops.decode_attention(q, kc, vc, lens, return_lse=True)
    expect = torch.arange(D, device="cuda", dtype=torch.float32).mul(1 / 64).to(torch.bfloat16).float()
    assert (o.float() - expect).abs().max().item() <= 2e-2
    assert (lse - lens.float().log().view(B, 1)).abs().max().item() <= 1e-3


# ------------------------------------------------------------------------------------------ K3 FusedMLP
def make_mlp(T, h, i, act, seed=0, bias=True, std=0.02, dtype=BF16):
    g = torch.Generator(device="cuda").manual_seed(seed)
    r = lambda *s, sc=1.0: (torch.randn(*s, device="cuda", generator=g) * sc).to(dtype)
    x = r(T, h)
    wu, wd = r(i, h, sc=std), r(h, i, sc=std)
    bu, bd = (r(i, sc=0.1), r(h, sc=0.1)) if bias else (None, None)
    wg = bg = None
    if act == "swiglu":
        wg = r(i, h, sc=std)
        bg = r(i, sc=0.1) if bias else None
    return x, wu, bu, wd, bd, wg, bg


MLP_CASES = [
    (512, 768, 3072, "gelu_tanh", True),     # GPT-2 layer shape, reduced T
    (1024, 1024, 2816, "swiglu", True),
    (77, 256, 512, "relu", True),            # ragged T
    (256, 512, 1024, "gelu", True),          # exact erf GELU (bare FusedMLP)
    (300, 4096, 11008, "swiglu", False),     # Llama-2 layer shape, bias-less (HF Llama)
    (1, 768, 3072, "gelu_tanh", True),       # single token
    (130, 264, 520, "swiglu", True),         # nothing a multiple of the tile
    (64, 4096, 11008, "swiglu", True),       # decode-sized T at Llama-2 widths: split-K path in both GEMMs
    (8, 768, 3072, "gelu_tanh", True),       # decode-sized T at GPT-2 widths
]


@pytest.mark.parametrize(*with_dtypes("T,h,i,act,bias", MLP_CASES))
def test_fused_mlp_vs_oracle(ops, T, h, i, act, bias, dtype):
    x, wu, bu, wd, bd, wg, bg = make_mlp(T, h, i, act, bias=bias, dtype=dtype)
    y = ops.fused_mlp(x, wu, bu, wd, bd, act, wg, bg)
    c = lambda t: None if t is None else t.cpu()
    ref = orc.mlp_ref(c(x), c(wu), c(bu), c(wd), c(bd), act, c(wg), c(bg))
    check_out(y, ref, dtype, "2d")


FUSED_LAUNCH_CASES = [
    # T, h, i, act, bias — prefill-sized (T >= 1024): one launch, up(+gate) and down projection interleaved by row groups
    (1024, 512, 1408, "swiglu", True),
    (1500, 768, 3072, "gelu_tanh", True),      # ragged last row-block, GPT-2 widths (intermediate L2-resident mode)
    (4096 + 77, 512, 1376, "swiglu", False),   # the tensor-parallel shard width of C3 at tp=8, ragged T, bias-less
    (2048, 1024, 4096, "relu", True),
    (8192, 768, 3072, "gelu", True),           # several row groups: P1 -> P2 dependency counters cross group boundaries
    (2304, 264, 520, "swiglu", True),          # nothing a multiple of the tile
]


@pytest.mark.parametrize(*with_dtypes("T,h,i,act,bias", FUSED_LAUNCH_CASES))
def test_fused_mlp_single_launch_vs_oracle_and_two_launch(ops, T, h, i, act, bias, dtype, monkeypatch):
    """Row a6: fused_mlp_pair_kernel (ONE launch; the bf16 intermediate is handed from the up to the down projection
    through per-row-block counters) against the oracle, and bit-identical to the two-launch path on the same tiles."""
    x, wu, bu, wd, bd, wg, bg = make_mlp(T, h, i, act, bias=bias, dtype=dtype)
    monkeypatch.setenv("B200_MLP_FUSED", "1")
    y = ops.fused_mlp(x, wu, bu, wd, bd, act, wg, bg)
    assert ops.last_gemm_kernel().startswith("fused_mlp_pair_kernel")
    for g, lag in ((1, 1), (2, 3), (3, 1)):   # stress the tile list: tiny groups, long and short P1 -> P2 lags
        monkeypatch.setenv("B200_FUSED_G", str(g)); monkeypatch.setenv("B200_FUSED_LAG", str(lag))
        assert torch.equal(ops.fused_mlp(x, wu, bu, wd, bd, act, wg, bg), y), f"group {g} lag {lag} changes the result"
    monkeypatch.setenv("B200_FUSED_G", "0"); monkeypatch.setenv("B200_FUSED_LAG", "0")
    monkeypatch.setenv("B200_MLP_FUSED", "0")
    y2 = ops.fused_mlp(x, wu, bu, wd, bd, act, wg, bg)
    two = ops.last_gemm_kernel()
    assert not two.startswith("fused_mlp")
    if two.startswith("gemm_act_pair_kernel"):   # same 256x256 tiles, same k order: bit-identical
        assert torch.equal(y, y2)
    c = lambda t: None if t is None else t.cpu()
    ref = orc.mlp_ref(c(x), c(wu), c(bu), c(wd), c(bd), act, c(wg), c(bg))
    check_out(y, ref, dtype, "2d")


def test_fused_mlp_single_launch_repeated_calls_and_streams(ops, monkeypatch):
    """The dependency counters live in the caller's workspace and are re-zeroed per launch: back-to-back calls (same
    workspace) and a call on a side stream must all give the same bits."""
    monkeypatch.setenv("B200_MLP_FUSED", "1")
    x, wu, bu, wd, bd, wg, bg = make_mlp(3000, 512, 1024, "swiglu", bias=True)
    ys = [ops.fused_mlp(x, wu, bu, wd, bd, "swiglu", wg, bg) for _ in range(5)]
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        ys.append(ops.fused_mlp(x, wu, bu, wd, bd, "swiglu", wg, bg))
    torch.cuda.synchronize()
    for y in ys[1:]:
        assert torch.equal(y, ys[0])


@pytest.mark.parametrize(*with_dtypes("act", [None, "gelu_tanh", "gelu", "relu", "swiglu"]))
def test_linear_act_vs_oracle(ops, act, dtype):
    T, K, N = 300, 768, 1024
    x, w, b, _, _, wg, bg = make_mlp(T, K, N, act or "relu", seed=4, std=0.05, dtype=dtype)
    y = ops.linear_act(x, w, b, act, wg, bg)
    c = lambda t: None if t is None else t.cpu()
    ref = orc.linear_act_ref(c(x), c(w), c(b), act, c(wg), c(bg))
    check_out(y, ref, dtype, "2d")


def test_fused_mlp_golden_reference_vectors(ops, golden_dir):
    """The reference's own module outputs (tests/golden, generated by running the reference on CPU)."""
    vecs = torch.load(os.path.join(golden_dir, "mlp_reference_vectors.pt"))
    for name, act in (("FusedTransformerMLP_gelu", "gelu_tanh"), ("FusedTransformerMLP_relu", "relu"),
                      ("FusedTransformerMLP_swiglu", "swiglu")):
        d = vecs[name]
        sd = {k: v.to("cuda", torch.bfloat16) for k, v in d["state_dict"].items()}
        y = ops.fused_mlp(d["x"].to("cuda", torch.bfloat16), sd["mlp.fc1.weight"], sd["mlp.fc1.bias"], sd["mlp.fc2.weight"],
                          sd["mlp.fc2.bias"], act, sd.get("mlp.fc1_gate.weight"), sd.get("mlp.fc1_gate.bias"))
        check_out(y, d["y"], BF16, "2d", mean_rel=2e-2, max_rel=3e-2)  # inputs themselves are rounded to bf16 here


def test_attention_golden_reference_vectors(ops, golden_dir):
    vecs = torch.load(os.path.join(golden_dir, "attention_reference_vectors.pt"))
    for name, causal in (("ring_fallback_noncausal", False), ("ring_fallback_causal_finite_mask", True),
                         ("ring_fallback_cross", False)):
        d = vecs[name]
        q, k, v = (d[n].permute(0, 2, 1, 3).to("cuda", torch.bfloat16) for n in ("q", "k", "v"))
        o = ops.flash_attn_fwd(q, k, v, causal=causal)
        B, S, H, D = o.shape
        check_out(o.reshape(B, S, H * D), d["y"], BF16, "2d", mean_rel=2e-2, max_rel=3e-2)


def test_mlp_full_size_linearity(ops):
    """C3 MLP shape (T=32768, 4096 -> 11008 SwiGLU) checked by properties: rows are independent (a row block equals
    the same rows computed alone) and the down projection is linear in the intermediate (zero W_down -> bias)."""
    T, h, i = 32768, 4096, 11008
    x, wu, bu, wd, bd, wg, bg = make_mlp(T, h, i, "swiglu", seed=9)
    y = ops.fused_mlp(x, wu, bu, wd, bd, "swiglu", wg, bg)
    rows = slice(20000, 20256)
    y_rows = ops.fused_mlp(x[rows].contiguous(), wu, bu, wd, bd, "swiglu", wg, bg)
    # the 256-row problem takes the split-K path (different fp32 summation order): equal up to bf16 rounding
    assert (y[rows].float() - y_rows.float()).abs().max().item() <= 2e-2 * max(1.0, y_rows.float().abs().max().item() / 4)
    c = lambda t: t.cpu()
    ref = orc.mlp_ref(c(x[rows]), c(wu), c(bu), c(wd), c(bd), "swiglu", c(wg), c(bg))
    check_out(y_rows, ref, BF16, "2d")
    y0 = ops.fused_mlp(x[:512].contiguous(), wu, bu, torch.zeros_like(wd), bd, "swiglu", wg, bg)
    assert torch.equal(y0, bd.view(1, -1).expand(512, -1))  # zero weights: exactly the bias on every path


# ------------------------------------------------------------------------------------------ LayerNorm (f3)
@pytest.mark.parametrize(*with_dtypes("rows,cols,res,bias", [(300, 768, False, True), (257, 4096, True, True), (5, 8192, True, False),
                                                (1, 64, False, True), (1000, 1032, True, True),
                                                # persistent CTA-per-row kernel: more rows than resident CTAs (several
                                                # rows per CTA with the next row prefetched), every ITERS instantiation,
                                                # ragged widths, with and without residual
                                                (3001, 2048, True, True), (2500, 2056, False, False), (1777, 4104, True, True),
                                                (1300, 6152, False, True), (1201, 8192, False, True), (700, 3000, True, False)]))
def test_layernorm_vs_oracle(ops, rows, cols, res, bias, dtype):
    g = torch.Generator(device="cuda").manual_seed(3)
    r = lambda *s: torch.randn(*s, device="cuda", generator=g).to(dtype)
    x, w = r(rows, cols) * 2 + 0.5, r(cols)
    b = r(cols) if bias else None
    rs = r(rows, cols) if res else None
    y = ops.layernorm(x, w, b, 1e-5, rs, 0.7)
    c = lambda t: None if t is None else t.cpu()
    ref = orc.layernorm_ref(c(x), c(w), c(b), 1e-5, c(rs), 0.7)
    check_out(y, ref, dtype, "2d")


def test_layernorm_golden_and_shim(ops, golden_dir):
    from kernels.triton.layernorm_kernels import triton_layernorm

    vecs = torch.load(os.path.join(golden_dir, "layernorm_reference_vectors.pt"))
    d = vecs["pytorch_layernorm_residual"]
    cu = lambda t: t.to("cuda", torch.bfloat16)
    y = triton_layernorm(cu(d["x"]), cu(d["w"]), cu(d["b"]), d["eps"], cu(d["r"]), d["alpha"])
    assert y.shape == d["y"].shape
    check_out(y, d["y"], BF16, "2d", mean_rel=1e-2, max_rel=2e-2)  # inputs rounded to bf16 (|y| up to 6)


# ------------------------------------------------------------------------------------------ guard rows (own bounds checks)
def _guarded(shape, dtype, rows_dim, guard=3, fill=-7.0):
    """A tensor of `shape` that is a view into a larger buffer with `guard` sentinel slices before and after along rows_dim."""
    big_shape = list(shape)
    big_shape[rows_dim] += 2 * guard
    big = torch.full(big_shape, fill, device="cuda", dtype=dtype)
    idx = [slice(None)] * len(shape)
    idx[rows_dim] = slice(guard, guard + shape[rows_dim])
    return big, big[tuple(idx)], idx


def _guards_untouched(big, idx, rows_dim, guard=3, fill=-7.0):
    lo = [slice(None)] * big.dim(); hi = [slice(None)] * big.dim()
    lo[rows_dim] = slice(0, guard); hi[rows_dim] = slice(big.shape[rows_dim] - guard, None)
    return bool((big[tuple(lo)] == fill).all()) and bool((big[tuple(hi)] == fill).all())


@pytest.mark.parametrize(*with_dtypes("pair", ["0", "1"]))
def test_kernels_write_only_their_rows(ops, monkeypatch, pair, dtype):
    """Outputs are views into larger buffers with sentinel rows on both sides: ragged row counts (partial last tiles, more
    rows than resident CTAs, persistent loops with a prefetched next row) must not write a byte outside their rows —
    attention (both prefill kernels), GQA decode (both staging variants), LayerNorm (warp and CTA kernels), linear."""
    monkeypatch.setenv("B200_FA_PAIR", pair)
    monkeypatch.setenv("B200_GQA_RING", pair)
    bf = dtype
    # prefill attention: the sequence dimension is guarded ([B, S, H, D] view with the same strides as the buffer)
    q, k, v = rand_qkv(2, 333, 333, 4, 2, 128, dtype, seed=9)
    big, out, idx = _guarded((2, 333, 4, 128), bf, rows_dim=1)
    ops.flash_attn_fwd(q, k, v, causal=True, out=out)
    ro, _ = orc.attention_ref(q.cpu(), k.cpu(), v.cpu(), causal=True)
    check_out(out, ro, dtype)
    assert _guards_untouched(big, idx, 1)
    # decode (GQA 4:1): the batch dimension is guarded
    g = torch.Generator(device="cuda").manual_seed(4)
    qd = torch.randn(3, 16, 128, device="cuda", dtype=bf, generator=g)
    kc = torch.randn(3, 777, 4, 128, device="cuda", dtype=bf, generator=g); vc = torch.randn_like(kc)
    lens = torch.tensor([777, 1, 300], device="cuda", dtype=torch.int32)
    big, out, idx = _guarded((3, 16, 128), bf, rows_dim=0)
    ops.decode_attention(qd, kc, vc, lens, out=out)
    rd, _ = orc.decode_attention_ref(qd.cpu(), kc.cpu(), vc.cpu(), lens.cpu())
    check_out(out, rd, dtype, "decode", 4)
    assert _guards_untouched(big, idx, 0)
    # LayerNorm: warp-per-row (768), CTA-per-row with more rows than resident CTAs (4104 columns, ragged width)
    for rows, cols in ((1237, 768), (2111, 4104), (999, 2048)):
        x = torch.randn(rows, cols, device="cuda", dtype=bf); r_ = torch.randn_like(x)
        w_ = torch.randn(cols, device="cuda", dtype=bf); b_ = torch.randn(cols, device="cuda", dtype=bf)
        big, out, idx = _guarded((rows, cols), bf, rows_dim=0)
        ops.layernorm(x, w_, b_, 1e-5, residual=r_, out=out)
        ref = orc.layernorm_ref(x.cpu(), w_.cpu(), b_.cpu(), 1e-5, r_.cpu(), 1.0)
        check_out(out, ref, dtype, "2d")
        assert _guards_untouched(big, idx, 0)
    # linear (ragged T: the last 128-row tile is partial; TMA store clips)
    x = torch.randn(300, 512, device="cuda", dtype=bf); w_ = (torch.randn(1024, 512, device="cuda") * 0.05).to(bf)
    big, out, idx = _guarded((300, 1024), bf, rows_dim=0)
    ops.linear_act(x, w_, None, None, out=out)
    ref = x.float().cpu() @ w_.float().cpu().t()
    check_out(out, ref, dtype, "2d")
    assert _guards_untouched(big, idx, 0)
