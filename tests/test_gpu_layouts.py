"""Operand layouts the C-ABI accepts besides dense ``randn`` tensors, with the memory around every operand poisoned.

Every operand here is a view into a larger buffer (row strides wider than the row, batch / head / sequence gaps, interleaved
and time-major KV caches, paged caches with padding slots, unused blocks and other layers). Whatever an operation must not
read holds NaN or +Inf, so a read of the wrong row, block or layer cannot hide inside a tolerance; whatever it must not write
holds a finite sentinel, compared bit for bit afterwards. Each case is checked twice:

  (a) tile by tile against the fp32 oracle at the thresholds of test_gpu_parity.py, the oracle receiving only the logical
      values of each view;
  (b) bit for bit against the same call on dense copies: the same kernel, the same split count and the same tiling, so a
      wrong stride or a read past the end changes bits.

Keys past ``kv_lens`` / ``context_lens`` must never affect a result: the padding rows are poisoned too, and the result must
equal the call with those rows zeroed. The last group pins the ``out=`` contract of the wrappers: an ``out`` either receives
the result or the call raises ValueError.

GPU tests are marked one by one; the helpers' self-test runs without a GPU.
"""
import pytest
import torch

from oracle import attn_mlp_oracle as orc
from test_gpu_parity import BF16, DTYPES, FP16, check_lse, check_out, make_mlp, rand_qkv

gpu = pytest.mark.gpu
DT_IDS = {BF16: "bf16", FP16: "fp16"}
NAN, INF = float("nan"), float("inf")
FILLS = [NAN, INF]
FILL_IDS = {NAN: "nan", INF: "inf"}.get
SENTINEL = -3.25                  # what output buffers hold outside the view (exact in bf16, fp16 and fp32)
INT_VIEW = {1: torch.uint8, 2: torch.int16, 4: torch.int32, 8: torch.int64}


@pytest.fixture(scope="module")
def ops(built_lib):
    assert torch.cuda.is_available(), "gpu tests need CUDA"
    from ml_inference_optimizer_b200 import ops as _ops

    assert _ops.arch_ok(), "gpu tests need an sm_100 device"
    return _ops


# ------------------------------------------------------------------------------------------------- helpers
def poisoned_view(shape, dtype, pads, fill, values=None, device="cuda"):
    """A ``shape`` view into a larger buffer whose every element outside the view holds ``fill``. ``pads[i]`` is the extra
    extent of dimension i: an int (after the view) or ``(before, after)``. Returns ``(view, buffer)``; ``values`` fills the
    view."""
    pads = [(0, p) if isinstance(p, int) else tuple(p) for p in pads]
    assert len(pads) == len(shape)
    buf = torch.full([n + a + b for n, (a, b) in zip(shape, pads)], fill, dtype=dtype, device=device)
    view = buf[tuple(slice(a, a + n) for n, (a, _) in zip(shape, pads))]
    if values is not None:
        view.copy_(values)
    return view, buf


def _bits(t):
    return t.contiguous().view(INT_VIEW[t.element_size()])


def same_bits(a, b):
    """Equal shapes, dtypes and bit patterns (NaN compares equal to the same NaN)."""
    return a.shape == b.shape and a.dtype == b.dtype and torch.equal(_bits(a).cpu(), _bits(b).cpu())


def untouched(buf, view, fill):
    """True if every element of the contiguous ``buf`` outside ``view`` still holds ``fill``, compared bit for bit."""
    assert buf.is_contiguous()
    idx = torch.arange(buf.numel(), device=buf.device).as_strided(view.shape, view.stride(),
                                                                  view.storage_offset() - buf.storage_offset())
    outside = torch.ones(buf.numel(), dtype=torch.bool, device=buf.device)
    outside[idx.reshape(-1)] = False
    want = _bits(torch.tensor([fill], dtype=buf.dtype)).to(buf.device)
    return bool((_bits(buf).reshape(-1)[outside] == want).all())


def logical(t):
    """What the oracle receives: the values of the view only."""
    return t.clone().cpu()


# ------------------------------------------------------------------------------------------------- CPU self-test
def test_poisoned_view_and_untouched_self_test():
    """The gaps hold the poison and the view holds the given values; ``untouched`` passes an untouched buffer (a NaN fill
    included, which a float comparison would reject) and catches one stray write, a NaN written among finite sentinels
    included."""
    vals = torch.randn(3, 5, 2, 16).to(BF16)
    for fill in (NAN, INF, SENTINEL):
        view, buf = poisoned_view(vals.shape, BF16, ((1, 2), 3, (0, 1), (0, 8)), fill, values=vals, device="cpu")
        assert view.shape == vals.shape and buf.shape == (6, 8, 3, 24)
        assert view.data_ptr() != buf.data_ptr() and same_bits(logical(view), vals)
        assert untouched(buf, view, fill)
        mask = torch.ones(buf.shape, dtype=torch.bool)
        mask[1:4, :5, :2, :16] = False
        gaps = buf[mask]
        assert gaps.numel() == buf.numel() - vals.numel()
        assert (torch.isnan(gaps).all() if fill != fill else (gaps == fill).all())
        for stray in ((0, 0, 0, 0), (5, 7, 2, 23), (2, 1, 1, 16), (3, 5, 0, 3)):   # corners, one past the row, past the seq
            for value in (0.0, NAN):
                if fill != fill and value != value:
                    continue
                b2 = buf.clone()
                v2 = b2[1:4, :5, :2, :16]
                b2[stray] = value
                assert not untouched(b2, v2, fill), (fill, stray, value)
        view[1, 2, 1, 3] = 0.0                          # writes inside the view are not its business
        assert untouched(buf, view, fill)
    acc, abuf = poisoned_view((2, 3, 4), torch.float32, (1, (2, 0), 4), SENTINEL, device="cpu")
    assert untouched(abuf, acc, SENTINEL)
    abuf.view(torch.int32)[0, 0, 7] = 0x7FC00001       # a NaN with a payload
    assert not untouched(abuf, acc, SENTINEL)


# ------------------------------------------------------------------------------------------------- 1. prefill
def _fa_name(pair):
    return "fa_fwd_pair_kernel" if pair else "fa_fwd_kernel"


@gpu
@pytest.mark.parametrize("fill", FILLS, ids=FILL_IDS)
@pytest.mark.parametrize("D", [64, 128, 80])
@pytest.mark.parametrize("pair", [False, True])
@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS.get)
def test_prefill_strided_operands(ops, monkeypatch, dtype, pair, D, fill):
    """q / k / v with poisoned batch, sequence and head gaps and poisoned columns past D; out, o_acc and lse_acc as views
    of sentinel buffers. Plain output (with LSE) and two accumulate steps over key slices of the poisoned views."""
    monkeypatch.setenv("B200_FA_PAIR", "1" if pair else "0")
    name = _fa_name(pair)
    B, Sq, Sk, Hq, Hkv = 2, 300, 420, 4, 2
    coff = Sk - Sq - 150                                # the first rows see no key
    q0, k0, v0 = rand_qkv(B, Sq, Sk, Hq, Hkv, D, dtype, seed=D + pair)
    q, _ = poisoned_view(q0.shape, dtype, ((1, 1), (2, 3), (0, 1), 8), fill, values=q0)
    k, _ = poisoned_view(k0.shape, dtype, (1, (1, 5), (1, 1), 16), fill, values=k0)
    v, _ = poisoned_view(v0.shape, dtype, ((1, 0), (3, 2), 2, 8), fill, values=v0)
    ro, rl = orc.attention_ref(logical(q), logical(k), logical(v), causal=True, causal_offset=coff)
    dense = [t.contiguous() for t in (q, k, v)]

    out, obuf = poisoned_view((B, Sq, Hq, D), dtype, (1, (1, 2), (1, 0), 8), SENTINEL)
    o, lse = ops.flash_attn_fwd(q, k, v, causal=True, causal_offset=coff, return_lse=True, out=out)
    assert ops.last_kernel() == name and o.data_ptr() == out.data_ptr()
    check_out(out, ro, dtype, lse=lse, ref_lse=rl)
    assert untouched(obuf, out, SENTINEL), "out: written outside the view"
    od, ld = ops.flash_attn_fwd(*dense, causal=True, causal_offset=coff, return_lse=True)
    assert ops.last_kernel() == name
    assert same_bits(out, od) and same_bits(lse, ld), "strided operands changed the result"

    acc, abuf = poisoned_view((B, Sq, Hq, D), torch.float32, ((1, 0), 3, 1, 4), SENTINEL)
    lacc, lbuf = poisoned_view((B, Hq, Sq), torch.float32, (1, (1, 1), 5), SENTINEL)
    dacc, dlacc = torch.empty(B, Sq, Hq, D, device="cuda"), torch.empty(B, Hq, Sq, device="cuda")
    for i, (a, b) in enumerate(((0, 128), (128, Sk))):
        for (qq, kk, vv), oa, la in (((q, k, v), acc, lacc), (dense, dacc, dlacc)):
            ops.flash_attn_fwd_accum(qq, kk[:, a:b], vv[:, a:b], oa, la, init=(i == 0), causal=True, causal_offset=coff - a)
            assert ops.last_kernel() == name
    check_out(acc, ro, dtype, lse=lacc, ref_lse=rl)
    assert untouched(abuf, acc, SENTINEL) and untouched(lbuf, lacc, SENTINEL), "accumulator written outside the view"
    assert same_bits(acc, dacc) and same_bits(lacc, dlacc), "strided operands changed the accumulated result"


@gpu
@pytest.mark.parametrize("fill", FILLS, ids=FILL_IDS)
@pytest.mark.parametrize("D", [64, 128, 80])
@pytest.mark.parametrize("pair", [False, True])
@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS.get)
def test_prefill_poisoned_right_padding(ops, monkeypatch, dtype, pair, D, fill):
    """Right padding: every K / V row at or past ``kv_lens[b]`` is poisoned. The result must be finite, bit-identical to the
    call with those rows zeroed, and equal to the oracle; plain and accumulate output."""
    monkeypatch.setenv("B200_FA_PAIR", "1" if pair else "0")
    name = _fa_name(pair)
    lens = [384, 0, 1, 200, 129]
    B, Sq, Sk, Hq, Hkv = len(lens), 200, 384, 4, 2
    q, k0, v0 = rand_qkv(B, Sq, Sk, Hq, Hkv, D, dtype, seed=7 * D + pair)
    k, _ = poisoned_view(k0.shape, dtype, (1, 2, 0, 8), fill, values=k0)
    v, _ = poisoned_view(v0.shape, dtype, (1, 2, 0, 8), fill, values=v0)
    kz, vz = k0.clone(), v0.clone()
    for b, n in enumerate(lens):
        k[b, n:], v[b, n:] = fill, fill
        kz[b, n:], vz[b, n:] = 0, 0
    kvl = torch.tensor(lens, device="cuda", dtype=torch.int32)
    ro, rl = orc.attention_ref(q.cpu(), kz.cpu(), vz.cpu(), kv_lens=kvl.cpu())
    o, lse = ops.flash_attn_fwd(q, k, v, kv_lens=kvl, return_lse=True)
    assert ops.last_kernel() == name
    oz, lz = ops.flash_attn_fwd(q, kz, vz, kv_lens=kvl, return_lse=True)
    assert torch.isfinite(o).all(), f"keys past kv_lens reached the output in {int((~torch.isfinite(o)).sum())} elements"
    assert same_bits(o, oz) and same_bits(lse, lz), "keys past kv_lens changed the result"
    check_out(o, ro, dtype, lse=lse, ref_lse=rl)
    accs = []
    for kk, vv in ((k, v), (kz, vz)):
        oa, la = torch.empty(B, Sq, Hq, D, device="cuda"), torch.empty(B, Hq, Sq, device="cuda")
        ops.flash_attn_fwd_accum(q, kk, vv, oa, la, init=True, kv_lens=kvl)
        assert ops.last_kernel() == name
        accs.append((oa, la))
    assert torch.isfinite(accs[0][0]).all(), "keys past kv_lens reached the accumulator"
    assert same_bits(accs[0][0], accs[1][0]) and same_bits(accs[0][1], accs[1][1])
    check_out(accs[0][0], ro, dtype, lse=accs[0][1], ref_lse=rl)


# ------------------------------------------------------------------------------------------------- 2. paged cache
TAIL_ENTRIES = (-1, 2 ** 31 - 1)   # block-table entries past a sequence's last block


def paged_cache(K, V, lens, block_size, max_blocks, num_layers, layer, fill, tail, spare=3):
    """A paged cache ``[num_blocks, L, block_size, Hkv, D]`` holding ``K[b, :lens[b]]`` / ``V[b, :lens[b]]`` through a
    block table, and ``fill`` everywhere else: the other layers, ``spare`` blocks no table names, the slots past the
    context in each last block. Table entries past a sequence's last block hold ``tail``. The table depends only on the
    arguments, so two calls that differ in ``fill`` share it."""
    B, _, Hkv, D = K.shape
    need = [(n + block_size - 1) // block_size for n in lens]
    nblk = sum(need) + spare
    perm = torch.randperm(nblk, generator=torch.Generator().manual_seed(block_size * 131 + len(lens)))
    bt = torch.full((B, max_blocks), tail, dtype=torch.int32)
    used = 0
    for b, m in enumerate(need):
        bt[b, :m] = perm[used:used + m].to(torch.int32)
        used += m
    kc = torch.full((nblk, num_layers, block_size, Hkv, D), fill, dtype=K.dtype, device=K.device)
    vc = torch.full_like(kc, fill)
    for b, n in enumerate(lens):
        t = torch.arange(n)
        blk, slot = bt[b, t // block_size].long().to(K.device), (t % block_size).to(K.device)
        kc[blk, layer, slot] = K[b, :n]
        vc[blk, layer, slot] = V[b, :n]
    return kc, vc, bt.to(K.device)


def paged_lens(block_size, target=320):
    """Table width and context lengths: 0, 1, a block boundary - 1 and + 1, and a full table."""
    max_blocks = max(2, -(-target // block_size))
    cap = max_blocks * block_size
    b0 = block_size * (max_blocks // 2)
    return max_blocks, cap, [0, 1, b0 - 1, b0 + 1, cap]


@gpu
@pytest.mark.parametrize("fill", FILLS, ids=FILL_IDS)
@pytest.mark.parametrize("block_size", [8, 16, 32, 64, 128])
@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS.get)
def test_paged_prefill_poisoned_cache(ops, dtype, block_size, fill):
    """Paged prefill reads only what a sequence owns: the result on a cache poisoned everywhere else is finite, equal to
    the call on the same cache with the poison zeroed, and equal to the oracle."""
    max_blocks, cap, lens = paged_lens(block_size)
    B, Sq, Hq, Hkv, D, L, layer = len(lens), 40, 4, 2, 128, 3, 1
    g = torch.Generator(device="cuda").manual_seed(block_size)
    r = lambda *s: torch.randn(*s, device="cuda", generator=g).to(dtype)
    q, K, V = r(B, Sq, Hq, D), r(B, cap, Hkv, D), r(B, cap, Hkv, D)
    ctx = torch.tensor(lens, device="cuda", dtype=torch.int32)
    for tail in TAIL_ENTRIES:
        kc, vc, bt = paged_cache(K, V, lens, block_size, max_blocks, L, layer, fill, tail)
        kz, vz, btz = paged_cache(K, V, lens, block_size, max_blocks, L, layer, 0.0, tail)
        assert torch.equal(bt, btz)
        o, lse = ops.paged_prefill_attention(q, kc, vc, bt, ctx, layer_idx=layer, causal=True, return_lse=True)
        assert ops.last_kernel() == "fa_fwd_kernel"
        oz, lz = ops.paged_prefill_attention(q, kz, vz, bt, ctx, layer_idx=layer, causal=True, return_lse=True)
        assert torch.isfinite(o).all(), f"tail {tail}: slots past the context reached the output"
        assert same_bits(o, oz) and same_bits(lse, lz), f"tail {tail}: memory the sequences do not own changed the result"
        ro, rl = orc.paged_prefill_attention_ref(q.cpu(), kz.cpu(), vz.cpu(), bt.cpu(), ctx.cpu(), layer_idx=layer,
                                                 causal=True)
        check_out(o, ro, dtype, lse=lse, ref_lse=rl)


def _decode_name(G, ring, splits):
    if splits > 1:
        return "decode_reduce_kernel"
    return "decode_kernel" if G <= 2 else "decode_gqa_ring_kernel" if ring else "decode_gqa_mma_kernel"


@gpu
@pytest.mark.parametrize("fill", FILLS, ids=FILL_IDS)
@pytest.mark.parametrize("G", [1, 2, 4, 16])
@pytest.mark.parametrize("block_size", [1, 8, 16, 24, 64, 128, 256])
@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS.get)
def test_paged_decode_and_append_poisoned_cache(ops, monkeypatch, dtype, block_size, G, fill):
    """Paged decode (power-of-two and division addressing, block sizes from 1 to wider than a key tile) on a cache poisoned
    everywhere a sequence does not own: for the same split count, bit-identical to decode on a contiguous cache holding
    the same keys (poisoned past the context), and equal to the oracle. kv_append then changes exactly one slot of each
    non-empty sequence."""
    max_blocks, cap, lens = paged_lens(block_size)
    B, Hkv, D, L, layer = len(lens), 2, 128, 3, 2
    g = torch.Generator(device="cuda").manual_seed(block_size * 17 + G)
    r = lambda *s: torch.randn(*s, device="cuda", generator=g).to(dtype)
    q, K, V = r(B, Hkv * G, D), r(B, cap, Hkv, D), r(B, cap, Hkv, D)
    ctx = torch.tensor(lens, device="cuda", dtype=torch.int32)
    kd, vd = K.clone(), V.clone()
    for b, n in enumerate(lens):
        kd[b, n:], vd[b, n:] = fill, fill
    ro, rl = orc.decode_attention_ref(q.cpu(), K.cpu(), V.cpu(), ctx.cpu())
    for tail in TAIL_ENTRIES:
        kc, vc, bt = paged_cache(K, V, lens, block_size, max_blocks, L, layer, fill, tail)
        for ring in ((False, True) if G >= 3 else (False,)):
            monkeypatch.setenv("B200_GQA_RING", "1" if ring else "0")
            for splits in (1, 3):
                o, lse = ops.decode_attention(q, kc, vc, ctx, block_tables=bt, layer_idx=layer, num_splits=splits,
                                              return_lse=True)
                assert ops.last_kernel() == _decode_name(G, ring, splits)
                check_out(o, ro, dtype, "decode", Hkv, lse=lse, ref_lse=rl)
                od, ld = ops.decode_attention(q, kd, vd, ctx, num_splits=splits, return_lse=True)
                assert ops.last_kernel() == _decode_name(G, ring, splits)
                assert same_bits(o, od) and same_bits(lse, ld), f"tail {tail} ring {ring} splits {splits}: paged != contiguous"
        key, val = r(B, Hkv, D), r(B, Hkv, D)
        ek, ev = kc.cpu(), vc.cpu()
        orc.kv_append_ref(key.cpu(), val.cpu(), ek, ev, ctx.cpu(), bt.cpu(), layer)
        ops.kv_append(key, val, kc, vc, ctx, block_tables=bt, layer_idx=layer)
        assert ops.last_kernel() == "kv_append_kernel"
        assert same_bits(kc, ek) and same_bits(vc, ev), f"tail {tail}: kv_append changed more or less than one slot"


# ------------------------------------------------------------------------------------------------- 3. contiguous caches
def kv_buffers(layout, B, S, Hkv, D, dtype, fill, device="cuda"):
    shapes = {"interleaved": [(B, S, 2, Hkv, D)], "time_major": [(S, B, Hkv, D)] * 2, "batch_slice": [(B + 3, S, Hkv, D)] * 2}
    return [torch.full(s, fill, dtype=dtype, device=device) for s in shapes[layout]]


def kv_views(layout, bufs, B):
    """(k_cache, v_cache) ``[B, S, Hkv, D]`` views of the buffers: k / v interleaved per token (token stride 2 Hkv D), a
    time-major cache (batch stride < token stride), or the first B rows of a larger cache."""
    if layout == "interleaved":
        return bufs[0][:, :, 0], bufs[0][:, :, 1]
    if layout == "time_major":
        return bufs[0].transpose(0, 1), bufs[1].transpose(0, 1)
    return bufs[0][:B], bufs[1][:B]


@gpu
@pytest.mark.parametrize("fill", FILLS, ids=FILL_IDS)
@pytest.mark.parametrize("D", [64, 128])
@pytest.mark.parametrize("layout", ["interleaved", "time_major", "batch_slice"])
@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS.get)
def test_contiguous_cache_layouts(ops, monkeypatch, dtype, layout, D, fill):
    """Decode and kv_append on strided contiguous caches, positions past the context and unused rows poisoned. An idle slot
    (context 0) gives O = 0 and LSE = -inf in both decode kernels, with and without splits."""
    lens = [0, 1, 17, 299, 300]
    B, S, Hkv = len(lens), 300, 2
    g = torch.Generator(device="cuda").manual_seed(D + len(layout))
    r = lambda *s: torch.randn(*s, device="cuda", generator=g).to(dtype)
    K, V = r(B, S, Hkv, D), r(B, S, Hkv, D)
    bufs = kv_buffers(layout, B, S, Hkv, D, dtype, fill)
    k, v = kv_views(layout, bufs, B)
    for b, n in enumerate(lens):
        k[b, :n], v[b, :n] = K[b, :n], V[b, :n]
    ctx = torch.tensor(lens, device="cuda", dtype=torch.int32)
    kd, vd = k.contiguous(), v.contiguous()
    for G in (1, 4):
        q = r(B, Hkv * G, D)
        ro, rl = orc.decode_attention_ref(q.cpu(), K.cpu(), V.cpu(), ctx.cpu())
        for ring in ((False, True) if G >= 3 else (False,)):
            monkeypatch.setenv("B200_GQA_RING", "1" if ring else "0")
            for splits in (1, 3):
                o, lse = ops.decode_attention(q, k, v, ctx, num_splits=splits, return_lse=True)
                assert ops.last_kernel() == _decode_name(G, ring, splits)
                check_out(o, ro, dtype, "decode", Hkv, lse=lse, ref_lse=rl)
                assert _bits(o[0]).eq(0).all() and torch.isneginf(lse[0]).all(), "idle slot: O must be +0, LSE -inf"
                od, ld = ops.decode_attention(q, kd, vd, ctx, num_splits=splits, return_lse=True)
                assert same_bits(o, od) and same_bits(lse, ld), f"G {G} ring {ring} splits {splits}: layout changed the result"
    key, val = r(B, Hkv, D), r(B, Hkv, D)
    expect = [t.cpu() for t in bufs]
    orc.kv_append_ref(key.cpu(), val.cpu(), *kv_views(layout, expect, B), ctx.cpu())
    ops.kv_append(key, val, k, v, ctx)
    assert ops.last_kernel() == "kv_append_kernel"
    assert all(same_bits(t, e) for t, e in zip(bufs, expect)), "kv_append changed more or less than one slot per sequence"


# ------------------------------------------------------------------------------------------------- 4. GEMM / FusedMLP
GEMM_PATHS = {   # path -> (op, T, environment, GEMM kernel, split-K reduce)
    "gemm_act": ("linear", 300, {"B200_GEMM_K_SPLITS": "1"}, "gemm_act_kernel<GELU_TANH>", False),
    "split_k2": ("linear", 300, {"B200_GEMM_K_SPLITS": "2"}, "gemm_act_kernel<GELU_TANH>", True),
    "split_k5": ("linear", 300, {"B200_GEMM_K_SPLITS": "5"}, "gemm_act_kernel<GELU_TANH>", True),
    "pair_1wg": ("linear", 1100, {"B200_GEMM_K_SPLITS": "1", "B200_GEMM_EPI_WGS": "1"}, "gemm_act_pair_kernel<GELU_TANH>", False),
    "pair_2wg": ("linear", 1100, {"B200_GEMM_K_SPLITS": "1", "B200_GEMM_EPI_WGS": "2"}, "gemm_act_pair_kernel<GELU_TANH,2wg>",
                 False),
    "fused": ("mlp", 1100, {"B200_MLP_FUSED": "1"}, "fused_mlp_pair_kernel<GELU_TANH>", False),
    "two_launch": ("mlp", 300, {"B200_MLP_FUSED": "0", "B200_GEMM_K_SPLITS": "1"}, "gemm_act_kernel<NONE>", False),
}


@gpu
@pytest.mark.parametrize("fill", FILLS, ids=FILL_IDS)
@pytest.mark.parametrize("path", list(GEMM_PATHS))
@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS.get)
def test_gemm_row_strides(ops, monkeypatch, dtype, path, fill):
    """x a column slice of a poisoned 640-wide buffer at the ragged K = 584 (NaN / Inf right behind the last 8-column
    k-block) with a poisoned spare row; out a column slice of a sentinel buffer (ldy > N). Every GEMM path."""
    op, T, env, gemm_name, reduce = GEMM_PATHS[path]
    for key, val in env.items():
        monkeypatch.setenv(key, val)
    K, N = 584, (520 if op == "linear" else 1032)
    x0, w1, b1, w2, b2, _, _ = make_mlp(T, K, N, "gelu_tanh", seed=T + len(path), std=0.05, dtype=dtype)
    x, _ = poisoned_view((T, K), dtype, ((1, 2), 640 - K), fill, values=x0)
    n_out = N if op == "linear" else K
    out, obuf = poisoned_view((T, n_out), dtype, (1, 16), SENTINEL)

    def run(xx, o=None):
        if op == "linear":
            y = ops.linear_act(xx, w1, b1, "gelu_tanh", out=o)
        else:
            y = ops.fused_mlp(xx, w1, b1, w2, b2, "gelu_tanh", out=o)
        assert ops.last_gemm_kernel() == gemm_name
        assert (ops.last_kernel() == "splitk_reduce_kernel") == reduce
        return y

    y = run(x, out)
    assert y.data_ptr() == out.data_ptr()
    c = lambda t: t.cpu()
    ref = (orc.linear_act_ref(logical(x), c(w1), c(b1), "gelu_tanh") if op == "linear"
           else orc.mlp_ref(logical(x), c(w1), c(b1), c(w2), c(b2), "gelu_tanh"))
    check_out(out, ref, dtype, "2d")
    assert untouched(obuf, out, SENTINEL), "out: written outside the view"
    assert same_bits(out, run(x.contiguous())), "row strides changed the result"


# ------------------------------------------------------------------------------------------------- 5. LayerNorm
@gpu
@pytest.mark.parametrize("fill", FILLS, ids=FILL_IDS)
@pytest.mark.parametrize("cols", [768, 4104])
@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS.get)
def test_layernorm_row_strides(ops, dtype, cols, fill):
    """x, residual and out with three different row strides and poisoned gaps, in the warp-per-row kernel (768 columns)
    and the CTA-per-row kernel (4104 columns)."""
    rows = 301
    g = torch.Generator(device="cuda").manual_seed(cols)
    r = lambda *s: torch.randn(*s, device="cuda", generator=g).to(dtype)
    x, _ = poisoned_view((rows, cols), dtype, (2, 8), fill, values=r(rows, cols) * 2 + 0.5)
    res, _ = poisoned_view((rows, cols), dtype, ((1, 0), 24), fill, values=r(rows, cols))
    w, b = r(cols), r(cols)
    out, obuf = poisoned_view((rows, cols), dtype, ((0, 1), 16), SENTINEL)
    y = ops.layernorm(x, w, b, 1e-5, res, 0.7, out=out)
    assert ops.last_kernel() == "layernorm_kernel" and y.data_ptr() == out.data_ptr()
    check_out(out, orc.layernorm_ref(logical(x), w.cpu(), b.cpu(), 1e-5, logical(res), 0.7), dtype, "2d")
    assert untouched(obuf, out, SENTINEL), "out: written outside the view"
    assert same_bits(out, ops.layernorm(x.contiguous(), w, b, 1e-5, res.contiguous(), 0.7)), "row strides changed the result"


# ------------------------------------------------------------------------------------------------- 6. lse_merge / cast_out
@gpu
@pytest.mark.parametrize("fill", FILLS, ids=FILL_IDS)
@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS.get)
def test_lse_merge_and_cast_out_strided(ops, dtype, fill):
    """lse_merge reads o_b as a transposed [B,H,S,D] view with poisoned gaps; cast_out writes into a strided view of a
    sentinel buffer, byte-exact against Tensor.to."""
    B, S, H, D = 2, 200, 4, 128
    g = torch.Generator(device="cuda").manual_seed(3)
    ob_bhsd, _ = poisoned_view((B, H, S, D), dtype, (0, 1, (1, 2), 8), fill,
                               values=torch.randn(B, H, S, D, device="cuda", generator=g).to(dtype))
    ob = ob_bhsd.transpose(1, 2)
    oa, la = torch.randn(B, S, H, D, device="cuda", generator=g), torch.randn(B, H, S, device="cuda", generator=g)
    lb = torch.randn(B, H, S, device="cuda", generator=g)
    la[0, 0, :5] = float("-inf")
    lb[0, 1, :5] = float("-inf")
    la[1, 2, :3] = lb[1, 2, :3] = float("-inf")
    ro, rl = orc.lse_merge_ref(oa.cpu(), la.cpu(), logical(ob), lb.cpu())
    oa2, la2 = oa.clone(), la.clone()
    ops.lse_merge(oa, la, ob, lb)
    assert ops.last_kernel() == "lse_merge_kernel"
    assert (oa.cpu() - ro).abs().max().item() <= 1e-5
    check_lse(la, rl)
    ops.lse_merge(oa2, la2, ob.contiguous(), lb)
    assert same_bits(oa, oa2) and same_bits(la, la2), "a strided o_b changed the merge"

    out, obuf = poisoned_view((B, S, H, D), dtype, ((1, 0), 2, 1, 8), SENTINEL)
    res = ops.cast_out(oa, dtype, out=out)
    assert ops.last_kernel() == "cast_out_kernel" and res.data_ptr() == out.data_ptr()
    assert same_bits(out, oa.cpu().to(dtype)), "cast_out is not Tensor.to"
    assert untouched(obuf, out, SENTINEL), "out: written outside the view"


# ------------------------------------------------------------------------------------------------- 7. out= contract
def lands_or_raises(call, out, want):
    """``call()`` either returns ``out`` holding exactly ``want`` or raises ValueError before writing anything; it never
    returns a right answer computed in a copy while ``out`` stays unwritten."""
    before = out.clone()
    try:
        res = call()
    except ValueError:
        assert same_bits(out, before), "raised ValueError after writing into out"
        return
    assert res.data_ptr() == out.data_ptr(), "the result is not out"
    assert same_bits(out, want), "out does not hold the result"


@gpu
@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS.get)
def test_out_argument_lands_or_raises(ops, dtype):
    """linear_act, fused_mlp and layernorm with an out that cannot be viewed as [rows, N] (``buf[:, :S]`` of a
    [B, S+3, N] buffer), of the wrong dtype and of the wrong shape; decode_attention with a strided and an fp32 out;
    cast_out with a wrong-shaped out. Every wrong-shaped out is a view inside a larger buffer, so nothing is written
    outside an allocation even where the shape is not checked."""
    B, S, K, N, I = 2, 40, 256, 264, 512
    x, w1, b1, w2, b2, _, _ = make_mlp(B * S, K, I, "gelu_tanh", seed=11, std=0.05, dtype=dtype)
    x = x.view(B, S, K)
    wl, bl = w1[:N].contiguous(), b1[:N].contiguous()

    def cases(width, call):
        want = call(None)
        assert want.shape == (B, S, width)
        buf = torch.full((B, S + 3, width), SENTINEL, dtype=dtype, device="cuda")
        lands_or_raises(lambda: call(buf[:, :S]), buf[:, :S], want)                       # rows of two strides
        assert untouched(buf, buf[:, :S], SENTINEL)
        wrong_dt = torch.full((B, S, width), SENTINEL, dtype=torch.float32, device="cuda")
        lands_or_raises(lambda: call(wrong_dt), wrong_dt, want)
        big = torch.full((B, S, width + 8), SENTINEL, dtype=dtype, device="cuda")
        lands_or_raises(lambda: call(big[..., :width - 8]), big[..., :width - 8], want)   # 8 columns short

    cases(N, lambda o: ops.linear_act(x, wl, bl, "gelu_tanh", out=o))
    cases(K, lambda o: ops.fused_mlp(x, w1, b1, w2, b2, "gelu_tanh", out=o))
    lw, lb = torch.randn(K, device="cuda").to(dtype), torch.randn(K, device="cuda").to(dtype)
    cases(K, lambda o: ops.layernorm(x, lw, lb, out=o))

    Hq, Hkv, D = 8, 2, 128
    g = torch.Generator(device="cuda").manual_seed(12)
    q = torch.randn(B, Hq, D, device="cuda", generator=g).to(dtype)
    kc = torch.randn(B, 64, Hkv, D, device="cuda", generator=g).to(dtype)
    vc = torch.randn_like(kc)
    ctx = torch.tensor([64, 30], device="cuda", dtype=torch.int32)
    want = ops.decode_attention(q, kc, vc, ctx)
    dbuf = torch.full((B, Hq, D + 8), SENTINEL, dtype=dtype, device="cuda")
    lands_or_raises(lambda: ops.decode_attention(q, kc, vc, ctx, out=dbuf[..., :D]), dbuf[..., :D], want)
    assert untouched(dbuf, dbuf[..., :D], SENTINEL)
    d32 = torch.full((B, Hq, D), SENTINEL, dtype=torch.float32, device="cuda")
    lands_or_raises(lambda: ops.decode_attention(q, kc, vc, ctx, out=d32), d32, want)

    acc = torch.randn(B, S, 4, D, device="cuda", generator=g)
    want = acc.to(dtype)
    cbuf = torch.full((B, S, 4, D), SENTINEL, dtype=dtype, device="cuda")
    lands_or_raises(lambda: ops.cast_out(acc, dtype, out=cbuf[:, :S - 1]), cbuf[:, :S - 1], want)   # one row short
    assert untouched(cbuf, cbuf[:, :S - 1], SENTINEL)
