"""FP8 (e4m3) paged KV cache: the quantizing append (b200_kv_append_fp8), the FP8 decode kernels (b200_fa_decode_fp8) and
the serving path on top of them (PagedKVCache, generate_paged, TransformerInferenceRunner).

CPU: the reference quantizer (fp8_quantize_ref, below) on hand-computed bytes, the error codes of the entry points, the
cache's shape and size, and the inventory of the b200::decode::fp8 kernels. GPU (marked one by one): byte-exact append,
decode against the oracle on the dequantized cache, and generation end to end.
"""
import copy
import ctypes
import math
import os
import re
import shutil
import subprocess

import pytest
import torch

from oracle import attn_mlp_oracle as orc
from test_gpu_parity import BF16, DTYPES, FP16, ROW_MEAN_REL, TILE_MAX_REL, WORST, check_out
from test_gpu_precision import _instantiations

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FP8 = torch.float8_e4m3fn
gpu = pytest.mark.gpu
P = "tests/test_kv_fp8.py::"
# Decode on the dequantized cache uses the 16-bit decode thresholds of test_gpu_parity (ROW_MEAN_REL, TILE_MAX_REL,
# LSE_MAX_ABS). Worst values measured here on a B200 (1000 W), bf16 / fp16: row mean rel 1.7e-3 / 2.4e-4, tile max rel
# 3.4e-3 / 4.4e-4, LSE abs 1.7e-6.
# Logits of an FP8 step vs a 16-bit step on the dequantized cache: each step carries its own 16-bit decode rounding (the
# 16-bit GQA kernel rounds P to bf16, the FP8 one to f16), so their difference is held to twice the bf16 decode thresholds.
# Worst measured on a B200 (1000 W): mean rel 7.3e-3 (Llama, G = 4).
LOGITS_MEAN_REL, LOGITS_MAX_REL = 2 * ROW_MEAN_REL[BF16], 2 * TILE_MAX_REL[BF16]


# ---- reference of the FP8 cache format (include/b200_attn_mlp.h), torch on the CPU ----
def fp8_quantize_ref(x: torch.Tensor, scale: float) -> torch.Tensor:
    """The stored byte: e4m3(x / scale), correctly rounded fp32 division, saturating to +-448 (+-inf included), NaN kept."""
    return (x.float() / torch.tensor(scale, dtype=torch.float32)).clamp(-448, 448).to(FP8)


def fp8_dequantize_ref(b: torch.Tensor, scale: float) -> torch.Tensor:
    """The value a stored byte stands for: byte * scale, fp32."""
    return b.float() * torch.tensor(scale, dtype=torch.float32)


def kv_append_fp8_ref(key, value, k_cache, v_cache, context_lens, block_tables, layer_idx, k_scale, v_scale) -> None:
    """In place on FP8 paged caches: row i of key / value ``[B,n,Hkv,D]`` goes, quantized, to position
    ``context_lens[b] - n + i``; positions below 0 or past the block table's capacity are dropped."""
    B, n = key.shape[:2]
    bs = k_cache.shape[2]
    capacity = block_tables.shape[1] * bs
    for b in range(B):
        for i in range(n):
            pos = int(context_lens[b]) - n + i
            if pos < 0 or pos >= capacity:
                continue
            blk = int(block_tables[b, pos // bs])
            k_cache[blk, layer_idx, pos % bs] = fp8_quantize_ref(key[b, i], k_scale)
            v_cache[blk, layer_idx, pos % bs] = fp8_quantize_ref(value[b, i], v_scale)


def _fp8_instantiations():
    """Every b200::decode::fp8 kernel instantiation -> the test here that launches it."""
    t = {}
    for dt in ("__nv_bfloat16", "__half"):
        t[f"decode::fp8::kv_append_kernel<{dt}>"] = P + "test_append_byte_exact"
        for D in (64, 128):
            for G in (1, 2):
                t[f"decode::fp8::decode_kernel<{D},{G},{dt}>"] = P + "test_decode_vs_oracle"
            t[f"decode::fp8::decode_gqa_mma_kernel<{D},{dt}>"] = P + "test_decode_vs_oracle"
    return t


@pytest.fixture(scope="module")
def ops(built_lib):
    assert torch.cuda.is_available(), "gpu tests need CUDA"
    from ml_inference_optimizer_b200 import ops as _ops

    assert _ops.arch_ok(), "gpu tests need an sm_100 device"
    return _ops


@pytest.fixture(scope="module", autouse=True)
def _report_worst():
    WORST.clear()
    yield
    for (metric, dt), val in sorted(WORST.items()):
        print(f"[worst fp8] {metric} {dt} {val:.3e}")


# ------------------------------------------------------------------------------------------------- CPU
def test_reference_quantizer_hand_computed_bytes():
    x = torch.tensor([448.0, 464.0, 1e9, -1e9, float("inf"), float("-inf"), float("nan"), 2.0 ** -9, -2.0 ** -9, 2.0 ** -10,
                      3 * 2.0 ** -10, 1.0625, 1.1875, 0.0])
    want = [0x7E, 0x7E, 0x7E, 0xFE, 0x7E, 0xFE, None, 0x01, 0x81, 0x00, 0x02, 0x38, 0x3A, 0x00]
    got = fp8_quantize_ref(x, 1.0)
    assert got.dtype == FP8
    b = got.view(torch.uint8).tolist()
    for i, w in enumerate(want):
        if w is None:
            assert math.isnan(got[i].float().item())
        else:
            assert b[i] == w, (i, x[i].item(), hex(b[i]), hex(w))
    # the scale divides first (correctly rounded fp32): 3.0 / 0.5 = 6.0 -> 0x4C; 448 * 4 saturates at scale 2
    assert fp8_quantize_ref(torch.tensor([3.0, 3584.0]), 0.5).view(torch.uint8).tolist() == [0x4C, 0x7E]
    assert fp8_dequantize_ref(torch.tensor([0x4C], dtype=torch.uint8).view(FP8), 0.5).item() == 3.0


def test_round_trip_error_inside_normal_range():
    g = torch.Generator().manual_seed(0)
    for scale in (1.0, 0.05, 3.0):
        mag = torch.exp(torch.empty(100000).uniform_(math.log(2.0 ** -6), math.log(448.0), generator=g)) * scale
        x = mag * torch.where(torch.rand(100000, generator=g) < 0.5, -1.0, 1.0)
        back = fp8_dequantize_ref(fp8_quantize_ref(x, scale), scale)
        assert ((back - x).abs() / x.abs()).max().item() <= 2.0 ** -4


def test_every_fp8_kernel_has_a_test(built_lib):
    """Every STB_GLOBAL kernel of the library, at any namespace depth, is in test_gpu_precision's table or in the FP8 table
    above; the FP8 kernels have no shared-memory-ring variant."""
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
        m = re.match(r"void b200::((?:\w+::)+)(\w+(?:<.*?>)?)\(", ln)
        if m:
            ns = m.group(1)[:-2]
            name = re.sub(r"\((?:int|bool)\)|\s", "", m.group(2))
            found.add(name if "::" not in ns else ns + "::" + name)   # b200::<ns>::name keeps test_gpu_precision's key
    fp8 = _fp8_instantiations()
    table = set(_instantiations()) | set(fp8)
    assert found - table == set(), "compiled kernels no test launches"
    assert table - found == set(), "listed kernels that are not compiled"
    assert {k for k in found if k.startswith("decode::fp8::")} == set(fp8)
    assert not any("ring" in k or re.match(r"decode::fp8::decode_gqa_mma_kernel<\d+,\w+,", k) for k in fp8)
    for target in set(fp8.values()):
        assert target.partition("::")[2] in globals(), target


def test_entry_points_return_documented_error_codes(built_lib):
    lib = built_lib
    d = ctypes.c_void_p(256)
    mis = ctypes.c_void_p(264)

    def dec(q=d, kc=d, layout=1, bt=d, D=128, Hq=8, Hkv=2, ks=1.0, vs=1.0, layer=0, bs=16):
        return lib.b200_fa_decode_fp8(q, kc, d, d, None, 2, Hq, Hkv, D, d, 64, 0.1, layout, bt, 4, bs, 2, layer, 1, None, 0, ks,
                                      vs, 0, None)

    def app(key=d, kc=d, bt=d, D=128, ks=1.0, vs=1.0, n=1, layer=0, dtype=0):
        return lib.b200_kv_append_fp8(key, d, kc, d, 2, n, 2, D, d, bt, 4, 16, 2, layer, ks, vs, dtype, None)

    bad = {"NULL": [dec(q=None), app(key=None)], "align": [dec(kc=mis), app(kc=mis)], "head_dim": [dec(D=96), app(D=32)],
           "group": [dec(Hq=34, Hkv=2)], "paged": [dec(bt=None), dec(layer=2), dec(bs=0), app(bt=None), app(layer=-1)],
           "scale": [dec(ks=0.0), dec(vs=-1.0), dec(ks=float("inf")), dec(vs=float("nan")), app(ks=0.0), app(vs=float("inf")),
                     app(ks=float("nan"))],
           "other": [app(n=0), app(dtype=2)]}
    for what, codes in bad.items():
        assert codes == [-1] * len(codes), (what, codes)
    assert dec(layout=0) == -2 and "paged" in _last_error()


def _last_error():
    from ml_inference_optimizer_b200 import _lib

    return _lib.last_error()


def test_paged_cache_fp8_allocation():
    from baseline.inference import PagedKVCache

    c8 = PagedKVCache(20, 16, 3, 4, 96, dtype=FP8, device="cpu", k_scale=[0.5, 1.0, 2.0], v_scale=0.25)
    c16 = PagedKVCache(20, 16, 3, 4, 96, dtype=torch.bfloat16, device="cpu")
    k, v = c8.get_physical_caches()
    assert k.shape == v.shape == (20, 3, 16, 4, 128) and k.dtype == v.dtype == FP8
    assert c8.get_memory_usage()["total_mb"] * 2 == c16.get_memory_usage()["total_mb"]
    assert c8.layer_scales(2) == (2.0, 0.25) and c16.layer_scales(0) == (1.0, 1.0)
    for kw in ({"k_scale": 0.0}, {"v_scale": float("inf")}, {"k_scale": [1.0, 2.0]}):
        with pytest.raises(ValueError):
            PagedKVCache(4, 16, 3, 4, 64, dtype=FP8, device="cpu", **kw)
    with pytest.raises(ValueError, match="FP8"):
        PagedKVCache(4, 16, 3, 4, 64, dtype=torch.bfloat16, device="cpu", k_scale=0.5)


# ------------------------------------------------------------------------------------------------- GPU: append
POISON = 0x5A


@gpu
@pytest.mark.parametrize("dtype", DTYPES, ids=["bf16", "fp16"])
@pytest.mark.parametrize("n", [1, 37])
@pytest.mark.parametrize("scale", [1.0, 0.05, 3.0])
def test_append_byte_exact(ops, dtype, n, scale):
    """n = 1 (decode) and n = S (prompt) rows, quantized byte for byte as fp8_quantize_ref does, saturating / infinite / NaN inputs
    included; every other byte of the cache keeps the poison, and rows past the block table's capacity are dropped."""
    g = torch.Generator(device="cuda").manual_seed(n)
    B, Hkv, D, bs, L = 3, 2, 128, 16, 2
    key = (torch.randn(B, n, Hkv, D, device="cuda", generator=g) * 40).to(dtype)
    val = (torch.randn(B, n, Hkv, D, device="cuda", generator=g) * 40).to(dtype)
    key[0, -1, 0, :6] = torch.tensor([1e4, -1e4, float("inf"), float("-inf"), float("nan"), 2.0 ** -12], dtype=dtype)
    val[1, 0, 1, :3] = torch.tensor([float("nan"), 6e4, -float("inf")], dtype=dtype)
    kc = torch.full((12, L, bs, Hkv, D), POISON, dtype=torch.uint8, device="cuda").view(FP8)
    vc = kc.clone()
    bt = torch.randperm(12, device="cuda")[:B * 3].view(B, 3).to(torch.int32).contiguous()   # capacity 48 tokens
    lens = torch.tensor([n, n + 5, 48 + n - 2], dtype=torch.int32, device="cuda")             # the last runs 2 rows past it
    rk, rv = kc.cpu().clone(), vc.cpu().clone()
    ops.kv_append(key if n > 1 else key[:, 0], val if n > 1 else val[:, 0], kc, vc, lens, bt, 1, k_scale=scale, v_scale=scale)
    assert ops.last_kernel() == "fp8_kv_append_kernel"
    kv_append_fp8_ref(key.cpu(), val.cpu(), rk, rv, lens.cpu(), bt.cpu(), 1, scale, scale)
    for got, ref in ((kc, rk), (vc, rv)):
        gb, rb = got.cpu().view(torch.uint8), ref.view(torch.uint8)
        nan_ref = torch.isnan(ref.float())
        assert torch.equal(torch.isnan(got.cpu().float()), nan_ref)
        assert torch.equal(gb[~nan_ref], rb[~nan_ref])
    assert (kc.cpu().view(torch.uint8)[:, 0] == POISON).all()           # the other layer


# ------------------------------------------------------------------------------------------------- GPU: decode
def _fp8_cache(B, Hkv, D, lens, bs, L, layer, ks, vs, seed, width=None):
    """A paged FP8 cache whose rows of each sequence are random values quantized by fp8_quantize_ref; NaN bytes (0x7f) everywhere else,
    slots past the context included. ``width`` < D: zero columns behind it (a narrow head in a wider cache)."""
    g = torch.Generator().manual_seed(seed)
    nblk_seq = max(1, math.ceil(max(lens) / bs))
    nblk = B * nblk_seq + 3
    bt = torch.randperm(nblk, generator=g)[:B * nblk_seq].view(B, nblk_seq).to(torch.int32)
    kc = torch.full((nblk, L, bs, Hkv, D), 0x7F, dtype=torch.uint8).view(FP8)
    vc = kc.clone()
    w = width or D
    for b, n in enumerate(lens):
        for t in range(n):
            blk = int(bt[b, t // bs])
            k, v = torch.zeros(Hkv, D), torch.zeros(Hkv, D)
            k[:, :w] = torch.randn(Hkv, w, generator=g) * 2
            v[:, :w] = torch.randn(Hkv, w, generator=g)
            kc[blk, layer, t % bs] = fp8_quantize_ref(k, ks)
            vc[blk, layer, t % bs] = fp8_quantize_ref(v, vs)
    return kc, vc, bt


DECODE_CASES = [(D, G) for D in (64, 128) for G in (1, 2, 4, 8, 16)]


@gpu
@pytest.mark.parametrize("dtype", DTYPES, ids=["bf16", "fp16"])
@pytest.mark.parametrize("D,G", DECODE_CASES)
def test_decode_vs_oracle(ops, D, G, dtype):
    """Decode over an FP8 cache against the oracle on the dequantized cache: forced 1 and 3 splits, block size 16 and 24,
    ragged lengths including 0 and 1, scales != 1, NaN bytes in every slot past the context."""
    B, Hkv, L, layer = 4, 2, 2, 1
    lens = [0, 1, 333, 700]
    for splits, bs, ks, vs in ((1, 16, 0.05, 3.0), (3, 24, 2.0, 0.125)):
        kc, vc, bt = _fp8_cache(B, Hkv, D, lens, bs, L, layer, ks, vs, seed=D * G + bs)
        q = torch.randn(B, Hkv * G, D, generator=torch.Generator().manual_seed(G)).to(dtype)
        ctx = torch.tensor(lens, dtype=torch.int32)
        o, lse = ops.decode_attention(q.cuda(), kc.cuda(), vc.cuda(), ctx.cuda(), block_tables=bt.cuda(), layer_idx=layer,
                                      num_splits=splits, return_lse=True, k_scale=ks, v_scale=vs)
        kern = "fp8_decode_gqa_mma_kernel" if G >= 3 else "fp8_decode_kernel"
        assert ops.last_kernel() == (kern if splits == 1 else "decode_reduce_kernel")
        ro, rl = orc.decode_attention_ref(q, fp8_dequantize_ref(kc, ks), fp8_dequantize_ref(vc, vs), ctx,
                                          block_tables=bt, layer_idx=layer)
        check_out(o, ro, dtype, "decode", Hkv, lse=lse, ref_lse=rl)


@gpu
@pytest.mark.parametrize("dtype", DTYPES, ids=["bf16", "fp16"])
@pytest.mark.parametrize("G", [1, 4])
def test_decode_head_dim_96_in_128_cache(ops, G, dtype):
    B, Hkv, L = 3, 2, 1
    lens = [5, 200, 64]
    kc, vc, bt = _fp8_cache(B, Hkv, 128, lens, 16, L, 0, 0.5, 0.25, seed=96 + G, width=96)
    q = torch.randn(B, Hkv * G, 96, generator=torch.Generator().manual_seed(9)).to(dtype)
    ctx = torch.tensor(lens, dtype=torch.int32)
    o = ops.decode_attention(q.cuda(), kc.cuda(), vc.cuda(), ctx.cuda(), block_tables=bt.cuda(), k_scale=0.5, v_scale=0.25)
    assert o.shape == (B, Hkv * G, 96)
    ro, _ = orc.decode_attention_ref(q, fp8_dequantize_ref(kc, 0.5)[..., :96], fp8_dequantize_ref(vc, 0.25)[..., :96],
                                     ctx, softmax_scale=1 / math.sqrt(96), block_tables=bt)
    check_out(o, ro, dtype, "decode", Hkv)


@gpu
def test_python_surface_refusals(ops):
    kc = torch.zeros(4, 1, 16, 2, 64, dtype=FP8, device="cuda")
    q = torch.randn(1, 2, 64, dtype=BF16, device="cuda")
    lens = torch.ones(1, dtype=torch.int32, device="cuda")
    with pytest.raises(NotImplementedError):
        ops.decode_attention(q, kc[:, 0], kc[:, 0], lens)
    with pytest.raises(NotImplementedError):
        ops.paged_prefill_attention(q[:, None], kc, kc, torch.zeros(1, 4, dtype=torch.int32, device="cuda"), lens)
    k16 = torch.zeros(4, 1, 16, 2, 64, dtype=BF16, device="cuda")
    with pytest.raises(ValueError, match="FP8"):
        ops.decode_attention(q, k16, k16, lens, block_tables=torch.zeros(1, 4, dtype=torch.int32, device="cuda"), k_scale=0.5)


# ------------------------------------------------------------------------------------------------- GPU: end to end
def _gpt2():
    from transformers import GPT2Config, GPT2LMHeadModel

    from ml_inference_optimizer import Optimizer

    torch.manual_seed(0)
    cfg = GPT2Config(n_layer=2, attn_implementation="eager")
    return Optimizer(GPT2LMHeadModel(cfg).eval().to("cuda", BF16)).optimize(), cfg.vocab_size


def _llama():
    from transformers import LlamaConfig, LlamaForCausalLM

    from ml_inference_optimizer import Optimizer

    torch.manual_seed(0)
    cfg = LlamaConfig(hidden_size=512, intermediate_size=1408, num_hidden_layers=2, num_attention_heads=8, num_key_value_heads=2,
                      vocab_size=1024, max_position_embeddings=512, attn_implementation="eager")
    return Optimizer(LlamaForCausalLM(cfg).eval().to("cuda", BF16)).optimize(), cfg.vocab_size


MODELS = {"gpt2": _gpt2, "llama": _llama}


@gpu
@pytest.mark.parametrize("name", list(MODELS))
def test_generate_paged_fp8_eager_equals_graph(ops, name):
    from baseline.inference import generate_paged

    model, vocab = MODELS[name]()
    ids = torch.randint(0, vocab, (2, 21), device="cuda", generator=torch.Generator(device="cuda").manual_seed(1))
    eager = generate_paged(model, ids, 14, kv_cache_dtype=FP8)
    graph = generate_paged(model, ids, 14, kv_cache_dtype=FP8, use_cuda_graph=True)
    assert eager.shape == (2, 35) and torch.equal(graph, eager)


@gpu
@pytest.mark.parametrize("name", list(MODELS))
def test_fp8_step_logits_match_16bit_step_on_dequantized_cache(ops, name, monkeypatch):
    """With a power-of-two scale every dequantized value is exact in bf16: one decode step over the FP8 cache and one over a
    16-bit copy of the dequantized cache (the new token's K,V rounded through e4m3 the same way) give the same logits within
    the bf16 decode tolerance of each of the two steps."""
    from baseline.inference import PagedKVCache, generate_paged
    from ml_inference_optimizer_b200.kernels.attention import flash_attention as fa

    model, vocab = MODELS[name]()
    adapters = [m for m in model.modules() if isinstance(m, fa._HFAttentionAdapter)]
    L, Hkv, hd = len(adapters), adapters[0].inner.num_kv_heads, adapters[0].inner.head_dim
    B, S, scale = 2, 21, 0.5
    ids = torch.randint(0, vocab, (B, S), device="cuda", generator=torch.Generator(device="cuda").manual_seed(2))
    c8 = PagedKVCache(8, 16, L, Hkv, hd, dtype=FP8, device="cuda", k_scale=scale, v_scale=scale)
    tok = generate_paged(model, ids, 1, cache=c8)[:, -1:]
    c16 = PagedKVCache(8, 16, L, Hkv, hd, dtype=BF16, device="cuda")
    c16.sequences = copy.deepcopy(c8.sequences)
    for dst, src in zip(c16.get_physical_caches(), c8.get_physical_caches()):
        dst.copy_((src.float() * scale).to(BF16))
        assert torch.equal(dst.float(), src.float() * scale)

    def step(cache):
        for sid in range(B):
            cache.append_token(sid)
        bt, lens = cache.device_tables(list(range(B)))
        fa.set_paged_context({"mode": "decode", "cache": cache, "seq_ids": list(range(B)), "block_tables": bt,
                              "context_lengths": lens})
        try:
            with torch.no_grad():
                return model(tok, position_ids=torch.full((B, 1), S, dtype=torch.long, device="cuda"), use_cache=False).logits[:, -1]
        finally:
            fa.set_paged_context(None)

    got = step(c8)
    real_append = ops.kv_append

    def append_through_e4m3(key, value, *a, **kw):
        rnd = lambda t: fp8_dequantize_ref(fp8_quantize_ref(t.cpu(), scale), scale).to(t.dtype).to(t.device)
        return real_append(rnd(key), rnd(value), *a, **kw)

    monkeypatch.setattr(ops, "kv_append", append_through_e4m3)
    ref = step(c16)
    e = orc.tile_errors(got.float(), ref.float(), "2d")
    print(f"[logits {name}] mean rel {e['mean_rel'].max().item():.3e} max rel {e['max_rel'].max().item():.3e}")
    check_out(got, ref, BF16, "2d", mean_rel=LOGITS_MEAN_REL, max_rel=LOGITS_MAX_REL)


@gpu
def test_runner_fp8_cache_twice_the_blocks_and_serves(ops):
    from transformers import GPT2Config, GPT2LMHeadModel

    from baseline.inference import TransformerInferenceRunner

    torch.manual_seed(0)
    cfg = GPT2Config(n_layer=2, attn_implementation="eager")
    model = GPT2LMHeadModel(cfg).eval().to("cuda", BF16)
    r16 = TransformerInferenceRunner(copy.deepcopy(model), "cuda", "bf16", kv_cache_num_gpu_blocks=16)
    r8 = TransformerInferenceRunner(copy.deepcopy(model), "cuda", "bf16", kv_cache_num_gpu_blocks=16, kv_cache_dtype=FP8)
    assert r8.paged_kv_cache.get_physical_caches()[0].dtype == FP8
    assert r8.paged_kv_cache.get_memory_usage()["total_mb"] * 2 == r16.paged_kv_cache.get_memory_usage()["total_mb"]
    n16, n8 = r16._calculate_num_gpu_blocks(), r8._calculate_num_gpu_blocks()   # the free-memory rule, same device state
    assert n16 > 0 and n8 in (2 * n16, 2 * n16 + 1), (n16, n8)
    ids = torch.randint(0, cfg.vocab_size, (2, 19), device="cuda")
    for graph in (False, True):
        r8.use_cuda_graph = graph
        out, _ = r8.run_inference({"input_ids": ids}, max_new_tokens=8)
        assert out.shape == (2, 27) and torch.equal(out[:, :19], ids)
