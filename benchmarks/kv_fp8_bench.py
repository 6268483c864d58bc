"""Decode attention over an FP8 (e4m3) paged KV cache against the bf16 paged cache, at bench.py's decode shapes.

C3 (B 64, 8K context, Hq = Hkv = 32, D 128: MHA, the CUDA-core kernel) and C4 (Hq 32 / Hkv 8: GQA, the mma.sync kernel),
paged with 16-token blocks. Each repetition times the bf16 paged cache, the FP8 paged cache and the bf16 contiguous cache
one after the other in the same process, after warm-up; the caches (1.1-8.6 GB of KV per call) are far larger than the
126 MB L2, so every call streams its bytes from HBM. Reports the median µs per call and algorithmic bandwidth
(2·B·S·Hkv·D·bytes per element / time), with the card's name and power limit read in the same run.

    python benchmarks/kv_fp8_bench.py --out profiles/kv_fp8_decode.jsonl
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

SHAPES = {"C3": (64, 8192, 32, 32, 128), "C4": (64, 8192, 32, 8, 128)}   # B, context, Hq, Hkv, D


def card():
    name = torch.cuda.get_device_name(0)
    try:
        power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                               capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        power = "unknown"
    return name, power


def time_calls(fn, iters):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) * 1e3 / iters


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--shapes", default="C3,C4")
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=None, help="append the JSON lines to this file")
    args = ap.parse_args()
    from ml_inference_optimizer_b200 import ops

    name, power = card()
    bs = 16
    lines = []
    for tag in args.shapes.split(","):
        B, S, Hq, Hkv, D = SHAPES[tag]
        g = torch.Generator(device="cuda").manual_seed(0)
        nb = B * S // bs
        bt = torch.randperm(nb, device="cuda", generator=g).view(B, S // bs).to(torch.int32).contiguous()
        lens = torch.full((B,), S, dtype=torch.int32, device="cuda")
        q = torch.randn(B, Hq, D, device="cuda", dtype=torch.bfloat16, generator=g)
        kp = torch.empty(nb, 1, bs, Hkv, D, device="cuda", dtype=torch.bfloat16).normal_(generator=g)
        vp = torch.empty_like(kp).normal_(generator=g)

        def fp8_bytes():   # finite e4m3 values of either sign in [2^-6, 2]
            b = torch.randint(0x08, 0x40, (nb, 1, bs, Hkv, D), device="cuda", dtype=torch.uint8, generator=g)
            return (b | (torch.randint(0, 2, b.shape, device="cuda", dtype=torch.uint8, generator=g) << 7)).view(torch.float8_e4m3fn)

        k8, v8 = fp8_bytes(), fp8_bytes()
        kc = kp.view(B, S, Hkv, D)   # the same bytes read as a contiguous [B, S, Hkv, D] cache
        vc = vp.view(B, S, Hkv, D)
        legs = {
            "bf16_paged": (lambda: ops.decode_attention(q, kp, vp, lens, block_tables=bt), 2),
            "fp8_paged": (lambda: ops.decode_attention(q, k8, v8, lens, block_tables=bt, k_scale=0.5, v_scale=0.25), 1),
            "bf16_contiguous": (lambda: ops.decode_attention(q, kc, vc, lens), 2),
        }
        kernels = {}
        for leg, (fn, _) in legs.items():
            for _ in range(args.warmup):
                fn()
            kernels[leg] = ops.last_kernel()
        torch.cuda.synchronize()
        times = {leg: [] for leg in legs}
        for _ in range(args.reps):
            for leg, (fn, _) in legs.items():
                times[leg].append(time_calls(fn, args.iters))
        for leg, (_, elem) in legs.items():
            us = statistics.median(times[leg])
            nbytes = 2 * B * S * Hkv * D * elem
            rec = {"bench": "kv_fp8_decode", "shape": tag, "leg": leg, "B": B, "context": S, "Hq": Hq, "Hkv": Hkv, "D": D,
                   "block_size": bs, "kernel": kernels[leg], "us_per_call": round(us, 2),
                   "us_all_reps": [round(t, 2) for t in times[leg]], "kv_bytes": nbytes,
                   "algorithmic_GBps": round(nbytes / us / 1e3, 1), "gpu": name, "power_limit": power}
            lines.append(rec)
            print(json.dumps(rec), flush=True)
        b16, f8 = statistics.median(times["bf16_paged"]), statistics.median(times["fp8_paged"])
        rec = {"bench": "kv_fp8_decode", "shape": tag, "leg": "speedup_fp8_over_bf16_paged", "ratio": round(b16 / f8, 3),
               "gpu": name, "power_limit": power}
        lines.append(rec)
        print(json.dumps(rec), flush=True)
        del kp, vp, k8, v8, kc, vc
        torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "a") as f:
            for rec in lines:
                f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
