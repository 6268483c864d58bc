"""BASELINE configs[0] through the product path: GPT-2 small (124M, random-init — no checkpoints offline), 64-token
prompt, greedy generation of 128 tokens.

    python benchmarks/decode_bench.py [--new-tokens 128] [--cpu-tokens 24]

Legs (one JSON line each): the reference's path = HF eager attention + MLP in fp32 on the host cores (what
``baseline/inference.py`` wraps; timed on a bounded number of tokens), HF generate on the GPU (bf16, its own KV cache),
and this repo's paged-KV generation (``generate_paged``: K1 prefill, ``b200_kv_append`` + K2 decode, K3 MLP) eager and
with the decode step captured in a CUDA graph. Wall clock around the whole call with a device synchronize, as
``InferenceRunner.run_inference`` measures (reference baseline/inference.py:684-702).
"""
import argparse
import json
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--new-tokens", type=int, default=128)
    ap.add_argument("--prompt", type=int, default=64)
    ap.add_argument("--batch", type=int, default=1)
    ap.add_argument("--cpu-tokens", type=int, default=24)
    ap.add_argument("--kv-cache-dtype", choices=["bf16", "fp8"], default="bf16",
                    help="paged KV cache of the b200 legs: bf16, or fp8 (e4m3, scales 1.0)")
    args = ap.parse_args()
    kv_dtype = torch.float8_e4m3fn if args.kv_cache_dtype == "fp8" else None
    from transformers import GPT2Config, GPT2LMHeadModel

    from ml_inference_optimizer_b200.baseline.inference import generate_paged
    from ml_inference_optimizer_b200.optimizer import Optimizer

    torch.manual_seed(0)
    cfg = GPT2Config(attn_implementation="eager")
    base = GPT2LMHeadModel(cfg).eval()
    ids = torch.randint(0, cfg.vocab_size, (args.batch, args.prompt))

    def emit(leg, tokens, seconds, **extra):
        print(json.dumps({"bench": "gpt2_small_generate", "leg": leg, "batch": args.batch, "prompt": args.prompt,
                          "kv_cache_dtype": args.kv_cache_dtype, "new_tokens": tokens, "seconds": seconds, "tokens_per_s": args.batch * tokens / seconds, **extra}),
              flush=True)

    if args.cpu_tokens > 0:
        torch.set_num_threads(os.cpu_count() or 1)
        with torch.no_grad():
            base.generate(ids, max_new_tokens=2, do_sample=False, pad_token_id=0)
            t0 = time.perf_counter()
            base.generate(ids, max_new_tokens=args.cpu_tokens, do_sample=False, pad_token_id=0)
            emit("cpu_hf_eager_fp32 (reference path)", args.cpu_tokens, time.perf_counter() - t0, cores=torch.get_num_threads())

    dev = torch.device("cuda:0")
    gids = ids.to(dev)
    hf = GPT2LMHeadModel(cfg).eval()
    hf.load_state_dict(base.state_dict())
    hf = hf.to(dev, torch.bfloat16)

    def timed(fn):
        fn()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        out = fn()
        torch.cuda.synchronize()
        return out, time.perf_counter() - t0

    with torch.no_grad():
        ref, sec = timed(lambda: hf.generate(gids, max_new_tokens=args.new_tokens, do_sample=False, pad_token_id=0))
    emit("gpu_hf_generate_bf16", args.new_tokens, sec)
    import copy
    ours = Optimizer(copy.deepcopy(hf)).optimize(use_flash_attention=True, use_fused_mlp=True)
    out_e, sec = timed(lambda: generate_paged(ours, gids, args.new_tokens, kv_cache_dtype=kv_dtype))
    emit("b200_paged_eager_launches", args.new_tokens, sec, agree_with_hf=float((out_e == ref).float().mean()))
    try:
        out_g, sec = timed(lambda: generate_paged(ours, gids, args.new_tokens, use_cuda_graph=True,
                                                       kv_cache_dtype=kv_dtype))
        from ml_inference_optimizer_b200.baseline.inference import LAST_DECODE_STATS as st
        emit("b200_paged_cuda_graph", args.new_tokens, sec, agree_with_eager=float((out_g == out_e).float().mean()),
             capture_seconds=st.get("capture_s"), replay_steps=st.get("replay_steps"), replay_ms=st.get("replay_ms"),
             steady_tokens_per_s=args.batch * st["replay_steps"] / (st["replay_ms"] / 1e3) if st.get("replay_ms") else None)
    except Exception as exc:  # report, do not hide
        print(json.dumps({"bench": "gpt2_small_generate", "leg": "b200_paged_cuda_graph", "error": repr(exc)[:400]}), flush=True)


if __name__ == "__main__":
    main()
