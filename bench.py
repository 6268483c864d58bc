#!/usr/bin/env python
"""bench.py — the contract benchmark of the attention + FusedMLP hot path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload c3|c2] [--no-secondary]
                    [--dump-outputs DIR]

A "step" is one pass of the hot path over one batch of synthetic input at the Llama-2-7B layer shapes of
BASELINE.json configs[2] (the configuration the metric's "SwiGLU-MLP" is quoted on and the largest single-GPU one):
causal FlashAttention forward (B=4, S=8192, 32x128 heads, bf16) followed by the SwiGLU FusedMLP (T=32768,
4096 -> 11008 -> 4096). ``--workload c2`` runs configs[1] (GPT-2 small: B=8, S=4096, 12x64 heads, GELU MLP).

N = 1: the step on one GPU.
N > 1: the SAME step (same total work: strong scaling) sharded the way the reference shards it — tensor parallelism
  (parallelism/tensor_parallel.py): attention over Hq/N heads per rank (no collective inside attention), FusedMLP with
  W_up/W_gate rows and W_down columns /N and ONE all-reduce of the [T, h] partial outputs per step INSIDE the timed
  region (tensor_parallel.py:296-302) — done by this repo's in-switch reduction kernel K6 over symmetric memory,
  overlapped with the GEMMs of the next token chunk (NCCL if symmetric memory cannot be set up; the line says which).
  The same run also times BASELINE configs[4] — RingAttention over one causal 128K-token sequence, sequence-sharded
  with the KV blocks circulating over NVLink — and reports it as ``ring_c5`` with T1/(N*TN).
  Before timing, every rank checks its ring shard and its TP output on reduced shapes against the fp32 oracle
  (``parity``); a failed check aborts the run.

Prints ONE JSON line (rank 0). ``value`` = algorithmic TFLOP/s of the whole job with inputs resident in HBM;
``e2e`` = the same through the public nn.Module API with pinned HOST buffers (H2D of the inputs and D2H of the results
inside the timed region); ``roofline`` = the dominant kernel against the measured bf16 peak (DRAM traffic read from
the committed ncu summary under profiles/); ``secondary`` (N=1) = decode attention, FusedMLP vs unfused cuBLAS,
isolated attention and the C2 layer step; ``cpu_baseline`` = the fp32 oracle timed on this box's host cores on a
bounded sample of the same workload.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: B, S, Hq, Hkv, D, hidden, intermediate, activation
    "c3": dict(name="llama2-7b-layer prefill: causal attn B4 S8192 H32 D128 + SwiGLU MLP 4096->11008 (BASELINE configs[2])",
               B=4, S=8192, Hq=32, Hkv=32, D=128, h=4096, i=11008, act="swiglu"),
    "c2": dict(name="gpt2-small-layer prefill: causal attn B8 S4096 H12 D64 + GELU MLP 768->3072 (BASELINE configs[1])",
               B=8, S=4096, Hq=12, Hkv=12, D=64, h=768, i=3072, act="gelu_tanh"),
}
METRIC = "fwd attention + FusedMLP TFLOP/s (causal attn + MLP layer step)"
NVLINK_GBS = 770.0  # measured peer-copy bandwidth per direction per GPU on this pool (B200_PROFILING.md)


def flops_of(w, B=None, S=None):
    B = w["B"] if B is None else B
    S = w["S"] if S is None else S
    T = B * S
    attn = 4.0 * B * w["Hq"] * S * S * w["D"] * 0.5          # causal
    mlp = (6.0 if w["act"] == "swiglu" else 4.0) * T * w["h"] * w["i"]
    return attn, mlp


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            d = json.load(open(path))
            return dict(tflops_burst=float(d["bf16_tflops"]), tflops_sustained=float(d.get("bf16_tflops_sustained", d["bf16_tflops"])),
                        hbm_gbs=float(d["hbm_gbs"]), source="measured")
        except Exception:  # noqa: BLE001
            pass
    return dict(tflops_burst=1590.0, tflops_sustained=1400.0, hbm_gbs=6650.0, source="fallback")


def committed_traffic(kernel_name):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of ``kernel_name`` from the committed ncu --set full
    summary (profiles/kernel_traffic.json, written by tests/ncu_summary.py from the .ncu-rep). None if no capture of
    that kernel is committed — never a literal."""
    path = os.path.join(ROOT, "profiles", "kernel_traffic.json")
    try:
        table = json.load(open(path))
    except Exception:  # noqa: BLE001
        return None, None
    for key, rec in table.items():
        if key == kernel_name or kernel_name.startswith(key):
            return rec.get("dram_bytes"), rec.get("source")
    return None, None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons. The sampler is started before the warm-up (nvidia-smi needs a moment to
    start); only samples whose arrival time falls inside [t_start, t_end] of the timed region are summarised."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu_index, self.proc, self.lines = gpu_index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20",
                                          "-i", str(self.gpu_index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self, t_start=None, t_end=None):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.05)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:  # noqa: BLE001
            self.proc.kill()

        def parse(rows):
            sm, smax, reasons, power = [], [], set(), []
            for _, ln in rows:
                f = [x.strip() for x in ln.split(",")]
                if len(f) < 8:
                    continue
                try:
                    sm.append(float(f[1])); smax.append(float(f[2])); power.append(float(f[3]))
                except ValueError:
                    continue
                for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
            return sm, smax, reasons, power

        inside = [(t, l) for t, l in self.lines if t_start is None or (t_start <= t <= t_end + 0.03)]
        window = "timed region"
        if not inside:  # region shorter than the sampling period: fall back to the whole run (warm-up + timed)
            inside, window = self.lines, "warm-up + timed region"
        sm, smax, reasons, power = parse(inside)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(smax), "power_w_max": max(power), "samples": len(sm),
                "window": window, "reasons": sorted(reasons)}


def bind_to_gpu_numa_node(dev_index):
    """Pin this process (and therefore the first-touch placement of its pinned host buffers) to the CPUs of the NUMA
    node the GPU hangs off. With 8 ranks allocating on node 0 the e2e leg of round 1 ran at 0.25 efficiency."""
    try:
        import pynvml
        pynvml.nvmlInit()
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        phys = int(vis.split(",")[dev_index]) if vis and all(t.strip().isdigit() for t in vis.split(",")) else dev_index
        bus = pynvml.nvmlDeviceGetPciInfo(pynvml.nvmlDeviceGetHandleByIndex(phys)).busId
        bus = bus.decode() if isinstance(bus, bytes) else bus
        bdf = bus.lower()
        if len(bdf.split(":")[0]) == 8:  # nvml prints an 8-digit domain, sysfs a 4-digit one
            bdf = bdf[4:]
        node = int(open(f"/sys/bus/pci/devices/{bdf}/numa_node").read().strip())
        if node < 0:
            return {"numa_node": node, "note": "single NUMA domain: nothing to bind"}
        cpus = []
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.extend(range(int(a), int(b or a) + 1))
        allowed = os.sched_getaffinity(0)
        use = sorted(set(cpus) & allowed)
        if use:
            os.sched_setaffinity(0, use)
            return {"numa_node": node, "cpus": len(use)}
        return {"numa_node": node, "note": "no allowed CPU on the GPU's node"}
    except Exception as e:  # noqa: BLE001
        return {"error": f"{type(e).__name__}: {e}"[:120]}


# ---------------------------------------------------------------------------------------------------------------
# reference arm / cpu_baseline: the fp32 oracle on the host cores, bounded sample
# ---------------------------------------------------------------------------------------------------------------
def cpu_oracle_rate(w, steps, warmup, sample_S=None, sample_B=1):
    import torch
    from oracle import attn_mlp_oracle as orc

    cores = os.cpu_count() or 1
    try:
        cores = len(os.sched_getaffinity(0))
    except Exception:  # noqa: BLE001
        pass
    torch.set_num_threads(cores)
    S = sample_S or min(w["S"], 2048)
    B = sample_B
    torch.manual_seed(0)
    q = torch.randn(B, S, w["Hq"], w["D"])
    k = torch.randn(B, S, w["Hkv"], w["D"])
    v = torch.randn(B, S, w["Hkv"], w["D"])
    x = torch.randn(B * S, w["h"])
    wu = torch.randn(w["i"], w["h"]) * 0.02
    wd = torch.randn(w["h"], w["i"]) * 0.02
    bu, bd = torch.zeros(w["i"]), torch.zeros(w["h"])
    wg = torch.randn(w["i"], w["h"]) * 0.02 if w["act"] == "swiglu" else None
    bg = torch.zeros(w["i"]) if w["act"] == "swiglu" else None

    def step():
        o, _ = orc.attention_ref(q, k, v, causal=True)
        y = orc.mlp_ref(x, wu, bu, wd, bd, w["act"], wg, bg)
        return o, y

    for _ in range(warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = (time.perf_counter() - t0) / steps
    fa, fm = flops_of(w, B=B, S=S)
    return dict(value=(fa + fm) / dt / 1e12, seconds_per_step=dt, cores=torch.get_num_threads(),
                sample=f"fp32 oracle (torch CPU eager), B={B} S={S} of the workload's B={w['B']} S={w['S']}, same heads/widths")


def run_reference(args, w):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps, warmup = max(1, args.steps), max(1, min(args.warmup, 2))
    r = cpu_oracle_rate(w, steps=min(steps, 5), warmup=warmup)
    line = {
        "impl": "reference", "metric": METRIC, "value": r["value"],
        "unit": "TFLOP/s", "n_gpus": args.gpus, "steps": min(steps, 5), "warmup": warmup, "ms_per_step": r["seconds_per_step"] * 1e3,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": w["name"], "arm": "reference CPU eager path (oracle port of HF-eager attention + MLP)"},
        "cpu_baseline": {"value": r["value"], "unit": "TFLOP/s", "cores": r["cores"], "kind": "port", "sample": r["sample"]},
        "e2e": {"value": r["value"], "unit": "TFLOP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------------------------------
class Ctx:
    """Per-process state shared by the legs of the benchmark."""

    def __init__(self):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.rank = int(os.environ.get("RANK", "0"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py needs a GPU: there is no CPU fallback for the product path (use --impl reference for the CPU arm)")
        torch.cuda.set_device(self.local_rank)
        self.dev = torch.device("cuda", self.local_rank)
        self.numa = bind_to_gpu_numa_node(self.local_rank)
        if self.world > 1:
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            os.environ.setdefault("TORCH_NCCL_HIGH_PRIORITY", "1")
            dist.init_process_group("nccl", device_id=self.dev,
                                    pg_options=dist.ProcessGroupNCCL.Options(is_high_priority_stream=True))

    def ev(self):
        return self.torch.cuda.Event(enable_timing=True)

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, values):
        if self.world == 1:
            return list(values)
        t = self.torch.tensor(list(values), device=self.dev, dtype=self.torch.float64)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return t.tolist()

    def timed(self, fn, warmup, iters, flush=None):
        """Mean device time of fn() in ms (CUDA events on the current stream, max over ranks). ``flush`` is a callable
        run (untimed: its own event pair is subtracted by timing each iteration separately) before every iteration."""
        torch = self.torch
        for _ in range(warmup):
            if flush:
                flush()
            fn()
        self.barrier()
        total = 0.0
        if flush is None:
            s, e = self.ev(), self.ev()
            s.record()
            for _ in range(iters):
                fn()
            e.record()
            torch.cuda.synchronize()
            total = s.elapsed_time(e) / iters
        else:
            pairs = []
            for _ in range(iters):
                flush()
                s, e = self.ev(), self.ev()
                s.record(); fn(); e.record()
                pairs.append((s, e))
            torch.cuda.synchronize()
            total = statistics.mean(s.elapsed_time(e) for s, e in pairs)
        return self.max_over_ranks([total])[0]


def parity_check(cx):
    """Reduced-shape checks of the two sharded paths against the fp32 oracle (the checker, on CPU), on every rank, before
    anything is timed. Returns max-abs errors (max over ranks); raises if a bound is exceeded."""
    torch, dist = cx.torch, cx.dist
    from ml_inference_optimizer_b200 import ops
    from ml_inference_optimizer_b200.parallelism import communication as comm
    from ml_inference_optimizer_b200.parallelism.ring import ring_attention_forward
    from oracle import attn_mlp_oracle as orc  # checker only

    n, r, dev = cx.world, cx.rank, cx.dev
    g = torch.Generator().manual_seed(7)
    # ring attention, causal zigzag, GQA
    B, S, Hq, Hkv, D = 1, 512 * max(n, 1), 8, 2, 128
    q, k, v = (torch.randn(B, S, H, D, generator=g).bfloat16() for H in (Hq, Hkv, Hkv))
    full, lse_full = orc.attention_ref(q, k, v, causal=True)
    part = "zigzag" if n > 1 else "contiguous"
    sh = lambda t: comm.scatter_along_sequence_dim(t, n, partition=part, rank=r).contiguous().to(dev)
    o, lse = ring_attention_forward(sh(q), sh(k), sh(v), causal=True, partition=part, return_lse=True)
    want = comm.scatter_along_sequence_dim(full, n, partition=part, rank=r)
    want_lse = comm.scatter_along_sequence_dim(lse_full.transpose(1, 2), n, partition=part, rank=r).transpose(1, 2)
    ring_o = (o.float().cpu() - want).abs().max().item()
    ring_l = (lse.cpu() - want_lse).abs().max().item()
    # tensor-parallel SwiGLU MLP through the module (symmetric all-reduce path when available)
    T, h, i = 512, 512, 1024 * n
    rn = lambda *s, sc=1.0: (torch.randn(*s, generator=g) * sc).bfloat16()
    x, wu, bu, wg, bg, wd, bd = rn(T, h), rn(i, h, sc=0.03), rn(i, sc=0.1), rn(i, h, sc=0.03), rn(i, sc=0.1), rn(h, i, sc=0.03), rn(h, sc=0.1)
    ref, partial_abs = orc.tp_mlp_ref(x, wu, bu, wd, bd, "swiglu", n, wg, bg, return_partial_abs_sum=True)
    c = lambda t: t.to(dev)
    reduce_impl = "none"
    if n > 1:
        import torch.nn.functional as F
        from ml_inference_optimizer_b200.parallelism import parallel_utils as pu
        from ml_inference_optimizer_b200.parallelism.tensor_parallel import TensorParallelConfig, TensorParallelMLP
        pu.initialize_tensor_parallel(n)
        cfg = TensorParallelConfig(world_size=n, tp_size=n)
        m = TensorParallelMLP.from_dense(c(wu), c(bu), c(wd), c(bd), cfg, F.silu, c(wg), c(bg))
        y = m(c(x))
        reduce_impl = m.last_reduce
        # the chunked pipeline (prefill-sized input) must agree with the oracle as well
        m.overlap_min_tokens = 256
        y2 = m(c(x))
        tp_err = max((y.float().cpu() - ref).abs().max().item(), (y2.float().cpu() - ref).abs().max().item())
    else:
        y = ops.fused_mlp(c(x), c(wu), c(bu), c(wd), c(bd), "swiglu", c(wg), c(bg))
        tp_err = (y.float().cpu() - ref).abs().max().item()
    tp_scale = ref.abs().max().item()
    tp_tol = orc.tp_mlp_tolerance(ref, partial_abs, n, multicast="multicast" in reduce_impl)
    ring_o, ring_l, tp_err = cx.max_over_ranks([ring_o, ring_l, tp_err])
    out = {"ring_max_abs": ring_o, "ring_lse_max_abs": ring_l, "tp_max_abs": tp_err, "tp_ref_max_abs": tp_scale,
           "bounds": {"ring_max_abs": 2e-2, "ring_lse_max_abs": 1e-2, "tp_max_abs": tp_tol,
                      "tp_rule": "2e-2*max(1,|ref|max/4) + 2^-9*max sum_r|partial_r| (bf16 partials) + 2^-8*|ref|max (switch rounding); oracle.tp_mlp_tolerance"},
           "shapes": f"ring: causal {part} B{B} S{S} Hq{Hq} Hkv{Hkv} D{D}; tp: SwiGLU T{T} {h}->{i}->{h}",
           "tp_reduce": reduce_impl, "checker": "oracle/attn_mlp_oracle.py (fp32, CPU)"}
    ok = ring_o <= 2e-2 and ring_l <= 1e-2 and tp_err <= tp_tol
    if not ok:
        raise SystemExit(f"parity check failed before timing: {json.dumps(out)}")
    return out


def build_step(cx, w, args):
    """Allocate the workload (sharded for N>1) and return (step(record), state)."""
    torch = cx.torch
    from ml_inference_optimizer_b200 import ops
    n, r, dev = cx.world, cx.rank, cx.dev
    B, S, Hq, Hkv, D, h, i, act = (w[k] for k in ("B", "S", "Hq", "Hkv", "D", "h", "i", "act"))
    if Hq % n or Hkv % n or i % (n * 8):
        raise SystemExit(f"workload does not shard over {n} ranks (Hq={Hq}, Hkv={Hkv}, i={i})")
    T = B * S
    bf = torch.bfloat16
    g = torch.Generator(device=dev).manual_seed(1234)  # same stream on every rank: replicated tensors agree
    hq, hkv = Hq // n, Hkv // n
    # q/k/v: this rank's heads (what a column-parallel QKV projection leaves on the rank)
    q = torch.randn(B, S, hq, D, device=dev, dtype=bf, generator=g)
    k = torch.randn(B, S, hkv, D, device=dev, dtype=bf, generator=g)
    v = torch.randn(B, S, hkv, D, device=dev, dtype=bf, generator=g)
    x = torch.randn(T, h, device=dev, dtype=bf, generator=g)  # replicated activation
    il = i // n
    wu = (torch.randn(il, h, device=dev, generator=g) * 0.02).to(bf)
    wd = (torch.randn(h, il, device=dev, generator=g) * 0.02).to(bf)
    bu = (torch.randn(il, device=dev, generator=g) * 0.02).to(bf)
    bd = (torch.randn(h, device=dev, generator=g) * 0.02).to(bf)
    wg = bg = None
    if act == "swiglu":
        wg = (torch.randn(il, h, device=dev, generator=g) * 0.02).to(bf)
        bg = (torch.randn(il, device=dev, generator=g) * 0.02).to(bf)
    o = torch.empty_like(q)
    st = dict(q=q, k=k, v=v, x=x, o=o, wu=wu, wd=wd, bu=bu, bd=bd, wg=wg, bg=bg, T=T, events=[])
    if n == 1:
        y = torch.empty(T, h, device=dev, dtype=bf)
        st["y"] = y

        def step(record=False):
            if record:
                e = [cx.ev() for _ in range(4)]
                e[0].record()
                ops.flash_attn_fwd(q, k, v, causal=True, out=o)
                ops.fused_mlp(x, wu, bu, wd, bd, act, wg, bg, out=y, timing_events=(e[1], e[2], e[3]))
                st["events"].append(e)
            else:
                ops.flash_attn_fwd(q, k, v, causal=True, out=o)
                ops.fused_mlp(x, wu, bu, wd, bd, act, wg, bg, out=y)
        st["mlp_module"] = None
    else:
        import torch.nn.functional as F
        from ml_inference_optimizer_b200.parallelism import parallel_utils as pu
        from ml_inference_optimizer_b200.parallelism.tensor_parallel import TensorParallelConfig, TensorParallelMLP
        pu.initialize_tensor_parallel(n)
        cfg = TensorParallelConfig(world_size=n, tp_size=n)
        mlp = TensorParallelMLP(h, i, cfg, F.silu if act == "swiglu" else F.gelu, gated=(act == "swiglu")).to(dev, bf)
        if act != "swiglu":
            mlp.activation = "gelu_tanh"
        with torch.no_grad():
            mlp.dense_h_to_4h.weight.copy_(wu); mlp.dense_h_to_4h.bias.copy_(bu)
            mlp.dense_4h_to_h.weight.copy_(wd); mlp.dense_4h_to_h.bias.copy_(bd)
            if wg is not None:
                mlp.dense_h_to_4h_gate.weight.copy_(wg); mlp.dense_h_to_4h_gate.bias.copy_(bg)
        mlp.symmetric_output = "view"  # the step's output stays in the peer-mapped buffer (two rotate)
        st["mlp_module"] = mlp
        st["wu"], st["wd"], st["wg"] = mlp.dense_h_to_4h.weight, mlp.dense_4h_to_h.weight, (mlp.dense_h_to_4h_gate.weight if wg is not None else None)

        def step(record=False):
            if record:
                e = [cx.ev() for _ in range(3)]
                e[0].record()
                ops.flash_attn_fwd(q, k, v, causal=True, out=o)
                e[1].record()
                st["y"] = mlp(x)
                e[2].record()
                st["events"].append(e)
            else:
                ops.flash_attn_fwd(q, k, v, causal=True, out=o)
                st["y"] = mlp(x)
    return step, st


DUMP_ROWS = 1024  # token rows kept per output: the C3 step's two [T, 4096] outputs come to 32 MB as float32


def dump_outputs(cx, st, out_dir):
    """Write what the last timed step computed as float32 .npy files: ``attn_out`` (the attention output O as
    [tokens, Hq*D]) and ``mlp_out`` (the MLP output y as [tokens, h]). Both keep the same DUMP_ROWS token rows, drawn
    with a fixed seed, so two builds run with the same arguments can be compared element for element."""
    import numpy as np
    torch = cx.torch
    T = st["T"]
    rows = np.sort(np.random.default_rng(0).choice(T, size=min(T, DUMP_ROWS), replace=False))
    idx = torch.from_numpy(rows).to(cx.dev)
    o = st["o"].reshape(T, -1).index_select(0, idx)
    if cx.world > 1:  # every rank holds Hq/N heads: put the job's heads side by side, rank order
        parts = [torch.empty_like(o) for _ in range(cx.world)]
        cx.dist.all_gather(parts, o)
        o = torch.cat(parts, dim=1)
    y = st["y"].reshape(T, -1).index_select(0, idx)
    if cx.rank == 0:
        os.makedirs(out_dir, exist_ok=True)
        np.save(os.path.join(out_dir, "attn_out.npy"), o.float().cpu().numpy())
        np.save(os.path.join(out_dir, "mlp_out.npy"), y.float().cpu().numpy())


def e2e_leg(cx, w, st, args):
    """End to end through the public nn.Module API with pinned HOST buffers: every step copies its inputs host -> device
    and its results device -> host inside the timed region (three streams, double-buffered device tensors)."""
    torch, dist = cx.torch, cx.dist
    from ml_inference_optimizer_b200.kernels.attention.flash_attention import FlashAttention3, FlashAttentionConfig
    from ml_inference_optimizer_b200.kernels.mlp.fused_mlp import FusedMLP, FusedMLPConfig, FusedMLPSwiGLU
    n, r, dev = cx.world, cx.rank, cx.dev
    bf = torch.bfloat16
    q, k, v, x, T = st["q"], st["k"], st["v"], st["x"], st["T"]
    attn = FlashAttention3(FlashAttentionConfig(causal=True, precision="bf16"))
    if n == 1:
        cfg = FusedMLPConfig(activation_fn="gelu_tanh" if w["act"] != "swiglu" else "gelu", precision="bf16")
        mlp = (FusedMLPSwiGLU if w["act"] == "swiglu" else FusedMLP)(w["h"], w["i"], cfg).to(dev, bf)
        with torch.no_grad():
            mlp.fc1.weight.copy_(st["wu"]); mlp.fc1.bias.copy_(st["bu"]); mlp.fc2.weight.copy_(st["wd"]); mlp.fc2.bias.copy_(st["bd"])
            if st["wg"] is not None:
                mlp.fc1_gate.weight.copy_(st["wg"]); mlp.fc1_gate.bias.copy_(st["bg"])
        rows = T
    else:
        mlp = st["mlp_module"]
        rows = T // n  # every rank uploads T/N rows of the activation; an all-gather over NVLink replicates it
    pin = lambda t: torch.empty(t.shape, dtype=t.dtype, pin_memory=True).copy_(t)
    x_rows = x[r * rows:(r + 1) * rows] if n > 1 else x
    hq, hk, hv, hx = pin(q), pin(k), pin(v), pin(x_rows)
    ho = torch.empty(q.shape, dtype=bf, pin_memory=True)
    hy = torch.empty((rows, w["h"]), dtype=bf, pin_memory=True)
    sets = [tuple(torch.empty_like(t) for t in (q, k, v, x_rows)) for _ in range(2)]
    xfull = [torch.empty_like(x) for _ in range(2)] if n > 1 else None
    outs = [None, None]
    s_h2d, s_cmp, s_d2h = torch.cuda.Stream(dev), torch.cuda.Stream(dev), torch.cuda.Stream(dev)

    def run(n_steps):
        h2d_done, cmp_done, d2h_done = {}, {}, {}
        for s_ in range(n_steps):
            dq, dk, dv, dx = sets[s_ % 2]
            with torch.cuda.stream(s_h2d):
                if s_ >= 2:
                    s_h2d.wait_event(cmp_done[s_ - 2])  # the kernels of step s-2 have consumed this input set
                dq.copy_(hq, non_blocking=True); dk.copy_(hk, non_blocking=True); dv.copy_(hv, non_blocking=True)
                dx.copy_(hx, non_blocking=True)
                h2d_done[s_] = torch.cuda.Event(); h2d_done[s_].record(s_h2d)
            with torch.cuda.stream(s_cmp):
                s_cmp.wait_event(h2d_done[s_])
                if s_ >= 2:
                    s_cmp.wait_event(d2h_done[s_ - 2])  # the results of step s-2 have left the device
                do = attn(dq, dk, dv)
                if n > 1:
                    dist.all_gather_into_tensor(xfull[s_ % 2], dx)
                    dy = mlp(xfull[s_ % 2])
                    dy = dy[r * rows:(r + 1) * rows]
                else:
                    dy = mlp(dx)
                outs[s_ % 2] = (do, dy)
                cmp_done[s_] = torch.cuda.Event(); cmp_done[s_].record(s_cmp)
            with torch.cuda.stream(s_d2h):
                s_d2h.wait_event(cmp_done[s_])
                ho.copy_(do, non_blocking=True); hy.copy_(dy, non_blocking=True)
                d2h_done[s_] = torch.cuda.Event(); d2h_done[s_].record(s_d2h)
        for s in (s_h2d, s_cmp, s_d2h):
            torch.cuda.current_stream(dev).wait_stream(s)

    if n > 1:
        mlp.symmetric_output = "view"
    steps = max(4, min(args.steps, 10))
    run(2)
    cx.barrier()
    s2, e2 = cx.ev(), cx.ev()
    for s in (s_h2d, s_cmp, s_d2h):
        s.wait_stream(torch.cuda.current_stream(dev))
    s2.record()
    for s in (s_h2d, s_cmp, s_d2h):
        s.wait_event(s2)
    run(steps)
    e2.record()
    cx.barrier()
    ms = cx.max_over_ranks([s2.elapsed_time(e2)])[0] / steps
    h2d = sum(t.numel() * t.element_size() for t in (hq, hk, hv, hx)) * n
    d2h = sum(t.numel() * t.element_size() for t in (ho, hy)) * n
    return dict(ms=ms, steps=steps, h2d=h2d, d2h=d2h)


def ring_c5_leg(cx, args):
    """BASELINE configs[4]: causal attention over one 128K-token sequence (32x128 heads, bf16), sequence-sharded zigzag
    ring with the KV hop overlapped with the local tile. T1 (one GPU, whole sequence) is measured in the same run on
    rank 0 so that the efficiency T1 / (N * TN) is self-contained."""
    torch = cx.torch
    from ml_inference_optimizer_b200 import ops
    from ml_inference_optimizer_b200.parallelism.ring import ring_attention_forward
    n, dev = cx.world, cx.dev
    S, H, D = 131072, 32, 128
    flops = 4.0 * H * S * S * D * 0.5
    iters = 3
    out = {"workload": "RingAttention causal 128K tokens, 32x128 heads, bf16 (BASELINE configs[4])", "seq": S, "n_gpus": n,
           "flops": flops}
    g = torch.Generator(device=dev).manual_seed(99 + cx.rank)
    if n > 1:
        Sl = S // n
        q, k, v = (torch.randn(1, Sl, H, D, device=dev, dtype=torch.bfloat16, generator=g) for _ in range(3))
        ms = cx.timed(lambda: ring_attention_forward(q, k, v, causal=True, partition="zigzag", overlap=True), 2, iters)
        ms_no = cx.timed(lambda: ring_attention_forward(q, k, v, causal=True, partition="zigzag", overlap=False), 1, 2)
        del q, k, v
        out.update({"partition": "zigzag", "ms": ms, "tflops_total": flops / ms / 1e9, "ms_without_overlap": ms_no,
                    "kv_bytes_per_hop": 2 * Sl * H * D * 2, "hops": n - 1,
                    "nvlink_ms_per_hop_at_770GBs": 2 * Sl * H * D * 2 / NVLINK_GBS / 1e6})
    t1 = None
    if cx.rank == 0:
        q, k, v = (torch.randn(1, S, H, D, device=dev, dtype=torch.bfloat16, generator=g) for _ in range(3))
        o = torch.empty_like(q)
        fn = lambda: ops.flash_attn_fwd(q, k, v, causal=True, out=o)
        fn(); torch.cuda.synchronize()
        s, e = cx.ev(), cx.ev()
        s.record()
        for _ in range(iters):
            fn()
        e.record()
        torch.cuda.synchronize()
        t1 = s.elapsed_time(e) / iters
        del q, k, v, o
    cx.barrier()
    if cx.rank == 0:
        out["t1_ms"] = t1
        out["t1_tflops"] = flops / t1 / 1e9
        if n > 1:
            out["efficiency_T1_over_N_TN"] = t1 / (n * out["ms"])
        else:
            out["ms"] = t1
            out["tflops_total"] = flops / t1 / 1e9
    torch.cuda.empty_cache()
    return out


def tp_breakdown_leg(cx, w, st, args):
    """N > 1: the components of the sharded step timed alone, to name the limiter from data."""
    torch = cx.torch
    from ml_inference_optimizer_b200 import ops
    mlp, x, n = st["mlp_module"], st["x"], cx.world
    q, k, v, o = st["q"], st["k"], st["v"], st["o"]
    act = w["act"]
    up, down, gate = mlp.dense_h_to_4h, mlp.dense_4h_to_h, mlp.dense_h_to_4h_gate
    gw, gb = (gate.weight, gate.bias) if gate is not None else (None, None)
    y = torch.empty(st["T"], w["h"], device=cx.dev, dtype=torch.bfloat16)
    fa = cx.timed(lambda: ops.flash_attn_fwd(q, k, v, causal=True, out=o), 2, 5)
    gemms = cx.timed(lambda: ops.fused_mlp(x, up.weight, up.bias, down.weight, None, act, gw, gb, out=y), 2, 5)
    out = {"fa_ms": fa, "mlp_gemms_alone_ms": gemms}
    payload = st["T"] * w["h"] * 2
    pool = mlp._symmetric_pool(payload, cx.dev) if mlp.reduce_impl != "nccl" else None
    if pool is not None:
        buf = pool["bufs"][0]
        t = buf.view((st["T"], w["h"]), torch.bfloat16)
        ar = cx.timed(lambda: buf.all_reduce_(t, down.bias, max_ctas=mlp.comm_ctas_single), 2, 5)
        buf.check()
        out.update({"allreduce_alone_ms": ar, "allreduce_impl": "K6 " + ("multicast" if buf.multicast else "peer"),
                    "allreduce_ctas": mlp.comm_ctas_single or "one per SM (co-resident with the GEMM CTAs)"})
    nccl = cx.timed(lambda: cx.dist.all_reduce(y), 2, 5)
    out["nccl_allreduce_alone_ms"] = nccl
    bus = 2.0 * (n - 1) / n * payload
    out["allreduce_payload_bytes"] = payload
    out["allreduce_bus_bytes_per_gpu"] = bus
    out["nvlink_floor_ms_at_770GBs"] = bus / 2 / NVLINK_GBS / 1e6  # reduce and broadcast halves move in opposite directions
    return out


def secondary_leg(cx, args):
    """N = 1: the other numbers BASELINE.json's configs name, measured by the driver's own run instead of builder logs."""
    torch = cx.torch
    import torch.nn.functional as F
    from ml_inference_optimizer_b200 import ops
    dev, bf = cx.dev, torch.bfloat16
    peaks = measured_peaks()
    out = {}
    flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    flush = lambda: flush_buf.fill_(1)  # 256 MB write: evicts the 126 MB L2

    # ---- decode attention (HBM-bound): C3 MHA and C4 GQA, batch 64 against an 8K KV cache ----
    for tag, Hq, Hkv in (("decode_c3_mha_b64_s8192", 32, 32), ("decode_c4_gqa_b64_s8192", 32, 8)):
        B, S, D = 64, 8192, 128
        kc = torch.randn(B, S, Hkv, D, device=dev, dtype=bf)
        vc = torch.randn(B, S, Hkv, D, device=dev, dtype=bf)
        qd = torch.randn(B, Hq, D, device=dev, dtype=bf)
        lens = torch.full((B,), S, device=dev, dtype=torch.int32)
        od = torch.empty_like(qd)
        ms = cx.timed(lambda: ops.decode_attention(qd, kc, vc, lens, out=od), 3, 10, flush=flush)
        nbytes = 2.0 * B * S * Hkv * D * 2
        out[tag] = {"ms": ms, "gbs": nbytes / ms / 1e6, "frac_of_hbm_peak": nbytes / ms / 1e6 / peaks["hbm_gbs"],
                    "bytes": nbytes, "l2": "flushed (256 MB write) before every iteration"}
        del kc, vc
    torch.cuda.empty_cache()

    # ---- isolated causal attention: C3 / C2 shapes ----
    for tag, (B, S, H, D), Hkv in (("attn_c3_causal", (4, 8192, 32, 128), 32), ("attn_c4_gqa_causal", (4, 8192, 32, 128), 8),
                                   ("attn_c2_causal", (8, 4096, 12, 64), 12)):
        q = torch.randn(B, S, H, D, device=dev, dtype=bf)
        k, v = (torch.randn(B, S, Hkv, D, device=dev, dtype=bf) for _ in range(2))
        o = torch.empty_like(q)
        ms = cx.timed(lambda: ops.flash_attn_fwd(q, k, v, causal=True, out=o), 3, 10)
        fl = 4.0 * B * H * S * S * D * 0.5
        rec = {"ms": ms, "tflops": fl / ms / 1e9, "frac_of_burst_peak": fl / ms / 1e9 / peaks["tflops_burst"]}
        try:  # same-GPU comparator: cuDNN SDPA
            from torch.nn.attention import SDPBackend, sdpa_kernel
            qt, kt, vt = (t.transpose(1, 2) for t in (q, k, v))
            if Hkv != H:  # the comparator gets K/V already expanded to the query heads (no GQA saving on its side)
                kt, vt = (t.repeat_interleave(H // Hkv, dim=1) for t in (kt, vt))
            with sdpa_kernel(SDPBackend.CUDNN_ATTENTION):
                ms_c = cx.timed(lambda: F.scaled_dot_product_attention(qt, kt, vt, is_causal=True), 3, 10)
            rec["cudnn_sdpa_tflops"] = fl / ms_c / 1e9
        except Exception as e:  # noqa: BLE001
            rec["cudnn_sdpa_tflops"] = None
            rec["cudnn_note"] = type(e).__name__
        out[tag] = rec
        del q, k, v, o
    torch.cuda.empty_cache()

    # ---- FusedMLP vs unfused cuBLAS + elementwise ----
    def mlp_case(tag, T, h, i, act, iters, use_graph=False):
        x = torch.randn(T, h, device=dev, dtype=bf)
        wu = (torch.randn(i, h, device=dev) * 0.02).to(bf); wd = (torch.randn(h, i, device=dev) * 0.02).to(bf)
        bu = (torch.randn(i, device=dev) * 0.02).to(bf); bd = (torch.randn(h, device=dev) * 0.02).to(bf)
        wg = bg = None
        if act == "swiglu":
            wg = (torch.randn(i, h, device=dev) * 0.02).to(bf); bg = (torch.randn(i, device=dev) * 0.02).to(bf)
        y = torch.empty(T, h, device=dev, dtype=bf)

        def ours():
            ops.fused_mlp(x, wu, bu, wd, bd, act, wg, bg, out=y)

        def unfused():
            if act == "swiglu":
                return F.linear(F.silu(F.linear(x, wg, bg)) * F.linear(x, wu, bu), wd, bd)
            return F.linear(F.gelu(F.linear(x, wu, bu), approximate="tanh"), wd, bd)

        if use_graph:  # decode-sized: launch overhead would dominate either side
            def graphed(fn):
                fn(); torch.cuda.synchronize()
                gr = torch.cuda.CUDAGraph()
                with torch.cuda.graph(gr):
                    for _ in range(10):
                        fn()
                return lambda: gr.replay()
            ours_g, unf_g = graphed(ours), graphed(unfused)
            ms_o = cx.timed(ours_g, 3, iters) / 10
            ms_u = cx.timed(unf_g, 3, iters) / 10
        else:
            ms_o = cx.timed(ours, 3, iters)
            ms_u = cx.timed(unfused, 3, iters)
        fl = (6.0 if act == "swiglu" else 4.0) * T * h * i
        out[tag] = {"ms": ms_o, "tflops": fl / ms_o / 1e9, "unfused_cublas_ms": ms_u, "speedup_vs_unfused": ms_u / ms_o,
                    "kernel": ops.last_gemm_kernel(), "timing": "CUDA graph of 10 calls" if use_graph else "events"}
        torch.cuda.empty_cache()

    mlp_case("mlp_c3_swiglu_T32768_4096_11008", 32768, 4096, 11008, "swiglu", 10)
    mlp_case("mlp_c4_swiglu_T32768_4096_14336", 32768, 4096, 14336, "swiglu", 10)
    mlp_case("mlp_c2_gelu_T32768_768_3072", 32768, 768, 3072, "gelu_tanh", 20)
    mlp_case("mlp_decode_swiglu_T64_4096_11008", 64, 4096, 11008, "swiglu", 10, use_graph=True)

    # ---- C2 layer step (attention + GELU MLP) ----
    w = WORKLOADS["c2"]
    B, S, H, D, h, i = w["B"], w["S"], w["Hq"], w["D"], w["h"], w["i"]
    q, k, v = (torch.randn(B, S, H, D, device=dev, dtype=bf) for _ in range(3))
    x = torch.randn(B * S, h, device=dev, dtype=bf)
    wu = (torch.randn(i, h, device=dev) * 0.02).to(bf); wd = (torch.randn(h, i, device=dev) * 0.02).to(bf)
    bu = torch.zeros(i, device=dev, dtype=bf); bd = torch.zeros(h, device=dev, dtype=bf)
    o, y = torch.empty_like(q), torch.empty_like(x)

    def c2_step():
        ops.flash_attn_fwd(q, k, v, causal=True, out=o)
        ops.fused_mlp(x, wu, bu, wd, bd, "gelu_tanh", out=y)
    ms = cx.timed(c2_step, 3, 20)
    fa, fm = flops_of(w)
    out["c2_layer_step"] = {"ms": ms, "tflops": (fa + fm) / ms / 1e9, "workload": w["name"]}
    del flush_buf
    torch.cuda.empty_cache()
    return out


def run_ours(args, w):
    cx = Ctx()
    torch, dist = cx.torch, cx.dist
    from ml_inference_optimizer_b200 import ops
    assert ops.arch_ok(), "needs an sm_100 device"
    n = cx.world
    if args.group_rows:
        ops.set_gemm_group_rows(args.group_rows)

    parity = parity_check(cx)
    step, st = build_step(cx, w, args)

    sampler = ClockSampler(cx.local_rank)
    if cx.rank == 0:
        sampler.start()
    warm = max(args.warmup, 3)
    for _ in range(warm):
        step()
    cx.barrier()
    start, end = cx.ev(), cx.ev()
    launches0 = ops.launch_count()
    cx.barrier()
    t_start = time.time()
    start.record()
    for _ in range(args.steps):
        step(record=True)
    end.record()
    cx.barrier()
    t_end = time.time()
    launches = ops.launch_count() - launches0
    elapsed_ms = start.elapsed_time(end)
    clocks = sampler.stop(t_start, t_end) if cx.rank == 0 else None
    ev = st["events"]
    fa_ms = statistics.mean(e[0].elapsed_time(e[1]) for e in ev)
    if n == 1:
        gemm1_ms = statistics.mean(e[1].elapsed_time(e[2]) for e in ev)
        gemm2_ms = statistics.mean(e[2].elapsed_time(e[3]) for e in ev)
        mlp_ms = gemm1_ms + gemm2_ms
    else:
        mlp_ms = statistics.mean(e[1].elapsed_time(e[2]) for e in ev)
    gemm_kernel = ops.last_gemm_kernel()
    if st["mlp_module"] is not None and st["mlp_module"].last_reduce.startswith("symmetric"):
        pool = st["mlp_module"]._symmetric_pool(1, cx.dev)
        for b in pool["bufs"]:
            b.check()
    elapsed_ms, fa_ms, mlp_ms = cx.max_over_ranks([elapsed_ms, fa_ms, mlp_ms])
    if args.dump_outputs:
        dump_outputs(cx, st, args.dump_outputs)

    e2e = e2e_leg(cx, w, st, args)
    breakdown = tp_breakdown_leg(cx, w, st, args) if n > 1 else None
    reduce_impl = st["mlp_module"].last_reduce if st["mlp_module"] is not None else None
    chunks = st["mlp_module"].overlap_chunks if st["mlp_module"] is not None else None
    comm_ctas = (st["mlp_module"].comm_ctas or "one per SM, co-resident with the GEMM CTAs") if st["mlp_module"] is not None else None
    T = st["T"]
    del st, step
    torch.cuda.empty_cache()
    ring = ring_c5_leg(cx, args) if not args.no_ring else None
    secondary = secondary_leg(cx, args) if (n == 1 and not args.no_secondary) else None

    fa, fm = flops_of(w)
    total_flops = fa + fm  # strong scaling: the job is the same at every N
    ms_per_step = elapsed_ms / args.steps
    value = total_flops / (ms_per_step * 1e-3) / 1e12
    e2e_value = total_flops / (e2e["ms"] * 1e-3) / 1e12

    if cx.rank == 0:
        peaks = measured_peaks()
        peak = peaks["tflops_sustained"]  # kernels timed inside a long step
        h, i, act = w["h"], w["i"], w["act"]
        line = {
            "metric": METRIC, "value": value, "unit": "TFLOP/s",
            "n_gpus": n, "steps": args.steps, "warmup": warm, "ms_per_step": ms_per_step,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": w["name"],
                       "parallelism": ("single GPU" if n == 1 else
                                       f"tp{n}: attention over {w['Hq'] // n} of {w['Hq']} heads per rank, FusedMLP W_up/W_gate rows and "
                                       f"W_down columns /{n}, one all-reduce of [T,h] bf16 per step inside the timed region"),
                       "l2": "inputs (q,k,v,x) exceed the 126 MB L2" if n <= 2 else "per-rank q,k,v shrink with N; x (268 MB) and the weights exceed L2",
                       "attn_flops_per_step": fa, "mlp_flops_per_step": fm, "numa_binding": cx.numa},
            "parity": parity,
            "e2e": {"value": e2e_value, "unit": "TFLOP/s", "h2d_bytes_per_step": e2e["h2d"], "d2h_bytes_per_step": e2e["d2h"],
                    "ms_per_step": e2e["ms"], "steps": e2e["steps"],
                    "api": "FlashAttention3.forward + " + ("FusedMLP*.forward" if n == 1 else "TensorParallelMLP.forward (x rows uploaded T/N per rank, all-gathered over NVLink)"),
                    "pipeline": "3 streams (H2D / kernels / D2H), double-buffered device tensors, pinned host buffers on the GPU's NUMA node; bytes are whole-job totals"},
            "gpu_launches": int(launches),
            "gpu_launches_note": "counted by the library (b200_launch_count) inside the timed region, this rank",
            "clocks": clocks,
            # the other halves of BASELINE.json's metric ("% B200 bf16 peak; prefill tok/s at 1-8 GPU"): the same timed
            # region expressed as tokens through the layer step per second (whole job) and as fractions of the dense bf16 peak
            "prefill_tokens_per_s": T / (ms_per_step * 1e-3),
            "pct_of_bf16_peak": {"measured_burst": 100.0 * value / (n * peaks["tflops_burst"]),
                                 "measured_sustained": 100.0 * value / (n * peaks["tflops_sustained"]),
                                 "nominal_2250": 100.0 * value / (n * 2250.0), "peak_source": peaks["source"]},
        }
        if n == 1:
            gemm1_flops = (4.0 if act == "swiglu" else 2.0) * T * h * i
            achieved = gemm1_flops / (gemm1_ms * 1e-3) / 1e12
            k1 = gemm_kernel.replace("NONE", "SWIGLU" if act == "swiglu" else "GELU_TANH")
            traffic, tsrc = committed_traffic(k1)
            line["roofline"] = {
                "kernel": f"{k1} (FusedMLP up{'+gate' if act == 'swiglu' else ''} GEMM, activation fused in the epilogue)",
                "bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
                "peak_source": f"MEASURED_PEAKS.json bf16_tflops_sustained ({peaks['source']}): kernel timed inside a long step",
                "ms_per_launch": gemm1_ms, "flops_per_launch": gemm1_flops, "traffic": traffic, "traffic_source": tsrc,
                "algorithmic_bytes": 2.0 * (T * h + (2 if act == "swiglu" else 1) * i * h + T * i)}
            fa_traffic, fa_src = committed_traffic("fa_fwd_kernel")
            line["roofline_attention"] = {
                "kernel": "fa_fwd_kernel (causal prefill attention)", "bound": "tensor", "achieved": fa / fa_ms / 1e9, "peak": peak,
                "unit": "TFLOP/s", "frac": fa / fa_ms / 1e9 / peak, "ms_per_launch": fa_ms, "flops_per_launch": fa,
                "traffic": fa_traffic, "traffic_source": fa_src, "timing": "CUDA events around the launch inside the timed step"}
            line["roofline"]["other_kernels_ms"] = {"fa_fwd_kernel": fa_ms, gemm_kernel + " (down projection)": gemm2_ms}
        else:
            mlp_flops_rank = fm / n
            payload = T * h * 2
            bus = 2.0 * (n - 1) / n * payload
            t_flops = mlp_flops_rank / (peak * 1e12) * 1e3
            t_link = bus / 2 / NVLINK_GBS / 1e6
            line["roofline"] = {
                "kernel": f"TensorParallelMLP step: {gemm_kernel} GEMMs on the shard + {reduce_impl} all-reduce, {chunks} token chunks overlapped",
                "bound": "tensor", "achieved": mlp_flops_rank / mlp_ms / 1e9, "peak": peak, "unit": "TFLOP/s",
                "frac": mlp_flops_rank / mlp_ms / 1e9 / peak, "ms_per_launch": mlp_ms, "flops_per_launch": mlp_flops_rank,
                "target_ms": max(t_flops, t_link), "target_rule": "max(FLOPs / measured GEMM peak, NVLink bytes per direction / 770 GB/s)",
                "achieved_over_target": max(t_flops, t_link) / mlp_ms, "traffic": None,
                "other_kernels_ms": {"fa_fwd_kernel": fa_ms}}
            line["collective"] = {"impl": reduce_impl, "payload_bytes_per_step": payload, "bus_bytes_per_gpu_per_step": bus,
                                  "comm_ctas": comm_ctas, "chunks": chunks}
            line["breakdown_ms"] = breakdown
            comp = {"attention": breakdown["fa_ms"], "mlp_gemms": breakdown["mlp_gemms_alone_ms"],
                    "allreduce": breakdown.get("allreduce_alone_ms", breakdown["nccl_allreduce_alone_ms"])}
            exposed = ms_per_step - comp["attention"] - comp["mlp_gemms"]
            line["limiter"] = {"largest_component": max(comp, key=comp.get), "components_ms": comp,
                               "allreduce_exposed_ms": exposed,
                               "note": "exposed = step - attention alone - GEMMs alone: the part of the all-reduce (and of the SMs given to it) that the chunk overlap does not hide"}
        if ring is not None:
            line["ring_c5"] = ring
        if secondary is not None:
            line["secondary"] = secondary
        if n == 1 and not args.no_cpu_baseline:
            cpu = cpu_oracle_rate(w, steps=2, warmup=1)
            line["cpu_baseline"] = {"value": cpu["value"], "unit": "TFLOP/s", "cores": cpu["cores"], "kind": "port",
                                    "sample": cpu["sample"]}
        print(json.dumps(line), flush=True)
    if n > 1:
        cx.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c3", choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true")
    ap.add_argument("--no-ring", action="store_true")
    ap.add_argument("--group-rows", type=int, default=0, help="override the GEMM L2 raster group (rows)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the last step's outputs (a fixed row sample) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl ours)")
    w = WORKLOADS[args.workload]
    if args.impl == "reference":
        run_reference(args, w)
    else:
        run_ours(args, w)


if __name__ == "__main__":
    main()
