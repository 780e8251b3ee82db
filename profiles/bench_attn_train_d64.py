"""Training attention at head dim 64 (the width-256 MixLogCDF model): the tcgen05 kernels (flowk_attention_train_tc_fwd /
_bwd) against the torch route (tc_autograd.ATTENTION_TC = False with _lib.ALLOW_LIBRARY = True: bmm + softmax + dropout in
ATen at torch's default fp32 matmul settings), alternated in one process, three rounds each.

  1. level-1 attention core, B = 64, S = 256, C = 256, 4 heads, p = 0.2: forward, and forward + backward, CUDA events over
     `--reps` calls after warm-up.  Algorithmic FLOPs per (image, head) pair: forward 4 S^2 D (Q K^T and P V), backward
     8 S^2 D (S recomputed, dP = dO V^T, dQ, dK, dV; the flash-style recompute of S is counted, torch's saved P is not);
     TFLOP/s = FLOPs / time.
  2. cfg2-shaped training step at width 256 (L = 3, K = 4, B = 64, drop_prob 0.2), ShardedTrainer with CUDA graphs:
     ms per step, the peak allocated memory while each route's trainer was built and warmed up (above what was allocated
     before), and the loss after the timed steps.

python profiles/bench_attn_train_d64.py [--reps 50] [--steps 20] [--out profiles/r11_attn_train_d64.json]"""
import argparse
import copy
import json
import os
import subprocess
import sys

import numpy as np
import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import flowk  # noqa: E402,F401
from flowk import _lib, sharding, tc_autograd  # noqa: E402
from flowk.marscf import MarScfFlow  # noqa: E402

ROUNDS = 3


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()[0]
    name, power, clock = [s.strip() for s in q.split(",")]
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def time_events(fn, reps):
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps          # ms per call


def torch_core(proj, heads, p):
    """GatedAttn's library route (flow_modules/mixlogcdf_nn.py, training mode) from the in_proj rows to the attention."""
    b, s, c3 = proj.shape
    c = c3 // 3
    d = c // heads
    kvq = proj.view(b, s, 3, heads, d).permute(2, 0, 3, 1, 4).contiguous()
    k, v, q = kvq[0], kvq[1], kvq[2] * (d ** -0.5)
    w = F.dropout(torch.softmax(q @ k.transpose(-1, -2), dim=-1), p, True)
    return (w @ v).permute(0, 2, 1, 3).reshape(b, s, c)


def core(dev, reps):
    B, S, C, heads, p = 64, 256, 256, 4, 0.2
    D = C // heads
    pairs = B * heads
    flop_fwd, flop_bwd = 4.0 * S * S * D * pairs, 8.0 * S * S * D * pairs
    g = torch.Generator().manual_seed(0)
    qkv = torch.randn(B, S, 3 * C, generator=g).to(dev).requires_grad_()
    dout = torch.randn(B, S, C, generator=g).to(dev)
    routes = {"flowk_tc": lambda x: tc_autograd.attention_core(x, heads, p, 3), "torch": lambda x: torch_core(x, heads, p)}
    out = {"shape": {"B": B, "S": S, "C": C, "heads": heads, "p": p},
           "flop_fwd": flop_fwd, "flop_fwd_bwd": flop_fwd + flop_bwd}
    for name, f in routes.items():                   # warm-up (module loads, cuBLAS algorithm choice)
        for _ in range(10):
            f(qkv).backward(dout)
    for rnd in range(ROUNDS):
        for name, f in routes.items():
            with torch.no_grad():
                ms_f = time_events(lambda: f(qkv), reps)

            def fb():
                qkv.grad = None
                f(qkv).backward(dout)
            ms_fb = time_events(fb, reps)
            out.setdefault(name + "_fwd_us", []).append(round(ms_f * 1e3, 1))
            out.setdefault(name + "_fwd_bwd_us", []).append(round(ms_fb * 1e3, 1))
            out.setdefault(name + "_fwd_tflops", []).append(round(flop_fwd / (ms_f * 1e-3) / 1e12, 2))
            out.setdefault(name + "_fwd_bwd_tflops", []).append(round((flop_fwd + flop_bwd) / (ms_fb * 1e-3) / 1e12, 2))
            print("core", name, rnd, round(ms_f * 1e3, 1), round(ms_fb * 1e3, 1), flush=True)
    return out


def set_route(name):
    tc_autograd.ATTENTION_TC = name == "flowk_tc"
    _lib.ALLOW_LIBRARY = name != "flowk_tc"


def step(dev, steps):
    B = 64
    gen = torch.Generator().manual_seed(200)
    xs = [(torch.randint(0, 256, (B, 3, 32, 32), generator=gen).float() / 255.0 - 0.5).to(dev) for _ in range(4)]
    torch.manual_seed(0)
    np.random.seed(0)
    base = MarScfFlow(B, (32, 32, 3), "mixlogcdf", 3, 4, 256).to(dev)
    base.train()
    with torch.no_grad():
        base(xs[0])                                  # ActNorm data-dependent init
    out = {"config": "mixlogcdf, 32x32x3, L=3, K=4, width 256, drop_prob 0.2, B=64", "steps": steps, "graphs": True}
    trainers = {}
    for name in ("flowk_tc", "torch"):               # the route is fixed when the step is captured
        set_route(name)
        torch.cuda.synchronize()
        before = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        tr = sharding.ShardedTrainer(copy.deepcopy(base), lr=1e-4, warm_up=10000, global_batch=B)
        for i in range(4):                           # 2 eager steps, capture, 1 replay
            tr.step(xs[i % len(xs)])
        torch.cuda.synchronize()
        out[name + "_peak_alloc_mb"] = round((torch.cuda.max_memory_allocated() - before) / 2 ** 20, 1)
        trainers[name] = tr
    for rnd in range(ROUNDS):
        for name, tr in trainers.items():
            set_route(name)
            loss = [None]

            def one(i=[0]):
                loss[0] = tr.step(xs[i[0] % len(xs)])
                i[0] += 1
            ms = time_events(one, steps)
            out.setdefault(name + "_ms_per_step", []).append(round(ms, 3))
            out.setdefault(name + "_loss_bits_per_dim", []).append(round(float(loss[0]), 5))
            print("step", name, rnd, round(ms, 3), flush=True)
    set_route("flowk_tc")
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    res = dict(gpu_info())
    res["core"] = core(dev, args.reps)
    res["train_step"] = step(dev, args.steps)
    print(json.dumps(res))
    if args.out:
        os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
