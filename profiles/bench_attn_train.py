"""Training `Transformer_attn` on the flowk kernels vs the torch-op form (flow_modules.transformer.KERNEL_TRAINING).

  python profiles/bench_attn_train.py --out profiles/r3_attn_train.json

1. Per layer: forward + backward of one Transformer_attn at the cfg2 level shapes, B = 64, CUDA events over --reps
   repetitions after warm-up, both routes alternated, two rounds.
2. Training step: cfg2 (MixLogCDF, width 96, L = 3, K = 4, B = 64) with attn=True under ShardedTrainer (forward + backward
   and the update replayed as CUDA graphs), --steps steps per route, routes alternated, two rounds.
3. Kernels per training step: eager steps under torch.profiler (CUDA activities), after the timed legs.
Device name and power limit are read in the same run.
"""
import argparse
import copy
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import flowk  # noqa: E402,F401
from flowk import sharding  # noqa: E402
from flowk.flow_modules import transformer  # noqa: E402
from flowk.marscf import MarScfFlow  # noqa: E402

ROUTES = (("kernel", True), ("torch_ops", False))
LEVELS = ((12, 16), (24, 8), (48, 4))            # cfg2 level shapes (C, H = W)


def device_info():
    info = {"device": torch.cuda.get_device_name(0)}
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=60).stdout.strip()
        info["power_limit"], info["sm_max_clock"] = [s.strip() for s in out.split(",")]
    except Exception as e:                      # the number is still reported, marked as missing its power limit
        info["power_limit"] = "unavailable (%s)" % type(e).__name__
    return info


def time_events(fn, reps):
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def per_layer(dev, B, reps):
    res = []
    for C, H in LEVELS:
        torch.manual_seed(C)
        m = transformer.Transformer_attn(C).to(dev)
        x = torch.randn(B, C, H, H, device=dev, requires_grad=True)
        ld0 = torch.zeros(B, device=dev, requires_grad=True)
        gy, gl = torch.randn(B, C, H, H, device=dev), torch.randn(B, device=dev)

        def step():
            y, ld = m(x, logdet=ld0)
            torch.autograd.backward([y, ld], [gy, gl])
        row = {"C": C, "H": H, "B": B, "reps": reps}
        for rnd in range(2):
            for name, on in ROUTES:
                transformer.KERNEL_TRAINING = on
                for _ in range(20):
                    step()
                row.setdefault(name + "_us", []).append(round(time_events(step, reps) * 1e3, 2))
        transformer.KERNEL_TRAINING = True
        res.append(row)
        print("layer", row, flush=True)
    return res


def cfg2_model(dev, B, seed=0):
    torch.manual_seed(seed)
    np.random.seed(seed)
    model = MarScfFlow(B, (32, 32, 3), "mixlogcdf", 3, 4, 96, attn=True).to(dev)
    model.train()
    return model


def batches(dev, B, n=4):
    gen = torch.Generator().manual_seed(200)
    return [(torch.randint(0, 256, (B, 3, 32, 32), generator=gen).float() / 255.0 - 0.5).to(dev) for _ in range(n)]


def train_steps(dev, B, steps):
    xs = batches(dev, B)
    base = cfg2_model(dev, B)
    with torch.no_grad():
        base(xs[0])                                 # ActNorm data-dependent init
    trainers = {}
    for name, on in ROUTES:                         # the route is fixed when the step is captured
        transformer.KERNEL_TRAINING = on
        model = copy.deepcopy(base)
        tr = sharding.ShardedTrainer(model, lr=1e-4, warm_up=10000, global_batch=B)
        for i in range(4):                          # 2 eager steps, capture, 1 replay
            tr.step(xs[i % len(xs)])
        trainers[name] = tr
    transformer.KERNEL_TRAINING = True
    out = {"steps": steps, "batch": B, "config": "cfg2 (mixlogcdf, 32x32x3, L=3, K=4, width 96) attn=True",
           "graphs": True}
    for rnd in range(2):
        for name, _ in ROUTES:
            tr = trainers[name]
            loss = [None]

            def one(i=[0]):
                loss[0] = tr.step(xs[i[0] % len(xs)])
                i[0] += 1
            ms = time_events(one, steps)
            out.setdefault(name + "_ms_per_step", []).append(round(ms, 3))
            out.setdefault(name + "_images_per_s", []).append(round(B / (ms / 1e3), 1))
            out.setdefault(name + "_loss_bits_per_dim", []).append(round(float(loss[0]), 5))
            print("train", name, rnd, ms, flush=True)
    return out


def kernels_per_step(dev, B, steps=2):
    from torch.profiler import ProfilerActivity, profile
    xs = batches(dev, B)
    base = cfg2_model(dev, B)
    with torch.no_grad():
        base(xs[0])
    out = {"steps": steps, "mode": "eager steps (forward + backward + fused Adamax), torch.profiler CUDA activities"}
    for name, on in ROUTES:
        transformer.KERNEL_TRAINING = on
        tr = sharding.ShardedTrainer(copy.deepcopy(base), lr=1e-4, warm_up=10000, global_batch=B, use_graph=False)
        for i in range(2):
            tr.step(xs[i])
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for i in range(steps):
                tr.step(xs[i % len(xs)])
            torch.cuda.synchronize()
        kern = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA
                and not e.name.lower().startswith(("memcpy", "memset"))]
        out[name + "_kernels_per_step"] = len(kern) / steps
        out[name + "_patch_attention_kernels_per_step"] = sum("patch_attention" in e.name for e in kern) / steps
        print("kernels", name, out[name + "_kernels_per_step"], flush=True)
    transformer.KERNEL_TRAINING = True
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=200)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--out", default=None, help="write the JSON here as well as to stdout")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_attn_train.py measures on a CUDA device; none is available")
    dev = torch.device("cuda:0")
    res = dict(device_info())
    res["per_layer_fwd_bwd"] = per_layer(dev, args.batch, args.reps)
    res["train_step"] = train_steps(dev, args.batch, args.steps)
    res["kernels"] = kernels_per_step(dev, args.batch)
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
