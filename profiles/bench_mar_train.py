"""Training with the mAR channel prior: the prior on flowk kernels (autograd through mar_prior.cuda_path) vs the torch
layers (cuda_path.ENABLED = False, cuDNN with TF32 off).

  python profiles/bench_mar_train.py --out profiles/r7_mar_train.json

1. Training step: cfg2 (MixLogCDF, 32x32x3, L = 3, K = 4, width 96, B = 64) with prior="mar" under ShardedTrainer (forward +
   backward and the update replayed as CUDA graphs), --steps steps per route after warm-up, the two routes alternated,
   three rounds; the standard-prior step of the same model as context.
2. Where the prior's time goes: one eager forward + backward of each prior level at B = 64 with a CUDA-event pair around
   every flowk call (_lib.TIMING), summed per entry point; the recurrent GEMMs (forward PRE_LSTM steps and the per-step
   dgrad of the backward, B images each) are reported apart from the batched ones (T*B images).
3. Kernels per eager training step (torch.profiler, CUDA activities), in a separate leg after the timed ones.
Device name, power limit and SM clock are read in the same run.
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
from flowk import _lib, sharding  # noqa: E402
from flowk.mar_prior import ChannelPriorUniScale, cuda_path  # noqa: E402
from flowk.marscf import MarScfFlow  # noqa: E402

ROUTES = (("flowk", True), ("torch_layers", False))


def device_info():
    info = {"device": torch.cuda.get_device_name(0)}
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm,clocks.sm", "--format=csv,noheader",
                              "-i", "0"], capture_output=True, text=True, timeout=60).stdout.strip()
        info["power_limit"], info["sm_max_clock"], info["sm_clock_at_start"] = [s.strip() for s in out.split(",")]
    except Exception as e:                      # the number is still reported, marked as missing its power limit
        info["power_limit"] = "unavailable (%s)" % type(e).__name__
    return info


def set_route(on):
    cuda_path.ENABLED = on
    torch.backends.cudnn.allow_tf32 = False          # the torch layers in fp32 (the flowk route does not use cuDNN)


def time_events(fn, reps):
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def cfg2_model(dev, B, prior, seed=0):
    torch.manual_seed(seed)
    np.random.seed(seed)
    model = MarScfFlow(B, (32, 32, 3), "mixlogcdf", 3, 4, 96, prior=prior).to(dev)
    model.train()
    return model


def batches(dev, B, n=4):
    gen = torch.Generator().manual_seed(200)
    return [(torch.randint(0, 256, (B, 3, 32, 32), generator=gen).float() / 255.0 - 0.5).to(dev) for _ in range(n)]


def trainer_for(model, B, xs, graph=True):
    tr = sharding.ShardedTrainer(model, lr=1e-4, warm_up=10000, global_batch=B, use_graph=graph)
    for i in range(4):                              # 2 eager steps, capture, 1 replay
        tr.step(xs[i % len(xs)])
    return tr


def train_steps(dev, B, steps, rounds):
    xs = batches(dev, B)
    base = cfg2_model(dev, B, "mar")
    with torch.no_grad():
        base(xs[0])                                 # ActNorm data-dependent init
    trainers = {}
    for name, on in ROUTES:                         # the route is fixed when the step is captured
        set_route(on)
        trainers[name] = trainer_for(copy.deepcopy(base), B, xs)
    cuda_path.ENABLED = True
    std = cfg2_model(dev, B, None)
    with torch.no_grad():
        std(xs[0])
    trainers["standard_prior"] = trainer_for(std, B, xs)
    out = {"steps": steps, "batch": B, "graphs": True,
           "config": "cfg2 (mixlogcdf, 32x32x3, L=3, K=4, width 96) prior='mar' (3 ConvLSTM layers, hidden 32)",
           "torch_layers_route": "cuda_path.ENABLED = False, torch.backends.cudnn.allow_tf32 = False"}
    for rnd in range(rounds):
        for name in [r for r, _ in ROUTES] + ["standard_prior"]:
            tr = trainers[name]
            loss = [None]

            def one(i=[0]):
                loss[0] = tr.step(xs[i[0] % len(xs)])
                i[0] += 1
            for _ in range(3):
                one()
            ms = time_events(one, steps)
            out.setdefault(name + "_ms_per_step", []).append(round(ms, 3))
            out.setdefault(name + "_images_per_s", []).append(round(B / (ms / 1e3), 1))
            out.setdefault(name + "_loss_bits_per_dim", []).append(round(float(loss[0]), 5))
            print("train", name, rnd, ms, flush=True)
    return out


def prior_breakdown(dev, B):
    """Per level: device time per flowk entry point over one eager prior forward + backward (events around each call)."""
    res = []
    for level in (1, 2, 3):
        torch.manual_seed(level)
        prior = ChannelPriorUniScale(B, 3, 32, 32, level, 3, hidden_size=32, num_layers=3, dp_rate=0).to(dev)
        z2 = torch.randn(B, prior.nc, prior.height, prior.width, device=dev, requires_grad=True)
        z1 = torch.randn(B, prior.nc, prior.height, prior.width, device=dev, requires_grad=True) if level < 3 else None

        def step():
            prior((z1, z2) if z1 is not None else z2).sum().backward()
        for _ in range(3):
            step()
        row = {"level": level, "T": prior.nc, "map": prior.height, "B": B}
        row["fwd_bwd_ms"] = round(time_events(step, 10), 3)
        _lib.TIMING = {}
        try:
            step()
            torch.cuda.synchronize()
            per = {}
            for name, calls in _lib.TIMING.items():
                for start, end, meta in calls:
                    key = name
                    if name == "flowk_conv_gemm":
                        key += " recurrent (B images)" if meta[0] == B else " batched (T*B images)"
                    t = per.setdefault(key, [0, 0.0])
                    t[0] += 1
                    t[1] += start.elapsed_time(end)
        finally:
            _lib.TIMING = None
        row["per_entry_point"] = {k: {"calls": c, "ms": round(ms, 3)} for k, (c, ms) in sorted(per.items())}
        row["timed_calls_ms"] = round(sum(ms for _, ms in per.values()), 3)
        res.append(row)
        print("prior", row, flush=True)
    return res


def kernels_per_step(dev, B, steps=2):
    from torch.profiler import ProfilerActivity, profile
    xs = batches(dev, B)
    base = cfg2_model(dev, B, "mar")
    with torch.no_grad():
        base(xs[0])
    out = {"steps": steps, "mode": "eager steps (forward + backward + fused Adamax), torch.profiler CUDA activities"}
    for name, on in ROUTES:
        set_route(on)
        tr = trainer_for(copy.deepcopy(base), B, xs, graph=False)
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for i in range(steps):
                tr.step(xs[i % len(xs)])
            torch.cuda.synchronize()
        kern = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA
                and not e.name.lower().startswith(("memcpy", "memset"))]
        out[name + "_kernels_per_step"] = len(kern) / steps
        out[name + "_library_conv_kernels_per_step"] = sum(
            any(s in e.name.lower() for s in ("cudnn", "xmma", "implicit_convolve", "conv2d_")) for e in kern) / steps
        print("kernels", name, out[name + "_kernels_per_step"], flush=True)
    cuda_path.ENABLED = True
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r7_mar_train.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_mar_train.py measures on a CUDA device; none is available")
    dev = torch.device("cuda:0")
    res = dict(device_info())
    res["train_step"] = train_steps(dev, args.batch, args.steps, args.rounds)
    res["prior_fwd_bwd"] = prior_breakdown(dev, args.batch)
    res["kernels"] = kernels_per_step(dev, args.batch)
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
