"""Sampling from the mAR channel prior at cfg2 (3x32x32, MixLogCDF, L3 K4 C96, B = 64, prior="mar", ActNorm initialised as in
bench.py's mar_prior_leg), in one process:

  eager      `model(None, None, reverse=True)` (host noise in the reference's order, one AncestralSampler per level)
  graphed    `GraphedSampler` with 1 lane and with --depth lanes replayed round-robin (device noise inside the graph)
  launches   flowk launches per replay
  levels     per-level prior time from CUDA events around the prior calls of an eager run
  standard   the standard-prior `GraphedSampler` on the same flow, for context

Prints one JSON object and writes it to --out.  `--eager-only` runs only the eager leg (e.g. on another tree for an A/B);
`--parent-json` folds such a run's result into this one's JSON."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

B, IMAGE, L, K, C = 64, (32, 32, 3), 3, 4, 96


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = ""
    return q or torch.cuda.get_device_name(0)


def build(prior, dev):
    from flowk.marscf import MarScfFlow
    torch.manual_seed(0)
    np.random.seed(0)
    model = MarScfFlow(B, IMAGE, "mixlogcdf", L, K, C, prior=prior).to(dev)
    gen = torch.Generator().manual_seed(300)                   # bench.py synthetic_batches(4, B, IMAGE, seed=300)[0]
    x = torch.rand(B, IMAGE[2], IMAGE[0], IMAGE[1], generator=gen) - 0.5
    model.train()
    with torch.no_grad():
        model(x.to(dev))                                       # ActNorm data-dependent init
    return model.eval()


def rate(fn, steps, warmup):
    """images/s of `steps` calls of fn() after `warmup`, host clock around work that ends in a device synchronise."""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(steps):
        fn()
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    return {"images_per_s": B * steps / dt, "ms_per_batch": 1e3 * dt / steps}


def eager_leg(model, args):
    from flowk import _lib
    with torch.no_grad():
        r = rate(lambda: model(None, None, reverse=True), args.steps, args.warmup)
        before = _lib.LAUNCHES
        model(None, None, reverse=True)
        r["flowk_launches_per_batch"] = _lib.LAUNCHES - before
    return r


def level_times(model, reps):
    """ms per prior call by level, CUDA events around each call of an eager decode (median over `reps` decodes)."""
    flow = model.flow
    times = {}

    def timed(z, level, **kw):
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        out = flow.c_prior(z, level, **kw)
        e.record()
        times.setdefault(level, []).append((s, e))
        return out

    with torch.no_grad():
        for _ in range(reps):
            flow.decode(None, prior=timed)
    torch.cuda.synchronize()
    return {"level%d" % lvl: float(np.median([s.elapsed_time(e) for s, e in ev[1:]])) for lvl, ev in sorted(times.items())}


def graphed_leg(model, depth, steps, warmup):
    from flowk.graphs import GraphedSampler
    lanes = [GraphedSampler(model, B, IMAGE) for _ in range(depth)]
    i = [0]

    def submit():                                  # each lane replays on its own stream; rate() synchronises the device
        lanes[i[0] % depth].run()
        i[0] += 1

    r = rate(submit, steps * depth, warmup * depth)
    r["flowk_launches_per_replay"] = int(lanes[0].flowk_launches)
    r["lanes"] = depth
    return r


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--depth", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r6_mar_sampling.json"))
    ap.add_argument("--eager-only", action="store_true")
    ap.add_argument("--parent-json", default=None, help="JSON of an --eager-only run on the parent tree to include")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_mar_sampling.py needs a CUDA device (none found)")
    import flowk  # noqa: F401
    dev = torch.device("cuda:0")
    res = {"card": card(), "workload": "cfg2 3x32x32 MixLogCDF L3 K4 C96 B64, prior=mar (hidden 32, 3 layers)",
           "steps": args.steps, "warmup": args.warmup}
    model = build("mar", dev)
    res["eager"] = eager_leg(model, args)
    if not args.eager_only:
        res["eager_prior_ms_by_level"] = level_times(model, 5)
        res["graphed_1_lane"] = graphed_leg(model, 1, args.steps, args.warmup)
        res["graphed_%d_lanes" % args.depth] = graphed_leg(model, args.depth, args.steps, args.warmup)
        del model
        std = build(None, dev)
        res["standard_prior_graphed_1_lane"] = graphed_leg(std, 1, args.steps, args.warmup)
        res["standard_prior_graphed_%d_lanes" % args.depth] = graphed_leg(std, args.depth, args.steps, args.warmup)
    if args.parent_json:
        with open(args.parent_json) as f:
            res["parent_eager"] = json.load(f)["eager"]
        res["parent_eager"]["note"] = "the parent commit's tree, same GPU call, run just before this one"
    text = json.dumps(res, indent=1)
    print(text)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(text + "\n")


if __name__ == "__main__":
    main()
