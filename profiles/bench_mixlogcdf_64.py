"""The MixLogCDF model on 64x64 images (L = 4, level 1 = 32x32 maps, 1024 tokens per attention), in one process:

  1. level-1 attention launch, B = 64, HW = 1024, 4 heads, C in {96, 128, 160, 256}: flowk_attention_long_tc (tcgen05)
     against the mma.sync kernel called directly (flowk_attention_f16), alternated, ROUNDS rounds of CUDA events over
     `--reps` launches each.  Both write fp16 (hi, lo) pairs.  Algorithmic FLOPs: 4 S^2 d per (image, head) pair.
     qkv is 201 MB at C = 256 (more than the 126 MB L2), so the launches read it from HBM.
  2. the 64x64 model (L = 4, K = 4, B = 64) at widths 128 and 256, eval mode: forward images/s through a DensityPipeline
     (two graph lanes), sampling images/s through a GraphedSampler, flowk launches per replay, and (in a separate
     torch.profiler run of one eager forward) the share of device kernel time spent in the level-1 attention kernel.
  3. a 64x64 training step, width 256, B = 16, ShardedTrainer with CUDA graphs: ms per step and peak allocated memory.
  4. one default `bench.py` line.

python profiles/bench_mixlogcdf_64.py [--reps 50] [--out profiles/r12_mixlogcdf_64.json]"""
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
import flowk  # noqa: E402,F401
from flowk import _lib, sharding  # noqa: E402
from flowk.graphs import DensityPipeline, GraphedSampler  # noqa: E402
from flowk.marscf import MarScfFlow  # noqa: E402

ROUNDS = 3
IMAGE = (64, 64, 3)


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


def attention_launch(dev, reps):
    B, HW, heads = 64, 1024, 4
    stream = torch.cuda.current_stream().cuda_stream
    out = {"shape": {"B": B, "HW": HW, "heads": heads}}
    for C in (96, 128, 160, 256):
        d = C // heads
        flop = 4.0 * HW * HW * d * B * heads
        g = torch.Generator().manual_seed(C)
        qkv = (torch.randn(B * HW, 3 * C, generator=g) * 1.5).to(dev)
        hi = torch.empty(B * HW, C, device=dev, dtype=torch.float16)
        lo = torch.empty_like(hi)
        status = torch.zeros(1, dtype=torch.int32, device=dev)
        routes = {
            "long_tc": lambda: _lib.call("flowk_attention_long_tc", qkv.data_ptr(), hi.data_ptr(), lo.data_ptr(), 1, B, HW,
                                         C, heads, status.data_ptr(), None, stream),
            "mma_sync": lambda: _lib.call("flowk_attention_f16", qkv.data_ptr(), hi.data_ptr(), lo.data_ptr(), B, HW, C,
                                          heads, stream),
        }
        res = {"d": d, "flop": flop}
        outs = {}
        for name, f in routes.items():
            for _ in range(5):
                f()
            torch.cuda.synchronize()
            outs[name] = hi.float() + lo.float()
        res["max_abs_diff"] = float((outs["long_tc"] - outs["mma_sync"]).abs().max())
        for rnd in range(ROUNDS):
            for name, f in routes.items():
                ms = time_events(f, reps)
                res.setdefault(name + "_us", []).append(round(ms * 1e3, 1))
                res.setdefault(name + "_tflops", []).append(round(flop / (ms * 1e-3) / 1e12, 2))
                print("attn C=%d" % C, name, rnd, round(ms * 1e3, 1), flush=True)
        res["status"] = int(status.item())
        out["C%d" % C] = res
        del qkv, hi, lo
    return out


def make_model(dev, B, hidden, seed=0, train=False):
    torch.manual_seed(seed)
    np.random.seed(seed)
    model = MarScfFlow(B, IMAGE, "mixlogcdf", 4, 4, hidden).to(dev)
    gen = torch.Generator().manual_seed(seed + 1)
    x = (torch.randint(0, 256, (B, 3, 64, 64), generator=gen).float() / 255.0 - 0.5).to(dev)
    model.train()
    with torch.no_grad():
        model(x)                                         # ActNorm data-dependent init
    if not train:
        model.eval()
    return model, x


def model_eval(dev, hidden, reps):
    B = 64
    model, x = make_model(dev, B, hidden)
    res = {"config": "mixlogcdf, 64x64x3, L=4, K=4, width %d, B=%d, eval" % (hidden, B)}
    pipe = DensityPipeline(model, x, depth=2)
    res["forward_flowk_launches"] = pipe.flowk_launches
    sampler = GraphedSampler(model, B, IMAGE)
    res["sampling_flowk_launches"] = sampler.flowk_launches
    for _ in range(3):
        pipe.submit(x)
        sampler.run()
    torch.cuda.synchronize()
    for rnd in range(ROUNDS):
        t0 = time.perf_counter()
        for _ in range(reps):
            pipe.submit(x)
        pipe.drain()
        torch.cuda.synchronize()
        fwd = reps * B / (time.perf_counter() - t0)
        t0 = time.perf_counter()
        for _ in range(reps):
            sampler.run()
        torch.cuda.synchronize()
        smp = reps * B / (time.perf_counter() - t0)
        res.setdefault("forward_images_per_s", []).append(round(fwd, 1))
        res.setdefault("sampling_images_per_s", []).append(round(smp, 1))
        print("model", hidden, rnd, round(fwd, 1), round(smp, 1), flush=True)
    # one eager forward under the profiler: device time of the level-1 attention kernel over all kernel time
    with torch.no_grad():
        model(x)
        torch.cuda.synchronize()
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            model(x)
            torch.cuda.synchronize()
    total = attn = 0.0
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None)
        if t is None:
            t = e.cuda_time_total
        if e.key.startswith("cuda") or "Memcpy" in e.key or "Memset" in e.key:
            continue
        total += t
        if "attention_long_tc_kernel" in e.key:
            attn += t
    res["eager_forward_kernel_us"] = round(total, 1)
    res["eager_forward_level1_attention_us"] = round(attn, 1)
    res["eager_forward_level1_attention_share"] = round(attn / max(total, 1e-9), 4)
    del pipe, sampler, model
    torch.cuda.empty_cache()
    return res


def train_step(dev, steps):
    B = 16
    model, x = make_model(dev, B, 256, seed=3, train=True)
    gen = torch.Generator().manual_seed(7)
    xs = [(torch.randint(0, 256, (B, 3, 64, 64), generator=gen).float() / 255.0 - 0.5).to(dev) for _ in range(4)]
    torch.cuda.synchronize()
    before = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    tr = sharding.ShardedTrainer(model, lr=1e-4, warm_up=10000, global_batch=B)
    for i in range(4):                                   # 2 eager steps, capture, 1 replay
        tr.step(xs[i % len(xs)])
    torch.cuda.synchronize()
    res = {"config": "mixlogcdf, 64x64x3, L=4, K=4, width 256, drop_prob 0.2 (default), B=%d, CUDA graphs" % B,
           "steps": steps, "peak_alloc_mb": round((torch.cuda.max_memory_allocated() - before) / 2 ** 20, 1)}
    for rnd in range(ROUNDS):
        loss = [None]

        def one(i=[0]):
            loss[0] = tr.step(xs[i[0] % len(xs)])
            i[0] += 1
        ms = time_events(one, steps)
        res.setdefault("ms_per_step", []).append(round(ms, 2))
        res.setdefault("loss_bits_per_dim", []).append(round(float(loss[0]), 5))
        print("train", rnd, round(ms, 2), flush=True)
    return res


def bench_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")], capture_output=True, text=True, cwd=ROOT)
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    return json.loads(lines[-1]) if lines else {"error": r.stderr[-2000:]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--model-reps", type=int, default=10)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--skip-bench", action="store_true")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    res = dict(gpu_info())
    res["attention_launch"] = attention_launch(dev, args.reps)
    res["model"] = {"C%d" % h: model_eval(dev, h, args.model_reps) for h in (128, 256)}
    res["train_step"] = train_step(dev, args.steps)
    if not args.skip_bench:
        res["bench_default"] = bench_line()
    print(json.dumps(res))
    if args.out:
        os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
