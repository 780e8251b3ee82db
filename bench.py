#!/usr/bin/env python
"""Benchmark of the mAR-SCF flow-step hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl flowk|reference] [--workload cfg2] [--dump-outputs DIR]

One "step" = one forward pass (z, log-det, bits/dim) of the whole flow stack over one batch of
synthetic images.  Default workload: cfg2 = CIFAR10-shape 3x32x32, MixLogCDF coupling, L=3 K=4 C=96,
batch 64 per GPU (BASELINE.json configs[1]).  Prints ONE JSON line on rank 0.

  value      images/s with the inputs resident in HBM (CUDA-graph replay of the stack)
  e2e        images/s through the public nn.Module API fed from pinned HOST buffers, H2D copy of the
             images and D2H read of the per-image bits/dim inside the timed region
  roofline   the dominant flowk kernel (MixLogCDF forward at the first level): algorithmic bytes per
             launch / CUDA-event time per launch, against MEASURED_PEAKS.json's HBM copy bandwidth
  cpu_baseline  the CPU oracle (a port of the reference's PyTorch code path, oracle/flow_oracle.py)
             timed on this box's host cores on a bounded sample of the same workload
  --impl reference   the same oracle as the reference arm (the reference is Python and cannot travel
             to the GPU box; see DESIGN.md)
  --dump-outputs DIR   after the timed steps of `value`, rank 0 writes what the last of them returned (latent z,
             per-image bits/dim) as float32 .npy files.  Weights and images come from fixed seeds; the
             dequantisation noise is drawn inside the CUDA graph from the seeded device generator, so it repeats
             for the same --warmup, --steps and --depth.  The same arguments give the same inputs on every run.
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (coupling, image HWC, L, K, hidden C, batch per GPU)
    "cfg1": ("affine", (32, 32, 3), 3, 4, 64, 32),
    "cfg2": ("mixlogcdf", (32, 32, 3), 3, 4, 96, 64),
    "cfg3": ("affine", (32, 32, 3), 3, 4, 256, 128),
    "cfg4": ("mixlogcdf", (32, 32, 3), 3, 4, 160, 64),
    "cfg5": ("affine", (64, 64, 3), 4, 4, 256, 32),
}
DESCRIBE = {
    "cfg1": "3x32x32 affine L3 K4 C64 B32 forward bits/dim+logdet",
    "cfg2": "CIFAR10-shape 3x32x32 MixLogCDF L3 K4 C96 B64/GPU forward bits/dim+logdet",
    "cfg3": "3x32x32 affine L3 K4 C256 B128 forward bits/dim+logdet",
    "cfg4": "ImageNet32-shape 3x32x32 MixLogCDF L3 K4 C160 B64/GPU forward bits/dim+logdet",
    "cfg5": "ImageNet64-shape 3x64x64 affine L4 K4 C256 B32/GPU forward bits/dim+logdet",
}
METRIC = "mAR-SCF CIFAR10 MixLogCDF fwd+logdet images/s"


def shared_config(workload, batch, world, depth):
    """The `config` object BOTH arms print (the driver compares them): workload, batch and what one step is."""
    return {"workload": DESCRIBE[workload], "batch_per_gpu": batch, "global_batch": batch * world,
            "step": "one forward pass (z, log-det, bits/dim) of the whole flow stack over one batch",
            "l2": "no explicit flush: inputs larger than L2 - one step streams the conditioner weight operands of 12 "
                  "couplings (cfg2: > 170 MB) through the 126 MB L2 and rotates over 8 input batches"}


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def tensor_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["bf16_tflops"]), "measured (MEASURED_PEAKS.json bf16_tflops, burst)"
    return 1590.0, "fallback (B200_PROFILING.md)"


def synthetic_batches(n, batch, image, seed):
    h, w, c = image
    gen = torch.Generator().manual_seed(seed)
    return [torch.rand(batch, c, h, w, generator=gen) - 0.5 for _ in range(n)]


def elementwise_bytes_per_image(coupling, image, L, K):
    """SURVEY.md section 8d: per tensor element of a level, 8 B for the fused ActNorm∘InvConv pass and
    12 B (affine) / 204 B (MixLogCDF incl. pass-through and flip) for the coupling."""
    h, w, c = image
    total = 0
    for lvl in range(L):
        c, h, w = c * 4, h // 2, w // 2
        n = c * h * w
        total += K * n * (8 + (204 if coupling == "mixlogcdf" else 12))
        if lvl < L - 1:
            c //= 2
    return total


# --------------------------------------------------------------------------------------------
# CPU oracle arm (cpu_baseline and --impl reference)
# --------------------------------------------------------------------------------------------
def oracle_state(coupling, image, L, K, hidden, batch):
    """Random-init weights of the named architecture, built on the CPU from the oracle's own key
    layout (no flowk import: the reference arm must not touch the product)."""
    from oracle import flow_oracle as O
    gen = torch.Generator().manual_seed(0)
    rng = np.random.RandomState(0)
    sd = {}
    h, w, c = image
    idx = 0
    for lvl in range(L):
        c, h, w = c * 4, h // 2, w // 2
        idx += 1                                    # squeeze layer
        for _ in range(K):
            pre = "flow.layers.%d." % idx
            sd[pre + "actnormlayer.bias"] = torch.randn(1, c, 1, 1, generator=gen) * 0.1
            sd[pre + "actnormlayer.logs"] = torch.randn(1, c, 1, 1, generator=gen) * 0.1
            q = np.linalg.qr(rng.randn(c, c))[0].astype(np.float32)
            import scipy.linalg
            p_, l_, u_ = scipy.linalg.lu(q)
            s_ = np.diag(u_)
            sd[pre + "invert_1x1_layer.p"] = torch.from_numpy(p_.astype(np.float32))
            sd[pre + "invert_1x1_layer.l"] = torch.from_numpy(l_.astype(np.float32))
            sd[pre + "invert_1x1_layer.u"] = torch.from_numpy(np.triu(u_, 1).astype(np.float32))
            sd[pre + "invert_1x1_layer.sign_s"] = torch.from_numpy(np.sign(s_).astype(np.float32))
            sd[pre + "invert_1x1_layer.log_s"] = torch.from_numpy(np.log(np.abs(s_)).astype(np.float32))
            cp = pre + "coupling."
            half = c // 2

            def rnd(*shape, std=0.05):
                return torch.randn(*shape, generator=gen) * std

            if coupling == "affine":
                sd[cp + "NN_net.conv1.weight"] = rnd(hidden, half, 3, 3)
                sd[cp + "NN_net.conv2.weight"] = rnd(hidden, hidden, 1, 1)
                for n_ in ("conv1", "conv2"):
                    sd[cp + "NN_net.%s.actnorm.bias" % n_] = rnd(1, hidden, 1, 1)
                    sd[cp + "NN_net.%s.actnorm.logs" % n_] = rnd(1, hidden, 1, 1)
                sd[cp + "NN_net.conv3.weight"] = rnd(c, hidden, 3, 3, std=0.01)
                sd[cp + "NN_net.conv3.bias"] = rnd(c, std=0.01)
                sd[cp + "NN_net.conv3.logs"] = rnd(c, 1, 1, std=0.01)
            else:
                def wn(key, *shape, bias=True):
                    sd[cp + key + "weight_v"] = rnd(*shape)
                    sd[cp + key + "weight_g"] = torch.ones(shape[0], *([1] * (len(shape) - 1)))
                    if bias:
                        sd[cp + key + "bias"] = rnd(shape[0], std=0.01)
                wn("nn.in_conv.conv.", hidden, half, 3, 3)
                for blk in range(10):
                    bp = "nn.mid_convs.%d." % blk
                    wn(bp + "conv.conv.conv.", hidden, 2 * hidden, 3, 3)
                    wn(bp + "conv.gate.conv.", 2 * hidden, 2 * hidden, 1, 1)
                    wn(bp + "attn.in_proj.", 3 * hidden, hidden, bias=False)
                    wn(bp + "attn.gate.", 2 * hidden, hidden)
                    for nm in ("norm_1", "norm_2"):
                        sd[cp + bp + nm + ".weight"] = torch.ones(hidden)
                        sd[cp + bp + nm + ".bias"] = torch.zeros(hidden)
                wn("nn.out_conv.conv.", 98 * half, hidden, 3, 3)
                sd[cp + "nn.rescale.weight_g"] = torch.ones(half, 1, 1)
                sd[cp + "nn.rescale.weight_v"] = torch.ones(half, 1, 1)
            idx += 1
        if lvl < L - 1:
            idx += 1                                # split layer
            c //= 2
    return sd


def time_oracle(sd, coupling, image, L, K, sample, steps, warmup):
    from oracle import flow_oracle as O
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    xs = synthetic_batches(2, sample, image, seed=0)
    noise = synthetic_batches(1, sample, image, seed=1)[0] + 0.5
    times = []
    with torch.no_grad():
        for i in range(warmup + steps):
            t0 = time.perf_counter()
            O.normal_flow(sd, xs[i % 2], noise, L, K, coupling)
            dt = time.perf_counter() - t0
            if i >= warmup:
                times.append(dt)
    return sample / (sum(times) / len(times)), cores, sum(times) / len(times)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    coupling, image, L, K, hidden, batch = WORKLOADS[args.workload]
    sample = args.cpu_sample or batch               # the SAME batch the flowk arm steps over (cfg2: 64 images)
    sd = oracle_state(coupling, image, L, K, hidden, sample)
    ips, cores, sec = time_oracle(sd, coupling, image, L, K, sample, args.steps, args.warmup)
    line = {
        "impl": "reference", "metric": METRIC, "value": ips, "unit": "images/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": shared_config(args.workload, sample, 1, 1),
        "note": "CPU oracle = port of the reference's PyTorch code path (the reference is a Python tree that cannot "
                "travel to the GPU box); all host cores through torch's intra-op threads; rank 0 only",
        "cpu_baseline": {"value": ips, "unit": "images/s", "cores": cores, "kind": "port",
                         "sample": "%d images per step (the full batch), %d steps" % (sample, args.steps)},
        "e2e": {"value": ips, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


# --------------------------------------------------------------------------------------------
# clocks
# --------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag, self.max_mhz = index, [], set(), False, None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {"hw_slowdown": nv.nvmlClocksThrottleReasonHwSlowdown,
                 "hw_thermal_slowdown": nv.nvmlClocksThrottleReasonHwThermalSlowdown,
                 "sw_thermal_slowdown": nv.nvmlClocksThrottleReasonSwThermalSlowdown,
                 "sw_power_cap": nv.nvmlClocksThrottleReasonSwPowerCap}
        while not self.stop_flag:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.handle, nv.NVML_CLOCK_SM))
                mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle)
                for k, bit in names.items():
                    if mask & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            time.sleep(0.02)

    def summary(self):
        med = float(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


# --------------------------------------------------------------------------------------------
# flowk arm
# --------------------------------------------------------------------------------------------
def build_model(workload, device):
    import flowk  # noqa: F401
    from flowk.marscf import MarScfFlow
    coupling, image, L, K, hidden, batch = WORKLOADS[workload]
    torch.manual_seed(0)
    np.random.seed(0)
    model = MarScfFlow(batch, image, coupling, L, K, hidden).to(device)
    x0 = synthetic_batches(1, batch, image, seed=0)[0].to(device)
    model.train()
    with torch.no_grad():
        model(x0)                                   # ActNorm data-dependent init (reference: first train batch)
    model.eval()
    return model


def kernel_table(timing):
    """name -> (launches, mean microseconds, int args of the first launch)."""
    out = {}
    for name, recs in timing.items():
        groups = {}
        for s, e, meta in recs:
            groups.setdefault(meta, []).append(s.elapsed_time(e) * 1e3)
        out[name] = {str(k): (len(v), float(np.mean(v))) for k, v in groups.items()}
    return out


def run_flowk(args):
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: the flowk arm needs a CUDA device (no CPU fallback); use --impl reference")
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=device)

    import flowk  # noqa: F401
    from flowk import _lib
    from flowk.graphs import DensityPipeline, GraphedDensity

    coupling, image, L, K, hidden, batch = WORKLOADS[args.workload]
    model = build_model(args.workload, device)
    host = [t.pin_memory() for t in synthetic_batches(8, batch, image, seed=100 + rank)]
    pool = [t.to(device) for t in host]
    graphed = DensityPipeline(model, pool[0], depth=args.depth) if args.depth > 1 else GraphedDensity(model, pool[0])
    single = graphed.lanes[0] if args.depth > 1 else graphed
    nll_sum = torch.zeros(1, device=device)
    host_out = [torch.empty(batch, pin_memory=True) for _ in range(8)]

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def reduce_bits(nll):
        if dist is not None:                      # the path's only exchange in evaluation: the bits/dim sum
            nll_sum.copy_(nll.sum().reshape(1))
            dist.all_reduce(nll_sum)

    lane_sums = {}

    def reduce_on_lane(lane):                     # runs on the lane's stream right after its replay
        if dist is not None:
            buf = lane_sums.get(id(lane))
            if buf is None:
                buf = lane_sums[id(lane)] = torch.zeros(1, device=device)
            buf.copy_(lane.static_nll.sum().reshape(1))
            dist.all_reduce(buf)

    def resident_step(i):
        if args.depth > 1:
            graphed.submit(pool[i % len(pool)], after=reduce_on_lane)
            return
        _, nll = graphed.run(pool[i % len(pool)])
        reduce_bits(nll)

    def e2e_step(i):
        if args.depth > 1:                                    # H2D, replay and D2H all on the lane's stream
            graphed.submit(host[i % len(host)], host_out[i % len(host_out)], after=reduce_on_lane)
            return
        _, nll = graphed.run(host[i % len(host)])             # H2D from pinned memory, then replay
        host_out[i % len(host_out)].copy_(nll, non_blocking=True)   # D2H of the per-image bits/dim
        reduce_bits(nll)

    def latency_step(i):                                      # one batch at a time, same stream: per-batch latency
        _, nll = single.run(pool[i % len(pool)])
        reduce_bits(nll)

    def finish_steps():
        if args.depth > 1:
            graphed.drain()

    def timed(step_fn):
        for i in range(args.warmup):
            step_fn(i)
        finish_steps()
        barrier()
        sampler = ClockSampler(local_rank)
        sampler.start()
        start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        start.record()
        for i in range(args.steps):
            step_fn(i)
        finish_steps()
        end.record()
        barrier()
        sampler.stop_flag = True
        sampler.join()
        ms = start.elapsed_time(end)
        if dist is not None:
            t = torch.tensor([ms], device=device)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t)
        return ms, sampler.summary()

    ms_res, clocks = timed(resident_step)
    if args.dump_outputs and rank == 0:             # before the e2e and latency legs replay the same graphs
        last = graphed.lanes[(graphed.i - 1) % args.depth] if args.depth > 1 else graphed
        dump_outputs(args.dump_outputs, {"z": last.static_z, "bits_per_dim": last.static_nll})
    ms_e2e, _ = timed(e2e_step)
    ms_lat, _ = timed(latency_step)
    images = batch * world * args.steps
    value = images / (ms_res / 1e3)
    e2e = images / (ms_e2e / 1e3)

    # ---- per-kernel CUDA-event timing of the flowk launches over the same K steps (eager, rank 0) -------
    hbm_peak, peak_src = peaks()
    roofline = roofline_elementwise = kernels = None
    if rank == 0:
        with torch.no_grad():
            for i in range(3):
                model(pool[i % len(pool)])
            torch.cuda.synchronize()
            _lib.TIMING = {}
            for i in range(args.steps):
                model(pool[i % len(pool)])
            torch.cuda.synchronize()
            kernels = kernel_table(_lib.TIMING)
            _lib.TIMING = None
        dom = "flowk_mixlogcdf_fwd" if coupling == "mixlogcdf" else "flowk_affine_coupling_fwd"
        per_elem = 204 if coupling == "mixlogcdf" else 12
        best = None
        for meta, (n, us) in kernels[dom].items():
            bb, cc, hw = eval(meta)
            nbytes = per_elem * bb * cc * hw
            if best is None or nbytes > best[0]:
                best = (nbytes, us, n, (bb, cc, hw))
        nbytes, us, n, shape = best
        achieved = nbytes / (us * 1e-6) / 1e9
        traffic = None
        prof = os.path.join(ROOT, "profiles", "r1_mixlogcdf_fwd_tma_ncu.json")
        if coupling == "mixlogcdf" and os.path.exists(prof) and shape == (64, 12, 256):
            with open(prof) as f:
                traffic = json.load(f)["dram_bytes_per_launch"]
        roofline_elementwise = {
            "bound": "hbm", "kernel": dom + " B,C,HW=%s" % (shape,), "achieved": achieved, "peak": hbm_peak,
            "unit": "GB/s", "frac": achieved / hbm_peak, "traffic": traffic, "bytes_per_launch": nbytes,
            "us_per_launch": us, "launches_timed": n, "peak_source": peak_src,
            "note": "eager launches timed with CUDA events (includes the launch gap); operands were just written by "
                    "the conditioner and partly sit in L2 at this batch size; roofline_large is the HBM-resident figure"}
        # dominant kernel of the step: the tcgen05 implicit-GEMM conditioner layer with the most work (launches x flops)
        roofline = roofline_elementwise
        if "flowk_conv_gemm" in kernels:
            tf_peak, tf_src = tensor_peak()
            top = None
            for meta, (n, us) in kernels["flowk_conv_gemm"].items():
                gb, gh, gw, cin, nn, taps, pre = eval(meta)
                work = n * 2.0 * gb * gh * gw * nn * taps * cin      # eager per-launch times are host-launch-bound (all
                if top is None or work > top[0]:                     # ~equal): rank the layers by algorithmic work
                    top = (work, n, us, (gb, gh, gw, cin, nn, taps, pre))
            _, n, us_eager, (gb, gh, gw, cin, nn, taps, pre) = top
            flops = 2.0 * gb * gh * gw * nn * taps * cin
            from flowk import conditioner_tc
            cin_op = cin                                      # channels of the operand the kernel was called with
            us, us_l2, rot_bytes = time_conv_gemm_isolated(device, gb, gh, gw, cin_op, nn, taps, conditioner_tc.F16)
            ach = flops / (us * 1e-6) / 1e12
            gemm_traffic = None            # dram bytes of this launch from the committed ncu --set full capture
            prof = os.path.join(ROOT, "profiles", "r2_conv_gemm_f16_ncu_summary.json")
            if os.path.exists(prof) and (gb, gh, gw, cin, nn, taps, pre) == (64, 16, 16, 192, 96, 9, 0):
                try:
                    with open(prof) as f:
                        gemm_traffic = float(json.load(f)["dram_bytes_per_launch"])
                except (KeyError, ValueError, IndexError):
                    gemm_traffic = None
            roofline = {
                "bound": "tensor", "kernel": "flowk_conv_gemm %s Cin=%d N=%d @%dx%d B=%d" % (
                    "3x3" if taps == 9 else "1x1", cin, nn, gh, gw, gb),
                "achieved": ach, "peak": tf_peak, "unit": "TFLOP/s", "frac": ach / tf_peak, "traffic": gemm_traffic,
                "flops_per_launch": flops, "us_per_launch": us, "us_per_launch_l2_resident": us_l2,
                "us_per_launch_eager_in_step": us_eager, "launches_in_step": n, "rotating_working_set_mb": rot_bytes / 1e6,
                "algorithmic_bytes_per_launch": 4.0 * (gb * gh * gw * cin + nn * taps * cin + gb * gh * gw * nn),
                "peak_source": tf_src,
                "note": "algorithmic flops 2*M*N*K of the fp32 convolution; the kernel runs 3 tcgen05 kind::f16 passes over "
                        "fp16 (hi, lo) operand pairs (two-term split for the 1e-4 fp32 parity budget), i.e. its own ceiling is "
                        "peak/3; timed in isolation: 10 back-to-back launches per CUDA-graph replay on rotating operand / "
                        "output buffers larger than L2, CUDA events on the launching stream; us_per_launch_eager_in_step "
                        "is the per-launch event time inside the eager step (includes the host launch gap)"}

    # ---- the same kernel with a working set far beyond L2 (true HBM-bound figure) --------------------------
    roofline_large = None
    if rank == 0 and coupling == "mixlogcdf" and not args.no_large:
        from flowk import ops
        bl, c, hw = 1024, 12, 256
        x = torch.randn(bl, c, 16, 16, device=device)
        raw = torch.randn(bl, 98 * (c // 2), 16, 16, device=device)
        res = torch.ones(c // 2, device=device)
        ldj = torch.zeros(bl, device=device)
        for _ in range(3):
            ops.mixlogcdf_coupling(x, raw, res, ldj, False, True, 32)
        torch.cuda.synchronize()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = 10
        s.record()
        for _ in range(reps):
            ops.mixlogcdf_coupling(x, raw, res, ldj, False, True, 32)
        e.record()
        torch.cuda.synchronize()
        us = s.elapsed_time(e) * 1e3 / reps
        nbytes = 204 * bl * c * hw
        roofline_large = {"kernel": "flowk_mixlogcdf_fwd B,C,HW=(%d, %d, %d)" % (bl, c, hw), "bound": "hbm",
                          "achieved": nbytes / (us * 1e-6) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                          "frac": nbytes / (us * 1e-6) / 1e9 / hbm_peak, "bytes_per_launch": nbytes,
                          "us_per_launch": us, "working_set_mb": nbytes / 1e6}
        del x, raw

    # ---- CPU baseline: the oracle on this box's host cores, bounded sample, rank 0 at N=1 only ---------------
    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        sample = args.cpu_sample or batch
        sd = {k: v.detach().cpu() for k, v in model.state_dict().items()}
        ips, cores, sec = time_oracle(sd, coupling, image, L, K, sample, 3, 1)
        cpu_baseline = {"value": ips, "unit": "images/s", "cores": cores, "kind": "port",
                        "sample": "%d images per step (the full batch), 3 timed steps after 1 warm-up (%.2f s/step)"
                                  % (sample, sec)}

    # ---- training step (fwd + bwd + Adamax + gradient all-reduce), the metric's second half ---------------------------
    train = train_strong = None
    if not args.no_train:
        train = train_leg(args, device, rank, world, dist, "weak")
        if world > 1 and WORKLOADS[args.workload][5] % world == 0:
            train_strong = train_leg(args, device, rank, world, dist, "strong")
        elif train is not None:
            train_strong = dict(train, scaling="strong", note="N = 1: strong and weak scaling coincide")

    # ---- inverse pass (sampling), every rank -------------------------------------------------------------------------
    inverse = None
    if not args.no_inverse:
        inverse = inverse_leg(args, model, device, rank, world, dist)

    other = None
    if rank == 0 and world == 1 and not args.no_other_configs:
        other = other_configs_leg(args, device)

    mar = None
    if not args.no_mar:
        mar = mar_prior_leg(args, device, rank, world, dist)

    # ---- HBM rooflines of the flow-level kernels, working set >> L2 (rank 0) ----------------------------------------------
    roofline_flow_kernels = None
    if rank == 0 and not args.no_large:
        roofline_flow_kernels = elementwise_rooflines(device, hbm_peak)

    if rank == 0:
        ew_bytes = elementwise_bytes_per_image(coupling, image, L, K)
        line = {
            "metric": METRIC, "value": value, "unit": "images/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_res / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": shared_config(args.workload, batch, world, args.depth),
            "run": {"batches_in_flight": args.depth,
                    "l2": "no explicit flush: one step streams the conditioner weight operands of 12 couplings (cfg2: "
                          ">170 MB) through the 126 MB L2 and rotates over 8 input batches",
                    "prior": "standard normal (the mAR ConvLSTM prior is a plug-in outside the north-star path)",
                    "conditioner": "flowk tcgen05 implicit GEMMs + attention kernel, inside the CUDA graph",
                    "bits_dim_allreduce": "every step, on the replaying stream (N > 1)"},
            "e2e": {"value": e2e, "unit": "images/s", "h2d_bytes_per_step": int(host[0].numel() * 4),
                    "d2h_bytes_per_step": int(batch * 4), "ms_per_step": ms_e2e / args.steps},
            "single_stream": {"value": images / (ms_lat / 1e3), "unit": "images/s", "ms_per_step": ms_lat / args.steps,
                              "note": "one batch in flight: the per-batch latency of the stack"},
            "gpu_launches": int(graphed.flowk_launches * args.steps),
            "flowk_launches_per_step": int(graphed.flowk_launches),
            "clocks": clocks,
            "roofline": roofline,
            "roofline_elementwise": roofline_elementwise,
            "roofline_large": roofline_large,
            "cpu_baseline": cpu_baseline,
            "train": train,
            "train_strong": train_strong,
            "inverse": inverse,
            "mar_prior": mar,
            "other_configs": other,
            "roofline_flow_kernels": roofline_flow_kernels,
            "elementwise_bytes_per_image": ew_bytes,
            "kernels": kernels,
        }
        print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()


def dump_outputs(out_dir, arrays):
    """Writes each tensor as `<out_dir>/<name>.npy` in float32, so that two builds can be compared output for output."""
    host = {name: t.detach().float().cpu().numpy() for name, t in arrays.items()}
    assert sum(a.nbytes for a in host.values()) <= 64 << 20
    os.makedirs(out_dir, exist_ok=True)
    for name, a in host.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def time_conv_gemm_isolated(device, gb, gh, gw, cin, nn, taps, f16=True, sets=10, reps=5):
    """The dominant conditioner GEMM on its own: `sets` launches on DIFFERENT operand / output buffers (together larger
    than the 126 MB L2, so no launch finds its activations cached) captured in one CUDA graph - back-to-back launches on
    one stream with no host launch gap - and timed with CUDA events on that stream.  Returns (us per launch with rotating
    buffers, us per launch re-using one L2-resident buffer set)."""
    from flowk import tc
    m = gb * gh * gw
    k = 3 if taps == 9 else 1
    w = torch.randn(nn, cin, k, k, device=device) / (taps * cin) ** 0.5
    bias = torch.randn(nn, device=device)
    if f16:
        w_hi, w_lo, sc = tc.conv_weight_operand_f16(w)
    else:
        (w_hi, w_lo), sc = tc.conv_weight_operand(w), None
    odt = torch.float16 if f16 else torch.float32
    bufs = []
    for _ in range(sets):
        a = torch.randn(m, cin, device=device)
        a_hi, a_lo = tc.split_rows_f16(a) if f16 else tc.split_rows(a)
        bufs.append((a_hi, a_lo, torch.empty(m, 2 * nn, device=device, dtype=odt), torch.empty(m, 2 * nn, device=device, dtype=odt)))

    def launch(b):
        tc.conv_gemm(b[0], b[1], w_hi, w_lo, gb, gh, gw, cin, nn, taps, tc.PRE_BIAS, tc.OUT_HILO_CELU, bias=bias,
                     out_hi=b[2], out_lo=b[3], acc_scale=sc)

    def timed(seq):
        for b in seq:
            launch(b)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            for b in seq:
                launch(b)
        g.replay()
        torch.cuda.synchronize()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for _ in range(reps):
            g.replay()
        e.record()
        torch.cuda.synchronize()
        return s.elapsed_time(e) * 1e3 / (reps * len(seq))

    per_set = sum(t.numel() * t.element_size() for t in bufs[0])
    return timed(bufs), timed([bufs[0]] * sets), per_set * sets


def inverse_leg(args, model, device, rank, world, dist):
    """Sampling throughput (the inverse pass the north star names; marscf_main.py:167-175,223-231): latents drawn from
    N(0,1) on the device, `FlowNet.decode_latents`, NaN/clamp post-processing, all inside one CUDA graph per lane;
    `e2e` adds the D2H copy of the images into pinned host memory.  Weak scaling: every rank samples its own batch."""
    from flowk.graphs import GraphedSampler
    coupling, image, L, K, hidden, batch = WORKLOADS[args.workload]
    depth = max(1, args.depth)
    lanes = [GraphedSampler(model, batch, image) for _ in range(depth)]
    host_img = [torch.empty(batch, image[2], image[0], image[1], pin_memory=True) for _ in range(depth)]

    def run(steps, to_host, single):
        for i in range(steps):
            lane = lanes[0] if single else lanes[i % depth]
            lane.run(host_img[i % depth] if to_host else None)
        for lane in lanes:
            torch.cuda.current_stream().wait_stream(lane.stream)

    def timed(to_host, single):
        run(max(3, args.warmup), to_host, single)
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        run(args.steps, to_host, single)
        e.record()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()
        ms = s.elapsed_time(e)
        if dist is not None:
            t = torch.tensor([ms], device=device)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t)
        return ms

    ms_res, ms_e2e, ms_single = timed(False, False), timed(True, False), timed(False, True)
    images = batch * world * args.steps
    finite = bool(torch.isfinite(lanes[0].images).all())
    return {"value": images / (ms_res / 1e3), "unit": "images/s", "ms_per_step": ms_res / args.steps,
            "e2e": {"value": images / (ms_e2e / 1e3), "unit": "images/s", "h2d_bytes_per_step": 0,
                    "d2h_bytes_per_step": int(host_img[0].numel() * 4)},
            "single_stream": {"value": images / (ms_single / 1e3), "ms_per_step": ms_single / args.steps},
            "batches_in_flight": depth, "batch_per_gpu": batch, "flowk_launches_per_step": int(lanes[0].flowk_launches),
            "finite": finite,
            "note": "sampling = inverse pass of the whole stack incl. drawing the latents; MixLogCDF: register-resident "
                    "per-element bisection (log_dist.py:43-72), affine: closed form"}


def other_configs_leg(args, device):
    """Driver-visible numbers for the BASELINE.json configs the headline does not run (rank 0, one GPU, a few seconds
    each): forward (z, log-det, bits/dim) and inverse (sampling) images/s by CUDA-graph replay, `depth` batches in flight.
    Parity of each config at its real width is tests/test_gpu_parity.py::test_baseline_config_vs_oracle."""
    from flowk.graphs import DensityPipeline, GraphedSampler
    out = {}
    for name in ("cfg1", "cfg3", "cfg4", "cfg5"):
        if name == args.workload:
            continue
        coupling, image, L, K, hidden, batch = WORKLOADS[name]
        model = build_model(name, device)
        xs = [t.to(device) for t in synthetic_batches(4, batch, image, seed=400)]
        depth = max(1, args.depth)
        pipe = DensityPipeline(model, xs[0], depth=depth)
        lanes = [GraphedSampler(model, batch, image) for _ in range(depth)]

        def fwd(steps):
            for i in range(steps):
                pipe.submit(xs[i % len(xs)])
            pipe.drain()

        def inv(steps):
            for i in range(steps):
                lanes[i % depth].run()
            for lane in lanes:
                torch.cuda.current_stream().wait_stream(lane.stream)

        res = {}
        for key, fn in (("forward", fwd), ("inverse", inv)):
            fn(3)
            torch.cuda.synchronize()
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            fn(args.steps)
            e.record()
            torch.cuda.synchronize()
            ms = s.elapsed_time(e)
            res[key] = {"value": batch * args.steps / (ms / 1e3), "unit": "images/s", "ms_per_step": ms / args.steps}
        res["workload"] = DESCRIBE[name]
        res["batch"] = batch
        res["batches_in_flight"] = depth
        out[name] = res
        del pipe, lanes, model
        torch.cuda.empty_cache()
    return out


def mar_prior_leg(args, device, rank, world, dist):
    """The same forward step with the reference's REAL objective: the mAR ConvLSTM channel prior (marscf_main.py:147-148,
    159-164) instead of N(0,1) - bits/dim as the reference computes it.  The prior's convolutions and LSTM cells run on
    the flowk tensor-core kernels (mar_prior/cuda_path.py); the whole step is one CUDA graph per lane."""
    import flowk  # noqa: F401
    from flowk.graphs import DensityPipeline
    from flowk.marscf import MarScfFlow
    coupling, image, L, K, hidden, batch = WORKLOADS[args.workload]
    torch.manual_seed(0)
    np.random.seed(0)
    model = MarScfFlow(batch, image, coupling, L, K, hidden, prior="mar").to(device)
    xs = [t.to(device) for t in synthetic_batches(4, batch, image, seed=300 + rank)]
    model.train()
    with torch.no_grad():
        model(xs[0])
    model.eval()
    pipe = DensityPipeline(model, xs[0], depth=max(1, args.depth))

    def run(steps):
        for i in range(steps):
            pipe.submit(xs[i % len(xs)])
        pipe.drain()

    run(max(3, args.warmup))
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    run(args.steps)
    e.record()
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    ms = s.elapsed_time(e)
    if dist is not None:
        t = torch.tensor([ms], device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t)
    return {"value": batch * world * args.steps / (ms / 1e3), "unit": "images/s", "ms_per_step": ms / args.steps,
            "batches_in_flight": max(1, args.depth), "flowk_launches_per_step": int(pipe.flowk_launches),
            "bits_per_dim_first_image": float(pipe.lanes[0].static_nll[0]),
            "note": "forward (z, log-det, bits/dim) with the mAR ConvLSTM channel prior (hidden 32, 3 layers; k=5 dil 2 / "
                    "k=5 / k=3; sequence over 6 / 12 / 48 channels) evaluated on the flowk tcgen05 kernels, random-init prior"}


def elementwise_rooflines(device, hbm_peak):
    """HBM rooflines of the flow-level kernels with working sets far beyond the 126 MB L2 (SURVEY.md section 8d bytes:
    8 B per element for the fused ActNorm∘InvConv channel mix, 12 B per element for the affine coupling)."""
    from flowk import ops
    out = {}

    def time_us(fn, reps=10):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for _ in range(reps):
            fn()
        e.record()
        torch.cuda.synchronize()
        return s.elapsed_time(e) * 1e3 / reps

    for c, hw in ((12, 16), (24, 8), (48, 4), (96, 4)):
        bl = min(65535, (512 << 20) // (c * hw * hw * 4))      # <= 512 MB input + as much output (grid.y = batch)
        x = torch.randn(bl, c, hw, hw, device=device)
        mat = torch.linalg.qr(torch.randn(c, c, device=device))[0].contiguous()
        bias = torch.randn(c, device=device)
        ldj = torch.zeros(bl, device=device)
        add = torch.ones(1, device=device)
        us = time_us(lambda: ops.channel_mix(x, mat, bias, ldj, add, False, False))
        nbytes = 8 * x.numel()
        out["channel_mix_C%d" % c] = {"bound": "hbm", "kernel": "flowk_channel_mix B,C,H,W=(%d, %d, %d, %d)" % (bl, c, hw, hw),
                                      "achieved": nbytes / (us * 1e-6) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                                      "frac": nbytes / (us * 1e-6) / 1e9 / hbm_peak, "bytes_per_launch": nbytes,
                                      "us_per_launch": us, "flop_per_byte": 2.0 * c * c / (8.0 * c)}
        del x
    bl, c, hw = 16384, 12, 16
    x = torch.randn(bl, c, hw, hw, device=device)
    h = torch.randn(bl, c, hw, hw, device=device)
    ldj = torch.zeros(bl, device=device)
    for name, rev in (("affine_fwd", False), ("affine_inv", True)):
        us = time_us(lambda: ops.affine_coupling(x, h, ldj, rev))
        nbytes = 12 * x.numel()
        out[name] = {"bound": "hbm", "kernel": "flowk_affine_coupling_%s B,C,H,W=(%d, %d, %d, %d)" % (
                         "inv" if rev else "fwd", bl, c, hw, hw),
                     "achieved": nbytes / (us * 1e-6) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                     "frac": nbytes / (us * 1e-6) / 1e9 / hbm_peak, "bytes_per_launch": nbytes, "us_per_launch": us}
    return out


def train_leg(args, device, rank, world, dist, scaling="weak"):
    """Training images/s on the same workload: the reference's step (marscf_main.py:331-347) with the batch sharded
    over ranks (64 images per GPU, weak scaling) and the gradients all-reduced over NCCL in flat buckets."""
    import flowk  # noqa: F401
    from flowk import sharding
    from flowk.marscf import MarScfFlow
    coupling, image, L, K, hidden, batch = WORKLOADS[args.workload]
    if scaling == "strong":                             # the reference divides ONE global batch (marscf_main.py:290)
        assert batch % world == 0
        batch = batch // world
    torch.manual_seed(0)
    np.random.seed(0)
    model = MarScfFlow(batch, image, coupling, L, K, hidden).to(device)
    model.train()
    xs = [t.to(device) for t in synthetic_batches(4, batch, image, seed=200 + rank)]
    with torch.no_grad():
        model(xs[0])                                    # ActNorm data-dependent init on the first batch
    sharding.broadcast_module(model)
    trainer = sharding.ShardedTrainer(model, lr=1e-4, warm_up=10000, global_batch=batch * world)
    steps = max(2, args.train_steps)
    for i in range(4):                                  # 2 eager steps, graph capture, 1 replay
        trainer.step(xs[i % len(xs)])
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for i in range(steps):
        loss = trainer.step(xs[i % len(xs)])
    e.record()
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    ms = s.elapsed_time(e)
    if dist is not None:
        t = torch.tensor([ms], device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t)
    return {"value": batch * world * steps / (ms / 1e3), "unit": "images/s", "ms_per_step": ms / steps, "steps": steps,
            "warmup": 4, "scaling": scaling, "batch_per_gpu": batch, "global_batch": batch * world,
            "grad_allreduce_mb": trainer.buckets.nbytes() / 1e6,
            "loss_bits_per_dim": float(loss),
            "note": "fwd+bwd+Adamax(+NCCL all-reduce of flat gradient buckets); forward+backward and the optimizer update "
                    "replayed as CUDA graphs (the all-reduces are nodes of the backward graph); conditioner convs/linears: "
                    "forward, input- and weight-gradients on the flowk tcgen05 kernels (3xTF32); attention core "
                    "(with dropout) forward/backward on the flowk mma.sync kernels; weight norm, concat-ELU, GLU, "
                    "residual+LayerNorm, bias gradients and Adamax as fused flowk kernels; flow ops through the flowk "
                    "forward/backward kernels"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="flowk", choices=["flowk", "reference"])
    ap.add_argument("--workload", default="cfg2", choices=sorted(WORKLOADS))
    ap.add_argument("--cpu-sample", type=int, default=0, help="images per CPU-oracle step (0 = default)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-large", action="store_true")
    ap.add_argument("--depth", type=int, default=10, help="batches in flight (graph instances on separate streams)")
    ap.add_argument("--no-train", action="store_true")
    ap.add_argument("--train-steps", type=int, default=20)
    ap.add_argument("--no-inverse", action="store_true")
    ap.add_argument("--no-mar", action="store_true")
    ap.add_argument("--no-other-configs", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the latent z and the per-image bits/dim of the last timed step (rank 0) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "flowk":
        ap.error("--dump-outputs writes the outputs of the flowk arm")
    args.warmup = max(args.warmup, 3) if args.impl == "flowk" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    else:
        run_flowk(args)


if __name__ == "__main__":
    main()
