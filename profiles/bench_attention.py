"""Time the attention kernels in isolation (CUDA graph of back-to-back launches) and print the tcgen05 kernels' phase stamps.

The level-1 shapes (seq 256, C = 96 and 160) run on both tcgen05 kernels: the one-wave kernel (attention_tc_v2_kernel,
two CTAs per SM) where it takes the shape, and the one-CTA-per-SM kernel (attention_tc_kernel).  The two are timed in the
same process, alternating, over several rounds; each line gives the median and the range over the rounds."""
import ctypes
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import flowk  # noqa: E402,F401
from flowk import _lib, tc  # noqa: E402

dev = torch.device("cuda:0")
B, heads = 64, 4
ROUNDS, LAUNCHES = 7, 20


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = ""
    return q or torch.cuda.get_device_name(0)


def graph_of(qkv, HW, C):
    for _ in range(3):
        tc.attention(qkv, B, HW, C, heads, True)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(LAUNCHES):
            tc.attention(qkv, B, HW, C, heads, True)
    g.replay()
    torch.cuda.synchronize()
    return g


def time_graph(g):
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    g.replay()
    e.record()
    torch.cuda.synchronize()
    return s.elapsed_time(e) * 1e3 / LAUNCHES


def stamps(qkv, HW, C):
    trace = torch.zeros(8, dtype=torch.int64, device=dev)
    tc.attention(qkv, B, HW, C, heads, True, trace=trace)
    torch.cuda.synchronize()
    t = trace.cpu().tolist()
    return "stage %d  S-mma %d  max-pass %d  exp-pass %d  rest %d  epilogue %d" % (
        t[1] - t[0], t[2] - t[1], t[3] - t[2], t[4] - t[3], t[5] - t[4], t[6] - t[5])


def set_route(name):
    tc.ATTENTION_TC = name != "mma.sync"
    tc.ATTENTION_TC_V2 = name == "tcgen05-1wave"


print("device: %s" % card())
print("B = %d, %d heads, fp16 operand-pair output; %d rounds of a graph of %d launches, routes alternated; "
      "median [min, max] us per launch" % (B, heads, ROUNDS, LAUNCHES))
for HW, C in ((256, 96), (256, 160), (64, 96), (16, 96)):
    qkv = torch.randn(B * HW, 3 * C, device=dev)
    routes = []
    for name in ("tcgen05-1wave", "tcgen05", "mma.sync"):
        set_route(name)
        if name == "tcgen05-1wave" and not tc.attention_tc_v2_supported(HW, C, heads):
            continue
        if name == "tcgen05" and not tc.attention_tc_supported(HW, C, heads):
            continue
        routes.append((name, graph_of(qkv, HW, C)))
    times = {name: [] for name, _ in routes}
    for _ in range(ROUNDS):
        for name, g in routes:
            times[name].append(time_graph(g))
    for name, _ in routes:
        set_route(name)
        v = sorted(times[name])
        line = "%-13s seq %4d C %3d: %6.1f us [%5.1f, %5.1f]" % (name, HW, C, v[len(v) // 2], v[0], v[-1])
        if name.startswith("tcgen05"):
            line += "   cycles: " + stamps(qkv, HW, C)
        if name == "tcgen05-1wave":
            n, smem = ctypes.c_int(0), ctypes.c_int(0)
            _lib.check(_lib.lib.flowk_attention_tc_v2_occupancy(HW, C, heads, ctypes.byref(n), ctypes.byref(smem)))
            line += "   (%d CTAs per SM, %d B dynamic smem)" % (n.value, smem.value)
        print(line, flush=True)
set_route("tcgen05-1wave")
tc.ATTENTION_TC, tc.ATTENTION_TC_V2 = True, True
