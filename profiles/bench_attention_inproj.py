"""Per-launch cost of the fused in_proj + attention route at cfg2 level 1 (B = 64, 16 x 16, C = 96, 4 heads).

Two routes from the same conv-3x3 output, timed in one process, alternating, as CUDA graphs of back-to-back repeats:
  chained: gate GEMM with the in_proj GEMM chained in its epilogue (fp32 q, k, v rows) + the one-wave attention kernel;
  fused:   gate GEMM writing the normalised rows + positional encoding as an fp16 pair + flowk_attention_inproj_tc.
Each launch is also timed alone.  Prints the card, median [min, max] us per route over the rounds, the fused CTA's phase
cycles (projection, drain, first S, softmax passes, the rest) and the two routes' largest output difference."""
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import flowk  # noqa: E402,F401
from flowk import tc  # noqa: E402

dev = torch.device("cuda:0")
B, H, W, C, heads = 64, 16, 16, 96, 4
HW, M = H * W, B * H * W
ROUNDS, LAUNCHES = 7, 20


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = ""
    return q or torch.cuda.get_device_name(0)


g = torch.Generator(device="cpu").manual_seed(0)
a_hi, a_lo = tc.split_rows_f16((torch.randn(M, 2 * C, generator=g)).to(dev))
w_hi, w_lo, sc = tc.conv_weight_operand_f16((torch.randn(2 * C, 2 * C, generator=g) / 14).to(dev))
w3_hi, w3_lo, sc3 = tc.conv_weight_operand_f16((torch.randn(3 * C, C, generator=g) / 10).to(dev))
bias, res = torch.randn(2 * C, generator=g).to(dev), torch.randn(M, C, generator=g).to(dev)
gamma, beta = torch.ones(C, device=dev), torch.zeros(C, device=dev)
pos = (torch.randn(HW, C, generator=g) * 0.1).to(dev)
x1, qkv = torch.empty(M, C, device=dev), torch.empty(M, 3 * C, device=dev)
p_hi, p_lo = torch.empty(M, C, device=dev, dtype=torch.float16), torch.empty(M, C, device=dev, dtype=torch.float16)
common = dict(bias=bias, res=res, gamma=gamma, beta=beta, pos=pos, out_f32=x1, acc_scale=sc)
out = {}


def gate_chained():
    tc.conv_gemm(a_hi, a_lo, w_hi, w_lo, B, H, W, 2 * C, 2 * C, 1, tc.PRE_GLU_RES_LN, tc.OUT_F32,
                 w2_hi=w3_hi, w2_lo=w3_lo, out2_f32=qkv, n2=3 * C, acc_scale2=sc3, **common)


def attn_v2():
    out["chained"] = tc.attention(qkv, B, HW, C, heads, True)


def gate_pair():
    tc.conv_gemm(a_hi, a_lo, w_hi, w_lo, B, H, W, 2 * C, 2 * C, 1, tc.PRE_GLU_RES_LN, tc.OUT_F32 | tc.OUT_HILO_POS,
                 out_hi=p_hi, out_lo=p_lo, **common)


def attn_fused(trace=None):
    out["fused"] = tc.attention_inproj(p_hi, p_lo, w3_hi, w3_lo, sc3, B, HW, C, heads, trace=trace)


ROUTES = {
    "chained gate + one-wave attention": lambda: (gate_chained(), attn_v2()),
    "pair gate + fused attention": lambda: (gate_pair(), attn_fused()),
    "  chained gate alone": gate_chained,
    "  one-wave attention alone": attn_v2,
    "  pair gate alone": gate_pair,
    "  fused attention alone": attn_fused,
}


def graph_of(fn):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    gr = torch.cuda.CUDAGraph()
    with torch.cuda.graph(gr):
        for _ in range(LAUNCHES):
            fn()
    gr.replay()
    torch.cuda.synchronize()
    return gr


def time_graph(gr):
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    gr.replay()
    e.record()
    torch.cuda.synchronize()
    return s.elapsed_time(e) * 1e3 / LAUNCHES


print("device: %s" % card())
print("cfg2 level 1: B = %d, %dx%d, C = %d, %d heads; %d rounds of a graph of %d repeats, routes alternated; "
      "median [min, max] us" % (B, H, W, C, heads, ROUNDS, LAUNCHES))
graphs = {name: graph_of(fn) for name, fn in ROUTES.items()}
times = {name: [] for name in ROUTES}
for _ in range(ROUNDS):
    for name, gr in graphs.items():
        times[name].append(time_graph(gr))
for name in ROUTES:
    v = sorted(times[name])
    print("%-36s %6.1f us [%5.1f, %5.1f]" % (name, v[len(v) // 2], v[0], v[-1]), flush=True)

gate_chained()
attn_v2()
gate_pair()
trace = torch.zeros(8, dtype=torch.int64, device=dev)
attn_fused(trace)
torch.cuda.synchronize()
t = trace.cpu().tolist()
print("fused CTA cycles: projection %d  drain %d  first S %d  max-pass %d  exp-pass %d  rest %d  epilogue %d" % tuple(
    t[i + 1] - t[i] for i in range(7)))
ref = sum(x.double() for x in out["chained"])
got = sum(x.double() for x in out["fused"])
print("max |fused - chained| = %.3e (max |chained| = %.3e)" % (float((got - ref).abs().max()), float(ref.abs().max())))
