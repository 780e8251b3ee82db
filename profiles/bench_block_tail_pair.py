"""Per-launch cost of the level-1 block tail in one launch of two-CTA clusters (flowk_block_tail_pair_tc) at cfg2's level 1
(16 x 16, C = 96, 4 heads) and the benchmark's B = 64.

Two routes from the same conv-3x3 output (the c1 pair), timed in one process, alternating, as CUDA graphs of back-to-back
repeats:
  three launches: gate GEMM (GLU + residual + LayerNorm, x1 and the (x1 + pos) fp16 pair) + flowk_attention_inproj_tc +
                  attention-gate GEMM (concat-ELU output), the route of FLOWK_BLOCK_TAIL_PAIR=0;
  fused:          flowk_block_tail_pair_tc.
Each launch of the three-launch route is also timed alone.  Prints the card, median [min, max] us per route over the rounds,
the fused CTA's phase cycles and the largest output difference of the two routes.

    python profiles/bench_block_tail_pair.py [out.txt]
"""
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import flowk  # noqa: E402,F401
from flowk import tc  # noqa: E402

dev = torch.device("cuda:0")
C, heads = 96, 4
ROUNDS, LAUNCHES = 7, 20
lines = []


def say(s):
    print(s, flush=True)
    lines.append(s)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm", "--format=csv,noheader",
                            "-i", "0"], capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = ""
    return q or torch.cuda.get_device_name(0)


def level(H, B):
    W, HW, M = H, H * H, B * H * H
    g = torch.Generator(device="cpu").manual_seed(H)

    def rnd(*shape, s=1.0):
        return (torch.randn(*shape, generator=g) * s).to(dev)
    c1_hi, c1_lo = tc.split_rows_f16(rnd(M, 2 * C, s=0.8))
    gate = tc.conv_weight_operand_f16(rnd(2 * C, 2 * C, s=(2 * C) ** -0.5))
    in_proj = tc.conv_weight_operand_f16(rnd(3 * C, C, s=C ** -0.5))
    attn_gate = tc.conv_weight_operand_f16(rnd(2 * C, C, s=C ** -0.5))
    bias_g, bias_a, x, pos = rnd(2 * C, s=0.1), rnd(2 * C, s=0.1), rnd(M, C), rnd(HW, C, s=0.1)
    ln1 = (torch.ones(C, device=dev), torch.zeros(C, device=dev))
    ln2 = (torch.ones(C, device=dev), torch.zeros(C, device=dev))
    x1, x2 = torch.empty(M, C, device=dev), torch.empty(M, C, device=dev)
    p_hi = torch.empty(M, C, device=dev, dtype=torch.float16)
    p_lo = torch.empty_like(p_hi)
    n_hi = torch.empty(M, 2 * C, device=dev, dtype=torch.float16)
    n_lo = torch.empty_like(n_hi)
    out = {}

    def gate_gemm():
        tc.conv_gemm(c1_hi, c1_lo, gate[0], gate[1], B, H, W, 2 * C, 2 * C, 1, tc.PRE_GLU_RES_LN,
                     tc.OUT_F32 | tc.OUT_HILO_POS, bias=bias_g, res=x, gamma=ln1[0], beta=ln1[1], pos=pos, out_f32=x1,
                     out_hi=p_hi, out_lo=p_lo, acc_scale=gate[2])

    def attention():
        out["t"] = tc.attention_inproj(p_hi, p_lo, in_proj[0], in_proj[1], in_proj[2], B, HW, C, heads)

    def attn_gate_gemm():
        t_hi, t_lo = out["t"]
        tc.conv_gemm(t_hi, t_lo, attn_gate[0], attn_gate[1], B, H, W, C, 2 * C, 1, tc.PRE_GLU_RES_LN,
                     tc.OUT_F32 | tc.OUT_HILO_CELU, bias=bias_a, res=x1, gamma=ln2[0], beta=ln2[1], out_f32=x2,
                     out_hi=n_hi, out_lo=n_lo, acc_scale=attn_gate[2])

    def fused(trace=None):
        out["fused"] = tc.block_tail_pair(c1_hi, c1_lo, gate, bias_g, x, ln1, pos, in_proj, attn_gate, bias_a, ln2, B, HW,
                                          C, heads, True, trace=trace)

    routes = {
        "three launches": lambda: (gate_gemm(), attention(), attn_gate_gemm()),
        "fused pair block tail": fused,
        "  gate GEMM alone": gate_gemm,
        "  in_proj + attention alone": attention,
        "  attention gate alone": attn_gate_gemm,
    }
    gate_gemm()
    attention()                                    # out["t"] exists before the attention gate is captured alone
    graphs = {name: graph_of(fn) for name, fn in routes.items()}
    times = {name: [] for name in routes}
    for _ in range(ROUNDS):
        for name, gr in graphs.items():
            times[name].append(time_graph(gr))
    say("cfg2 %dx%d: B = %d, C = %d, %d heads, M = %d (%d clusters of two 128-row CTAs)" % (H, W, B, C, heads, M, M // 256))
    for name in routes:
        v = sorted(times[name])
        say("  %-30s %6.1f us [%5.1f, %5.1f]" % (name, v[len(v) // 2], v[0], v[-1]))
    gate_gemm()
    attention()
    attn_gate_gemm()
    trace = torch.zeros(8, dtype=torch.int64, device=dev)
    fused(trace)
    torch.cuda.synchronize()
    t = trace.cpu().tolist()
    say("  fused CTA cycles (rank 0 of image 0): gate GEMM %d  GLU/LN 1 %d  in_proj %d  first S %d  rest of attention %d  "
        "attention gate %d  GLU/LN 2 + write-out %d  (total %d)" % (tuple(t[i + 1] - t[i] for i in range(7)) + (t[7] - t[0],)))
    f_x2, f_hi, f_lo = out["fused"]
    for name, a, b in (("x2", f_x2.double(), x2.double()),
                       ("concat-ELU pair", f_hi.double() + f_lo.double(), n_hi.double() + n_lo.double())):
        say("  max |fused - three launches| %s = %.3e (max |ref| = %.3e)" % (name, float((a - b).abs().max()),
                                                                           float(b.abs().max())))


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


say("device (name, power limit, max SM clock, SM clock): %s" % card())
say("%d rounds of a CUDA graph of %d repeats per route, routes alternated; median [min, max] us per repeat"
    % (ROUNDS, LAUNCHES))
level(16, 64)
say("device after the runs: %s" % card())
if len(sys.argv) > 1:
    with open(sys.argv[1], "w") as f:
        f.write("$ python profiles/bench_block_tail_pair.py\n" + "\n".join(lines) + "\n")
