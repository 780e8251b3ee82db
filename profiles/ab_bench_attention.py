"""Same-call A/B of the level-1 attention route on the flagship benchmark.

Runs `bench.py --no-cpu-baseline --no-other-configs --no-mar --no-train --steps 200` ROUNDS times per route, alternating
VAR=0 and VAR=1, each with --dump-outputs into a temporary directory, then compares the dumped z and bits/dim of the two
routes against the parity budget |got - ref| <= 1e-4 max(1, max|ref|) and |bits/dim| difference <= 1e-3.  Prints every
bench line, the median and range of `value`, `single_stream` and `inverse` per route, and writes everything as JSON to
argv[1] (default: stdout only).  VAR (argv[3]) is FLOWK_ATTENTION_TC_V2 by default (one CTA per SM vs the one-wave
kernel); FLOWK_ATTENTION_INPROJ compares the in_proj GEMM + one-wave kernel with the fused kernel.

    python profiles/ab_bench_attention.py [out.json] [rounds] [VAR]
"""
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ARGS = ["--no-cpu-baseline", "--no-other-configs", "--no-mar", "--no-train", "--steps", "200"]


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                               "-i", "0"], capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def run(var, v2, dump):
    env = dict(os.environ, **{var: str(v2)})
    out = subprocess.run([sys.executable, "bench.py"] + ARGS + ["--dump-outputs", dump], cwd=ROOT, env=env,
                         capture_output=True, text=True)
    lines = [ln for ln in out.stdout.splitlines() if ln.startswith("{")]
    if out.returncode != 0 or not lines:
        sys.stderr.write(out.stdout[-4000:] + out.stderr[-4000:])
        raise SystemExit("bench.py failed (%s=%d)" % (var, v2))
    return json.loads(lines[-1])


def summary(vals):
    v = sorted(vals)
    return {"median": v[len(v) // 2], "min": v[0], "max": v[-1], "all": vals}


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else None
    rounds = int(sys.argv[2]) if len(sys.argv) > 2 else 3
    var = sys.argv[3] if len(sys.argv) > 3 else "FLOWK_ATTENTION_TC_V2"
    res = {"device": card(), "args": ARGS, "variable": var, "runs": {"0": [], "1": []}}
    print("device:", res["device"], flush=True)
    with tempfile.TemporaryDirectory() as tmp:
        for r in range(rounds):
            for v2 in (0, 1):
                line = run(var, v2, os.path.join(tmp, "v2_%d" % v2))
                res["runs"][str(v2)].append(line)
                print("%s=%d round %d: value %.1f images/s (%.3f ms/step), single_stream %.1f images/s, inverse %.1f images/s"
                      % (var, v2, r, line["value"], line["ms_per_step"], line["single_stream"]["value"],
                         line["inverse"]["value"]), flush=True)
        parity = {}
        for name in ("z", "bits_per_dim"):
            ref = np.load(os.path.join(tmp, "v2_0", name + ".npy")).astype(np.float64)
            got = np.load(os.path.join(tmp, "v2_1", name + ".npy")).astype(np.float64)
            parity[name] = {"max_abs_diff": float(np.abs(got - ref).max()), "max_abs_ref": float(np.abs(ref).max())}
        res["parity"] = parity
        res["parity_ok"] = (parity["z"]["max_abs_diff"] <= 1e-4 * max(1.0, parity["z"]["max_abs_ref"])
                            and parity["bits_per_dim"]["max_abs_diff"] <= 1e-3)
    for v2 in ("0", "1"):
        runs = res["runs"][v2]
        res["value_" + v2] = summary([ln["value"] for ln in runs])
        res["single_stream_" + v2] = summary([ln["single_stream"]["value"] for ln in runs])
        res["inverse_" + v2] = summary([ln["inverse"]["value"] for ln in runs])
    print(json.dumps({k: v for k, v in res.items() if k != "runs"}, indent=1))
    if out_path:
        with open(out_path, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
