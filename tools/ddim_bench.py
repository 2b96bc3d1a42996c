"""DDIM vs DDPM sampling throughput on the headline workload (cfg3: 128x128 Family R with lsm, topography, cond field and season
labels, B = 256, linear schedule T = 1000), on one GPU, in one process.

    python tools/ddim_bench.py [--rounds 3] [--batch 256] [--steps 100,50,25] [--out FILE]

Every mode (DDPM `sample`, 999 evaluations; `sample_ddim` at each S) is warmed up first, then the modes alternate round by round
so that clock and power drift hit all of them alike.  Each timed window is bracketed by CUDA events and holds about two seconds
of work (the shorter DDIM runs are repeated).  Reported per mode: samples/s, ms per model evaluation and launches per evaluation
(`launch_count()`), as the median over the rounds; plus the card, its power limit and maximum SM clock, and the fp16 saturation
counter, which must stay 0.  Prints one JSON document (and writes it to --out)."""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from diffusionmodelscustom_b200 import DiffusionUtils  # noqa: E402
from diffusionmodelscustom_b200.configs import R_CASES, build_ours_r, inputs_r  # noqa: E402
from diffusionmodelscustom_b200.modules import NativeModel  # noqa: E402

T = 1000


def card():
    q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power, clock = ([s.strip() for s in q.stdout.strip().split(",")] + ["?", "?", "?"])[:3] if q.returncode == 0 else \
        (torch.cuda.get_device_name(0), "unknown", "unknown")
    return {"device": name, "power_limit": power, "max_sm_clock": clock}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--steps", default="100,50,25")
    ap.add_argument("--window-s", type=float, default=2.0, help="approximate device time per timed window")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    case = R_CASES["cfg3_full_128"]
    net, _ = build_ours_r(case, "cuda")
    _, d = inputs_r(case, a.batch, "cuda")
    du = DiffusionUtils(T, 1e-4, 0.02, "cuda", "linear")
    args = (d["x"], net, d["y"], d["cond"], d["lsm"], d["topo"])
    modes = [("ddpm", T - 1)] + [(f"ddim_S{s}", int(s)) for s in a.steps.split(",")]

    def run(mode, evals, k):
        if mode == "ddpm":
            return du.sample(*args, seed=1000 + k)
        return du.sample_ddim(*args, steps=evals, eta=0.0, seed=1000 + k)

    NativeModel.saturation_count(reset=True)
    reps, launches = {}, {}
    for mode, evals in modes:                       # warm-up: captures every graph pair, and sizes the windows
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        run(mode, evals, 0)
        e0.record()
        x0 = run(mode, evals, 0)
        e1.record()
        torch.cuda.synchronize()
        assert torch.isfinite(x0).all(), mode
        launches[mode] = net.launch_count()
        reps[mode] = max(1, round(a.window_s * 1e3 / e0.elapsed_time(e1)))
    times = {m: [] for m, _ in modes}
    for r in range(a.rounds):
        for mode, evals in modes:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for k in range(reps[mode]):
                x0 = run(mode, evals, 1 + r * 100 + k)
            e1.record()
            torch.cuda.synchronize()
            times[mode].append(e0.elapsed_time(e1) / reps[mode])
    sat = NativeModel.saturation_count()
    res = {"tool": "tools/ddim_bench.py", "workload": f"cfg3_full_128 (Family R 128x128, lsm + topo + cond + 4 season classes), "
           f"B = {a.batch}, linear schedule T = {T}, eta = 0, Philox noise", **card(), "rounds": a.rounds, "modes": {}}
    for mode, evals in modes:
        ms = statistics.median(times[mode])
        res["modes"][mode] = {"evals_per_sample": evals, "calls_per_window": reps[mode], "ms_per_call": ms,
                              "ms_per_call_all_rounds": times[mode], "samples_per_s": a.batch / (ms / 1e3),
                              "ms_per_eval": ms / evals, "launches_per_eval": launches[mode] / evals}
    base = res["modes"]["ddpm"]
    for mode, evals in modes[1:]:
        m = res["modes"][mode]
        m["ms_per_eval_vs_ddpm"] = m["ms_per_eval"] / base["ms_per_eval"]
        m["throughput_vs_ddpm"] = m["samples_per_s"] / base["samples_per_s"]
        m["ideal_throughput_vs_ddpm"] = (T - 1) / evals
    res["fp16_saturations"] = sat
    text = json.dumps(res, indent=1)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")
    if sat != 0:
        raise SystemExit("fp16 saturation counter is not 0")


if __name__ == "__main__":
    main()
