#!/usr/bin/env python
"""Headline benchmark: samples/s for full T=1000 DDPM sampling (999 UNet evaluations + posterior updates per sample).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload cfg3|cfg2|cfg4|cfg1|cfg5]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

Headline workload = BASELINE.json configs[2] (cfg3): the conditional Family-R UNet of ddpm_DANRA_conditional_wValid__128x128
(LSM + topography + conditioning image + season classes, 128x128), GLOBAL batch 256, T=1000, STRONG-scaled over the N GPUs
(256/N samples per GPU, no data-path collective, one NCCL all_gather of the final fields per step).  A "step" is ONE pass of the
hot path over that global batch: DiffusionUtils.sample (T-1 = 999 reverse steps, graph-replayed).  The other BASELINE
configurations ride along as `secondary` objects (fewer steps; cfg2 64x64 batch 64/GPU, cfg4 Family D batch 64/GPU, both weak).

`value`      : device-resident throughput (inputs already in HBM), CUDA events on the launching stream, max over ranks.
`e2e`        : the same metric through the reference-facing API with pinned HOST buffers (DiffusionUtils.sample_host ->
               b2d_sample_host): H2D of x_T + conditioning and D2H of the fields inside the timed region.
`roofline`   : the dominant kernel class of one reverse step, timed live with CUDA events between launches (b2d_profile_step,
               each launch in isolation => the BURST peaks of MEASURED_PEAKS.json); `roofline_classes` carries every class.
`cpu_baseline`: the UNMODIFIED reference (oracle/_ref, staged by oracle/stage_ref.py; `kind` "reference") on the host cores for
               a bounded sample, or the oracle port (`kind` "port") when the staged copy is absent.
`--impl reference`: that same reference CPU implementation as its own arm — identical `config`, each step = one call of the
               reference's own DiffusionUtils.sample bounded to a few reverse steps of a sub-batch (`cpu_baseline.sample` says
               which); `ms_per_step` is the time actually measured, `value` the extrapolation to 999 steps per sample.
`--dump-outputs DIR`: after the timed steps, the fields x_0 that the last timed step of the headline workload returned (the whole
               global batch) go to DIR/x0.npy as float32 [B, C, H, W].  Inputs, weights and noise seeds depend only on the
               arguments, so two builds run with the same arguments can be compared field for field.  Compare with a
               tolerance: atomic reductions make two runs of one build differ in the last bits (cfg3, 256 fields on one B200
               at its 1000 W limit: 7e-6 relative L2).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

T_STEPS = 1000
METRIC = "samples_per_s_T1000_ddpm_sampling"
WORKLOADS = {
    # name: case (diffusionmodelscustom_b200/configs.py), global batch, scaling, FLOPs per sample per reverse step [BASELINE.md §3]
    "cfg1": dict(case="cfg1_uncond_64", global_batch=4, scaling="weak", flops=1.381e9),
    "cfg2": dict(case="cfg2_lsmtopo_64", global_batch=64, scaling="weak", flops=1.398e9),
    "cfg3": dict(case="cfg3_full_128", global_batch=256, scaling="strong", flops=12.527e9),
    "cfg4": dict(case="cfg4_downscale_64", global_batch=64, scaling="weak", flops=17.75e9),   # 64 per GPU = 512 on 8 GPUs
    "cfg5": dict(case="cfg5_flexible_128", global_batch=256, scaling="strong", flops=12.527e9),
}
# BASELINE configs[4]: 1024-member ensemble through the native generation driver (b2d_ensemble_run): dates x members per date
ENSEMBLE = dict(case="cfg5_flexible_128", dates=16, members=64, sub_batch=128, flops=12.527e9)
# reference arm / cpu_baseline: (sub-batch, reverse steps per timed call) sized for ~1-2 s per call on 16 host cores
REF_SAMPLE = {"cfg1": (4, 8), "cfg2": (8, 4), "cfg3": (4, 2), "cfg4": (4, 2), "cfg5": (4, 2)}
HEAD_DIM_OF_CLASS = {"attn_tc": 16, "attn_tc32": 32}
SFU_PEAK_TEXP = 4.63     # measured on this pool's B200s: tools/ub/mufu.cu (ex2.approx.ftz.f32, all SMs)
NCU_TRAFFIC = {}         # filled from profiles/r2_ncu_traffic.json when present (dram bytes per launch, per kernel class)
DUMP_BYTES = 64 << 20    # --dump-outputs writes at most this much


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sustained=d["bf16_tflops_sustained"], src="measured")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sustained=1400.0, src="fallback (B200_PROFILING.md)")


def dump_outputs(path, x0):
    """x0 as <path>/x0.npy (float32).  A batch above DUMP_BYTES is cut to a fixed sample of whole fields (seeded by 0, kept in
    batch order), the same for every run with the same arguments."""
    import numpy as np
    x0 = x0.float().cpu()
    if x0.numel() * 4 > DUMP_BYTES:
        keep = torch.randperm(x0.shape[0], generator=torch.Generator().manual_seed(0))[:DUMP_BYTES // (x0[0].numel() * 4)]
        x0 = x0[keep.sort().values]
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "x0.npy"), x0.numpy())


def workload_config(name, world):
    """The `config` object — built from the workload name and the GPU count only, so both arms emit it identically."""
    from diffusionmodelscustom_b200.configs import D_CASES, R_CASES
    w = WORKLOADS[name]
    is_d = w["case"] in D_CASES
    case = D_CASES[w["case"]] if is_d else R_CASES[w["case"]]
    gb = w["global_batch"] * (world if w["scaling"] == "weak" else 1)
    if is_d:
        desc = (f"{name}: Family D UNet_downscale (DDPM_clean_application/src/unet_ms.py), {case['hw']}x{case['hw']}, c_in={case['c_in']} "
                f"(x + {case['lowres']}x{case['lowres']} low-res field, bicubic), global batch {gb}, T={T_STEPS} linear beta")
    else:
        desc = (f"{name}: Family R DiffusionNet ({case.get('module', 'modules_DANRA_conditional')}), {case['hw']}x{case['hw']}, "
                f"c_in={case['c_in']} (lsm={case['has_lsm']}, topo={case['has_topo']}, cond={case['has_cond']}, "
                f"classes={case['num_classes']}), global batch {gb}, T={T_STEPS} linear beta")
    return {"workload": desc, "T": T_STEPS, "unet_evals_per_sample": T_STEPS - 1, "global_batch": gb, "img_size": case["hw"],
            "scaling": w["scaling"]}, case, is_d, gb


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in self.rows if len(r) >= 7 for n, v in zip(names, r[3:7]) if v.lower().startswith("active")})
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


# ----------------------------------------------------------------------------------------------- CPU arms
def cpu_port_steps(case_name, batch, rev_steps, repeats, warmup, threads):
    """Oracle port (FP32 torch on CPU): `repeats` timed calls of `rev_steps` reverse steps each."""
    from diffusionmodelscustom_b200 import synth
    from diffusionmodelscustom_b200.configs import D_CASES, R_CASES
    from oracle import ddpm_oracle as O
    torch.set_num_threads(threads)
    if case_name in D_CASES:
        case = D_CASES[case_name]
        sd = synth.synth_state_dict_d(case["c_in"], 1, seed=case["wseed"])
        inp = synth.synth_inputs(batch, case["hw"], seed=case["iseed"], lowres=case["lowres"])
        model_fn = lambda x, t: O.family_d_forward(sd, x, t, inp["y_lowres"])
    else:
        case = R_CASES[case_name]
        sd = synth.synth_state_dict_r(case["c_in"], 1, case["num_classes"], (case["hw"],) * 2, case["has_lsm"],
                                      case["has_topo"], seed=case["wseed"])
        inp = synth.synth_inputs(batch, case["hw"], seed=case["iseed"], has_lsm=case["has_lsm"], has_topo=case["has_topo"],
                                 has_cond=case["has_cond"], num_classes=case["num_classes"])
        model_fn = lambda x, t: O.family_r_forward(sd, x, t, inp["y"], inp["cond"], inp["lsm"], inp["topo"])
    betas, alphas, ahat = O.schedule_tables(T_STEPS, 1e-4, 0.02)
    g = torch.Generator().manual_seed(1)
    secs = []
    with torch.no_grad():
        for k in range(warmup + repeats):
            x = inp["x"].clone()
            t0 = time.perf_counter()
            for i in range(rev_steps, 0, -1):
                t = torch.full((batch,), i, dtype=torch.long)
                x = O.posterior_update(x, model_fn(x, t), torch.randn(x.shape, generator=g), i, betas, alphas, ahat)
            if k >= warmup:
                secs.append(time.perf_counter() - t0)
    t_rev = sum(secs) / len(secs) / rev_steps
    return batch / (t_rev * (T_STEPS - 1)), secs


def cpu_arm(workload, repeats, warmup):
    """The reference's CPU implementation of the path on this box's host cores, bounded sample.  Returns the cpu_baseline object
    and the per-call seconds."""
    from oracle import ref_runner
    case_name = WORKLOADS[workload]["case"]
    batch, rev_steps = REF_SAMPLE[workload]
    threads = os.cpu_count() or 1
    if ref_runner.ref_root() is not None:
        sps, secs = ref_runner.time_reference_steps(case_name, batch, rev_steps, repeats, warmup, threads, T=T_STEPS)
        kind = "reference"
        what = "the unmodified reference (oracle/_ref: its own DiffusionNet / UNet_downscale driven by its own DiffusionUtils.sample)"
    else:
        sps, secs = cpu_port_steps(case_name, batch, rev_steps, repeats, warmup, threads)
        kind = "port"
        what = "the oracle port (oracle/ddpm_oracle.py; oracle/_ref not staged on this box)"
    sample = (f"{repeats} timed calls (after {warmup} warm-up) of {what}, each {rev_steps} reverse steps of the same network at "
              f"batch {batch} with the T={T_STEPS} tables; samples/s = batch / (s per reverse step x {T_STEPS - 1}) — every "
              f"reverse step runs the identical code")
    return {"value": sps, "unit": "samples/s", "cores": threads, "kind": kind, "sample": sample}, secs


def run_reference(args, rank, world):
    if rank != 0:
        return
    cfg, _, _, _ = workload_config(args.workload, world)
    t0 = time.perf_counter()
    cpu, secs = cpu_arm(args.workload, max(args.steps, 1), max(args.warmup, 1))
    line = {"impl": "reference", "metric": METRIC, "value": cpu["value"], "unit": "samples/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * sum(secs) / len(secs), "higher_is_better": True,
            "scaling": cfg["scaling"], "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": cfg,
            "cpu_baseline": cpu,
            "e2e": {"value": cpu["value"], "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0, "wall_s": time.perf_counter() - t0}
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------- our arm
class Bench:
    def __init__(self, rank, world, dev):
        self.rank, self.world, self.dev = rank, world, dev
        self.flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)   # > 126 MB L2

    def barrier(self):
        import torch.distributed as dist
        if self.world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(self, fn, steps, warmup, clocks=None):
        import torch.distributed as dist
        for k in range(warmup):
            fn(k)
        self.barrier()
        if clocks:
            clocks.start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        w0 = time.perf_counter()
        e0.record()
        out = None
        for k in range(steps):
            self.flush.zero_()                    # L2 flush between timed iterations
            out = fn(warmup + k)
        e1.record()
        self.barrier()
        wall = time.perf_counter() - w0
        ms = e0.elapsed_time(e1)
        if self.world > 1:
            t = torch.tensor([ms, wall * 1e3], device=self.dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms, wall = float(t[0].item()), float(t[1].item()) / 1e3
        return ms, wall, out

    def run_workload(self, name, steps, warmup, e2e_steps, clocks=None, profile=False, keep_output=False):
        """Device-resident and host end-to-end throughput of one workload; returns a dict (rank 0 fills the roofline).
        keep_output: res["output"] holds the global batch of x_0 of the last timed device step, on the host."""
        import torch.distributed as dist
        from diffusionmodelscustom_b200 import DiffusionUtils
        from diffusionmodelscustom_b200.configs import build_ours_d, build_ours_r, inputs_d, inputs_r
        rank, world, dev = self.rank, self.world, self.dev
        cfg, case, is_d, gb = workload_config(name, world)
        if gb % world:
            raise SystemExit(f"global batch {gb} does not divide over {world} GPUs")
        batch = gb // world
        if is_d:
            net, _ = build_ours_d(case, dev)
            host, d = inputs_d(dict(case, iseed=case["iseed"] + rank), batch, dev)
            for dd in (host, d):     # Family D: the low-res field travels in the cond_img slot of the sampler
                dd.update(cond=dd.pop("y_lowres"), lsm=None, topo=None, y=None)
        else:
            net, _ = build_ours_r(case, dev)
            host, d = inputs_r(dict(case, iseed=case["iseed"] + rank), batch, dev)
        du = DiffusionUtils(T_STEPS, 1e-4, 0.02, dev, "linear")
        gather = [torch.empty_like(d["x"]) for _ in range(world)] if world > 1 else None
        offset = rank * batch

        def step_device(k):
            x0 = du.sample(d["x"], net, d["y"], d["cond"], d["lsm"], d["topo"], seed=1234 + k, sample_offset=offset)
            if world > 1:
                dist.all_gather(gather, x0)
            return x0

        pinned = {k: (v.pin_memory() if v is not None else None) for k, v in host.items()}

        def step_host(k):
            return du.sample_host(pinned["x"], net, pinned["y"], pinned["cond"], pinned["lsm"], pinned["topo"], seed=1234 + k,
                                  sample_offset=offset, device=dev)

        net.saturation_count(reset=True)
        ms, wall, x0 = self.timed(step_device, steps, warmup, clocks)
        launches = net.launch_count() * steps
        assert torch.isfinite(x0).all(), "non-finite samples"
        value = gb * steps / (ms / 1e3)
        ms_e2e, wall_e2e, x0h = self.timed(step_host, e2e_steps, 1)
        assert torch.isfinite(x0h).all(), "non-finite samples (host path)"
        e2e_value = gb * e2e_steps / max(wall_e2e, ms_e2e / 1e3)
        res = {"name": name, "config": cfg, "per_gpu_batch": batch, "value": value, "ms_per_step": ms / steps, "steps": steps,
               "warmup": warmup,
               "e2e": {"value": e2e_value, "unit": "samples/s", "steps": e2e_steps,
                       "h2d_bytes_per_step": sum(v.numel() * v.element_size() for v in pinned.values() if v is not None) * world,
                       "d2h_bytes_per_step": pinned["x"].numel() * 4 * world},
               "gpu_launches": int(launches), "fp16_saturations": net.saturation_count(),
               "tflops_per_gpu": value * WORKLOADS[name]["flops"] * (T_STEPS - 1) / 1e12 / world}
        if keep_output:     # still the last timed device step: the host path writes neither x0 nor the gather buffers
            res["output"] = (torch.cat(gather) if world > 1 else x0).cpu()
        if profile and rank == 0:
            tt = torch.full((batch,), 500, dtype=torch.long)
            res["profile"] = net.profile_step(d["x"], tt, d["y"], d["cond"], d["lsm"], d["topo"], reps=5)
        del net
        torch.cuda.empty_cache()
        return res


def run_ensemble(B: "Bench"):
    """cfg5: 16 dates x 64 members = 1024 fields of the modules_DANRA_flexible network at 128x128 through generate_ensemble
    (host conditioning per date -> native sub-batch scheduler -> host fields); members sharded over the ranks."""
    import torch.distributed as dist
    from diffusionmodelscustom_b200 import DiffusionUtils, generate_ensemble, synth
    from diffusionmodelscustom_b200.configs import R_CASES, build_ours_r
    case = R_CASES[ENSEMBLE["case"]]
    net, _ = build_ours_r(case, B.dev)
    D, M, sb = ENSEMBLE["dates"], ENSEMBLE["members"], ENSEMBLE["sub_batch"]
    inp = synth.synth_inputs(D, case["hw"], seed=case["iseed"], has_lsm=True, has_topo=True, has_cond=True, num_classes=4)
    du = DiffusionUtils(T_STEPS, 1e-4, 0.02, B.dev, "linear")
    kw = dict(season=inp["y"], cond_img=inp["cond"], lsm=inp["lsm"], topo=inp["topo"], sub_batch=sb, device=B.dev, gather=False,
              return_stats=True)
    per_rank = D * M // B.world
    warm_members = max(1, min(sb, per_rank) * B.world // D)        # one sub-batch per rank: builds the program and the graphs
    generate_ensemble(net, du, D, warm_members, seed=1, **kw)
    B.barrier()
    t0 = time.perf_counter()
    out, st = generate_ensemble(net, du, D, M, seed=2, **kw)
    B.barrier()
    wall = time.perf_counter() - t0
    if B.world > 1:
        t = torch.tensor([wall], device=B.dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        wall = float(t.item())
    assert torch.isfinite(out).all()
    total = D * M
    del net
    torch.cuda.empty_cache()
    return {"name": "cfg5", "workload": (f"cfg5: Family R DiffusionNet (modules_DANRA_flexible), 128x128, full conditioning, {total}-member "
                                          f"ensemble = {D} dates x {M} members through generate_ensemble / b2d_ensemble_run, T={T_STEPS}"),
            "value": total / wall, "unit": "samples/s", "end_to_end": True, "wall_s": wall, "members": total,
            "sub_batch": sb, "sub_batches_per_rank": st["sub_batches"], "out_pinned": st["out_pinned"],
            "host_gather_ms": st["gather_ms"], "gpu_launches": st["launches"],
            "tflops_per_gpu": total / wall * ENSEMBLE["flops"] * (T_STEPS - 1) / 1e12 / B.world,
            "note": "host conditioning per date in, host fields out; timed by wall clock between barriers, max over ranks"}


def class_rooflines(prof, pk):
    """Per kernel class of one reverse step: share, launches, achieved TFLOP/s / GB/s / Texp/s against the burst peaks."""
    by = {}
    for p in prof:
        k = by.setdefault(p["klass"], dict(ms=0.0, flops=0.0, bytes=0.0, launches=0))
        k["ms"] += p["ms"]; k["flops"] += p["flops"]; k["bytes"] += p["bytes"]; k["launches"] += 1
    step_ms = sum(k["ms"] for k in by.values())
    out = {}
    for name, k in sorted(by.items(), key=lambda kv: -kv[1]["ms"]):
        sec = k["ms"] * 1e-3
        e = {"share": round(k["ms"] / step_ms, 4), "ms_per_step": round(k["ms"], 5), "launches": k["launches"],
             "avg_launch_ms": k["ms"] / k["launches"], "algorithmic_bytes_per_launch": k["bytes"] / k["launches"],
             "algorithmic_flops_per_launch": k["flops"] / k["launches"]}
        tf = k["flops"] / sec / 1e12 if k["flops"] else 0.0
        gbs = k["bytes"] / sec / 1e9
        if name in HEAD_DIM_OF_CLASS:        # large-L attention: one exponential per 4*head_dim MMA FLOPs
            texp = k["flops"] / (4.0 * HEAD_DIM_OF_CLASS[name]) / sec / 1e12
            e.update(bound="tensor", achieved=tf, peak=pk["tf_burst"], unit="TFLOP/s", frac=tf / pk["tf_burst"],
                     co_bound={"bound": "sfu_ex2", "achieved": texp, "peak": SFU_PEAK_TEXP, "unit": "Texp/s",
                               "frac": texp / SFU_PEAK_TEXP, "peak_source": "tools/ub/mufu.cu measured on this pool",
                               "note": "peak = every exponential on the SFU; the kernel evaluates half of them on the FMA pipe "
                                       "(packed-half polynomial), so frac may exceed 1 — the kernel is issue-bound, see profiles/"})
        elif k["flops"] and k["flops"] / max(k["bytes"], 1.0) > 150.0:   # above ~260 FLOP/B the tensor pipe is the roof; 150 keeps conv/attn blocks there
            e.update(bound="tensor", achieved=tf, peak=pk["tf_burst"], unit="TFLOP/s", frac=tf / pk["tf_burst"])
        else:
            e.update(bound="hbm", achieved=gbs, peak=pk["hbm"], unit="GB/s", frac=gbs / pk["hbm"])
            if k["flops"]:
                e["tflops"] = tf
        e["traffic"] = NCU_TRAFFIC.get(name)
        out[name] = e
    return out, step_ms


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg3", choices=list(WORKLOADS))
    ap.add_argument("--global-batch", type=int, default=0, help="override the workload's global batch")
    ap.add_argument("--secondary", default="cfg2,cfg4,cfg5", help="comma list of workloads carried as secondary objects ('' = none); "
                    "cfg5 = the 1024-member ensemble through the generation driver")
    ap.add_argument("--e2e-steps", type=int, default=0, help="timed host end-to-end steps (default min(steps, 3))")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write x_0 of the last timed step of the headline workload to DIR/x0.npy (float32, <= 64 MiB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    if args.global_batch:
        WORKLOADS[args.workload]["global_batch"] = args.global_batch
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        return run_reference(args, rank, world)

    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    tp = os.path.join(ROOT, "profiles", "r2_ncu_traffic.json")
    if os.path.exists(tp):
        NCU_TRAFFIC.update(json.load(open(tp)).get(args.workload, {}))
    B = Bench(rank, world, dev)
    sampler = ClockSampler(local_rank) if rank == 0 else None
    e2e_steps = args.e2e_steps or max(1, min(args.steps, 3))
    head = B.run_workload(args.workload, args.steps, args.warmup, e2e_steps, sampler, profile=True,
                          keep_output=bool(args.dump_outputs) and rank == 0)
    clocks = sampler.stop() if sampler else None
    if "output" in head:
        dump_outputs(args.dump_outputs, head.pop("output"))
    secondary = {}
    for name in [s for s in args.secondary.split(",") if s and s != args.workload]:
        if name == "cfg5":
            r = run_ensemble(B)
            if rank == 0:
                secondary[name] = r
            continue
        r = B.run_workload(name, min(args.steps, 2), 1, 1, None, profile=True)
        if rank == 0:
            pk = peaks()
            classes, _ = class_rooflines(r.pop("profile"), pk)
            top = next(iter(classes))
            r["roofline"] = dict(kernel=top, **{k: classes[top][k] for k in ("bound", "achieved", "peak", "unit", "frac")})
            r["kernel_shares"] = {k: v["share"] for k, v in classes.items()}
            r["note"] = "secondary line: 1 warm-up, <= 2 timed steps, 1 timed end-to-end step"
            secondary[name] = r

    if rank == 0:
        pk = peaks()
        classes, step_ms = class_rooflines(head.pop("profile"), pk)
        tname = next(iter(classes))
        roof = dict(kernel=tname, **classes[tname])
        roof["peak_source"] = pk["src"] + " burst bf16 (= fp16 rate): every launch is timed in isolation by CUDA events"
        roof["traffic_source"] = "profiles/r2_ncu_traffic.json (ncu dram__bytes per launch, cold cache)" if roof.get("traffic") else None
        whole = head["tflops_per_gpu"]
        cpu = None
        if not args.no_cpu_baseline and world == 1:
            cpu, _ = cpu_arm(args.workload, 4, 1)
        cfg = head["config"]
        line = {"metric": METRIC, "value": head["value"], "unit": "samples/s", "n_gpus": world,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": head["ms_per_step"], "higher_is_better": True,
                "scaling": cfg["scaling"], "vs_baseline": None, "dtype": "fp16 operands, fp32 accumulate (fp32 state/update)",
                "data": "synthetic", "config": cfg,
                "run": {"per_gpu_batch": head["per_gpu_batch"],
                        "parallelism": f"sample-sharded x{world}, no per-step collective, one all_gather of the fields per step",
                        "l2": "256 MiB buffer written between timed steps", "rng": "in-kernel Philox4x32-10",
                        "e2e_steps": e2e_steps},
                "e2e": head["e2e"], "gpu_launches": head["gpu_launches"], "fp16_saturations": head["fp16_saturations"],
                "clocks": clocks, "roofline": roof, "roofline_classes": classes,
                "whole_step": {"tflops_per_gpu": whole, "frac_of_burst_peak": whole / pk["tf_burst"],
                               "frac_of_sustained_peak": whole / pk["tf_sustained"],
                               "reverse_step_ms_graph": head["ms_per_step"] / (T_STEPS - 1),
                               "reverse_step_ms_sum_of_kernels": step_ms},
                "secondary": secondary, "cpu_baseline": cpu}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
