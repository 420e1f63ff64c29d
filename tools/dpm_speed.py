#!/usr/bin/env python3
"""Samples/s of the DPM-Solver++(2M) sampler at 10, 20 and 50 steps and of its SDE form (dpm++2m-sde) at 20, 50 and 80
steps against the reverse-SDE sampler at 300 steps, at the bench configuration (n = 1024 per job, CFG 1.5, t_end 0.005,
the bench's EMA weights: default init under seed 1, bf16 on the tcgen05 engine).  The seven jobs alternate in one process:
one warm-up round, then --reps timed rounds; each job is timed with CUDA events and ends in a device synchronise.  The card's name, power limit and SM clock (sampled during the
timed rounds) are recorded in the same run.

Also reported, for information only (no gate): the pre-clamp x0_hat rel-L2 between dpm++2m at 50 steps and the Heun ODE
at 300 steps from the same x_T (Philox, seed 1234).  The weights are untrained, so this says how closely the two solve the
same ODE, not what either does to sample quality.

    python tools/dpm_speed.py --out profiles/dpm_speed_b200.json
"""
import argparse
import ctypes as C
import json
import math
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "vae-diffusion-toy-crystals_b200"))
sys.path.insert(0, ROOT)
from toycrystals_b200 import _cabi  # noqa: E402
from toycrystals_b200.models import sde_score_model as shim  # noqa: E402
from bench import ClockSampler  # noqa: E402

N, CFG, T_END, SEED = 1024, 1.5, 0.005, 1234
JOBS = [("dpm++2m", 10), ("dpm++2m", 20), ("dpm++2m", 50), ("dpm++2m-sde", 20), ("dpm++2m-sde", 50),
        ("dpm++2m-sde", 80), ("sde", 300)]
SAMPLER_IDS = {"dpm++2m": _cabi.SAMPLER_DPMPP_2M, "dpm++2m-sde": _cabi.SAMPLER_DPMPP_2M_SDE, "ode": _cabi.SAMPLER_ODE,
               "sde": _cabi.SAMPLER_SDE}


def gpu_info():
    q = "name,power.limit,clocks.max.sm,clocks.sm,driver_version"
    try:
        r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"], capture_output=True,
                           text=True, timeout=30)
        vals = [v.strip() for v in r.stdout.strip().split(",")]
        return dict(zip(q.split(","), vals))
    except Exception as e:   # the card's name still comes from torch
        return {"error": repr(e)}


def x0_hat(model, sde, sampler, steps, yc, yk):
    """Pre-clamp projection of a whole job through the C ABI (no evaluation traces: 601 of them would not fit)."""
    h = model.engine_handle(sde)
    out = torch.empty((N, 1, 64, 64), device="cuda")
    x0 = torch.empty_like(out)
    a = _cabi.TcsSampleArgs()
    a.sampler, a.n, a.steps, a.guidance, a.t_end = SAMPLER_IDS[sampler], N, steps, CFG, T_END
    a.y_cat, a.y_cont, a.x_init, a.noise = yc.data_ptr(), yk.data_ptr(), None, None
    a.seed, a.global_index_offset = SEED, 0
    a.x_out, a.trace_eps, a.trace_x, a.x0_hat = out.data_ptr(), None, None, x0.data_ptr()
    a.beta_min, a.beta_max = sde.beta_min, sde.beta_max
    torch.cuda.synchronize()
    _cabi.check(_cabi.lib().tcs_sample(h, C.byref(a), None))
    torch.cuda.synchronize()
    return x0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="JSON result path")
    ap.add_argument("--reps", type=int, default=5, help="timed rounds (each times every job once)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("dpm_speed.py needs a B200 (there is no CPU path)")
    dev = torch.device("cuda", 0)
    torch.manual_seed(1)   # bench.py's weights: default init under seed 1 (the EMA model of its checkpoint layout)
    model = shim.CondUNetTiny(4, 4, 96, 128, 8, 8, precision="bf16").to(dev).eval()
    sde = shim.VPSDE(0.1, 30.0)
    yc, yk = shim.condition_grid(model, N, math.pi / 3.0, dev)

    def job(sampler, steps):
        return shim._SAMPLERS[sampler](model, sde, yc, yk, (N, 1, 64, 64), n_steps=steps, guidance_scale=CFG,
                                       t_end=T_END, seed=SEED)

    def timed(sampler, steps):
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        job(sampler, steps)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1)

    info = gpu_info()
    for sampler, steps in JOBS:   # warm-up: module load, graph capture, workspace of every job shape
        timed(sampler, steps)
    ms = {f"{s}@{k}": [] for s, k in JOBS}
    with ClockSampler(0) as clk:
        for _ in range(args.reps):
            for sampler, steps in JOBS:
                ms[f"{sampler}@{steps}"].append(timed(sampler, steps))
    jobs = {}
    for sampler, steps in JOBS:
        key = f"{sampler}@{steps}"
        med = statistics.median(ms[key])
        jobs[key] = {"sampler": sampler, "steps": steps, "nfe": int(_cabi.lib().tcs_nfe(SAMPLER_IDS[sampler], steps)),
            "ms_per_job": ms[key], "ms_median": med, "samples_per_sec": N / (med / 1e3),
            "ms_per_evaluation": med / (steps + 1)}   # every job here makes steps + 1 evaluations
    base = jobs["sde@300"]["samples_per_sec"]
    for v in jobs.values():
        v["speedup_vs_sde300"] = v["samples_per_sec"] / base
    a = x0_hat(model, sde, "dpm++2m", 50, yc, yk)
    b = x0_hat(model, sde, "ode", 300, yc, yk)
    rel = float((a.double() - b.double()).norm() / b.double().norm())
    res = {
        "tool": "tools/dpm_speed.py", "device": torch.cuda.get_device_name(dev), "nvidia_smi": info,
        "clocks_during_timing": clk.summary(),
        "config": {"n": N, "cfg": CFG, "t_end": T_END, "precision": "bf16", "engine": "tcgen05", "seed": SEED,
                   "weights": "default init under torch.manual_seed(1), as bench.py", "reps": args.reps},
        "jobs": jobs,
        "x0_hat_rel_l2_dpm50_vs_ode300": rel,
    }
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    for k, v in jobs.items():
        print(f"{k:>16}: {v['samples_per_sec']:8.1f} samples/s  ({v['ms_median']:.1f} ms/job, {v['nfe']} evaluations, "
              f"{v['ms_per_evaluation']:.2f} ms/evaluation, x{v['speedup_vs_sde300']:.2f} vs sde@300)")
    print(f"x0_hat rel-L2 dpm++2m@50 vs ode@300: {rel:.3e}")
    print(json.dumps({"device": res["device"], "nvidia_smi": info, "clocks": res["clocks_during_timing"]}))


if __name__ == "__main__":
    main()
