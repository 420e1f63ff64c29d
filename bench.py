#!/usr/bin/env python3
"""bench.py — headline benchmark of the ToyCrystals VP-SDE sampling hot path on B200.

    python bench.py --gpus N --steps K --warmup W [--impl reference]

Metric (BASELINE.json): 64x64 samples/sec, 300 reverse-SDE (Euler-Maruyama) steps, CFG 1.5, EMA
weights, t_end 0.005.  One bench "step" = ONE complete sampling job of `--n` samples per GPU
(configs[1]: n=1024 on 1 B200; weak scaling for N>1, final images all-gathered over NCCL inside the
timed region).  `value` = device-resident throughput (conditions already in HBM, Philox noise
in-kernel); `e2e` = the same job through the public Python API with HOST condition buffers and a
device->host read of the images, copies inside the timed region.

`--impl reference` times the reference algorithm's CPU implementation (the oracle port, which is
bit-identical to the reference module in fp32) on the host cores, on a bounded sample.

`--workload prior` (not the default; BASELINE configs[3], SURVEY 8f-1) benches the latent-diffusion-prior path with
the same contract: one "step" = one job of n=4096 samples per GPU = 50-step DDIM over the FiLM-MLP prior (T=1000, width
1024, z_dim 32, beta_end 0.05) followed by the CondVAE decode to 64x64.

`--dump-outputs DIR` writes the images the last timed step returned as DIR/images.npy (float32, [n_total, 1, 64, 64]).
Weights, conditions and the Philox seed are fixed, so two builds run with the same arguments can be compared output for
output.  Above DUMP_MAX_BYTES a fixed, seeded subset of the samples is written instead.
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

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "vae-diffusion-toy-crystals_b200"))

CONV_GFLOP_PER_FORWARD = 7.092          # per sample per network forward (SURVEY 8d, table a4-L)
# MMAC per image of the 15 convolutions the tcgen05 kernel executes, in tcs_score_profiled order (SURVEY a4-L)
TC_CONV_MMAC = [339.74, 151.00, 169.87, 339.74, 151.00, 84.93, 84.93, 28.31, 9.44, 339.74, 339.74, 84.93, 339.74,
                679.48, 339.74]
TC_CONV_NAMES = ["down1.net.3", "ds1", "down2.net.0", "down2.net.3", "ds2", "mid.net.0", "mid.net.3", "attn.qkv",
                 "attn.proj", "us2_conv", "up2.net.0", "up2.net.3", "us1_conv", "up1.net.0", "up1.net.3"]
ATTN_SDPA_MMAC = 25.17                   # q k^T and p v of the 4 heads (SURVEY a4-L), not part of the conv figure
SDE_STEPS, CFG, T_END = 300, 1.5, 0.005
PEAKS_FALLBACK = {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}
DUMP_MAX_BYTES = 64_000_000             # --dump-outputs: bytes written in all, .npy headers included


def shard_range(n_total: int, rank: int, world: int):
    """Contiguous block of global sample indices owned by `rank` (SURVEY 8e)."""
    base, rem = divmod(n_total, world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def gather_images(local, n_total: int, world: int):
    """All-gather of the per-rank image blocks -> [n_total,1,H,W] on every rank (the path's only collective)."""
    import torch
    import torch.distributed as dist
    if world == 1:
        return local
    sizes = [shard_range(n_total, r, world) for r in range(world)]
    if len({hi - lo for lo, hi in sizes}) == 1:
        out = local.new_empty((n_total,) + tuple(local.shape[1:]))
        dist.all_gather_into_tensor(out, local.contiguous())
        return out
    parts = [local.new_empty((hi - lo,) + tuple(local.shape[1:])) for lo, hi in sizes]
    dist.all_gather(parts, local.contiguous())
    return torch.cat(parts)


def max_over_ranks(value: float, device) -> float:
    import torch
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
        return value
    t = torch.tensor([value], dtype=torch.float64, device=device)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def nccl_logging():
    """stdout carries the ONE JSON line; NCCL's log (communicator init: 'comm ... rank r nranks N', NVLS, rings) goes to
    stderr via NCCL_DEBUG_FILE, so whoever launched the job can check that all N ranks joined.  An NCCL_DEBUG level set
    by the launcher is kept; below INFO the init subsystem is logged at INFO.  report_comm() adds one line per rank of its own."""
    if os.environ.get("NCCL_DEBUG", "").upper() not in ("INFO", "TRACE"):   # (this image presets NCCL_DEBUG=VERSION)
        os.environ["NCCL_DEBUG"] = "INFO"
        os.environ.setdefault("NCCL_DEBUG_SUBSYS", "INIT")
    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")


def report_comm(rank, world, local_rank, dev):
    """One line per rank on stderr once the communicator exists (whatever NCCL's own log level is): an all-reduce of ones
    over the new communicator must return the world size on every rank."""
    import torch
    import torch.distributed as dist
    t = torch.ones(1, device=dev)
    dist.all_reduce(t)
    ver = ".".join(str(v) for v in torch.cuda.nccl.version())
    print(f"[bench] NCCL {ver} comm rank {rank} nranks {world} cudaDev {local_rank} all_reduce(1) = {int(t.item())} "
          f"NCCL_DEBUG={os.environ.get('NCCL_DEBUG')} NCCL_DEBUG_FILE={os.environ.get('NCCL_DEBUG_FILE')}", file=sys.stderr, flush=True)
    assert int(t.item()) == world


def dump_outputs(out_dir: str, outputs: dict) -> None:
    """Write each tensor of `outputs` as <out_dir>/<name>.npy in float32.  The leading axis is the sample; when an array
    would take more than its share of DUMP_MAX_BYTES, a fixed (seed 0), sorted subset of its samples is written."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    budget = DUMP_MAX_BYTES // len(outputs) - 4096          # room for the .npy header
    for name, x in outputs.items():
        x = x.detach().float()
        n, row_bytes = x.shape[0], x[0].numel() * 4
        if n * row_bytes > budget:
            keep = torch.randperm(n, generator=torch.Generator().manual_seed(0))[:budget // row_bytes].sort().values
            x = x[keep.to(x.device)]
        np.save(os.path.join(out_dir, f"{name}.npy"), x.cpu().numpy())
        print(f"[bench] {name}: {x.shape[0]} of {n} samples -> {os.path.join(out_dir, name + '.npy')}", file=sys.stderr,
              flush=True)


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        d["_source"] = "measured"
        return d
    d = dict(PEAKS_FALLBACK)
    d["_source"] = "fallback"
    return d


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.index)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def __exit__(self, *a):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self):
        sm = [float(r[1]) for r in self.rows if len(r) >= 8 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 8 and r[2].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for k, n in enumerate(names) if any(len(r) >= 8 and r[4 + k].lower() == "active" for r in self.rows)]
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


# ---------------------------------------------------------------------------------------------------
# CPU arm: the reference algorithm (oracle port) on the host cores, bounded sample
# ---------------------------------------------------------------------------------------------------
def _reference_module():
    """The UNMODIFIED reference module staged under oracle/_ref (oracle/stage_ref.py), or None when it is absent."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    try:
        import stage_ref
        return stage_ref.import_reference()
    except Exception:  # noqa: BLE001
        return None


def _reference_job(ref, device, n, steps, seed_model=1):
    """Build the reference's own model (default init under torch.manual_seed(seed_model), i.e. the bench's EMA weights) and
    return a callable running its reverse-SDE sampler for `steps` steps (+ projection) on n samples."""
    import torch
    torch.manual_seed(seed_model)
    model = ref.CondUNetTiny(n_types=4, y_cont_dim=4, base_ch=96, emb_dim=128, cond_ch=8, time_ch=8).to(device).eval()
    sde = ref.VPSDE(beta_min=0.1, beta_max=30.0)
    y_cat = torch.tensor([i % 4 for i in range(n)], dtype=torch.long, device=device)       # save_sde_samples :317-321
    y_cont = torch.zeros((n, 4), dtype=torch.float32, device=device)
    y_cont[:, 1] = torch.linspace(0.0, 3.141592653589793 / 3.0, steps=n, device=device)

    def job():
        with torch.no_grad():
            return ref.sample_reverse_sde_euler_maruyama(model=model, sde=sde, y_cat=y_cat, y_cont=y_cont,
                                                         img_shape=(n, 1, 64, 64), n_steps=steps, guidance_scale=CFG,
                                                         t_end=T_END)
    return job


def cpu_reference_samples_per_sec(n: int = 16, steps: int = 3, repeats: int = 1):
    """Time `steps` reverse-SDE steps (+ final projection) of the reference on n samples on the host cores and
    extrapolate linearly to 300 steps (per-evaluation cost is constant).  Runs the unmodified reference module from
    oracle/_ref when it is staged (kind "reference"), else the oracle port (bit-identical to it in fp32; kind "port").
    Returns (samples/s, cores, kind, description)."""
    import torch
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    staged = _reference_module()
    if staged is not None:
        ref, man = staged
        job = _reference_job(ref, torch.device("cpu"), n, steps)
        kind = "reference"
        what = (f"UNMODIFIED reference sample_reverse_sde_euler_maruyama from oracle/_ref "
                f"(sde_score_model.py sha256 {man['files']['toycrystals/models/sde_score_model.py'][:12]})")
    else:
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import toycrystals_oracle as orc
        sd = orc.default_init_state_dict(1)
        y_cat, y_cont = orc.condition_grid(n, 4, 4)
        g = torch.Generator().manual_seed(1234)
        x0 = torch.randn((n, 1, 64, 64), generator=g)
        noise = [torch.randn((n, 1, 64, 64), generator=g) for _ in range(steps)]
        sch = orc.Schedule(0.1, 30.0)
        job = lambda: orc.sample(sd, orc.DEFAULT_CFG, sch, y_cat, y_cont, x0, "sde", steps, CFG, T_END, noise, keep_trace=False)  # noqa: E731
        kind, what = "port", "reference algorithm (oracle port; oracle/_ref not staged)"
    best = None
    for _ in range(repeats):
        t0 = time.perf_counter()
        job()
        dt = time.perf_counter() - t0
        best = dt if best is None else min(best, dt)
    per_eval = best / (steps + 1)
    sps = n / (per_eval * (SDE_STEPS + 1))
    desc = (f"{what}, torch {torch.__version__} CPU fp32, {torch.get_num_threads()} threads: "
            f"n={n}, {steps} reverse-SDE steps + projection = {steps + 1} CFG evaluations in {best:.2f}s, "
            f"extrapolated linearly to {SDE_STEPS + 1} evaluations")
    return sps, cores, kind, desc


def cuda_eager_reference_samples_per_sec(n: int = 1024, evals: int = 10, tf32: bool = True):
    """The reference's OWN sampler as eager PyTorch ON THE B200 (the baseline north_star's ">= 50x" is quoted against),
    at the benchmark's batch size: `evals` CFG evaluations timed after a warm-up run, extrapolated linearly to 301.
    tf32=True is PyTorch's default for cuDNN convolutions (the reference never touches the flags); tf32=False is IEEE fp32."""
    import torch
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    torch.backends.cudnn.allow_tf32 = tf32
    torch.backends.cuda.matmul.allow_tf32 = False       # PyTorch default
    staged = _reference_module()
    steps = evals - 1
    if staged is not None:
        ref, _ = staged
        job, warm = _reference_job(ref, dev, n, steps), _reference_job(ref, dev, n, 1)
        what = "UNMODIFIED reference module (oracle/_ref)"
    else:
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import toycrystals_oracle as orc
        sd = {k: v.to(dev) for k, v in orc.default_init_state_dict(1).items()}
        y_cat, y_cont = orc.condition_grid(n, 4, 4, device=dev)
        x0 = torch.randn((n, 1, 64, 64), device=dev)
        noise = [torch.randn((n, 1, 64, 64), device=dev) for _ in range(steps)]
        sch = orc.Schedule(0.1, 30.0)
        job = lambda: orc.sample(sd, orc.DEFAULT_CFG, sch, y_cat, y_cont, x0, "sde", steps, CFG, T_END, noise, keep_trace=False)  # noqa: E731
        warm = lambda: orc.sample(sd, orc.DEFAULT_CFG, sch, y_cat, y_cont, x0, "sde", 1, CFG, T_END, noise[:1], keep_trace=False)  # noqa: E731
        what = "oracle port of the reference (oracle/_ref not staged)"
    warm()
    torch.cuda.synchronize(dev)
    best = None
    for _ in range(2):
        t0 = time.perf_counter()
        job()
        torch.cuda.synchronize(dev)
        dt = time.perf_counter() - t0
        best = dt if best is None else min(best, dt)
    sps = n / (best / evals * (SDE_STEPS + 1))
    return {"value": sps, "unit": "samples/s", "tf32": tf32, "n": n, "evaluations_timed": evals,
            "sample": f"{what}, eager PyTorch {torch.__version__} on {torch.cuda.get_device_name(dev)}, n={n}, {evals} CFG "
                      f"evaluations in {best:.3f}s (best of 2 after a warm-up run), extrapolated linearly to {SDE_STEPS + 1}"}


# ---------------------------------------------------------------------------------------------------
# --workload prior: BASELINE configs[3]
# ---------------------------------------------------------------------------------------------------
PRIOR = dict(z_dim=32, n_types=4, y_cont_dim=4, t_emb_dim=64, width=1024, n_blocks=8, y_cat_emb_dim=64)
PRIOR_T, PRIOR_B0, PRIOR_B1, DDIM_STEPS = 1000, 1e-4, 0.05, 50
# tensor-core work per sample per DDIM step: fc1 + fc2 of the 8 blocks (the `cond` Linears are hoisted out of the loop)
PRIOR_GEMM_MFLOP_PER_STEP = 8 * 2 * 2 * 1024 * 4096 / 1e6
PRIOR_METRIC = "samples_per_sec_latent_prior_ddim50_vae_decode_64x64"


def prior_workload_config(args, n_per_gpu, world):
    return {"workload": f"latent diffusion prior (FiLM MLP, width 1024, 8 blocks, z_dim 32, T=1000, beta_end 0.05), "
                        f"{DDIM_STEPS}-step DDIM (eta 0), then CondVAE decode to 64x64, n={n_per_gpu} per GPU, random-init "
                        f"weights (BASELINE configs[3])",
            "n_per_gpu": n_per_gpu, "n_total": n_per_gpu * world, "ddim_steps": DDIM_STEPS, "precision": args.precision,
            "parallelism": f"dp{world} (batch sharded, all-gather of images)",
            "l2_policy": "inputs larger than L2: weights 206 MB bf16 + 268 MB FiLM table + activations per step >> 126 MB; "
                         "no explicit flush"}


def cpu_prior_samples_per_sec(n: int = 64, steps: int = 5):
    """The reference algorithm (oracle port) on the host cores: `steps` DDIM evaluations + one decode on n samples,
    the DDIM part extrapolated linearly to 50 steps."""
    import torch
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import latent_prior_oracle as po
    import toycrystals_oracle as orc
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    psd, vsd = po.prior_default_init(0), po.vae_default_init(2)
    y_cat, y_cont = orc.condition_grid(n, 4, 4)
    z = torch.randn((n, 32), generator=torch.Generator().manual_seed(1234))
    with torch.no_grad():
        t0 = time.perf_counter()
        for k in range(steps):
            t = torch.full((n,), 999 - 20 * k, dtype=torch.int64)
            eps = po.film_prior(psd, po.PRIOR_CFG, z, t, y_cat, y_cont)
            z = z - 0.01 * eps
        t1 = time.perf_counter()
        po.vae_decode(vsd, po.VAE_CFG, z, y_cat, y_cont)
        t2 = time.perf_counter()
    per_job = (t1 - t0) / steps * DDIM_STEPS + (t2 - t1)
    desc = (f"reference algorithm (oracle port, torch {torch.__version__} CPU fp32, {torch.get_num_threads()} threads): n={n}, "
            f"{steps} prior evaluations in {t1 - t0:.2f}s (extrapolated linearly to {DDIM_STEPS}) + decode {t2 - t1:.2f}s")
    return n / per_job, cores, desc


def run_reference_prior(args):
    if int(os.environ.get("RANK", "0")) != 0:
        return 0
    n = args.n or 4096
    vals = []
    for i in range(args.warmup + args.steps):
        sps, cores, desc = cpu_prior_samples_per_sec(n=max(args.cpu_n, 512), steps=max(2, args.cpu_steps // 3))
        if i >= args.warmup:
            vals.append(sps)
    v = statistics.mean(vals)
    print(json.dumps({
        "impl": "reference", "metric": PRIOR_METRIC, "value": v, "unit": "samples/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * args.cpu_n / v if v else None, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": prior_workload_config(args, n, args.gpus),
        "cpu_baseline": {"value": v, "unit": "samples/s", "cores": cores, "kind": "port", "sample": desc},
        "e2e": {"value": v, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}), flush=True)
    return 0


def run_gpu_prior(args):
    import ctypes as C
    import torch
    import torch.distributed as dist
    from toycrystals_b200 import _cabi
    from toycrystals_b200.models import diffusion_prior as pshim
    from toycrystals_b200.models import sde_score_model as shim
    from toycrystals_b200.models import vae as vshim

    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200: there is no CPU fallback for the product path")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        nccl_logging()
        dist.init_process_group("nccl", device_id=dev)
        report_comm(rank, world, local_rank, dev)
    n = args.n or 4096
    n_total = n * world
    lo, hi = shard_range(n_total, rank, world)
    torch.manual_seed(0)
    prior = pshim.DiffusionPriorFiLM(**PRIOR, precision=args.precision).to(dev).eval()
    torch.manual_seed(2)
    vae = vshim.CondVAE(z_dim=32, n_types=4, y_cont_dim=4).to(dev).eval()
    sched = pshim.DiffusionSchedule.linear(PRIOR_T, PRIOR_B0, PRIOR_B1, dev)
    # conditions exactly as save_diffusion_samples builds them, for this rank's block of global indices
    gi = torch.arange(lo, hi, device=dev)
    y_cat = (gi % 4).to(torch.int64)
    y_cont = torch.zeros((n, 4), device=dev)
    y_cont[:, 1] = torch.linspace(0.0, 3.141592653589793 / 3.0, steps=n_total, device=dev)[lo:hi]
    g = torch.Generator().manual_seed(7)
    h_mean = (torch.randn((32,), generator=g) * 0.3).pin_memory()
    h_std = (torch.rand((32,), generator=g) + 0.5).pin_memory()
    z_mean, z_std = h_mean.to(dev), h_std.to(dev)
    h_cat, h_cont = y_cat.cpu().pin_memory(), y_cont.cpu().pin_memory()
    h_img = torch.empty((n, 1, 64, 64), dtype=torch.float32).pin_memory()
    seed = 1234

    def job_device():
        x = pshim.sample_images(vae, prior, sched, y_cat, y_cont, z_mean, z_std, DDIM_STEPS, seed=seed, global_index_offset=lo)
        return gather_images(x, n_total, world)

    def job_e2e():
        yc, yk = h_cat.to(dev, non_blocking=True), h_cont.to(dev, non_blocking=True)
        zm, zs = h_mean.to(dev, non_blocking=True), h_std.to(dev, non_blocking=True)
        x = pshim.sample_images(vae, prior, sched, yc, yk, zm, zs, DDIM_STEPS, seed=seed, global_index_offset=lo)
        full = gather_images(x, n_total, world)
        h_img.copy_(full[lo:hi], non_blocking=True)
        torch.cuda.current_stream().synchronize()
        return float(h_img[0, 0, 0, 0])

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, k):
        """(ms over k calls of fn, max over ranks; what the last call returned)"""
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = None
        for _ in range(k):
            out = fn()
        e1.record()
        barrier()
        return max_over_ranks(e0.elapsed_time(e1), dev), out

    for _ in range(args.warmup):
        job_device()
    l0 = prior.launch_count() + vae.launch_count()
    with ClockSampler(local_rank) as clk:
        ms, images = timed(job_device, args.steps)
    launches = prior.launch_count() + vae.launch_count() - l0
    job_e2e()
    ms_e2e, _ = timed(job_e2e, args.steps)
    # decode alone (device events on the current stream; the library orders its stream against it)
    z = torch.randn((n, 32), device=dev)
    ms_dec = timed(lambda: vae.decode(z, y_cat, y_cont, z_mean=z_mean, z_std=z_std), 5)[0] / 5
    kms = (C.c_float * 4)()
    if rank == 0:
        _cabi.check(_cabi.lib().tcs_prior_profile(prior.engine_handle(sched), n, 20, kms))
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        sps, cores, desc = cpu_prior_samples_per_sec(n=max(args.cpu_n, 512), steps=max(2, args.cpu_steps // 3))
        cpu = {"value": sps, "unit": "samples/s", "cores": cores, "kind": "port", "sample": desc}
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, {"images": images})
    if rank == 0:
        peaks = load_peaks()
        value = n_total * args.steps / (ms / 1e3)
        e2e = n_total * args.steps / (ms_e2e / 1e3)
        burst = peaks.get("bf16_tflops", PEAKS_FALLBACK["bf16_tflops"])
        sustained = peaks.get("bf16_tflops_sustained", PEAKS_FALLBACK["bf16_tflops_sustained"])
        hbm = peaks.get("hbm_gbs", PEAKS_FALLBACK["hbm_gbs"])
        gemm_flop = 2.0 * n * 1024 * 4096
        gemm_ms = 0.5 * (kms[0] + kms[1])
        gemm_tflops = gemm_flop / (gemm_ms * 1e-3) / 1e12
        job_tflops = value / world * DDIM_STEPS * PRIOR_GEMM_MFLOP_PER_STEP / 1e6
        lnf_bytes = n * (1024 * 4 + 2 * 1024 * 4 + 1024 * (2 if args.precision == "bf16" else 4))
        line = {
            "metric": PRIOR_METRIC, "value": value, "unit": "samples/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": args.precision, "data": "synthetic", "config": prior_workload_config(args, n, world),
            "e2e": {"value": e2e, "unit": "samples/s",
                    "h2d_bytes_per_step": int(h_cat.numel() * 8 + h_cont.numel() * 4 + 2 * 32 * 4),
                    "d2h_bytes_per_step": int(h_img.numel() * 4)},
            "gpu_launches": int(launches), "clocks": clk.summary(),
            # dominant kernel = linear_tc_kernel (fc1 / fc2 of the FiLM blocks: 16 of the 25 launches of a DDIM step),
            # timed live with CUDA events on the library's stream (tcs_prior_profile)
            "roofline": {"bound": "tensor", "kernel": "tcs::linear_tc_kernel", "achieved": gemm_tflops, "peak": burst,
                         "unit": "TFLOP/s", "frac": gemm_tflops / burst, "traffic": None,
                         "peak_source": f"bf16_tflops burst ({peaks['_source']})", "launch_ms": gemm_ms,
                         "rows_per_launch": n, "fc1_ms": kms[0], "fc2_ms": kms[1],
                         "flop_per_launch": gemm_flop},
            "whole_job": {"achieved": job_tflops, "peak": sustained, "unit": "TFLOP/s", "frac": job_tflops / sustained,
                          "note": f"fc1+fc2 FLOPs of the job ({DDIM_STEPS} steps x {PRIOR_GEMM_MFLOP_PER_STEP:.1f} MFLOP/sample) / "
                                  f"time per GPU, vs bf16 sustained peak ({peaks['_source']}); decode and the per-call FiLM "
                                  f"table are inside the time but not the FLOP count"},
            "ln_film_kernel": {"bound": "hbm", "achieved": lnf_bytes / (kms[2] * 1e-3) / 1e9, "peak": hbm, "unit": "GB/s",
                               "frac": lnf_bytes / (kms[2] * 1e-3) / 1e9 / hbm, "launch_ms": kms[2],
                               "bytes_per_row": lnf_bytes // n},
            "tail_kernel_ms": kms[3], "decode_ms": ms_dec, "decode_share_of_job": ms_dec / (ms / args.steps),
            "cpu_baseline": cpu,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    vals = []
    for i in range(args.warmup + args.steps):
        sps, cores, kind, desc = cpu_reference_samples_per_sec(n=args.cpu_n, steps=args.cpu_steps)
        if i >= args.warmup:
            vals.append(sps)
    v = statistics.mean(vals)
    line = {
        "impl": "reference", "metric": "samples_per_sec_64x64_sde300_cfg1.5", "value": v, "unit": "samples/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * args.cpu_n / v if v else None, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, n_per_gpu=args.n or 1024, world=args.gpus),
        "cpu_baseline": {"value": v, "unit": "samples/s", "cores": cores, "kind": kind, "sample": desc},
        "e2e": {"value": v, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    try:   # context only (north_star quotes its target against the reference's CUDA eager sampler)
        import torch
        if torch.cuda.is_available() and not args.no_cuda_eager:
            n_eager = args.n or 1024
            line["reference_cuda_eager"] = [cuda_eager_reference_samples_per_sec(n=n_eager, tf32=True),
                                            cuda_eager_reference_samples_per_sec(n=n_eager, tf32=False)]
    except Exception as e:  # noqa: BLE001
        line["reference_cuda_eager"] = {"error": str(e)[:200]}
    print(json.dumps(line), flush=True)
    return 0


def workload_config(args, n_per_gpu, world):
    strong = getattr(args, "scaling", "weak") == "strong"
    cfg_name = "BASELINE configs[2]" if strong else "BASELINE configs[1]"
    size = (f"n_total={n_per_gpu * world} sharded over {world} GPU(s)" if strong else f"n={n_per_gpu} per GPU")
    d = {"workload": f"VP-SDE reverse-SDE Euler-Maruyama sampling, EMA weights (random-init seed 1), CFG {CFG}, "
                     f"{SDE_STEPS} steps, t_end {T_END}, 64x64x1, {size} ({cfg_name})",
         "n_per_gpu": n_per_gpu, "n_total": n_per_gpu * world, "sde_steps": SDE_STEPS, "cfg": CFG, "t_end": T_END,
         "sampler": "sde", "precision": args.precision, "parallelism": f"dp{world} (batch sharded, all-gather of images)",
         "l2_policy": "inputs larger than L2: per-step activation working set >> 126 MB; no explicit flush"}
    if getattr(args, "warmup_sde_steps", 0):
        d["warmup_note"] = (f"each warm-up job runs {args.warmup_sde_steps} of the {SDE_STEPS} steps (same n, same CUDA graph, "
                            f"same kernels); the timed jobs are complete")
    return d


# ---------------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------------
def run_gpu(args):
    import torch
    import torch.distributed as dist
    from toycrystals_b200.models import sde_score_model as shim

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200: there is no CPU fallback for the product path")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        nccl_logging()
        dist.init_process_group("nccl", device_id=dev)
        report_comm(rank, world, local_rank, dev)
    strong = args.scaling == "strong"
    if strong:       # BASELINE configs[2]: a fixed job (n_total) sharded over the ranks
        n_total = args.n_total or 65536
        lo, hi = shard_range(n_total, rank, world)
        n = hi - lo
    else:            # configs[1] per GPU
        n = args.n or 1024
        n_total = n * world
        lo, hi = shard_range(n_total, rank, world)

    # weights: default init, seed 0 = model, seed 1 = EMA (the sampled one); built without the oracle
    torch.manual_seed(1)
    model = shim.CondUNetTiny(4, 4, 96, 128, 8, 8, precision=args.precision, engine=args.engine, chunk=args.chunk).to(dev).eval()
    sde = shim.VPSDE(0.1, 30.0)
    y_cat, y_cont = shim.condition_grid(model, n, 3.141592653589793 / 3.0, dev, offset=lo, n_total=n_total)
    h_cat, h_cont = y_cat.cpu().pin_memory(), y_cont.cpu().pin_memory()
    h_img = torch.empty((n, 1, 64, 64), dtype=torch.float32).pin_memory()
    seed = 1234

    def job_device(steps=SDE_STEPS):
        x = shim.sample_reverse_sde_euler_maruyama(model, sde, y_cat, y_cont, (n, 1, 64, 64), n_steps=steps,
                                                   guidance_scale=CFG, t_end=T_END, seed=seed, global_index_offset=lo)
        return gather_images(x, n_total, world)

    def job_e2e():
        yc = h_cat.to(dev, non_blocking=True)
        yk = h_cont.to(dev, non_blocking=True)
        x = shim.sample_reverse_sde_euler_maruyama(model, sde, yc, yk, (n, 1, 64, 64), n_steps=SDE_STEPS,
                                                   guidance_scale=CFG, t_end=T_END, seed=seed, global_index_offset=lo)
        full = gather_images(x, n_total, world)
        h_img.copy_(full[lo:hi], non_blocking=True)
        torch.cuda.current_stream().synchronize()
        return float(h_img[0, 0, 0, 0])

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, k):
        """(ms over k calls of fn, max over ranks; what the last call returned)"""
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = None
        for _ in range(k):
            out = fn()
        e1.record()
        barrier()
        return max_over_ranks(e0.elapsed_time(e1), dev), out

    for _ in range(args.warmup):
        job_device(args.warmup_sde_steps or SDE_STEPS)
    launches0 = model.launch_count()
    with ClockSampler(local_rank) as clk:
        ms, images = timed(job_device, args.steps)
    launches = model.launch_count() - launches0
    if args.skip_e2e:
        ms_e2e = None
    else:
        if not args.warmup_sde_steps:   # (long strong-scaling jobs: the device jobs above already warmed everything)
            job_e2e()
        ms_e2e, _ = timed(job_e2e, args.steps)

    kern = profile_kernels(model, sde, dev, n=args.profile_n) if rank == 0 else None
    extra = {}
    if rank == 0 and world == 1 and not strong and not args.no_extra:
        extra = extra_lines(args, dev)
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        sps, cores, kind, desc = cpu_reference_samples_per_sec(n=args.cpu_n, steps=args.cpu_steps)
        cpu = {"value": sps, "unit": "samples/s", "cores": cores, "kind": kind, "sample": desc}
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, {"images": images})
    if rank == 0:
        peaks = load_peaks()
        value = n_total * args.steps / (ms / 1e3)
        e2e = n_total * args.steps / (ms_e2e / 1e3) if ms_e2e else None
        tflop_per_sample = 2 * (SDE_STEPS + 1) * CONV_GFLOP_PER_FORWARD / 1e3
        achieved = value / world * tflop_per_sample
        peak = peaks.get("bf16_tflops_sustained", PEAKS_FALLBACK["bf16_tflops_sustained"])
        burst = peaks.get("bf16_tflops", PEAKS_FALLBACK["bf16_tflops"])
        hbm = peaks.get("hbm_gbs", PEAKS_FALLBACK["hbm_gbs"])
        # the conv family is timed INSIDE a long step-like loop at the power cap (back-to-back 2048-image passes), so the
        # sustained figure is its denominator; `frac_of_burst` is printed beside it
        line = {
            "metric": "samples_per_sec_64x64_sde300_cfg1.5", "value": value, "unit": "samples/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": args.scaling, "vs_baseline": None, "dtype": args.precision, "data": "synthetic",
            "config": workload_config(args, n, world),
            "e2e": {"value": e2e, "unit": "samples/s", "h2d_bytes_per_step": int(h_cat.numel() * 8 + h_cont.numel() * 4),
                    "d2h_bytes_per_step": int(h_img.numel() * 4)},
            "gpu_launches": int(launches),
            "clocks": clk.summary(),
            # dominant kernel family = conv_tc_kernel (all 15 tcgen05 convolutions of one network pass, GroupNorm+SiLU
            # epilogues included), timed live with CUDA events on the library's stream (tcs_score_profiled) at the
            # PRODUCTION shape: one pass over images_per_launch images, each launch 0.2 - 1.3 ms
            "roofline": {"bound": "tensor", "kernel": "tcs::conv_tc_kernel", "achieved": kern["conv_tflops"],
                         "peak": peak, "unit": "TFLOP/s", "frac": kern["conv_tflops"] / peak,
                         "frac_of_burst": kern["conv_tflops"] / burst,
                         "traffic": kern.get("traffic"), "traffic_source": kern.get("traffic_source"),
                         "peak_source": f"bf16_tflops_sustained ({peaks['_source']}): the passes are timed back to back at the "
                                        f"power cap, like the job",
                         "launch_ms": kern["conv_ms"], "images_per_launch": kern["images"],
                         "flop_per_launch_set": kern["conv_flop"], "share_of_pass": kern["conv_share"],
                         "pass_ms": kern["pass_ms"], "conv_layers": kern.get("conv_layers"),
                         "attention_block_ms": kern.get("attention_block_ms"), "per_layer_tflops": kern["per_layer"]},
            "whole_job": {"achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
                          "note": f"conv FLOPs of the whole job ({tflop_per_sample:.3f} TFLOP/sample, 7.092 GFLOP/forward) / "
                                  f"time per GPU, vs bf16 sustained peak ({peaks['_source']})"},
            "step_kernel": {"bound": "hbm", "kernel": "tcs::step_kernel<SDE>", "achieved": kern["step_gbs"],
                            "peak": hbm, "unit": "GB/s", "frac": kern["step_gbs"] / hbm,
                            "bytes_per_sample": 3 * 16384, "samples_per_launch": kern["step_n"]},
            "cpu_baseline": cpu,
            "extra": extra,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def extra_lines(args, dev):
    """Driver-visible numbers for the other modes of the same path, each a complete (shorter) job with its own clock
    record: the fp32 (1e-4) mode on the tensor pipe (bf16x3 split) and the latent-prior row (configs[3])."""
    import torch
    from toycrystals_b200.models import sde_score_model as shim
    out = {}
    try:
        torch.manual_seed(1)
        n = 1024
        m = shim.CondUNetTiny(4, 4, 96, 128, 8, 8, precision="fp32", engine="tcgen05").to(dev).eval()
        sde = shim.VPSDE(0.1, 30.0)
        yc, yk = shim.condition_grid(m, n, 3.141592653589793 / 3.0, dev)
        run = lambda st: shim.sample_reverse_sde_euler_maruyama(m, sde, yc, yk, (n, 1, 64, 64), n_steps=st, guidance_scale=CFG,  # noqa: E731
                                                                t_end=T_END, seed=1234)
        run(5)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with ClockSampler(dev.index or 0) as clk:
            e0.record()
            run(SDE_STEPS)
            e1.record()
            torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        out["fp32_tensor_core_mode"] = {
            "value": n / (ms / 1e3), "unit": "samples/s", "ms_per_job": ms, "n": n, "sde_steps": SDE_STEPS,
            "precision": "fp32 operands as bf16 hi+lo pairs, 3 tcgen05 MMAs per product term set, fp32 accumulate; "
                         "per-evaluation eps rel-L2 <= 1e-4 vs the reference (tests/test_gpu_parity.py)",
            "clocks": clk.summary()}
        del m
        torch.cuda.empty_cache()
    except Exception as e:  # noqa: BLE001
        out["fp32_tensor_core_mode"] = {"error": str(e)[:300]}
    try:
        out["prior"] = prior_quick(dev)
    except Exception as e:  # noqa: BLE001
        out["prior"] = {"error": str(e)[:300]}
    return out


def prior_quick(dev, n=4096, seconds=6.0):
    """BASELINE configs[3] (latent prior, 50-step DDIM + VAE decode, n = 4096) for >= `seconds` of back-to-back jobs so that
    the nvidia-smi clock record has samples; the full contract line is `bench.py --workload prior`."""
    import torch
    from toycrystals_b200.models import diffusion_prior as pshim
    from toycrystals_b200.models import vae as vshim
    torch.manual_seed(0)
    prior = pshim.DiffusionPriorFiLM(**PRIOR, precision="bf16").to(dev).eval()
    torch.manual_seed(2)
    vae = vshim.CondVAE(z_dim=32, n_types=4, y_cont_dim=4).to(dev).eval()
    sched = pshim.DiffusionSchedule.linear(PRIOR_T, PRIOR_B0, PRIOR_B1, dev)
    gi = torch.arange(0, n, device=dev)
    y_cat = (gi % 4).to(torch.int64)
    y_cont = torch.zeros((n, 4), device=dev)
    y_cont[:, 1] = torch.linspace(0.0, 3.141592653589793 / 3.0, steps=n, device=dev)
    g = torch.Generator().manual_seed(7)
    z_mean, z_std = (torch.randn((32,), generator=g) * 0.3).to(dev), (torch.rand((32,), generator=g) + 0.5).to(dev)
    job = lambda: pshim.sample_images(vae, prior, sched, y_cat, y_cont, z_mean, z_std, DDIM_STEPS, seed=1234)  # noqa: E731
    for _ in range(3):
        job()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); job(); e1.record(); torch.cuda.synchronize()
    k = max(20, int(seconds * 1e3 / max(e0.elapsed_time(e1), 1e-3)))
    with ClockSampler(dev.index or 0) as clk:
        e0.record()
        for _ in range(k):
            job()
        e1.record()
        torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / k
    peaks = load_peaks()
    sustained = peaks.get("bf16_tflops_sustained", PEAKS_FALLBACK["bf16_tflops_sustained"])
    job_tflops = n / (ms / 1e3) * DDIM_STEPS * PRIOR_GEMM_MFLOP_PER_STEP / 1e6
    return {"metric": PRIOR_METRIC, "value": n / (ms / 1e3), "unit": "samples/s", "ms_per_job": ms, "jobs_timed": k, "n": n,
            "whole_job": {"achieved": job_tflops, "peak": sustained, "unit": "TFLOP/s", "frac": job_tflops / sustained},
            "clocks": clk.summary()}


def profile_kernels(model, sde, dev, n=1024):
    """Per-kernel numbers, measured live at the PRODUCTION shape: (a) the tcgen05 conv family of one network pass over
    2n images (n = 1024 with CFG = the 2048-image pass the job runs) via tcs_score_profiled — CUDA events on the library
    stream around each conv launch; at this size a launch lasts 0.2 - 1.3 ms, so host launch latency cannot leak into the
    event pairs (the round-1 probe timed ~100 us launches of 256 images and was host sensitive) — over `reps` back-to-back
    passes after warm-up passes; (b) the fused SDE update kernel alone."""
    import ctypes as C
    import torch
    from toycrystals_b200 import _cabi
    from toycrystals_b200.models import sde_score_model as shim
    L = _cabi.lib()
    h = model.engine_handle(sde)
    y_cat, y_cont = shim.condition_grid(model, n, 3.141592653589793 / 3.0, dev)
    x = torch.randn((n, 1, 64, 64), device=dev)
    t = torch.full((n,), 0.37, device=dev)
    eps = torch.empty_like(x)
    conv = (C.c_float * 15)()
    tot = C.c_float()
    acc, tots = [0.0] * 15, 0.0
    warm, reps = 6, 12
    for r in range(warm + reps):
        _cabi.check(L.tcs_score_profiled(h, x.data_ptr(), t.data_ptr(), y_cat.data_ptr(), y_cont.data_ptr(), n, CFG,
                                         eps.data_ptr(), conv, C.byref(tot), torch.cuda.current_stream(dev).cuda_stream))
        if r >= warm:
            acc = [a + float(c) for a, c in zip(acc, conv)]
            tots += float(tot.value)
    images = 2 * n
    conv_ms = [a / reps for a in acc]
    flops = [2e6 * m * images for m in TC_CONV_MMAC]
    per_layer = {k: round(f / (ms * 1e-3) / 1e12, 1) for k, f, ms in zip(TC_CONV_NAMES, flops, conv_ms) if ms > 5e-3}
    iq, ip = TC_CONV_NAMES.index("attn.qkv"), TC_CONV_NAMES.index("attn.proj")
    if conv_ms[ip] <= 5e-3:   # fused attention block (attn_tc.cu): norm + qkv + softmax(q k^T) v + proj in the attn.qkv slot
        per_layer.pop("attn.qkv", None)
        blk = flops[iq] + flops[ip] + 2e6 * ATTN_SDPA_MMAC * images
        per_layer["attn.block(norm+qkv+sdpa+proj)"] = round(blk / (conv_ms[iq] * 1e-3) / 1e12, 1)
    traffic, traffic_source = None, None   # DRAM bytes of the same 15 launches from the committed `ncu --set full` capture
    for name in ("r2_conv_ncu_full_fused.json", "r2_conv_ncu_full.json", "r1_conv_ncu_full.json"):
        tp = os.path.join(ROOT, "profiles", name)
        if os.path.exists(tp):
            tj = json.load(open(tp))
            if tj.get("images_per_pass") == images:
                traffic, traffic_source = tj["traffic_bytes_per_pass"], f"profiles/{name}"
                break
    fam_flops, fam_ms, attn_ms = list(flops), list(conv_ms), None
    if conv_ms[ip] <= 5e-3:   # the attention block is its own kernel (attn_tc.cu), not a conv_tc launch: the conv family
        attn_ms = conv_ms[iq]  # (the kernel the roofline is about) is the 13 remaining layers, as in the ncu capture
        for j in sorted((iq, ip), reverse=True):
            del fam_flops[j], fam_ms[j]
    out = {"conv_tflops": sum(fam_flops) / (sum(fam_ms) * 1e-3) / 1e12, "conv_ms": sum(fam_ms), "images": images,
           "conv_flop": sum(fam_flops), "conv_share": sum(fam_ms) / (tots / reps), "pass_ms": tots / reps,
           "conv_layers": len(fam_ms), "attention_block_ms": attn_ms,
           "per_layer": per_layer, "traffic": traffic, "traffic_source": traffic_source}
    # the fused VP-SDE update, Philox noise in registers: 48 KiB of algorithmic traffic per sample
    ns = 32768
    xs = torch.randn((ns, 1, 64, 64), device=dev)
    es = torch.randn_like(xs)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for r in range(3 + 20):
        if r == 3:
            e0.record()
        _cabi.check(L.tcs_sde_update(h, xs.data_ptr(), es.data_ptr(), None, ns, 0.5, 0.499, 1234, 0, r,
                                     torch.cuda.current_stream(dev).cuda_stream))
    e1.record()
    torch.cuda.synchronize()
    out["step_gbs"] = ns * 3 * 16384 / (e0.elapsed_time(e1) / 20 * 1e-3) / 1e9
    out["step_n"] = ns
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="sde", choices=["sde", "prior"],
                    help="sde = BASELINE configs[1] (the headline); prior = configs[3] (latent prior DDIM + VAE decode)")
    ap.add_argument("--n", type=int, default=0, help="samples per GPU per job (default 1024 for sde, 4096 for prior)")
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--engine", default="auto", choices=["auto", "simt", "tcgen05"],
                    help="auto = tcgen05 for bf16, FFMA for fp32; `--precision fp32 --engine tcgen05` = fp32 operands as bf16x3 on "
                         "the tensor pipe")
    ap.add_argument("--chunk", type=int, default=0)
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: --n samples per GPU (configs[1]); strong: --n-total samples sharded over the ranks (configs[2])")
    ap.add_argument("--n-total", type=int, default=0, help="strong scaling: total samples of the job (default 65536)")
    ap.add_argument("--warmup-sde-steps", type=int, default=0,
                    help="run the warm-up jobs with this many SDE steps instead of 300 (long strong-scaling jobs; stated in config)")
    ap.add_argument("--profile-n", type=int, default=1024, help="samples of the per-layer roofline pass (x2 images with CFG)")
    ap.add_argument("--skip-e2e", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the fp32-tensor-core and latent-prior extra jobs")
    ap.add_argument("--cpu-n", type=int, default=64)
    ap.add_argument("--cpu-steps", type=int, default=15)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-cuda-eager", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write the images of the last timed step to DIR/images.npy (float32) for output comparisons")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs records the B200 implementation's outputs; it does not apply to --impl reference")
    if args.workload == "prior":
        return run_reference_prior(args) if args.impl == "reference" else run_gpu_prior(args)
    if args.impl == "reference":
        return run_reference(args)
    return run_gpu(args)


if __name__ == "__main__":
    raise SystemExit(main())
