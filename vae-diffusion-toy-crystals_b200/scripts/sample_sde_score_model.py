#!/usr/bin/env python3
"""Same command line as the reference's scripts/sample_sde_score_model.py (:30-131): same flags,
defaults, checkpoint layout ({"config","model",["ema"]}), default output name and final print.
Additions: --precision {bf16,fp32}, --out-tensor (dump all n samples as a .pt tensor), --sampler dpm++2m
(DPM-Solver++(2M): one network evaluation per step; 20 steps is the usual choice) and --sampler dpm++2m-sde
(SDE-DPM-Solver++(2M): stochastic, second order, one evaluation per step).

    python scripts/sample_sde_score_model.py --out-dir runs/sde --steps 300 --cfg 1.5 \
        --t-end 0.005 --sampler sde --use-ema 1
"""
import argparse
import math
import os
import sys

import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
from toycrystals_b200.models.sde_score_model import (  # noqa: E402
    _SAMPLERS, CondUNetTiny, VPSDE, condition_grid, save_sde_samples)


def _infer_ckpt_path(out_dir: str, ckpt: str) -> str:
    if ckpt.endswith(".pt"):
        return ckpt
    if ckpt in ("last", "best"):
        return os.path.join(out_dir, "checkpoints", f"sde_score_model_{ckpt}.pt")
    raise ValueError("ckpt must be a .pt path or one of: last, best")


def main(argv=None) -> int:
    p = argparse.ArgumentParser()
    p.add_argument("--device", default="cuda", choices=["cpu", "cuda"])
    p.add_argument("--out-dir", required=True, help="Training output dir containing checkpoints/")
    p.add_argument("--ckpt", default="last", help="Checkpoint: last, best, or path/to/file.pt")
    p.add_argument("--steps", type=int, default=200)
    p.add_argument("--cfg", type=float, default=0.0)
    p.add_argument("--t-end", type=float, default=1e-3)
    p.add_argument("--theta-max", type=float, default=math.pi / 3.0)
    p.add_argument("--n", type=int, default=36)
    p.add_argument("--use-ema", type=int, default=0, choices=[0, 1], help="If checkpoint has EMA weights, sample using them.")
    p.add_argument("--sampler", type=str, default="ode", choices=list(_SAMPLERS))
    # fallback model / SDE config, used only when the checkpoint has no payload["config"]
    p.add_argument("--n-types", type=int, default=4)
    p.add_argument("--y-cont-dim", type=int, default=4)
    p.add_argument("--base-ch", type=int, default=96)
    p.add_argument("--emb-dim", type=int, default=128)
    p.add_argument("--cond-ch", type=int, default=8)
    p.add_argument("--time-ch", type=int, default=8)
    p.add_argument("--beta-min", type=float, default=0.1)
    p.add_argument("--beta-max", type=float, default=30.0)
    p.add_argument("--out-path", default=None, help="Where to save the sample grid png")
    # additions
    p.add_argument("--precision", default="bf16", choices=["bf16", "fp32"])
    p.add_argument("--out-tensor", default=None, help="also save all n samples as a [n,1,64,64] tensor (.pt)")
    args = p.parse_args(argv)
    if args.device == "cpu":
        raise RuntimeError("toycrystals_b200 has no CPU path; use the reference package for --device cpu")
    device = torch.device(args.device)

    ckpt_path = _infer_ckpt_path(args.out_dir, args.ckpt)
    if not os.path.exists(ckpt_path):
        raise FileNotFoundError(f"Checkpoint not found: {ckpt_path}")
    payload = torch.load(ckpt_path, map_location="cpu")
    cfg = payload.get("config", None)
    if cfg is None:
        cfg = dict(img_ch=1, n_types=args.n_types, y_cont_dim=args.y_cont_dim, base_ch=args.base_ch,
                   emb_dim=args.emb_dim, cond_ch=args.cond_ch, time_ch=args.time_ch, beta_min=args.beta_min,
                   beta_max=args.beta_max)
    model = CondUNetTiny(n_types=cfg["n_types"], y_cont_dim=cfg["y_cont_dim"], base_ch=cfg["base_ch"],
                         emb_dim=cfg["emb_dim"], cond_ch=cfg["cond_ch"], time_ch=cfg["time_ch"],
                         precision=args.precision).to(device)
    model.load_state_dict(payload["model"])
    if args.use_ema == 1 and ("ema" in payload):
        model.load_state_dict(payload["ema"])
    model.eval()
    sde = VPSDE(beta_min=cfg.get("beta_min", 0.1), beta_max=cfg.get("beta_max", 30.0))

    if args.out_path is None:
        os.makedirs(os.path.join(args.out_dir, "results"), exist_ok=True)
        args.out_path = os.path.join(
            args.out_dir, "results",
            f"samples_ckpt-{os.path.splitext(os.path.basename(ckpt_path))[0]}"
            f"_steps{args.steps}_cfg{args.cfg:.2f}_tend{args.t_end:g}_sampler{args.sampler}_ema{args.use_ema}.png")

    if args.out_tensor:
        y_cat, y_cont = condition_grid(model, args.n, args.theta_max, device)
        fn = _SAMPLERS[args.sampler]
        x = fn(model=model, sde=sde, y_cat=y_cat, y_cont=y_cont, img_shape=(args.n, 1, 64, 64), n_steps=args.steps,
               guidance_scale=args.cfg, t_end=args.t_end)
        torch.save(x.cpu(), args.out_tensor)
        from toycrystals_b200.models.sde_score_model import _write_grid_png
        _write_grid_png(x, args.out_path, f"{args.sampler} | steps={args.steps} | cfg={args.cfg:.2f} | t_end={args.t_end:g}")
    else:
        save_sde_samples(model=model, sde=sde, out_path=args.out_path, device=device, n=args.n,
                         theta_max=args.theta_max, steps=args.steps, cfg=args.cfg, t_end=args.t_end,
                         sampler=args.sampler)
    print(f"Saved samples -> {args.out_path}")
    return 0


if __name__ == "__main__":
    raise SystemExit(main())
