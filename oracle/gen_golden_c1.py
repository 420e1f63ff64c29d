#!/usr/bin/env python3
"""BASELINE configs[0] at FULL size on the reference itself: PF-ODE (Heun), n=36, 300 steps, cfg 1.5,
t_end 0.005, EMA weights = default init seed 1, x_init from torch.Generator(1234).  ~30-60 min on 8 cores.
Writes tests/golden/c1_ode_n36_s300.pt (x_init is regenerated from the seed, not stored; the image from x0_hat)."""
import os
import sys
import time

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "_stubs"))
sys.path.insert(0, "/root/reference/src")
sys.path.insert(0, HERE)
import toycrystals.models.sde_score_model as ref  # noqa: E402
import toycrystals_oracle as orc  # noqa: E402

torch.set_num_threads(int(os.environ.get("C1_THREADS", "6")))
n, steps = 36, 300
torch.manual_seed(1)
m = ref.CondUNetTiny(**orc.DEFAULT_CFG).eval()
sde = ref.VPSDE(0.1, 30.0)
y_cat, y_cont = orc.condition_grid(n, 4, 4)
x_init = torch.randn((n, 1, 64, 64), generator=torch.Generator().manual_seed(1234))
real = torch.randn
torch.randn = lambda *a, **k: x_init.clone()
x0_holder = {}
real_clamp = torch.clamp
t0 = time.time()
try:
    # capture the pre-clamp x0_hat: the reference computes (x - s*eps)/clamp(a) then maps to [0,1]
    real_pred = ref.predict_eps_cfg
    calls = []

    def logged(model, x_t, t, yc, yk, guidance_scale):
        e = real_pred(model, x_t, t, yc, yk, guidance_scale)
        calls.append(1)
        if len(calls) % 50 == 0:
            print(len(calls), "evaluations", round(time.time() - t0), "s", flush=True)
        x0_holder["x"], x0_holder["eps"], x0_holder["t"] = x_t.clone(), e.clone(), float(t[0])
        return e

    ref.predict_eps_cfg = logged
    img = ref.sample_probability_flow_ode(model=m, sde=sde, y_cat=y_cat, y_cont=y_cont, img_shape=(n, 1, 64, 64),
                                          n_steps=steps, guidance_scale=1.5, t_end=0.005)
finally:
    torch.randn = real
    ref.predict_eps_cfg = real_pred
tf = torch.tensor(x0_holder["t"])
a, s = sde.alpha(tf), sde.sigma(tf)
x0_hat = (x0_holder["x"] - s * x0_holder["eps"]) / torch.clamp(a, min=1e-6)
assert torch.equal(((x0_hat + 1.0) * 0.5).clamp(0.0, 1.0), img)
assert len(calls) == 2 * steps + 1
# the image follows from x0_hat (asserted above); the last evaluation's input and output are kept for every third sample
# (all four classes, the whole theta range), so that the file stays under 1 MB
keep = torch.arange(0, n, 3)
out = dict(n=n, steps=steps, cfg=1.5, t_end=0.005, seed_weights=1, seed_x=1234, x0_hat=x0_hat, final_index=keep,
           x_final=x0_holder["x"][keep].clone(), eps_final=x0_holder["eps"][keep].clone(), nfe=len(calls),
           seconds=time.time() - t0)
torch.save(out, os.path.join(os.path.dirname(HERE), "tests", "golden", "c1_ode_n36_s300.pt"))
print("done", out["seconds"], "s; |x0_hat| max", float(x0_hat.abs().max()))
