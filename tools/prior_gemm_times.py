#!/usr/bin/env python3
"""fc1 / fc2 / LN+FiLM / tail kernel times of the latent prior (tcs_prior_profile), n rows."""
import ctypes as C
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "vae-diffusion-toy-crystals_b200"))
from toycrystals_b200 import _cabi  # noqa: E402
from toycrystals_b200.models import diffusion_prior as pshim  # noqa: E402

n = int(sys.argv[1]) if len(sys.argv) > 1 else 4096
torch.manual_seed(0)
prior = pshim.DiffusionPriorFiLM(32, 4, 4, 64, 1024, 8, 64, precision="bf16").cuda().eval()
sched = pshim.DiffusionSchedule.linear(1000, 1e-4, 0.05, torch.device("cuda"))
y_cat = (torch.arange(n, device="cuda") % 4).to(torch.int64)
y_cont = torch.zeros((n, 4), device="cuda")
sched.ddim_sample(prior, y_cat, y_cont, n_steps=3, seed=1)
torch.cuda.synchronize()
ms = (C.c_float * 4)()
_cabi.check(_cabi.lib().tcs_prior_profile(prior.engine_handle(sched), n, 50, ms))
fl = 2.0 * n * 1024 * 4096
print(f"n={n} fc1 {ms[0]*1e3:.1f} us ({fl/ms[0]/1e9:.0f} TF)  "
      f"fc2 {ms[1]*1e3:.1f} us ({fl/ms[1]/1e9:.0f} TF)  lnf {ms[2]*1e3:.1f} us  tail {ms[3]*1e3:.1f} us")
