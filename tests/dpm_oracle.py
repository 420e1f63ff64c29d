"""CPU oracle of the DPM-Solver++(2M) sampler.  It is test infrastructure, like ``oracle/toycrystals_oracle.py``, whose
network, schedule and trace types it uses unchanged.

The reference has no such sampler, so this module is pinned by the closed-form tests of ``tests/test_cpu_dpm.py``
rather than by golden vectors: Gaussian data, where the exact eps and the exact probability-flow ODE solution are
known; and eps == 0, where the solver is exact.  It is dtype-generic: in float64 it is the "truth" of those tests, and
in float32 it is what the GPU path is compared against.
"""
from __future__ import annotations

import math
from typing import Optional

import torch

from toycrystals_oracle import SampleTrace, Schedule, StateDict, eps_cfg
# --------------------------------------------------------------------------
# DPM-Solver++(2M)
# --------------------------------------------------------------------------
def dpm_schedule(n_steps: int, t_end: float, sched: Schedule):
    """Time grid and per-step coefficients of ``sample_dpmpp_2m``.

    Times are uniform in log-SNR lambda(t) = log alpha(t) - log sigma(t) from t = 1 to t_end; each comes from the closed
    inverse t(lambda) and is rounded to fp32, and the endpoints are exactly 1 and fp32(t_end).  The coefficients of step
    i are computed in double from those fp32 times:
        h = lambda(t_{i+1}) - lambda(t_i),  a = sigma(t_{i+1})/sigma(t_i),  m = alpha(t_{i+1}) * (-expm1(-h)),
        (c0, c1) = (1, 0) on step 0 and, when n_steps < 15, on the last step; else r = h_{i-1}/h_i and
        (c0, c1) = (1 + 1/(2r), -1/(2r)).
    Returns (ts: n_steps+1 floats, rows: n_steps tuples (a, m, c0, c1)), all Python floats (double)."""
    bmin, d = float(sched.beta_min), float(sched.beta_max) - float(sched.beta_min)

    def alpha(t):
        return math.exp(-0.5 * (bmin * t + 0.5 * d * (t * t)))

    def sigma(t):
        a = alpha(t)
        return math.sqrt(max(1.0 - a * a, 1e-8))

    def lam(t):
        return math.log(alpha(t)) - math.log(sigma(t))

    def f32(v):
        return float(torch.tensor(v, dtype=torch.float64).float())

    l_start, l_end = lam(1.0), lam(float(t_end))
    ts = [1.0]
    for i in range(1, n_steps):
        lv = l_start + (i / n_steps) * (l_end - l_start)
        ib = math.log1p(math.exp(-2.0 * lv))
        ts.append(f32((-bmin + math.sqrt(bmin * bmin + 2.0 * d * ib)) / d if d > 0.0 else ib / bmin))
    if n_steps >= 1:
        ts.append(f32(float(t_end)))
    rows, h_prev = [], 0.0
    for i in range(n_steps):
        t0, t1 = ts[i], ts[i + 1]
        h = lam(t1) - lam(t0)
        a, m = sigma(t1) / sigma(t0), alpha(t1) * -math.expm1(-h)
        if i == 0 or (i == n_steps - 1 and n_steps < 15):
            c0, c1 = 1.0, 0.0
        else:
            r = h_prev / h
            c0, c1 = 1.0 + 1.0 / (2.0 * r), -1.0 / (2.0 * r)
        rows.append((a, m, c0, c1))
        h_prev = h
    return ts, rows


@torch.no_grad()
def sample_dpmpp_2m(sd: Optional[StateDict], cfg: Optional[dict], sched: Schedule, y_cat, y_cont, x_init: torch.Tensor,
                    n_steps: int, guidance: float, t_end: float, eps_fn=None, keep_trace: bool = True) -> SampleTrace:
    """DPM-Solver++(2M) (Lu et al. 2022, "DPM-Solver++", Algorithm 2) on the probability-flow ODE, then the same final
    projection as ``sample``: n_steps + 1 network evaluations.

    The reference has no such sampler, so there are no golden vectors for it: this function is pinned by the closed-form
    tests instead (Gaussian data, where the exact eps and the exact PF-ODE solution are known; and eps == 0, where the
    solver is exact).  ``eps_fn(x, t)``, if given, replaces the network (``sd``, ``cfg``, ``y_cat``, ``y_cont`` and
    ``guidance`` are then unused).  Every step, in the dtype of ``x_init`` (the coefficients of ``dpm_schedule`` are
    rounded to it once):
        x0 = (x - sigma_i eps) / alpha_i;  D = x0 (first-order rows) or c0 x0 + c1 x0_prev;  x <- a x + m D."""
    if not (0.0 < float(t_end) < 1.0):
        raise ValueError(f"t_end must be in (0,1), got {t_end}")
    x = x_init.clone()
    B = x.shape[0]
    ts_list, rows = dpm_schedule(n_steps, float(t_end), sched)
    if n_steps == 0:
        ts_list = [1.0]
    ts = torch.tensor(ts_list, dtype=torch.float64).to(device=x.device, dtype=x.dtype)
    coef = torch.tensor(rows, dtype=torch.float64).reshape(-1, 4).to(device=x.device, dtype=x.dtype)
    tr = SampleTrace(image=x, x0_hat=x, eps=[], x_in=[], t_in=[], ts=ts)

    def evaluate(xx, t):
        e = eps_fn(xx, t) if eps_fn is not None else eps_cfg(sd, cfg, xx, t, y_cat, y_cont, guidance)
        if keep_trace:
            tr.eps.append(e.clone()); tr.x_in.append(xx.clone()); tr.t_in.append(float(t[0]))
        return e

    x0_prev = None
    for i in range(n_steps):
        t = ts[i].expand(B)
        al = sched.alpha(t).view(B, 1, 1, 1)
        sg = sched.sigma(t).view(B, 1, 1, 1)
        x0 = (x - sg * evaluate(x, t)) / al
        a, m, c0, c1 = coef[i]
        D = x0 if float(c1) == 0.0 else c0 * x0 + c1 * x0_prev
        x = a * x + m * D
        x0_prev = x0

    t_fin = ts[-1].expand(B)
    a = sched.alpha(t_fin).view(B, 1, 1, 1)
    s = sched.sigma(t_fin).view(B, 1, 1, 1)
    x0_hat = (x - s * evaluate(x, t_fin)) / torch.clamp(a, min=1e-6)
    tr.x0_hat = x0_hat
    tr.image = ((x0_hat + 1.0) * 0.5).clamp(0.0, 1.0)
    return tr
