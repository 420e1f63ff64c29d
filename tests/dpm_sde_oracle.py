"""CPU oracle of the SDE-DPM-Solver++(2M) sampler, and the exact output variance of it and of Euler-Maruyama in the
linear-Gaussian case.  It is test infrastructure, like ``tests/dpm_oracle.py``, whose grid and (c0, c1) rule it uses
unchanged.

The reference has no such sampler, so this module is pinned by closed forms (``tests/test_cpu_dpm_sde.py``): with
Gaussian data and the exact eps, or with eps == 0, every sampler here is a linear recurrence driven by Gaussian noise,
so the variance of its output can be propagated exactly in fp64 and compared with Var(E[x0 | x_{t_end}]).
"""
from __future__ import annotations

import math
from typing import Optional

import numpy as np
import torch

from dpm_oracle import dpm_schedule
from toycrystals_oracle import SampleTrace, Schedule, StateDict, eps_cfg, time_grid


def dpm_sde_schedule(n_steps: int, t_end: float, sched: Schedule):
    """Time grid and per-step coefficients of ``sample_dpmpp_2m_sde``: the grid and (c0, c1) of ``dpm_schedule``, and
    per step, in double from the fp32 grid times, with h = lambda(t_{i+1}) - lambda(t_i):
        a = sigma(t_{i+1})/sigma(t_i) * exp(-h),  m = alpha(t_{i+1}) * (-expm1(-2h)),  g = sigma(t_{i+1}) * sqrt(-expm1(-2h)).
    Returns (ts: n_steps+1 floats, rows: n_steps tuples (a, m, c0, c1, g)), all Python floats (double)."""
    ts, ode_rows = dpm_schedule(n_steps, t_end, sched)
    bmin, d = float(sched.beta_min), float(sched.beta_max) - float(sched.beta_min)

    def alpha(t):
        return math.exp(-0.5 * (bmin * t + 0.5 * d * (t * t)))

    def sigma(t):
        a = alpha(t)
        return math.sqrt(max(1.0 - a * a, 1e-8))

    def lam(t):
        return math.log(alpha(t)) - math.log(sigma(t))

    rows = []
    for i, (_, _, c0, c1) in enumerate(ode_rows):
        t0, t1 = ts[i], ts[i + 1]
        h = lam(t1) - lam(t0)
        e2 = -math.expm1(-2.0 * h)
        rows.append((sigma(t1) / sigma(t0) * math.exp(-h), alpha(t1) * e2, c0, c1, sigma(t1) * math.sqrt(e2)))
    return ts, rows


@torch.no_grad()
def sample_dpmpp_2m_sde(sd: Optional[StateDict], cfg: Optional[dict], sched: Schedule, y_cat, y_cont,
                        x_init: torch.Tensor, noise: torch.Tensor, n_steps: int, guidance: float, t_end: float,
                        eps_fn=None, keep_trace: bool = True) -> SampleTrace:
    """SDE-DPM-Solver++(2M) (Lu et al. 2022, "DPM-Solver++", the SDE variant of Algorithm 2, eta = 1) on the reverse
    VP-SDE, then the same final projection as ``sample``: n_steps + 1 network evaluations.  ``noise`` [n_steps, B, 1, 64,
    64] is z of every step.  ``eps_fn(x, t)``, if given, replaces the network (``sd``, ``cfg``, ``y_cat``, ``y_cont`` and
    ``guidance`` are then unused).  Every step, in the dtype of ``x_init`` (the coefficients of ``dpm_sde_schedule`` are
    rounded to it once):
        x0 = (x - sigma_i eps) / alpha_i;  D = x0 (first-order rows) or c0 x0 + c1 x0_prev;  x <- a x + m D + g z."""
    if not (0.0 < float(t_end) < 1.0):
        raise ValueError(f"t_end must be in (0,1), got {t_end}")
    x = x_init.clone()
    B = x.shape[0]
    ts_list, rows = dpm_sde_schedule(n_steps, float(t_end), sched)
    if n_steps == 0:
        ts_list = [1.0]
    ts = torch.tensor(ts_list, dtype=torch.float64).to(device=x.device, dtype=x.dtype)
    coef = torch.tensor(rows, dtype=torch.float64).reshape(-1, 5).to(device=x.device, dtype=x.dtype)
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
        a, m, c0, c1, g = coef[i]
        D = x0 if float(c1) == 0.0 else c0 * x0 + c1 * x0_prev
        x = a * x + m * D + g * noise[i].to(x.dtype)
        x0_prev = x0

    t_fin = ts[-1].expand(B)
    a = sched.alpha(t_fin).view(B, 1, 1, 1)
    s = sched.sigma(t_fin).view(B, 1, 1, 1)
    x0_hat = (x - s * evaluate(x, t_fin)) / torch.clamp(a, min=1e-6)
    tr.x0_hat = x0_hat
    tr.image = ((x0_hat + 1.0) * 0.5).clamp(0.0, 1.0)
    return tr


def gaussian_output_variance(sampler: str, steps: int, s: Optional[float], var_init: float, t_end: float = 0.005,
                             sched: Schedule = Schedule(0.1, 30.0), first_order: bool = False):
    """Exact fp64 variance of the pre-clamp x0_hat of ``sampler`` ("dpm++2m-sde" or "sde", Euler-Maruyama on the
    quadratic grid of ``toycrystals_oracle.time_grid``) for zero-mean per-pixel data, from x_T ~ N(0, var_init).

    With data N(0, s^2) and the exact eps, or with eps == 0 (``s=None``), the data prediction is linear in x: x0 = k_i x
    with k_i = alpha_i s^2 / (alpha_i^2 s^2 + sigma_i^2), or k_i = 1/alpha_i.  Each step is then linear in the state
    (x, x0_prev) plus independent Gaussian noise, so its 2x2 covariance P propagates exactly: P <- M P M^T + diag(g^2, 0),
    M = [[a + m c0 k_i, m c1], [k_i, 0]].  ``first_order`` forces c1 = 0 (c0 = 1) on every row.  Returns
    (Var(x0_hat), t_end as the grid stores it); the true value for Gaussian data is ``true_posterior_mean_variance``."""
    bmin, d = float(sched.beta_min), float(sched.beta_max) - float(sched.beta_min)

    def alpha(t):
        return math.exp(-0.5 * (bmin * t + 0.5 * d * (t * t)))

    def sigma(t):
        a = alpha(t)
        return math.sqrt(max(1.0 - a * a, 1e-8))

    def k(t):
        return 1.0 / alpha(t) if s is None else alpha(t) * s * s / (alpha(t) ** 2 * s * s + sigma(t) ** 2)

    if sampler == "dpm++2m-sde":
        ts, rows = dpm_sde_schedule(steps, t_end, sched)
        P = np.array([[float(var_init), 0.0], [0.0, 0.0]])
        for i, (a, m, c0, c1, g) in enumerate(rows):
            if first_order:
                c0, c1 = 1.0, 0.0
            ki = k(ts[i])
            M = np.array([[a + m * c0 * ki, m * c1], [ki, 0.0]])
            P = M @ P @ M.T + np.diag([g * g, 0.0])
        v = P[0, 0]
    elif sampler == "sde":
        # x <- x + (-0.5 b x - b score) dt + sqrt(b) sqrt(|dt|) z, score = -eps/sigma = -(1 - alpha k) x / sigma^2
        ts = [float(t) for t in time_grid(steps, t_end).double()]
        v = float(var_init)
        for i in range(steps):
            t, dt = ts[i], ts[i + 1] - ts[i]
            b = bmin + t * d
            c = 1.0 + dt * (-0.5 * b + b * (1.0 - alpha(t) * k(t)) / sigma(t) ** 2)
            v = c * c * v + b * abs(dt)
    else:
        raise ValueError(f"unknown sampler {sampler!r}")
    return k(ts[-1]) ** 2 * v, ts[-1]


def true_posterior_mean_variance(s: float, t: float, sched: Schedule = Schedule(0.1, 30.0)) -> float:
    """Var(E[x0 | x_t]) for data N(0, s^2): alpha^2 s^4 / (alpha^2 s^2 + sigma^2)."""
    a = float(sched.alpha(torch.tensor(t, dtype=torch.float64)))
    g = float(sched.sigma(torch.tensor(t, dtype=torch.float64)))
    return a * a * s ** 4 / (a * a * s * s + g * g)


def true_marginal_variance(s: float, t: float, sched: Schedule = Schedule(0.1, 30.0)) -> float:
    """Var(x_t) for data N(0, s^2): alpha^2 s^2 + sigma^2."""
    a = float(sched.alpha(torch.tensor(t, dtype=torch.float64)))
    g = float(sched.sigma(torch.tensor(t, dtype=torch.float64)))
    return a * a * s * s + g * g
