"""CPU tests of the DPM-Solver++(2M) sampler: the solver of tests/dpm_oracle.py against the exact probability-flow ODE
solution of Gaussian data (second-order convergence), its exactness when eps == 0, and the library's host-side schedule
against the oracle's.  The reference has no such sampler, so these closed-form cases are what pins the oracle."""
import ctypes as C
import importlib.util
import math
import os

import numpy as np
import pytest
import torch

import dpm_oracle
import toycrystals_oracle as orc
from toycrystals_b200 import _cabi
from toycrystals_b200.models import sde_score_model as shim

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SCHED = orc.Schedule(0.1, 30.0)
T_END = 0.005
MU, S = 0.3, 0.2   # per-pixel data distribution N(MU, S^2)


def _gaussian_eps(x, t):
    """Exact eps of N(MU, S^2) data under the VP-SDE: sigma (x - alpha MU) / (alpha^2 S^2 + sigma^2)."""
    a = SCHED.alpha(t).view(-1, 1, 1, 1)
    g = SCHED.sigma(t).view(-1, 1, 1, 1)
    return g * (x - a * MU) / (a * a * S * S + g * g)


def _exact_pf_ode(x1, t):
    """x(t) = alpha MU + sqrt(v(t)/v(1)) (x_1 - alpha(1) MU), v = alpha^2 S^2 + sigma^2."""
    t, one = torch.tensor(t, dtype=torch.float64), torch.tensor(1.0, dtype=torch.float64)
    v = lambda u: SCHED.alpha(u) ** 2 * S * S + SCHED.sigma(u) ** 2
    return SCHED.alpha(t) * MU + torch.sqrt(v(t) / v(one)) * (x1 - SCHED.alpha(one) * MU)


def _x1():
    return torch.linspace(-3.0, 3.0, 2 * 4096, dtype=torch.float64).reshape(2, 1, 64, 64)


def _solve(steps, eps_fn, x1):
    tr = dpm_oracle.sample_dpmpp_2m(None, None, SCHED, None, None, x1, steps, 0.0, T_END, eps_fn=eps_fn)
    assert len(tr.x_in) == steps + 1 and tr.t_in[0] == 1.0
    return tr


def test_closed_form_gaussian_converges_at_second_order():
    x1 = _x1()
    errs = {}
    for steps in (20, 80, 160, 320):
        tr = _solve(steps, _gaussian_eps, x1)
        want = _exact_pf_ode(x1, float(tr.ts[-1]))   # the grid ends at fp32(t_end)
        errs[steps] = orc.rel_l2(tr.x_in[-1], want)   # x at t_end, the input of the final evaluation
    print({k: f"{v:.3e}" for k, v in errs.items()})
    assert errs[20] <= 1e-2, errs
    order = (math.log2(errs[80] / errs[160]), math.log2(errs[160] / errs[320]))
    assert min(order) >= 1.8, (order, errs)


@pytest.mark.parametrize("steps", [1, 2, 14, 15, 20])
def test_zero_eps_is_exact(steps):
    """eps == 0: x0 = x / alpha is constant along the solution, and the exponential integrator moves x exactly to
    x_T alpha(t_end) / alpha(1) (1, 2 and 14 steps take the lower-order final step, 15 and 20 do not)."""
    x1 = _x1() * 7.0 + 0.01
    tr = _solve(steps, lambda x, t: torch.zeros_like(x), x1)
    a_end, a_start = SCHED.alpha(tr.ts[-1]), SCHED.alpha(tr.ts[0])
    assert float(tr.ts[0]) == 1.0 and float(tr.ts[-1]) == float(np.float32(T_END))
    rel = lambda got, want: float(((got - want).abs() / want.abs()).max())
    assert rel(tr.x_in[-1], x1 * a_end / a_start) < 1e-13
    assert rel(tr.x0_hat, x1 / a_start) < 1e-13


def test_schedule_rows_follow_the_lower_order_final_rule():
    for steps in (1, 2, 14, 15, 20):
        ts, rows = dpm_oracle.dpm_schedule(steps, T_END, SCHED)
        first = [i for i, r in enumerate(rows) if r[3] == 0.0]
        want = [0] + ([steps - 1] if steps < 15 and steps > 1 else [])
        assert first == want, (steps, first)
        assert all(r[2] == 1.0 for r in rows if r[3] == 0.0)
        assert all(abs(r[2] + r[3] - 1.0) < 1e-15 for r in rows)
        lam = [math.log(float(SCHED.alpha(torch.tensor(t, dtype=torch.float64))))
               - math.log(float(SCHED.sigma(torch.tensor(t, dtype=torch.float64)))) for t in ts]
        h = np.diff(lam)
        assert np.all(h > 0) and np.allclose(h, h.mean(), rtol=1e-5), (steps, h)   # uniform in log-SNR


def _ulps(a, b):
    a, b = np.asarray(a, dtype=np.float32), np.asarray(b, dtype=np.float32)
    return int(np.abs(a.view(np.int32).astype(np.int64) - b.view(np.int32).astype(np.int64)).max())


@pytest.mark.parametrize("steps,t_end,beta_max", [(1, 0.005, 30.0), (2, 0.005, 30.0), (14, 0.005, 30.0),
                                                  (20, 0.005, 30.0), (50, 1e-3, 30.0), (300, 0.005, 30.0),
                                                  (20, 0.005, 20.0), (20, 0.005, 60.0)])
def test_host_schedule_matches_the_oracle(steps, t_end, beta_max):
    L = _cabi.lib()
    ts = (C.c_float * (steps + 1))()
    coef = (C.c_float * (4 * steps))()
    assert L.tcs_dpm_schedule_host(steps, t_end, 0.1, beta_max, ts, coef) == 0
    o_ts, o_rows = dpm_oracle.dpm_schedule(steps, t_end, orc.Schedule(0.1, beta_max))
    got_ts = np.frombuffer(ts, dtype=np.float32)
    got_k = np.frombuffer(coef, dtype=np.float32).reshape(steps, 4)
    assert _ulps(got_ts, np.array(o_ts)) <= 1
    assert _ulps(got_k, np.array(o_rows)) <= 1
    assert got_ts[0] == 1.0 and got_ts[-1] == np.float32(t_end)
    assert np.all(np.diff(got_ts) < 0)


def test_host_schedule_rejects_bad_arguments():
    L = _cabi.lib()
    ts, coef = (C.c_float * 4)(), (C.c_float * 12)()
    assert L.tcs_dpm_schedule_host(0, 0.005, 0.1, 30.0, ts, coef) == _cabi.ERR_BAD_ARGUMENT
    assert L.tcs_dpm_schedule_host(3, 1.0, 0.1, 30.0, ts, coef) == _cabi.ERR_BAD_ARGUMENT
    assert L.tcs_dpm_schedule_host(3, 0.005, 0.1, 30.0, None, coef) == _cabi.ERR_BAD_ARGUMENT


def test_nfe_shim_errors_and_cli_parser():
    L = _cabi.lib()
    for s in (1, 14, 20, 300):
        assert L.tcs_nfe(_cabi.SAMPLER_DPMPP_2M, s) == s + 1
    assert _cabi.SAMPLER_DPMPP_2M == 2
    m = shim.CondUNetTiny(**orc.DEFAULT_CFG)
    for bad in ("heun", "dpm++", "dpmpp_2m", "DPM++2M"):
        with pytest.raises(ValueError, match="Unknown sampler"):
            shim.save_sde_samples(m, shim.VPSDE(), "/tmp/x.png", torch.device("cpu"), sampler=bad)
    spec = importlib.util.spec_from_file_location(
        "tcs_cli", os.path.join(ROOT, "vae-diffusion-toy-crystals_b200", "scripts", "sample_sde_score_model.py"))
    cli = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(cli)
    # the parser accepts the sampler; the run then stops at the device check (there is no CPU path)
    with pytest.raises(RuntimeError, match="no CPU path"):
        cli.main(["--out-dir", "unused", "--device", "cpu", "--sampler", "dpm++2m", "--steps", "20"])
    with pytest.raises(SystemExit):
        cli.main(["--out-dir", "unused", "--device", "cpu", "--sampler", "dpm"])
