"""CPU tests of the SDE-DPM-Solver++(2M) sampler: the library's host-side schedule against the oracle's, the exact
output variance on Gaussian data against Euler-Maruyama (second-order convergence), the oracle's Monte-Carlo output
against that variance, and the C ABI / shim / CLI surface.  The reference has no such sampler, so these closed-form
cases are what pins the oracle."""
import ctypes as C
import importlib.util
import math
import os

import numpy as np
import pytest
import torch

import dpm_oracle
import dpm_sde_oracle as dso
import toycrystals_oracle as orc
from toycrystals_b200 import _cabi
from toycrystals_b200.models import sde_score_model as shim

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SCHED = orc.Schedule(0.1, 30.0)
T_END, S = 0.005, 0.5   # per-pixel data N(0, S^2)


def _ulps(a, b):
    a, b = np.asarray(a, dtype=np.float32), np.asarray(b, dtype=np.float32)
    return int(np.abs(a.view(np.int32).astype(np.int64) - b.view(np.int32).astype(np.int64)).max())


@pytest.mark.parametrize("steps", [1, 2, 14, 15, 20, 80, 300])
def test_host_schedule_matches_the_oracle_to_0_ulp(steps):
    L = _cabi.lib()
    ts = (C.c_float * (steps + 1))()
    coef = (C.c_float * (5 * steps))()
    assert L.tcs_dpm_sde_schedule_host(steps, T_END, 0.1, 30.0, ts, coef) == 0
    o_ts, o_rows = dso.dpm_sde_schedule(steps, T_END, SCHED)
    got_ts = np.frombuffer(ts, dtype=np.float32)
    got_k = np.frombuffer(coef, dtype=np.float32).reshape(steps, 5)
    assert _ulps(got_ts, np.array(o_ts)) == 0
    assert _ulps(got_k, np.array(o_rows)) == 0
    # the same grid and (c0, c1) as the ODE form
    ode_ts, ode_rows = dpm_oracle.dpm_schedule(steps, T_END, SCHED)
    assert o_ts == ode_ts and [r[2:4] for r in o_rows] == [r[2:4] for r in ode_rows]
    assert np.all(got_k[:, 4] > 0)


def test_host_schedule_rejects_bad_arguments():
    L = _cabi.lib()
    ts, coef = (C.c_float * 4)(), (C.c_float * 15)()
    assert L.tcs_dpm_sde_schedule_host(0, 0.005, 0.1, 30.0, ts, coef) == _cabi.ERR_BAD_ARGUMENT
    assert L.tcs_dpm_sde_schedule_host(3, 1.0, 0.1, 30.0, ts, coef) == _cabi.ERR_BAD_ARGUMENT
    assert L.tcs_dpm_sde_schedule_host(3, 0.005, 0.1, 30.0, None, coef) == _cabi.ERR_BAD_ARGUMENT
    assert L.tcs_dpm_sde_schedule_host(3, 0.005, 0.1, 30.0, ts, None) == _cabi.ERR_BAD_ARGUMENT
    assert L.tcs_dpm_sde_schedule_host(3, 0.005, 0.0, 30.0, ts, coef) == _cabi.ERR_BAD_ARGUMENT
    assert L.tcs_dpm_sde_schedule_host(3, 0.005, 0.5, 0.1, ts, coef) == _cabi.ERR_BAD_ARGUMENT
    assert "tcs_dpm_sde_schedule_host" in _cabi.last_error()


def _rel_err(sampler, steps, **kw):
    var_t = dso.true_marginal_variance(S, 1.0)   # x_T from the true marginal at t = 1
    v, t_end = dso.gaussian_output_variance(sampler, steps, S, var_t, T_END, SCHED, **kw)
    return v / dso.true_posterior_mean_variance(S, t_end) - 1.0


# relative error of Var(x0_hat) against Var(E[x0 | x_{t_end}]), s = 0.5, beta 0.1..30, t_end 0.005
TABLE = [("sde", 100, {}, 2.38e-2), ("sde", 300, {}, 7.83e-3), ("sde", 1000, {}, 2.34e-3),
         ("dpm++2m-sde", 20, {}, 6.41e-2), ("dpm++2m-sde", 40, {}, 2.31e-2), ("dpm++2m-sde", 80, {}, 6.09e-3),
         ("dpm++2m-sde", 160, {}, 1.54e-3), ("dpm++2m-sde", 320, {}, 3.86e-4),
         ("dpm++2m-sde", 80, {"first_order": True}, -1.26e-1)]


@pytest.mark.parametrize("sampler,steps,kw,want", TABLE)
def test_gaussian_output_variance_reproduces_the_closed_form_table(sampler, steps, kw, want):
    err = _rel_err(sampler, steps, **kw)
    assert abs(err / want - 1.0) < 0.01, (sampler, steps, kw, err, want)


def test_second_order_and_fewer_evaluations_than_euler_maruyama():
    e = {n: _rel_err("dpm++2m-sde", n) for n in (80, 160, 320)}
    order = (math.log2(e[80] / e[160]), math.log2(e[160] / e[320]))
    assert min(order) >= 1.9, (order, e)
    assert abs(e[80]) < abs(_rel_err("sde", 300)), e


def test_monte_carlo_output_matches_the_exact_variance():
    """The fp64 oracle on N(0, S^2) data with the exact eps, 256 x 4096 = 1.05e6 independent pixels, 20 steps: the
    sample variance of x0_hat (mean known to be 0) is within 5 standard errors of the propagated variance; at 20 steps
    that variance is 6.4 % above the truth, so this also tells the recurrence from the posterior it approximates."""
    n, steps = 256, 20
    var_t = dso.true_marginal_variance(S, 1.0)
    g = torch.Generator().manual_seed(5)
    x_T = torch.randn((n, 1, 64, 64), generator=g, dtype=torch.float64) * math.sqrt(var_t)
    noise = torch.randn((steps, n, 1, 64, 64), generator=g, dtype=torch.float64)

    def eps(x, t):
        a, s = SCHED.alpha(t).view(-1, 1, 1, 1), SCHED.sigma(t).view(-1, 1, 1, 1)
        return s * x / (a * a * S * S + s * s)

    tr = dso.sample_dpmpp_2m_sde(None, None, SCHED, None, None, x_T, noise, steps, 0.0, T_END, eps_fn=eps,
                                 keep_trace=False)
    want, _ = dso.gaussian_output_variance("dpm++2m-sde", steps, S, var_t, T_END, SCHED)
    npix = tr.x0_hat.numel()
    got = float((tr.x0_hat ** 2).mean())
    se = want * math.sqrt(2.0 / npix)
    print(f"MC Var(x0_hat) {got:.6e}, exact {want:.6e}, {(got - want) / se:+.2f} standard errors")
    assert abs(got - want) < 5 * se, (got, want, se)
    assert abs(float(tr.x0_hat.mean())) < 5 * math.sqrt(want / npix)
    assert abs(want / dso.true_posterior_mean_variance(S, float(tr.ts[-1])) - 1.0) > 20 * se / want


def test_nfe_shim_errors_and_cli_parser():
    L = _cabi.lib()
    assert _cabi.SAMPLER_DPMPP_2M_SDE == 3
    for s in (1, 14, 20, 80, 300):
        assert L.tcs_nfe(_cabi.SAMPLER_DPMPP_2M_SDE, s) == s + 1
    assert shim._SAMPLERS["dpm++2m-sde"] is shim.sample_dpmpp_2m_sde
    m = shim.CondUNetTiny(**orc.DEFAULT_CFG)
    for bad in ("heun", "dpm++", "dpmpp_2m", "DPM++2M"):
        with pytest.raises(ValueError, match="Unknown sampler"):
            shim.save_sde_samples(m, shim.VPSDE(), "/tmp/x.png", torch.device("cpu"), sampler=bad)
    # the name is accepted; the run then stops at the device check (there is no CPU path)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        shim.save_sde_samples(m, shim.VPSDE(), "/tmp/x.png", torch.device("cpu"), sampler="dpm++2m-sde")
    spec = importlib.util.spec_from_file_location(
        "tcs_cli", os.path.join(ROOT, "vae-diffusion-toy-crystals_b200", "scripts", "sample_sde_score_model.py"))
    cli = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(cli)
    with pytest.raises(RuntimeError, match="no CPU path"):
        cli.main(["--out-dir", "unused", "--device", "cpu", "--sampler", "dpm++2m-sde", "--steps", "80"])
    with pytest.raises(SystemExit):
        cli.main(["--out-dir", "unused", "--device", "cpu", "--sampler", "dpm++2m_sde"])
