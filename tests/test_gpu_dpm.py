"""GPU tests of the DPM-Solver++(2M) sampler (tcs_sample with TCS_SAMPLER_DPMPP_2M, shim.sample_dpmpp_2m): the update
kernel bit for bit against the PyTorch fp32 expression, the whole production-size job with eps == 0 against the exact
answer, the free-running sampler against the CPU oracle, and graph replay / seeding / sharding / CLI."""
import ctypes as C
import importlib.util
import math
import os

import pytest
import torch

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TOL_EPS = {"fp32": 1e-4, "bf16": 2e-2}
# free-running pre-clamp x0_hat rel-L2 against the fp32 CPU oracle (n = 4, CFG 1.5, 20 steps): fp32 modes at the
# project's free-running tolerance; bf16 at about 2x the value measured on a B200 (1.6e-3, DESIGN.md §4.2)
TOL_X0 = {("fp32", "simt"): 1e-3, ("fp32", "tcgen05"): 1e-3, ("bf16", "tcgen05"): 3.5e-3}


def _pu():
    import parity_utils as pu
    return pu


# ---- the update kernel ---------------------------------------------------------------------------------------------
def _dpm_update(h, x, x0_prev, eps, alpha, sigma, row):
    from toycrystals_b200 import _cabi
    a, m, c0, c1 = (float(v) for v in row)
    _cabi.check(_cabi.lib().tcs_dpm_update(h, x.data_ptr(), x0_prev.data_ptr(), eps.data_ptr(), x.shape[0],
                                           float(alpha), float(sigma), a, m, c0, c1, None))
    torch.cuda.synchronize()


def test_dpm_update_is_bit_exact_vs_torch_expression():
    """x0 = (x - sigma*eps)/alpha; D = c0*x0 + c1*x0_prev; x = a*x + m*D in torch fp32 (CPU, true division), on a
    first-order row at t = 1 (alpha = 5.4e-4), second-order rows mid-grid and at the end, |x| ~ 30."""
    pu = _pu()
    import dpm_oracle
    import toycrystals_oracle as orc
    from toycrystals_b200.models.sde_score_model import VPSDE
    m = pu.model("fp32", "simt")
    h = m.engine_handle(VPSDE(0.1, 30.0))
    sde = VPSDE(0.1, 30.0)
    ts, rows = dpm_oracle.dpm_schedule(20, 0.005, orc.Schedule(0.1, 30.0))
    g = torch.Generator().manual_seed(8)
    n = 5
    for i in (0, 1, 9, 18, 19):
        t = torch.tensor(ts[i], dtype=torch.float32)
        alpha, sigma = sde.alpha(t), sde.sigma(t)
        a, mm, c0, c1 = (torch.tensor(v, dtype=torch.float64).float() for v in rows[i])
        x = torch.randn((n, 1, 64, 64), generator=g) * 30
        eps = torch.randn((n, 1, 64, 64), generator=g)
        x0p = torch.randn((n, 1, 64, 64), generator=g) * 30 / alpha
        x0_want = (x - sigma * eps) / alpha
        d_want = c0 * x0_want + c1 * x0p
        x_want = a * x + mm * d_want
        xs, ps = x.cuda(), x0p.cuda()
        _dpm_update(h, xs, ps, eps.cuda(), alpha, sigma, (a, mm, c0, c1))
        assert torch.equal(xs.cpu(), x_want), (i, float((xs.cpu() - x_want).abs().max()))
        assert torch.equal(ps.cpu(), x0_want), i
    # first-order row: x0_prev is not read (NaN in, finite out)
    t = torch.tensor(ts[0], dtype=torch.float32)
    alpha, sigma = sde.alpha(t), sde.sigma(t)
    a, mm = (torch.tensor(v, dtype=torch.float64).float() for v in rows[0][:2])
    x, eps = torch.randn((n, 1, 64, 64), generator=g) * 30, torch.randn((n, 1, 64, 64), generator=g)
    x0_want = (x - sigma * eps) / alpha
    xs, ps = x.cuda(), torch.full_like(x, float("nan")).cuda()
    _dpm_update(h, xs, ps, eps.cuda(), alpha, sigma, (a, mm, 1.0, 0.0))
    assert torch.equal(xs.cpu(), a * x + mm * x0_want)
    assert torch.equal(ps.cpu(), x0_want)


# ---- production size, eps == 0 ---------------------------------------------------------------------------------------
def _zero_out_model(precision):
    """Model whose `out` conv is zero: eps == 0 (the whole network still runs, its output is multiplied by zero)."""
    pu = _pu()
    import toycrystals_oracle as orc
    from toycrystals_b200.models.sde_score_model import CondUNetTiny
    sd = orc.default_init_state_dict(1)
    sd["out.weight"].zero_(); sd["out.bias"].zero_()
    m = CondUNetTiny(**pu.CFG, precision=precision, chunk=2048)
    m.load_state_dict(sd)
    return m.cuda().eval()


def test_full_size_zero_eps_is_exact():
    """n = 1024 with CFG 1.5 (one 2048-image pass per evaluation), 20 steps: with eps == 0 the solver is exact, so the
    pre-clamp projection equals x_T / alpha(1) up to the fp32 rounding of the coefficients and of each update."""
    pu = _pu()
    from toycrystals_b200.models import sde_score_model as shim
    n, steps = 1024, 20
    m = _zero_out_model("bf16")
    sde = shim.VPSDE(0.1, 30.0)
    yc, yk = shim.condition_grid(m, n, math.pi / 3, "cuda")
    x_T = torch.randn((n, 1, 64, 64), generator=torch.Generator().manual_seed(12)).cuda()
    img, tr = shim.sample_dpmpp_2m(m, sde, yc, yk, (n, 1, 64, 64), n_steps=steps, guidance_scale=1.5, t_end=0.005,
                                   x_init=x_T, return_trace=True)
    assert tr.eps.shape[0] == steps + 1 and float(tr.eps.abs().max()) == 0.0
    want = x_T / sde.alpha(torch.tensor(1.0)).cuda()
    err = pu.rel_l2(tr.x0_hat, want)
    print(f"dpm++2m n={n} steps={steps} eps==0: x0_hat rel-L2 vs x_T/alpha(1) = {err:.3e}")
    assert err <= 1e-5, err
    assert torch.equal(img, ((tr.x0_hat + 1.0) * 0.5).clamp(0.0, 1.0))
    m._release()
    del m
    torch.cuda.empty_cache()


# ---- free-running against the oracle ---------------------------------------------------------------------------------
N, STEPS, CFG_SCALE, T_END = 4, 20, 1.5, 0.005


@pytest.fixture(scope="module")
def oracle_run():
    """The fp32 CPU oracle's DPM-Solver++(2M) run on the golden weights (seed 1) from an injected x_T."""
    import dpm_oracle
    import toycrystals_oracle as orc
    sd = orc.default_init_state_dict(1)
    y_cat, y_cont = orc.condition_grid(N, 4, 4)
    x_T = torch.randn((N, 1, 64, 64), generator=torch.Generator().manual_seed(31))
    tr = dpm_oracle.sample_dpmpp_2m(sd, orc.DEFAULT_CFG, orc.Schedule(0.1, 30.0), y_cat, y_cont, x_T, STEPS, CFG_SCALE,
                                    T_END)
    return sd, y_cat, y_cont, x_T, tr


@pytest.mark.parametrize("precision,engine", list(TOL_X0))
def test_free_running_and_teacher_forced_against_the_oracle(oracle_run, precision, engine):
    pu = _pu()
    import toycrystals_oracle as orc
    from toycrystals_b200.models import sde_score_model as shim
    sd, y_cat, y_cont, x_T, ref = oracle_run
    m = pu.model(precision, engine, seed=1)
    sde = shim.VPSDE(0.1, 30.0)
    img, tr = shim.sample_dpmpp_2m(m, sde, y_cat.cuda(), y_cont.cuda(), (N, 1, 64, 64), n_steps=STEPS,
                                   guidance_scale=CFG_SCALE, t_end=T_END, x_init=x_T.cuda(), return_trace=True)
    assert tr.eps.shape == (STEPS + 1, N, 1, 64, 64) and tr.x_in.shape == tr.eps.shape
    assert torch.equal(tr.x_in[0].cpu(), x_T)
    worst = 0.0
    for k in range(STEPS + 1):   # teacher forced: the oracle evaluates the x_t this run saw, at the grid's time
        want = orc.eps_cfg(sd, orc.DEFAULT_CFG, tr.x_in[k].cpu(), ref.ts[k].expand(N), y_cat, y_cont, CFG_SCALE)
        worst = max(worst, pu.rel_l2(tr.eps[k], want))
    x0_err = pu.rel_l2(tr.x0_hat, ref.x0_hat)
    print(f"dpm++2m {precision}/{engine}: x0_hat rel-L2 vs oracle {x0_err:.3e}, worst teacher-forced eps {worst:.3e}")
    assert worst < TOL_EPS[precision], worst
    assert x0_err <= TOL_X0[(precision, engine)], x0_err
    assert torch.equal(img, ((tr.x0_hat + 1.0) * 0.5).clamp(0.0, 1.0))


# ---- graph replay, seeding, sharding, errors, CLI --------------------------------------------------------------------
def test_graph_replay_equals_plain_launches_and_ragged_chunks():
    pu = _pu()
    import toycrystals_oracle as orc
    from toycrystals_b200.models import sde_score_model as shim
    sde = shim.VPSDE(0.1, 30.0)
    y_cat, y_cont = orc.condition_grid(5, 4, 4)
    yc, yk = y_cat.cuda(), y_cont.cuda()
    x0 = torch.randn((5, 1, 64, 64), generator=torch.Generator().manual_seed(2)).cuda()
    outs = []
    for chunk, graph in ((0, True), (0, False), (4, True), (6, False)):  # 5 samples x2 -> ragged passes
        m = pu.model("bf16", "tcgen05", seed=1, chunk=chunk, use_graph=graph)
        for steps, cfg in ((3, 1.5), (16, 0.0)):   # 16 steps: second-order last row
            outs.append(shim.sample_dpmpp_2m(m, sde, yc, yk, (5, 1, 64, 64), n_steps=steps, guidance_scale=cfg,
                                             t_end=0.005, x_init=x0))
    for k in range(2, len(outs)):
        assert torch.equal(outs[k], outs[k % 2]), k
    assert not torch.equal(outs[0], outs[1])


def test_seed_alone_reproduces_and_shards():
    pu = _pu()
    from toycrystals_b200.models import sde_score_model as shim
    m = pu.model("bf16", "tcgen05", seed=1)
    sde = shim.VPSDE(0.1, 30.0)
    n = 6

    def run(lo, hi, torch_seed):
        torch.manual_seed(torch_seed)
        c, k = shim.condition_grid(m, hi - lo, math.pi / 3, "cuda", offset=lo, n_total=n)
        return shim.sample_dpmpp_2m(m, sde, c, k, (hi - lo, 1, 64, 64), n_steps=5, guidance_scale=1.5, t_end=0.005,
                                    seed=42, global_index_offset=lo)
    full = run(0, n, 1)
    assert torch.equal(full, run(0, n, 2)), "seed= alone must fix the run"
    assert torch.equal(torch.cat([run(0, 4, 3), run(4, 6, 4)]), full), "sharded run differs"


def test_noise_is_rejected_and_trace_layout():
    pu = _pu()
    import toycrystals_oracle as orc
    from toycrystals_b200 import _cabi
    from toycrystals_b200.models import sde_score_model as shim
    m = pu.model("bf16", "tcgen05", seed=1)
    h = m.engine_handle(shim.VPSDE(0.1, 30.0))
    y_cat, y_cont = orc.condition_grid(2, 4, 4)
    yc, yk = y_cat.cuda(), y_cont.cuda()
    out = torch.empty((2, 1, 64, 64), device="cuda")
    noise = torch.zeros((3, 2, 1, 64, 64), device="cuda")
    a = _cabi.TcsSampleArgs()
    a.sampler, a.n, a.steps, a.guidance, a.t_end = _cabi.SAMPLER_DPMPP_2M, 2, 3, 1.5, 0.005
    a.y_cat, a.y_cont, a.x_init, a.noise = yc.data_ptr(), yk.data_ptr(), None, noise.data_ptr()
    a.seed, a.global_index_offset = 1, 0
    a.x_out, a.trace_eps, a.trace_x, a.x0_hat = out.data_ptr(), None, None, None
    assert _cabi.lib().tcs_sample(h, C.byref(a), None) == _cabi.ERR_BAD_ARGUMENT
    assert "noise must be NULL" in _cabi.last_error()
    with pytest.raises(ValueError, match=r"t_end must be in \(0,1\)"):
        shim.sample_dpmpp_2m(m, shim.VPSDE(0.1, 30.0), yc, yk, (2, 1, 64, 64), t_end=0.0)
    # the trace has the SDE sampler's layout: evaluation k saw x at grid time k; the last one is x(t_end)
    _, tr = shim.sample_dpmpp_2m(m, shim.VPSDE(0.1, 30.0), yc, yk, (2, 1, 64, 64), n_steps=4, guidance_scale=1.5,
                                 t_end=0.005, seed=3, return_trace=True)
    assert tr.eps.shape[0] == tr.x_in.shape[0] == 5 == _cabi.lib().tcs_nfe(_cabi.SAMPLER_DPMPP_2M, 4)


@pytest.mark.parametrize("out_tensor", [False, True])
def test_cli_end_to_end(tmp_path, out_tensor):
    import toycrystals_oracle as orc
    os.makedirs(tmp_path / "checkpoints")
    torch.save(orc.make_checkpoint(), tmp_path / "checkpoints" / "sde_score_model_last.pt")
    spec = importlib.util.spec_from_file_location(
        "tcs_cli", os.path.join(ROOT, "vae-diffusion-toy-crystals_b200", "scripts", "sample_sde_score_model.py"))
    cli = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(cli)
    argv = ["--out-dir", str(tmp_path), "--steps", "20", "--cfg", "1.5", "--t-end", "0.005", "--sampler", "dpm++2m",
            "--use-ema", "1", "--n", "36"]
    if out_tensor:
        argv += ["--out-tensor", str(tmp_path / "x.pt")]
    assert cli.main(argv) == 0
    png = tmp_path / "results" / "samples_ckpt-sde_score_model_last_steps20_cfg1.50_tend0.005_samplerdpm++2m_ema1.png"
    assert png.exists()
    if out_tensor:
        x = torch.load(tmp_path / "x.pt")
        assert x.shape == (36, 1, 64, 64) and float(x.min()) >= 0 and float(x.max()) <= 1
