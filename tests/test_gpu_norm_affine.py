"""Every GroupNorm and LayerNorm of both networks with per-channel affines (tests/norm_affine.py) instead of PyTorch's
identity init, on every path that consumes or routes an affine.  A trained checkpoint never has weight = 1, bias = 0,
and under the identity a gamma read at the wrong channel, a swapped weight / bias or one layer's affine used for another
all give exactly the right answer.  tests/test_cpu_norm_affine.py shows that each such fault moves what is compared here
by >= 10x the gate.  Run with -s for the per-layer numbers.

Score network (the per-layer checker of test_gpu_layer_chain.py, fp64 references from the pass's own input taps):
  A. the production bf16 pass (n = 1024 with CFG) on the fused conv + GroupNorm + SiLU path, per element;
  B. the unfused GroupNorm path, and the fused layers as whole-image groups (TCS_MAX_CTAS = 18): bit-identical;
  C. fp32 on the CUDA cores and on the tensor pipe (bf16x3 split) against the fp64 oracle, layer by layer, and CFG eps;
  D. norm weights written in place through .data are re-uploaded: bit-identical to a model built from them.
Prior: eps in both precisions at a ragged batch with per-sample timesteps and at n = 4096, a teacher-forced DDIM trace
(out_norm in the tail kernel's DDIM mode), and the in-place update."""
import time

import pytest
import torch

import latent_prior_oracle as po
import norm_affine as na
import test_gpu_layer_chain as lc
import toycrystals_oracle as orc

pytestmark = pytest.mark.gpu
SEED = 7
PRIOR_TOL = {"fp32": 1e-4, "bf16": 2e-2}
ACT_NAMES = list(lc.LAYERS)   # every activation tap of the chain, and eps


def _score_sd(seed=1):
    return na.affine_state_dict(orc.default_init_state_dict(seed), SEED)


# ---- A: the production pass, fused path ---------------------------------------------------------------------------
def test_production_pass_with_norm_affines():
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    sd = _score_sd()
    m = lc._fresh_model(sd, 2048)
    x, t, yc, yk = lc._inputs(1024, 1.0, 1.0)
    t0 = time.time()
    res = lc.chain(m, sd, x, t, yc, yk, 1)
    print(f"affine chain: worst err/bound over all layers {max(r['worst'] for r in res.values()):.3f}; "
          f"wall time {time.time() - t0:.1f} s")


# ---- B: the unfused GroupNorm path, and whole-image groups on the fused path -----------------------------------------
def test_unfused_and_whole_image_group_paths_with_norm_affines(monkeypatch):
    from toycrystals_b200 import _cabi
    sd = _score_sd()
    x, t, yc, yk = lc._inputs(75, 37.0, 0.37, seed=5)
    monkeypatch.delenv("TCS_MAX_CTAS", raising=False)
    m = lc._fresh_model(sd, 256)
    m._fuse_gn = False   # conv -> raw fp32 -> gn_apply (the first conv stays fused)
    lc.chain(m, sd, x, t, yc, yk, 1, stash=None)
    del m
    m = lc._fresh_model(sd, 256)
    resident = int(_cabi.lib().tcs_launch_mode(m.engine_handle())) >> 8
    base = {}
    lc.chain(m, sd, x, t, yc, yk, 1, taps=base)
    del m
    assert 18 < resident, f"resident CTAs {resident}"
    monkeypatch.setenv("TCS_MAX_CTAS", "18")
    m = lc._fresh_model(sd, 256)
    for nm in ACT_NAMES:
        got = lc.tap(m, nm, x, t, yc, yk, 1)
        assert torch.equal(got, base[nm]), f"TCS_MAX_CTAS=18: {nm} differs from the default grid " \
            f"(max |diff| {float((got - base[nm]).abs().max()):.3g})"


# ---- C: fp32 on the CUDA cores and on the tensor pipe ------------------------------------------------------------
@pytest.mark.parametrize("engine", ["simt", "tcgen05"])
def test_fp32_layers_with_norm_affines(engine):
    """Every tap of parity_utils.LAYERS against orc.score_net in fp64, gates of test_layers_against_oracle.  The only
    coverage of attn.norm's fp32 kernel (gn_image16_kernel) and of the bf16x3 GroupNorm routing (gn_split / gn_f32)."""
    import parity_utils as pu
    from toycrystals_b200.models.sde_score_model import predict_eps_cfg
    sd = _score_sd(0)
    m = lc._fresh_model(sd, 128, precision="fp32", engine=engine)
    x, t, yc, yk = lc._inputs(3, 37.0, 0.37, seed=9)
    taps = {}
    with torch.no_grad():
        orc.score_net(sd, pu.CFG, x.double(), t.double(), yc, yk.double(), taps)
    gate = 2e-5 if engine == "simt" else 5e-5
    errs = {}
    for name, C, res in pu.LAYERS:
        got = pu.debug_layer(m, name, x, t, yc, yk, C, res)
        errs[name] = pu.rel_l2(got, taps[name].permute(0, 2, 3, 1))
    print(f"fp32/{engine} per-layer rel-L2: " + ", ".join(f"{k} {v:.2e}" for k, v in errs.items()))
    bad = {k: v for k, v in errs.items() if not v < gate}
    # errors compound through the oracle's own chain: the first layer over the gate is the one at fault
    assert not bad, f"fp32/{engine}: first layer over {gate:g}: {next(iter(bad))} ({next(iter(bad.values())):.3e}); " \
        f"all: {bad}"
    with torch.no_grad():
        want = orc.eps_cfg(sd, pu.CFG, x.double(), t.double(), yc, yk.double(), 1.5)
    err = pu.rel_l2(predict_eps_cfg(m, x, t, yc, yk, 1.5), want)
    print(f"fp32/{engine} CFG eps rel-L2 {err:.2e}")
    assert err < 1e-4, err


# ---- D: norm weights updated in place --------------------------------------------------------------------------
def test_in_place_norm_update_is_uploaded():
    """The reference's EMA idiom writes through .data, which autograd's version counter does not see; after refresh()
    (the samplers call it themselves) the pass must equal, bit for bit, one of a model built from the new weights."""
    sd0 = orc.default_init_state_dict(1)
    sd = na.affine_state_dict(sd0, SEED)
    x, t, yc, yk = lc._inputs(16, 1.0, 0.6, seed=3)
    m = lc._fresh_model(sd0, 64)
    before = lc.tap(m, "eps", x, t, yc, yk, 1)
    params = dict(m.named_parameters())
    for k in na.norm_keys(sd):
        params[k].data.copy_(sd[k])
    m.refresh()
    fresh = lc._fresh_model(sd, 64)
    for nm in ACT_NAMES:
        got, want = lc.tap(m, nm, x, t, yc, yk, 1), lc.tap(fresh, nm, x, t, yc, yk, 1)
        assert torch.equal(got, want), f"{nm}: the in-place update was not uploaded"
    assert not torch.equal(before, want)


# ---- the prior ---------------------------------------------------------------------------------------------------
def _prior(precision, sd):
    from toycrystals_b200.models import diffusion_prior as pshim
    m = pshim.DiffusionPriorFiLM(**po.PRIOR_CFG, precision=precision)
    m.load_state_dict(sd)
    return m.cuda().eval()


def _prior_sd():
    return na.affine_state_dict(po.prior_default_init(0), SEED)


def _eps_check(what, precision, got, want):
    err = orc.rel_l2(got, want)
    rows = float(((got.double() - want).norm(dim=1) / want.norm(dim=1)).max())
    print(f"prior {precision} {what}: eps rel-L2 {err:.3e}, worst row {rows:.3e}")
    assert err <= PRIOR_TOL[precision], (what, err)
    assert rows <= 3 * PRIOR_TOL[precision], (what, rows)


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_prior_eps_with_norm_affines(precision):
    sd = _prior_sd()
    sdc = {k: v.cuda() for k, v in sd.items()}
    m = _prior(precision, sd)
    cfg = po.PRIOR_CFG
    # ragged batch (not a multiple of the 128-row tile), per-sample timesteps
    n = 261
    g = torch.Generator().manual_seed(5)
    z = (torch.randn((n, 32), generator=g) * 3.0).cuda()
    t = torch.randint(0, 1000, (n,), generator=g).cuda()
    yc, yk = (v.cuda() for v in orc.condition_grid(n, 4, 4))
    with torch.no_grad():
        want = po.film_prior(sdc, cfg, z.double(), t, yc, yk.double())
    _eps_check(f"n={n} per-sample t", precision, m(z, t, yc, yk), want)
    # the full-size batch at three timesteps
    n = 4096
    z = (torch.randn((n, 32), generator=g) * 2.0).cuda()
    yc, yk = (v.cuda() for v in orc.condition_grid(n, 4, 4))
    for tv in (999, 500, 0):
        t = torch.full((n,), tv, dtype=torch.int64, device="cuda")
        with torch.no_grad():
            want = po.film_prior(sdc, cfg, z.double(), t, yc, yk.double())
        _eps_check(f"n={n} t={tv}", precision, m(z, t, yc, yk), want)


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_prior_ddim_trace_with_norm_affines(precision):
    """Every evaluation of a 12-step DDIM run, teacher-forced at the z_t the GPU saw: out_norm runs in the tail kernel's
    DDIM mode here (the forward above uses its eps-only mode).  With these random weights the latents grow towards 1e6,
    in_proj(z) then dominates the residual stream, and from about the fourth step on even bf16 eps agrees to ~2e-7: the
    early steps check the blocks, every step checks out_norm."""
    from toycrystals_b200.models import diffusion_prior as pshim
    sd = _prior_sd()
    sdc = {k: v.cuda() for k, v in sd.items()}
    m = _prior(precision, sd)
    s = pshim.DiffusionSchedule.linear(T=1000, beta_start=1e-4, beta_end=0.05, device=torch.device("cuda"))
    n = 300
    yc, yk = (v.cuda() for v in orc.condition_grid(n, 4, 4))
    _, tr = s.ddim_sample(m, yc, yk, n_steps=12, seed=77, return_trace=True)
    assert tr.eps.shape[0] == 12
    for k in range(tr.eps.shape[0]):
        t = tr.timesteps[k].repeat(n).cuda()
        with torch.no_grad():
            want = po.film_prior(sdc, po.PRIOR_CFG, tr.z_in[k].double(), t, yc, yk.double())
        _eps_check(f"DDIM step {k} (t={int(tr.timesteps[k])})", precision, tr.eps[k], want)


def test_prior_in_place_norm_update_is_uploaded():
    from toycrystals_b200.models import diffusion_prior as pshim
    sd0 = po.prior_default_init(0)
    sd = na.affine_state_dict(sd0, SEED)
    n = 261
    g = torch.Generator().manual_seed(6)
    z = torch.randn((n, 32), generator=g).cuda()
    t = torch.randint(0, 1000, (n,), generator=g).cuda()
    yc, yk = (v.cuda() for v in orc.condition_grid(n, 4, 4))
    s = pshim.DiffusionSchedule.linear(T=1000, beta_start=1e-4, beta_end=0.05, device=torch.device("cuda"))
    m = _prior("bf16", sd0)
    before = m(z, t, yc, yk)
    params = dict(m.named_parameters())
    for k in na.norm_keys(sd):
        params[k].data.copy_(sd[k])
    m.refresh()
    fresh = _prior("bf16", sd)
    want = fresh(z, t, yc, yk)
    assert torch.equal(m(z, t, yc, yk), want), "the in-place update was not uploaded"
    assert not torch.equal(before, want)
    assert torch.equal(s.ddim_sample(m, yc, yk, n_steps=12, seed=77), s.ddim_sample(fresh, yc, yk, n_steps=12, seed=77))
