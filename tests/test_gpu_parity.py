"""GPU suite (-m gpu): the CUDA path, called through the C ABI, against the oracle and the golden
vectors generated from the reference.  Tolerances are BASELINE.json's north_star:
per-evaluation eps rel-L2 <= 1e-4 in fp32 mode, <= 2e-2 in bf16 mode (teacher-forced)."""
import math

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

TOL_EPS = {"fp32": 1e-4, "bf16": 2e-2}
# fp32/tcgen05 = the fp32 mode on the tensor pipe: operands as bf16 (hi, lo) pairs, three MMAs per product (bf16x3)
MODES = [("fp32", "simt"), ("bf16", "simt"), ("bf16", "tcgen05"), ("fp32", "tcgen05")]


def _pu():
    import parity_utils as pu
    return pu


# ---- single conv layers, every shape the network uses ------------------------------------------------
CONV_CASES = [  # (cin0, cin1, cout, k, stride, res_out)
    (96, 0, 96, 3, 1, 64), (96, 0, 96, 4, 2, 32), (96, 0, 192, 3, 1, 32), (192, 0, 192, 3, 1, 32),
    (192, 0, 192, 4, 2, 16), (192, 0, 192, 3, 1, 16), (192, 0, 576, 1, 1, 16), (192, 0, 192, 1, 1, 16),
    (192, 192, 96, 3, 1, 32), (96, 96, 96, 3, 1, 64),
]


@pytest.mark.parametrize("precision,engine", MODES)
@pytest.mark.parametrize("case", CONV_CASES)
def test_conv_layer(case, precision, engine):
    pu = _pu()
    c0, c1, cout, k, s, res = case
    g = torch.Generator().manual_seed(hash(case) % 1000)
    B = 3
    in0 = torch.randn((B, res * s, res * s, c0), generator=g)
    in1 = torch.randn((B, res * s, res * s, c1), generator=g) if c1 else None
    w = torch.randn((cout, c0 + c1, k, k), generator=g) / math.sqrt((c0 + c1) * k * k)
    b = torch.randn((cout,), generator=g)
    ref = pu.conv_reference(in0, in1, w, b, k, s, round_bf16=(precision == "bf16"))
    for epi in (0, 1, 2):
        out, stats = pu.debug_conv(engine, precision, in0.cuda(), None if in1 is None else in1.cuda(), w.cuda(),
                                   b.cuda(), k, s, epi)
        tol = 2e-5 if (precision == "fp32" or epi == 0) else 6e-3  # epi 1/2 round the output to bf16
        err = pu.rel_l2(out, ref)
        assert err < tol, (case, precision, engine, epi, err)
        if epi == 0 and cout in (96, 192):  # GroupNorm only ever follows 96/192-channel convs
            cpg = cout // 8
            r = ref.reshape(B, -1, 8, cpg)
            want = torch.stack([r.sum(dim=(1, 3)), (r * r).sum(dim=(1, 3))], dim=-1)
            assert pu.rel_l2(stats, want) < 1e-4, (case, precision, engine, "stats")


# ---- us1_conv / us2_conv with the bilinear x2 upsample fused into the conv's operand path ----------------------------
@pytest.mark.parametrize("case", [(96, 96, 32), (192, 192, 16)])   # (cin, cout, low resolution): us1_conv, us2_conv
def test_conv_with_fused_upsample(case):
    """nn.Upsample(scale_factor=2, mode="bilinear") + 3x3 circular conv (sde_score_model.py:217-222): the upsample clamps
    at the image edge, the conv wraps around it; B = 5 images x every tile position covers all border cases."""
    pu = _pu()
    cin, cout, lo = case
    g = torch.Generator().manual_seed(cin + lo)
    B = 5
    x = torch.randn((B, lo, lo, cin), generator=g).bfloat16().float()
    w = (torch.randn((cout, cin, 3, 3), generator=g) / math.sqrt(cin * 9)).bfloat16().float()
    b = torch.randn((cout,), generator=g)
    up = torch.nn.functional.interpolate(x.permute(0, 3, 1, 2).double(), scale_factor=2, mode="bilinear", align_corners=False)
    up16 = up.float().bfloat16().double()      # the stand-alone kernel rounded the upsampled tensor to bf16; so does the fused path
    want = pu.conv_reference(up16.permute(0, 2, 3, 1).float(), None, w, b, 3, 1)
    got = pu.debug_conv_ups(x.cuda(), w.cuda(), b.cuda())
    err = pu.rel_l2(got.cpu(), want)
    # rows / columns next to the image edge separately: that is where clamp (upsample) and wrap (conv) meet
    ring = torch.ones(2 * lo, 2 * lo, dtype=torch.bool); ring[2:-2, 2:-2] = False
    err_ring = pu.rel_l2(got.cpu()[:, ring], want[:, ring])
    print(f"fused upsample {case}: rel-L2 {err:.2e}, border ring {err_ring:.2e}")
    assert err < 6e-3 and err_ring < 6e-3, (case, err, err_ring)


# ---- the fused attention block (attn_tc.cu) in isolation -------------------------------------------------------
@pytest.mark.parametrize("B", [1, 3, 150])
def test_fused_attention_block(B):
    """GroupNorm -> qkv -> softmax(q k^T) v -> proj -> + x in one tcgen05 kernel against an fp64 SelfAttention2d
    (sde_score_model.py:136-167).  Inputs and weights are bf16-representable so that the gate measures the kernel's own
    rounding (bf16 Xn / q / k / v / P / y operands, fp32 accumulation, bf16 output); B = 150 > 74 clusters exercises
    the persistent image loop (weight re-fetch, barrier phases) and the halo is verified inside the hook."""
    pu = _pu()
    g = torch.Generator().manual_seed(100 + B)
    bf = lambda t: t.bfloat16().float()
    x = bf(torch.randn((B, 16, 16, 192), generator=g) * 1.5 + 0.3)
    gn_w, gn_b = 1.0 + 0.2 * torch.randn(192, generator=g), 0.1 * torch.randn(192, generator=g)
    qkv_w, qkv_b = bf(torch.randn((576, 192), generator=g) * (2.0 / math.sqrt(192))), 0.1 * torch.randn(576, generator=g)
    proj_w, proj_b = bf(torch.randn((192, 192), generator=g) / math.sqrt(192)), 0.1 * torch.randn(192, generator=g)
    args = (x, gn_w, gn_b, qkv_w, qkv_b, proj_w, proj_b)
    want, wd = pu.attn_block_reference(*args)
    got, d = pu.debug_attn_block(*args, want_dbg=True)
    errs = {k: pu.rel_l2(d[k].cpu(), wd[k][0]) for k in ("xn", "qkv", "y")}
    err = pu.rel_l2(got.cpu(), want)
    branch = pu.rel_l2(got.cpu().double() - x.double(), want - x.double())   # the attention branch without the residual
    print(f"fused attention B={B}: out {err:.2e}, branch {branch:.2e}, stages {errs}")
    assert errs["xn"] < 4e-3 and errs["qkv"] < 6e-3 and errs["y"] < 1.5e-2, errs
    assert err < 1e-2 and branch < 2e-2, (err, branch)


# ---- per-layer activations against the oracle's taps ---------------------------------------------------
@pytest.mark.parametrize("precision,engine", MODES)
def test_layers_against_oracle(precision, engine):
    pu = _pu()
    import toycrystals_oracle as orc
    g = pu.golden("score_fwd.pt")
    m = pu.model(precision, engine)
    sd = orc.default_init_state_dict(0)
    x, t = g["x"] * 37.0, torch.full((3,), 0.37)
    taps = {}
    with torch.no_grad():
        orc.score_net(sd, pu.CFG, x.double(), t.double(), g["y_cat"], g["y_cont"].double(), taps)
    worst = 0.0
    for name, C, res in pu.LAYERS:
        try:
            got = pu.debug_layer(m, name, x.cuda(), t.cuda(), g["y_cat"].cuda(), g["y_cont"].cuda(), C, res)
        except NotImplementedError:
            # the tcgen05 engine fuses GroupNorm+SiLU into the conv: the raw conv output never exists
            assert engine == "tcgen05" and name.endswith(".raw") and name != "down1.net.0.raw", name
            continue
        want = taps[name].permute(0, 2, 3, 1)
        err = pu.rel_l2(got, want)
        worst = max(worst, err)
        assert err < ((2e-5 if engine == "simt" else 5e-5) if precision == "fp32" else 1.5e-2), (name, err)
    print(f"{precision}/{engine}: worst layer rel-L2 {worst:.3e}")


# ---- network evaluations against the reference golden vectors -------------------------------------------
@pytest.mark.parametrize("precision,engine", MODES)
def test_score_against_reference_golden(precision, engine):
    pu = _pu()
    from toycrystals_b200.models.sde_score_model import predict_eps_cfg
    g = pu.golden("score_fwd.pt")
    m = pu.model(precision, engine)
    yc, yk = g["y_cat"].cuda(), g["y_cont"].cuda()
    for case in g["cases"]:
        x = (g["x"] * case["scale"]).cuda()
        t = torch.full((3,), case["t"]).cuda()
        e_c = m(x, t, yc, yk)
        e_u = m(x, t, torch.full_like(yc, 4), torch.zeros_like(yk))
        e_g = predict_eps_cfg(m, x, t, yc, yk, 1.5)
        for got, key in ((e_c, "eps_c"), (e_u, "eps_u"), (e_g, "eps_cfg15")):
            err = pu.rel_l2(got, case[key])
            assert err < TOL_EPS[precision], (case["t"], key, err)
        if precision == "fp32":  # doubled batch == two separate passes, combined in the same order
            assert pu.rel_l2(e_g, e_u + 1.5 * (e_c - e_u)) < 1e-6


@pytest.mark.parametrize("precision,engine", MODES)
def test_sampler_teacher_forced_and_free_running(precision, engine):
    """Per-evaluation eps at the reference's own x_t (teacher forced), then the free-running sampler."""
    pu = _pu()
    from toycrystals_b200.models import sde_score_model as shim
    gs = pu.golden("samplers.pt")
    m = pu.model(precision, engine, seed=1)
    sde = shim.VPSDE(0.1, 30.0)
    for key, g in gs.items():
        yc, yk = g["y_cat"].cuda(), g["y_cont"].cuda()
        k = g["x_in"][0].shape[0]          # the stored traces hold the first k samples of the run
        for e_ref, x_in, t_in in zip(g["eps"], g["x_in"], g["t_in"]):
            got = shim.predict_eps_cfg(m, x_in.cuda(), torch.full((k,), t_in).cuda(), yc[:k], yk[:k], g["cfg"])
            err = pu.rel_l2(got, e_ref)
            assert err < TOL_EPS[precision], (key, t_in, err)
        fn = shim.sample_probability_flow_ode if g["sampler"] == "ode" else shim.sample_reverse_sde_euler_maruyama
        kw = dict(x_init=g["x_init"].cuda(), return_trace=True)
        if g["sampler"] == "sde":
            kw["noise"] = torch.stack(g["noise"]).cuda()
        img, tr = fn(m, sde, yc, yk, (2, 1, 64, 64), n_steps=g["steps"], guidance_scale=g["cfg"], t_end=g["t_end"], **kw)
        assert tr.eps.shape[0] == len(g["eps"])
        x0_err = pu.rel_l2(tr.x0_hat, g["x0_hat"])
        mism = float(((img.cpu() - pu.image_of(g["x0_hat"])).abs() > 1.0 / 255).float().mean())
        print(f"{precision}/{engine} {key}: x0_hat rel-L2 {x0_err:.3e}, mismatched pixels {mism:.4%}")
        if precision == "fp32":
            # stated per-pixel tolerance for final samples (SURVEY 8c): pre-clamp rel-L2 <= 1e-3 and
            # |delta| > 1/255 on <= 0.5% of the (nearly binary) clamped pixels
            assert x0_err < 1e-3 and mism < 5e-3, (key, x0_err, mism)
        else:   # measured on B200: 1e-3 .. 3e-3 (2-sample, few-step runs of an expanding random-weight trajectory)
            assert x0_err < 1e-2, (key, x0_err)


# ---- the fused update kernel and its RNG ---------------------------------------------------------------
def test_sde_update_is_bit_exact_vs_torch_expression():
    pu = _pu()
    import ctypes as C
    from toycrystals_b200 import _cabi
    from toycrystals_b200.models.sde_score_model import VPSDE
    m = pu.model("fp32", "simt")
    h = m.engine_handle(VPSDE(0.1, 30.0))
    g = torch.Generator().manual_seed(5)
    n = 5
    x = (torch.randn((n, 1, 64, 64), generator=g) * 30).cuda()
    eps, z = torch.randn((n, 1, 64, 64), generator=g).cuda(), torch.randn((n, 1, 64, 64), generator=g).cuda()
    sde = VPSDE(0.1, 30.0)
    t, t_next = torch.tensor(0.3712, device="cuda"), torch.tensor(0.3651, device="cuda")
    beta, sigma = sde.beta(t), sde.sigma(t)
    dt = t_next - t
    want = x + ((-0.5 * beta * x) - (beta * (-eps / sigma))) * dt + torch.sqrt(beta) * torch.sqrt(torch.abs(dt)) * z
    got = x.clone()
    _cabi.check(_cabi.lib().tcs_sde_update(h, got.data_ptr(), eps.data_ptr(), z.data_ptr(), n, float(t), float(t_next),
                                           0, 0, 0, None))
    torch.cuda.synchronize()
    assert pu.rel_l2(got, want) < 2e-7
    assert float((got - want).abs().max()) <= 4 * float(torch.finfo(torch.float32).eps) * float(want.abs().max())


def test_philox_stream_matches_numpy_reference_and_is_shard_invariant():
    pu = _pu()
    import philox_ref
    from toycrystals_b200.models import sde_score_model as shim
    m = pu.model("bf16", "tcgen05", seed=1)
    sde = shim.VPSDE(0.1, 30.0)
    import toycrystals_oracle as orc
    y_cat, y_cont = orc.condition_grid(6, 4, 4)
    yc, yk = y_cat.cuda(), y_cont.cuda()
    # steps=0: image = projection of the Philox initial state only -> check the stream via trace_x
    _, tr = shim.sample_reverse_sde_euler_maruyama(m, sde, yc, yk, (6, 1, 64, 64), n_steps=1, guidance_scale=1.5,
                                                   t_end=0.005, x_init=None, seed=1234, return_trace=True)
    full, trf = shim.sample_reverse_sde_euler_maruyama(m, sde, yc, yk, (6, 1, 64, 64), n_steps=2, guidance_scale=1.5,
                                                       t_end=0.005, seed=99, return_trace=True)
    a, _ = shim.sample_reverse_sde_euler_maruyama(m, sde, yc[:4], yk[:4], (4, 1, 64, 64), n_steps=2, guidance_scale=1.5,
                                                  t_end=0.005, x_init=trf.x_in[0][:4], seed=99, global_index_offset=0,
                                                  return_trace=True)
    b, _ = shim.sample_reverse_sde_euler_maruyama(m, sde, yc[4:], yk[4:], (2, 1, 64, 64), n_steps=2, guidance_scale=1.5,
                                                  t_end=0.005, x_init=trf.x_in[0][4:], seed=99, global_index_offset=4,
                                                  return_trace=True)
    assert torch.equal(torch.cat([a, b]), full), "sharded run differs from the unsharded one"


def test_philox_initial_state_matches_numpy():
    pu = _pu()
    import ctypes as C
    import philox_ref
    from toycrystals_b200 import _cabi
    from toycrystals_b200.models import sde_score_model as shim
    import toycrystals_oracle as orc
    m = pu.model("bf16", "tcgen05", seed=1)
    h = m.engine_handle(shim.VPSDE(0.1, 30.0))
    y_cat, y_cont = orc.condition_grid(3, 4, 4)
    out = torch.empty((3, 1, 64, 64), device="cuda")
    tx = torch.empty((1, 3, 1, 64, 64), device="cuda")
    a = _cabi.TcsSampleArgs()
    a.sampler, a.n, a.steps, a.guidance, a.t_end = _cabi.SAMPLER_SDE, 3, 0, 0.0, 0.005
    yc, yk = y_cat.cuda(), y_cont.cuda()
    a.y_cat, a.y_cont, a.x_init, a.noise = yc.data_ptr(), yk.data_ptr(), None, None
    a.seed, a.global_index_offset = 1234, 5
    a.x_out, a.trace_eps, a.trace_x, a.x0_hat = out.data_ptr(), None, tx.data_ptr(), None
    _cabi.check(_cabi.lib().tcs_sample(h, C.byref(a), None))
    torch.cuda.synchronize()
    for i in range(3):
        want = philox_ref.normal_image(1234, 5 + i, 0)
        got = tx[0, i].flatten().double().cpu().numpy()
        assert np.abs(got - want).max() < 2e-5, i
    z = tx.flatten().double()
    assert abs(float(z.mean())) < 0.03 and abs(float(z.std()) - 1) < 0.03


def test_graph_replay_equals_plain_launches_and_ragged_chunks():
    pu = _pu()
    from toycrystals_b200.models import sde_score_model as shim
    import toycrystals_oracle as orc
    sde = shim.VPSDE(0.1, 30.0)
    y_cat, y_cont = orc.condition_grid(5, 4, 4)
    yc, yk = y_cat.cuda(), y_cont.cuda()
    x0 = torch.randn((5, 1, 64, 64), generator=torch.Generator().manual_seed(2)).cuda()
    outs = []
    for chunk, graph in ((0, True), (0, False), (4, True), (6, False)):  # 5 samples x2 -> ragged passes
        m = pu.model("bf16", "tcgen05", seed=1, chunk=chunk, use_graph=graph)
        outs.append(shim.sample_reverse_sde_euler_maruyama(m, sde, yc, yk, (5, 1, 64, 64), n_steps=3, guidance_scale=1.5,
                                                           t_end=0.005, x_init=x0, seed=7))
        outs.append(shim.sample_probability_flow_ode(m, sde, yc, yk, (5, 1, 64, 64), n_steps=2, guidance_scale=0.0,
                                                     t_end=0.005, x_init=x0))
    for k in range(2, len(outs)):
        assert torch.equal(outs[k], outs[k % 2]), k
    assert m.launch_count() > 0


def test_errors_and_cli_on_gpu(tmp_path):
    pu = _pu()
    import os
    import importlib.util
    import toycrystals_oracle as orc
    from toycrystals_b200.models import sde_score_model as shim
    m = pu.model("bf16", "tcgen05", seed=1)
    y_cat, y_cont = orc.condition_grid(2, 4, 4)
    with pytest.raises(ValueError, match=r"t_end must be in \(0,1\)"):
        shim.sample_reverse_sde_euler_maruyama(m, shim.VPSDE(), y_cat.cuda(), y_cont.cuda(), (2, 1, 64, 64), t_end=0.0)
    with pytest.raises(NotImplementedError):
        shim.sample_probability_flow_ode(m, shim.VPSDE(), y_cat.cuda(), y_cont.cuda(), (2, 1, 32, 32))
    os.makedirs(tmp_path / "checkpoints")
    torch.save(orc.make_checkpoint(), tmp_path / "checkpoints" / "sde_score_model_last.pt")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location(
        "tcs_cli", os.path.join(root, "vae-diffusion-toy-crystals_b200", "scripts", "sample_sde_score_model.py"))
    cli = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(cli)
    rc = cli.main(["--out-dir", str(tmp_path), "--steps", "2", "--cfg", "1.5", "--t-end", "0.005", "--sampler", "sde",
                   "--use-ema", "1", "--n", "36", "--out-tensor", str(tmp_path / "x.pt")])
    assert rc == 0
    png = tmp_path / "results" / "samples_ckpt-sde_score_model_last_steps2_cfg1.50_tend0.005_samplersde_ema1.png"
    assert png.exists()
    x = torch.load(tmp_path / "x.pt")
    assert x.shape == (36, 1, 64, 64) and float(x.min()) >= 0 and float(x.max()) <= 1


# ---- BASELINE-size runs through size-independent properties -------------------------------------------------
def _zero_out_model(precision):
    """Model whose `out` conv is zero: eps == 0, so both samplers reduce to x_final = f * x_init (per pixel)."""
    pu = _pu()
    import toycrystals_oracle as orc
    from toycrystals_b200.models.sde_score_model import CondUNetTiny
    sd = orc.default_init_state_dict(1)
    sd["out.weight"].zero_(); sd["out.bias"].zero_()
    m = CondUNetTiny(**pu.CFG, precision=precision, chunk=2048)
    m.load_state_dict(sd)
    return m.cuda().eval()


def test_full_size_zero_eps_is_the_analytic_linear_recurrence():
    """configs[1] size (n=1024, 300 steps, CFG 1.5): with eps == 0 the ODE (Heun) trajectory is a scalar recurrence
    in fp32; the whole network still runs (its output is multiplied by zero weights)."""
    pu = _pu()
    import toycrystals_oracle as orc
    from toycrystals_b200.models import sde_score_model as shim
    n, steps = 1024, 300
    m = _zero_out_model("bf16")
    sde = shim.VPSDE(0.1, 30.0)
    yc, yk = shim.condition_grid(m, n, math.pi / 3, "cuda")
    x0 = torch.randn((n, 1, 64, 64), generator=torch.Generator().manual_seed(11)).cuda()
    img, tr = shim.sample_probability_flow_ode(m, sde, yc, yk, (n, 1, 64, 64), n_steps=steps, guidance_scale=1.5,
                                               t_end=0.005, x_init=x0, return_trace=False), None
    sch = orc.Schedule(0.1, 30.0)
    ts = orc.time_grid(steps, 0.005)
    f = torch.tensor(1.0)
    for i in range(steps):   # the reference's fp32 operation order on a scalar
        b0, b1, dt = sch.beta(ts[i]), sch.beta(ts[i + 1]), ts[i + 1] - ts[i]
        d0 = -0.5 * b0 * f
        xe = f + d0 * dt
        d1 = -0.5 * b1 * xe
        f = f + 0.5 * (d0 + d1) * dt
    x0_hat = x0 * (f / torch.clamp(sch.alpha(ts[-1]), min=1e-6)).cuda()
    want = ((x0_hat + 1.0) * 0.5).clamp(0.0, 1.0)
    assert float((img - want).abs().max()) < 2e-3
    assert pu.rel_l2(img, want) < 1e-4


def test_full_size_determinism_and_condition_grid():
    pu = _pu()
    import toycrystals_oracle as orc
    from toycrystals_b200.models import sde_score_model as shim
    n = 1024
    m = pu.model("bf16", "tcgen05", seed=1, chunk=2048)
    sde = shim.VPSDE(0.1, 30.0)
    yc, yk = shim.condition_grid(m, n, math.pi / 3, "cuda")
    oc, ok = orc.condition_grid(n, 4, 4)
    assert torch.equal(yc.cpu(), oc)
    assert float((yk.cpu() - ok).abs().max()) < 2e-7     # torch CPU linspace is SIMD-vectorised: 1 ulp
    def run(seed):
        torch.manual_seed(77)   # x_init is one torch.randn from the global generator, exactly like the reference
        return shim.sample_reverse_sde_euler_maruyama(m, sde, yc, yk, (n, 1, 64, 64), n_steps=3, guidance_scale=1.5,
                                                      t_end=0.005, seed=seed)
    a, b, c = run(5), run(5), run(6)
    assert torch.equal(a, b), "two identical calls differ: the fused GroupNorm reduction must be order-fixed"
    assert not torch.equal(a, c)
    # sharded across "ranks" (same GPU): identical to the unsharded run
    x0 = torch.randn((n, 1, 64, 64), generator=torch.Generator().manual_seed(3)).cuda()
    full = shim.sample_reverse_sde_euler_maruyama(m, sde, yc, yk, (n, 1, 64, 64), n_steps=2, guidance_scale=1.5,
                                                  t_end=0.005, x_init=x0, seed=9)
    parts = []
    for lo, hi in ((0, 300), (300, 1024)):
        yc_s, yk_s = shim.condition_grid(m, hi - lo, math.pi / 3, "cuda", offset=lo, n_total=n)
        parts.append(shim.sample_reverse_sde_euler_maruyama(m, sde, yc_s, yk_s, (hi - lo, 1, 64, 64), n_steps=2,
                                                            guidance_scale=1.5, t_end=0.005, x_init=x0[lo:hi], seed=9,
                                                            global_index_offset=lo))
    assert torch.equal(torch.cat(parts), full)


def test_c1_full_config_against_the_reference(golden_dir):
    """BASELINE configs[0] at full size: PF-ODE (Heun), n=36, 300 steps, CFG 1.5, t_end 0.005, generated by the
    UNMODIFIED reference (oracle/gen_golden_c1.py).  601 CFG evaluations of a random-weight (expanding) trajectory:
    fp32 mode is held to the stated final-sample tolerance, bf16 mode is reported and loosely bounded."""
    import os
    pu = _pu()
    path = os.path.join(golden_dir, "c1_ode_n36_s300.pt")
    if not os.path.exists(path):
        pytest.skip("c1 golden not generated")
    g = torch.load(path, weights_only=False)
    import toycrystals_oracle as orc
    from toycrystals_b200.models import sde_score_model as shim
    y_cat, y_cont = orc.condition_grid(g["n"], 4, 4)
    x_init = torch.randn((g["n"], 1, 64, 64), generator=torch.Generator().manual_seed(g["seed_x"]))
    sde = shim.VPSDE(0.1, 30.0)
    for precision, engine in (("fp32", "simt"), ("fp32", "tcgen05"), ("bf16", "tcgen05")):
        m = pu.model(precision, engine, seed=1)
        img, tr = shim.sample_probability_flow_ode(m, sde, y_cat.cuda(), y_cont.cuda(), (g["n"], 1, 64, 64),
                                                   n_steps=g["steps"], guidance_scale=g["cfg"], t_end=g["t_end"],
                                                   x_init=x_init.cuda(), return_trace=True)
        assert tr.eps.shape[0] == g["nfe"] == 601
        x0_err = pu.rel_l2(tr.x0_hat, g["x0_hat"])
        mism = float(((img.cpu() - pu.image_of(g["x0_hat"])).abs() > 1.0 / 255).float().mean())
        # teacher-forced last evaluation at the reference's own x_{t_end} (stored for the samples in final_index)
        idx = g["final_index"]
        e = shim.predict_eps_cfg(m, g["x_final"].cuda(), torch.full((len(idx),), float(orc.time_grid(300, 0.005)[-1])).cuda(),
                                 y_cat[idx].cuda(), y_cont[idx].cuda(), g["cfg"])
        e_err = pu.rel_l2(e, g["eps_final"])
        print(f"C1 {precision}/{engine}: x0_hat rel-L2 {x0_err:.3e}, mismatched pixels {mism:.4%}, final eps (teacher-forced) {e_err:.3e}")
        assert e_err < TOL_EPS[precision]
        # stated per-pixel tolerance for final PF-ODE samples (measured on B200: fp32 3.8e-7 / 0 pixels, bf16 1.3e-3 / 0.08 %)
        if precision == "fp32" and engine == "simt":
            assert x0_err < 1e-5 and mism < 1e-4, (x0_err, mism)
        elif precision == "fp32":      # bf16x3 on the tensor pipe: the stated final-sample tolerance (SURVEY 8c)
            assert x0_err < 1e-3 and mism < 5e-3, (x0_err, mism)
        else:
            assert x0_err < 1e-2 and mism < 1e-2, (x0_err, mism)


def test_training_hook_accepts_a_foreign_module(tmp_path):
    """SURVEY 8(f) row 2: scripts/train_sde_score_model.py:263-279 calls save_sde_samples(model=<its own nn.Module>)."""
    import toycrystals_oracle as orc
    from toycrystals_b200.models import sde_score_model as shim
    P = _pu()

    class Foreign(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.inner = shim.CondUNetTiny(**orc.DEFAULT_CFG)
            self.inner.load_state_dict(orc.default_init_state_dict(1))
            self.n_types, self.y_cont_dim = 4, 4

        def state_dict(self, *a, **k):
            return self.inner.state_dict(*a, **k)

    f = Foreign().to("cuda")
    out = tmp_path / "grid.png"
    shim.save_sde_samples(model=f, sde=shim.VPSDE(0.1, 30.0), out_path=str(out), device=torch.device("cuda"), steps=2, cfg=1.5,
                          t_end=0.005, sampler="sde")
    assert out.exists() and out.stat().st_size > 1000
    y_cat, y_cont = (t.cuda() for t in orc.condition_grid(4, 4, 4))
    x = torch.randn((4, 1, 64, 64), device="cuda")
    t = torch.full((4,), 0.4, device="cuda")
    a = shim.predict_eps_cfg(f, x, t, y_cat, y_cont, 1.5)
    b = shim.predict_eps_cfg(P.model("bf16", seed=1), x, t, y_cat, y_cont, 1.5)
    assert torch.equal(a, b)


def test_output_conv_variants_agree(monkeypatch):
    """The 96 -> 1 output conv with the kx taps as GEMM columns (default) against the one-window-per-tap variant
    (TCS_EPS_KXN=0): same bf16 operands, fp32 accumulation in a different order."""
    import toycrystals_oracle as orc
    from toycrystals_b200.models import sde_score_model as shim
    sd = orc.default_init_state_dict(1)
    y_cat, y_cont = (t.cuda() for t in orc.condition_grid(5, 4, 4))
    g = torch.Generator().manual_seed(8)
    x = torch.randn((5, 1, 64, 64), generator=g).cuda()
    t = torch.full((5,), 0.3).cuda()
    outs = []
    for flag in ("1", "0"):
        monkeypatch.setenv("TCS_EPS_KXN", flag)
        m = shim.CondUNetTiny(**orc.DEFAULT_CFG, precision="bf16", chunk=64)
        m.load_state_dict(sd)
        m = m.to("cuda").eval()
        outs.append((shim.predict_eps_cfg(m, x, t, y_cat, y_cont, 1.5), shim.predict_eps_cfg(m, x, t, y_cat, y_cont, 0.0)))
        del m
    for a, b in zip(outs[0], outs[1]):
        assert orc.rel_l2(a, b) < 1e-5


@pytest.mark.gpu
def test_tma_store_epilogues_match_per_lane_stores(monkeypatch):
    """Every epilogue that stages 32x32 blocks and hands them to TMA (padded outputs at 64/32/16-pixel rows, the
    unpadded qkv rows, the fused GroupNorm layers) against the per-lane store path (TCS_DEBUG=4) and against single-CTA
    MMAs (TCS_CG=1; since the 64-channel K blocks only the 1x1 layers can run that way): the arithmetic is the same, only
    the way the bytes reach memory changes, so a whole CFG evaluation must be bit-identical; n = 5 gives a ragged number of
    image groups and CTA pairs."""
    import toycrystals_oracle as orc
    from toycrystals_b200.models import sde_score_model as shim
    sd = orc.default_init_state_dict(1)
    y_cat, y_cont = (t.cuda() for t in orc.condition_grid(5, 4, 4))
    g = torch.Generator().manual_seed(9)
    x = torch.randn((5, 1, 64, 64), generator=g).cuda()
    t = torch.full((5,), 0.6).cuda()
    outs = []
    for env in ({}, {"TCS_DEBUG": "4"}, {"TCS_CG": "1"}, {"TCS_GEO": "0"}, {"TCS_TB": "1"}):
        for k in ("TCS_DEBUG", "TCS_CG", "TCS_GEO", "TCS_TB"):
            monkeypatch.delenv(k, raising=False)
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        m = shim.CondUNetTiny(**orc.DEFAULT_CFG, precision="bf16", chunk=64)
        m.load_state_dict(sd)
        m = m.to("cuda").eval()
        outs.append(shim.predict_eps_cfg(m, x, t, y_cat, y_cont, 1.5).clone())
        del m
    assert torch.equal(outs[0], outs[1]), "TMA-store epilogues differ from per-lane stores"
    assert torch.equal(outs[0], outs[2]), "CTA-pair MMAs differ from single-CTA MMAs"
    # tap-shift geometry (one window per channel block, taps as descriptor shifts) against the per-kx row windows: the
    # MMAs accumulate in the same order, only the fp32 GroupNorm sums are added in a different order; the ~1e-5 that
    # moves the statistics flips bf16 roundings in ten normalised layers (measured 4.9e-3 on the final eps, half the bf16
    # error against the oracle: both are equally far from it)
    e = orc.rel_l2(outs[3], outs[0])
    print(f"tap-shift geometry vs row windows: eps rel-L2 {e:.3e}")
    assert e < 1e-2
    assert torch.equal(outs[0], outs[4]), "weight stages of one tap differ from stages of three taps"


def test_fused_blocks_agree_with_their_unfused_forms(monkeypatch):
    """The fused attention block (attn_tc.cu) and the upsample fused into us1_conv / us2_conv against the same network with
    the four-launch attention / the stand-alone upsample kernel (TCS_FUSE_ATTN=0, TCS_FUSE_UPS=0): one CFG evaluation of
    5 samples.  The fused upsample performs the same fp32 blend and the same single rounding, so it may only move bf16
    roundings (measured: bit-identical eps); the fused attention rounds q, k, v, P differently (fp16 P and V): measured
    5.5e-3 on eps, both forms are equally far (~9e-3) from the oracle."""
    import toycrystals_oracle as orc
    from toycrystals_b200.models import sde_score_model as shim
    sd = orc.default_init_state_dict(1)
    y_cat, y_cont = (t.cuda() for t in orc.condition_grid(5, 4, 4))
    g = torch.Generator().manual_seed(21)
    x = torch.randn((5, 1, 64, 64), generator=g).cuda()
    t = torch.full((5,), 0.4).cuda()
    outs = {}
    for name, env in (("fused", {}), ("ups_off", {"TCS_FUSE_UPS": "0"}), ("attn_off", {"TCS_FUSE_ATTN": "0"})):
        for k in ("TCS_FUSE_UPS", "TCS_FUSE_ATTN"):
            monkeypatch.delenv(k, raising=False)
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        m = shim.CondUNetTiny(**orc.DEFAULT_CFG, precision="bf16", chunk=64)
        m.load_state_dict(sd)
        m = m.to("cuda").eval()
        outs[name] = shim.predict_eps_cfg(m, x, t, y_cat, y_cont, 1.5).clone()
        n_launch = m.launch_count()
        del m
        outs[name + "_launches"] = n_launch
    e_ups, e_att = orc.rel_l2(outs["fused"], outs["ups_off"]), orc.rel_l2(outs["fused"], outs["attn_off"])
    print(f"fused vs stand-alone upsample: eps rel-L2 {e_ups:.2e}; fused vs four-launch attention: {e_att:.2e}; "
          f"launches {outs['fused_launches']} / {outs['ups_off_launches']} / {outs['attn_off_launches']}")
    assert e_ups < 5e-3 and e_att < 1e-2, (e_ups, e_att)
    assert outs["ups_off_launches"] == outs["fused_launches"] + 2 and outs["attn_off_launches"] == outs["fused_launches"] + 3


# ---- round 2: gaps named by the round-1 review ----------------------------------------------------------
def _oracle_on_cuda():
    """The oracle evaluated by PyTorch on the GPU in IEEE fp32 (TF32 off): seconds instead of minutes at n = 1024."""
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.set_float32_matmul_precision("highest")


@pytest.mark.parametrize("precision,engine", [("fp32", "simt"), ("fp32", "tcgen05"), ("bf16", "tcgen05")])
def test_full_size_pass_teacher_forced_against_the_oracle(precision, engine):
    """BASELINE configs[1] shape: n = 1024 with CFG 1.5 = ONE 2048-image pass (the production shape: 144/148-CTA grids,
    G-CTA lock step, CTA pairs), eps against the oracle (IEEE fp32 on the GPU) at t = 1, 0.37, 0.005."""
    pu = _pu()
    import toycrystals_oracle as orc
    from toycrystals_b200.models import sde_score_model as shim
    _oracle_on_cuda()
    n = 1024
    m = pu.model(precision, engine, seed=1, chunk=2048)
    sd = {k: v.cuda() for k, v in orc.default_init_state_dict(1).items()}
    yc, yk = shim.condition_grid(m, n, math.pi / 3, "cuda")
    g = torch.Generator().manual_seed(21)
    x = torch.randn((n, 1, 64, 64), generator=g).cuda()
    for scale, tval in ((1.0, 1.0), (37.0, 0.37), (900.0, 0.005)):
        t = torch.full((n,), tval, device="cuda")
        got = shim.predict_eps_cfg(m, x * scale, t, yc, yk, 1.5)
        with torch.no_grad():
            want = torch.cat([orc.eps_cfg(sd, pu.CFG, x[i:i + 256] * scale, t[i:i + 256], yc[i:i + 256], yk[i:i + 256], 1.5)
                              for i in range(0, n, 256)])
        err = pu.rel_l2(got, want)
        per_sample = ((got - want).flatten(1).norm(dim=1) / want.flatten(1).norm(dim=1)).max().item()
        print(f"{precision}/{engine} n={n} t={tval}: eps rel-L2 {err:.3e}, worst sample {per_sample:.3e}")
        assert err < TOL_EPS[precision], (tval, err)
        assert per_sample < 2.5 * TOL_EPS[precision], (tval, per_sample)


def test_ode_update_kernels_are_bit_exact_vs_torch_expressions():
    """_probflow_drift (:426-449), the Heun predictor / corrector (:490-493) and the final projection (:496-504) in the
    reference's fp32 operation order."""
    pu = _pu()
    from toycrystals_b200 import _cabi
    from toycrystals_b200.models.sde_score_model import VPSDE
    m = pu.model("fp32", "simt")
    h = m.engine_handle(VPSDE(0.1, 30.0))
    L = _cabi.lib()
    sde = VPSDE(0.1, 30.0)
    g = torch.Generator().manual_seed(6)
    n = 5
    # expectations in torch CPU fp32: libtcs evaluates the schedule (exp, sqrt) on the host; torch's CUDA exp may differ
    # from the CPU one by an ulp, and sigma(t_end) = sqrt(1 - alpha^2) amplifies an ulp of alpha 1000-fold
    x = torch.randn((n, 1, 64, 64), generator=g) * 30
    e0, e1 = torch.randn((n, 1, 64, 64), generator=g), torch.randn((n, 1, 64, 64), generator=g)
    t, t_next = torch.tensor(0.3712), torch.tensor(0.3651)
    dt = t_next - t

    def drift(xx, ee, tt):
        beta_t, sigma_t = sde.beta(tt), sde.sigma(tt)
        score = -ee / sigma_t
        return -0.5 * beta_t * xx - 0.5 * beta_t * score

    d_want = drift(x, e0, t)
    xe_want = x + d_want * dt
    x_want = x + 0.5 * (d_want + drift(xe_want, e1, t_next)) * dt
    xs, xp, d0 = x.cuda(), torch.empty_like(x).cuda(), torch.empty_like(x).cuda()
    e0c, e1c = e0.cuda(), e1.cuda()
    _cabi.check(L.tcs_ode_update(h, 1, xs.data_ptr(), xp.data_ptr(), d0.data_ptr(), e0c.data_ptr(), n, float(t), float(t_next), None))
    torch.cuda.synchronize()
    assert torch.equal(d0.cpu(), d_want) and torch.equal(xp.cpu(), xe_want) and torch.equal(xs.cpu(), x)
    _cabi.check(L.tcs_ode_update(h, 2, xs.data_ptr(), xp.data_ptr(), d0.data_ptr(), e1c.data_ptr(), n, float(t), float(t_next), None))
    torch.cuda.synchronize()
    assert torch.equal(xs.cpu(), x_want)
    # final projection at t_end
    te = torch.tensor(0.005)
    a, sg = sde.alpha(te), sde.sigma(te)
    x0_want = (x - sg * e0) / torch.clamp(a, min=1e-6)
    img_want = ((x0_want + 1.0) * 0.5).clamp(0.0, 1.0)
    xs = x.cuda()
    _cabi.check(L.tcs_ode_update(h, 3, xs.data_ptr(), xp.data_ptr(), d0.data_ptr(), e0c.data_ptr(), n, float(te), float(te), None))
    torch.cuda.synchronize()
    assert torch.equal(d0.cpu(), x0_want) and torch.equal(xp.cpu(), img_want)


def test_update_kernels_are_bit_identical_at_scale():
    """The update kernels divide by a launch-uniform sigma / alpha through a hoisted reciprocal (three FFMA per quotient,
    the fast path of IEEE division).  260k values per case, |x| up to 1e4 and eps up to 1e4 as on the random-weight
    trajectory, several times of the grid: every bit must equal torch's fp32 expression (CPU, true division)."""
    pu = _pu()
    from toycrystals_b200 import _cabi
    from toycrystals_b200.models.sde_score_model import VPSDE
    m = pu.model("fp32", "simt")
    h = m.engine_handle(VPSDE(0.1, 30.0))
    L = _cabi.lib()
    sde = VPSDE(0.1, 30.0)
    g = torch.Generator().manual_seed(16)
    n = 64
    for tv, tn, scale in ((1.0, 0.9934, 1.0), (0.3712, 0.3651, 300.0), (0.0051, 0.005, 1e4)):
        x = torch.randn((n, 1, 64, 64), generator=g) * scale
        eps = torch.randn((n, 1, 64, 64), generator=g) * (1.0 + scale)
        z = torch.randn((n, 1, 64, 64), generator=g)
        t, t_next = torch.tensor(tv), torch.tensor(tn)
        beta, sigma, dt = sde.beta(t), sde.sigma(t), t_next - t
        want = x + ((-0.5 * beta * x) - (beta * (-eps / sigma))) * dt + torch.sqrt(beta) * torch.sqrt(torch.abs(dt)) * z
        got, ec, zc = x.cuda(), eps.cuda(), z.cuda()
        _cabi.check(L.tcs_sde_update(h, got.data_ptr(), ec.data_ptr(), zc.data_ptr(), n, float(t), float(t_next), 0, 0, 0, None))
        torch.cuda.synchronize()
        assert torch.equal(got.cpu(), want), (tv, float((got.cpu() - want).abs().max()))
        a, sg = sde.alpha(t), sde.sigma(t)
        x0_want = (x - sg * eps) / torch.clamp(a, min=1e-6)
        xs, xp, d0 = x.cuda(), torch.empty_like(x).cuda(), torch.empty_like(x).cuda()
        _cabi.check(L.tcs_ode_update(h, 3, xs.data_ptr(), xp.data_ptr(), d0.data_ptr(), ec.data_ptr(), n, float(t), float(t), None))
        torch.cuda.synchronize()
        assert torch.equal(d0.cpu(), x0_want), tv


def test_graph_cache_follows_workspace_reallocation():
    """ADVICE r1 (high): the captured step graph holds the device pointers of per-call buffers that grow with `steps` and
    with tcs_score / tcs_debug_layer calls in between; a re-allocation must force a re-capture."""
    pu = _pu()
    import toycrystals_oracle as orc
    from toycrystals_b200.models import sde_score_model as shim
    sde = shim.VPSDE(0.1, 30.0)
    y_cat, y_cont = orc.condition_grid(4, 4, 4)
    yc, yk = y_cat.cuda(), y_cont.cuda()
    x0 = torch.randn((4, 1, 64, 64), generator=torch.Generator().manual_seed(3)).cuda()

    def run(m, steps):
        return shim.sample_reverse_sde_euler_maruyama(m, sde, yc, yk, (4, 1, 64, 64), n_steps=steps, guidance_scale=1.5,
                                                      t_end=0.005, x_init=x0, seed=0).clone()
    plain = pu.model("bf16", "tcgen05", seed=1, chunk=64, use_graph=False)   # no graph: the ground truth
    m = pu.model("bf16", "tcgen05", seed=1, chunk=64)
    a50 = run(m, 50)
    a300 = run(m, 300)           # tvec / tvals / coef grow -> the old graph would replay freed pointers
    assert torch.equal(a300, run(plain, 300))
    assert torch.equal(a50, run(plain, 50))
    # a large tcs_score between two identical sampling calls grows cvec / tvec / eps
    yc2, yk2 = shim.condition_grid(m, 600, math.pi / 3, "cuda")
    shim.predict_eps_cfg(m, torch.randn((600, 1, 64, 64), device="cuda"), torch.full((600,), 0.5, device="cuda"), yc2, yk2, 1.5)
    assert torch.equal(run(m, 50), a50)


def test_seed_alone_reproduces_and_shards():
    """ADVICE r1: with `seed=` and no x_init the initial state comes from Philox keyed (seed, global index), so a
    2-shard run equals the 1-shard run and does not depend on torch's generator."""
    pu = _pu()
    import toycrystals_oracle as orc
    from toycrystals_b200.models import sde_score_model as shim
    m = pu.model("bf16", "tcgen05", seed=1)
    sde = shim.VPSDE(0.1, 30.0)
    n = 6
    yc, yk = shim.condition_grid(m, n, math.pi / 3, "cuda")

    def run(lo, hi, torch_seed):
        torch.manual_seed(torch_seed)
        c, k = shim.condition_grid(m, hi - lo, math.pi / 3, "cuda", offset=lo, n_total=n)
        return shim.sample_reverse_sde_euler_maruyama(m, sde, c, k, (hi - lo, 1, 64, 64), n_steps=3, guidance_scale=1.5,
                                                      t_end=0.005, seed=42, global_index_offset=lo)
    full = run(0, n, 1)
    assert torch.equal(full, run(0, n, 2)), "seed= alone must fix the run"
    assert torch.equal(torch.cat([run(0, 4, 3), run(4, 6, 4)]), full), "sharded run differs"
    ode = shim.sample_probability_flow_ode(m, sde, yc, yk, (n, 1, 64, 64), n_steps=2, guidance_scale=1.5, t_end=0.005, seed=42)
    ode2 = shim.sample_probability_flow_ode(m, sde, yc, yk, (n, 1, 64, 64), n_steps=2, guidance_scale=1.5, t_end=0.005, seed=42)
    assert torch.equal(ode, ode2)


def test_weight_updates_through_data_are_seen():
    """ADVICE r1: the reference's EMA update writes p_ema.data in place (scripts/train_sde_score_model.py:239-240), which
    does not bump tensor._version; the samplers and the training hook must still pick the new weights up."""
    import toycrystals_oracle as orc
    from toycrystals_b200.models import sde_score_model as shim
    sd = orc.default_init_state_dict(1)
    sde = shim.VPSDE(0.1, 30.0)
    y_cat, y_cont = (t.cuda() for t in orc.condition_grid(3, 4, 4))
    x0 = torch.randn((3, 1, 64, 64), generator=torch.Generator().manual_seed(4)).cuda()

    def build():
        m = shim.CondUNetTiny(**orc.DEFAULT_CFG, precision="bf16", chunk=64)
        m.load_state_dict(sd)
        return m.cuda().eval()

    def run(model):
        return shim.sample_reverse_sde_euler_maruyama(model, sde, y_cat, y_cont, (3, 1, 64, 64), n_steps=2, guidance_scale=1.5,
                                                      t_end=0.005, x_init=x0, seed=1).clone()
    m = build()
    before = run(m)
    vers = [p._version for p in m.parameters()]
    with torch.no_grad():
        for p in m.parameters():
            p.data.mul_(0.999).add_(0.01 * torch.ones_like(p), alpha=0.001)
    assert [p._version for p in m.parameters()] == vers, "the premise of this test: .data updates are invisible to _version"
    after = run(m)
    assert not torch.equal(before, after), "stale weights: the .data update was not seen"
    ref = build()
    ref.load_state_dict(m.state_dict())
    assert torch.equal(after, run(ref))

    class Foreign(torch.nn.Module):       # the training script's own module: only its state dict is known
        def __init__(self, inner):
            super().__init__()
            self.inner = inner
            self.n_types, self.y_cont_dim = 4, 4

        def state_dict(self, *a, **k):
            return self.inner.state_dict(*a, **k)
    f = Foreign(build())
    t = torch.full((3,), 0.4, device="cuda")
    e0 = shim.predict_eps_cfg(f, x0, t, y_cat, y_cont, 1.5).clone()
    with torch.no_grad():
        for p in f.inner.parameters():
            p.data.mul_(0.99)
    e1 = shim.predict_eps_cfg(f, x0, t, y_cat, y_cont, 1.5)
    assert not torch.equal(e0, e1)


def test_unsupported_architectures_fail_at_construction():
    from toycrystals_b200.models.sde_score_model import CondUNetTiny
    with pytest.raises(NotImplementedError, match="base_ch=96"):
        CondUNetTiny(4, 4)            # the reference's own default base_ch=32
    with pytest.raises(ValueError):
        CondUNetTiny(4, 2, base_ch=96)


def test_fused_groupnorm_stash_range_is_guarded():
    """The fused conv+GroupNorm epilogue stages pre-norm values as fp16 (|v| <= 65504).  GroupNorm is scale invariant, so
    a conv whose weights are scaled by 3e5 must give the same eps: the kernel flags the launch and the shim re-runs the
    evaluation on the unfused path instead of returning clipped activations."""
    pu = _pu()
    import toycrystals_oracle as orc
    from toycrystals_b200.models import sde_score_model as shim
    sd = orc.default_init_state_dict(1)
    big = {k: v.clone() for k, v in sd.items()}
    for k in ("down1.net.3", "up1.net.0"):
        big[k + ".weight"] *= 3e5
        big[k + ".bias"] *= 3e5
    y_cat, y_cont = (t.cuda() for t in orc.condition_grid(5, 4, 4))
    x = torch.randn((5, 1, 64, 64), generator=torch.Generator().manual_seed(12)).cuda()
    t = torch.full((5,), 0.37).cuda()
    m = shim.CondUNetTiny(**orc.DEFAULT_CFG, precision="bf16", chunk=64)
    m.load_state_dict(big)
    m = m.cuda().eval()
    with pytest.warns(UserWarning, match="fp16 staging range"):
        got = shim.predict_eps_cfg(m, x, t, y_cat, y_cont, 1.5)
    with torch.no_grad():
        want = orc.eps_cfg(big, pu.CFG, x.cpu(), t.cpu(), y_cat.cpu(), y_cont.cpu(), 1.5)
    assert pu.rel_l2(got, want) < TOL_EPS["bf16"]
    assert m._fuse_gn is False
    # and the ordinary model never trips the guard
    m2 = pu.model("bf16", "tcgen05", seed=1)
    import warnings as W
    with W.catch_warnings():
        W.simplefilter("error")
        shim.predict_eps_cfg(m2, x * 900.0, torch.full((5,), 0.005).cuda(), y_cat, y_cont, 1.5)
    assert m2._fuse_gn is True


def test_pass_survives_a_busy_neighbour_stream():
    """The fused-GroupNorm CTAs poll each other's partial sums: the launch must stay correct (and must not hang) while a
    kernel of ANOTHER stream holds part of the SMs."""
    pu = _pu()
    import toycrystals_oracle as orc
    from toycrystals_b200 import _cabi
    from toycrystals_b200.models import sde_score_model as shim
    m = pu.model("bf16", "tcgen05", seed=1)
    n = 64
    yc, yk = shim.condition_grid(m, n, math.pi / 3, "cuda")
    x = torch.randn((n, 1, 64, 64), generator=torch.Generator().manual_seed(13)).cuda()
    t = torch.full((n,), 0.5).cuda()
    quiet = shim.predict_eps_cfg(m, x, t, yc, yk, 1.5).clone()
    mode = int(_cabi.lib().tcs_launch_mode(m.engine_handle()))
    print(f"launch mode: fused={mode & 1} cooperative+cluster={(mode >> 1) & 1} max resident CTAs={mode >> 8}")
    side = torch.cuda.Stream()
    a = torch.randn((8192, 8192), device="cuda", dtype=torch.bfloat16)
    for _ in range(3):
        with torch.cuda.stream(side):
            for _ in range(20):
                a @ a                      # keeps every SM busy from another stream
        got = shim.predict_eps_cfg(m, x, t, yc, yk, 1.5)
        torch.cuda.synchronize()
        assert torch.equal(got, quiet)
