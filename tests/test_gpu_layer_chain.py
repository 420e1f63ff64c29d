"""Every layer of the bf16 tcgen05 score pass, element by element, at the production batch and under other grids.

Each layer's reference is computed in fp64 from the pass's own taps of its inputs (the bf16 values the kernel read), so
errors do not compound and the per-element bound of tests/layer_bounds.py is the kernel's own roundings.  A violation is
reported with the layer, image, CFG row, CTA tile and channel group.  Run with -s for one line per layer."""
import math
import time

import pytest
import torch
import torch.nn.functional as F

import layer_bounds as lb

pytestmark = pytest.mark.gpu

U = lb.U_F32
CHUNK_IMAGES = 256       # fp64 reference chunk (images)
# attention block: per element |got - r| <= 2^-8 |r| + C_ATTN rms_image(r - x): SAFETY x the 4.6-sigma tail of the
# 49152 elements of an image x the 1.5e-2 rel-L2 gate of the attention output y in test_fused_attention_block
C_ATTN = lb.SAFETY * 4.6 * 1.5e-2
ATTN_BRANCH_GATE = 2e-2  # the branch gate of test_fused_attention_block, per image here

# name -> (input taps, kind, parameter key, GroupNorm key, CTA tile (rows, cols), channels)
LAYERS = {
    "down1.net.0.act": ((), "first", "down1.net.0", "down1.net.1", (32, 64), 96),   # FC_SPLIT = 2 bands per image
    "down1.net.3.act": (("down1.net.0.act",), "gn", "down1.net.3", "down1.net.4", (16, 16), 96),
    "ds1": (("down1.net.3.act",), "conv", "ds1", None, (8, 32), 96),
    "down2.net.0.act": (("ds1",), "gn", "down2.net.0", "down2.net.1", (16, 8), 192),
    "down2.net.3.act": (("down2.net.0.act",), "gn", "down2.net.3", "down2.net.4", (16, 8), 192),
    "ds2": (("down2.net.3.act",), "conv", "ds2", None, (8, 16), 192),
    "mid.net.0.act": (("ds2",), "gn", "mid.net.0", "mid.net.1", (16, 8), 192),
    "mid.net.3.act": (("mid.net.0.act",), "gn", "mid.net.3", "mid.net.4", (16, 8), 192),
    "attn": (("mid.net.3.act",), "attn", "attn", "attn.norm", (16, 16), 192),
    "us2_conv": (("attn",), "ups", "us2_conv", None, (16, 8), 192),
    "up2.net.0.act": (("us2_conv", "down2.net.3.act"), "gn", "up2.net.0", "up2.net.1", (16, 16), 96),
    "up2.net.3.act": (("up2.net.0.act",), "gn", "up2.net.3", "up2.net.4", (16, 16), 96),
    "us1_conv": (("up2.net.3.act",), "ups", "us1_conv", None, (16, 16), 96),
    "up1.net.0.act": (("us1_conv", "down1.net.3.act"), "gn", "up1.net.0", "up1.net.1", (16, 16), 96),
    "up1.net.3.act": (("up1.net.0.act",), "gn", "up1.net.3", "up1.net.4", (16, 16), 96),
    "eps": (("up1.net.3.act",), "eps", "out", None, (2, 64), 1),
}
RES = {"down1": 64, "ds1": 32, "down2": 32, "ds2": 16, "mid.": 16, "attn": 16, "us2_": 32, "up2.": 32, "us1_": 64,
       "up1.": 64, "eps": 64}
GN_LAYERS = [k for k, v in LAYERS.items() if v[1] in ("gn", "first")]


def _pu():
    import parity_utils as pu
    return pu


def tap(m, name, x, t, yc, yk, uncond):
    res = next(v for k, v in RES.items() if name.startswith(k))
    return _pu().debug_layer(m, name, x, t, yc, yk, LAYERS[name][5], res, uncond=uncond)


def _rows(n, uncond, yc, yk, t, n_types=4):
    """Per batch row: condition, time (rows alternate conditional / unconditional when uncond)."""
    if not uncond:
        return yc, yk, t
    yc2 = torch.stack([yc, torch.full_like(yc, n_types)], 1).flatten()
    yk2 = torch.stack([yk, torch.zeros_like(yk)], 1).flatten(0, 1)
    return yc2, yk2, t.repeat_interleave(2)


def _embed_with_error(sd, t, yc, yk):
    """The first conv's per-(row, channel) bias tvec + cvec as time_embed_kernel / cond_embed_kernel form it in fp32
    (kernels_embed.cu), in fp64, with a running bound of its error: every dot product of K terms (dot_row, :15-19) costs
    (K + 1) u32 of the sum of |terms|, silu_acc (:12) 4 u32 (expf 2 ulp, add, divide) and passes 1.1 times the input
    error on, expf / sinf / cosf 2 ulp each."""
    import toycrystals_oracle as orc
    dev = t.device
    W = lambda k: sd[k].to(dev).double()

    def lin(name, x, ex):
        w, b = W(name + ".weight"), W(name + ".bias")
        return x @ w.T + b, ex @ w.abs().T + (w.shape[1] + 1) * U * (x.abs() @ w.abs().T + b.abs())

    def silu(v, ev):
        s = F.silu(v)
        return s, lb.SILU_SLOPE * ev + 4 * U * s.abs()

    emb = orc.time_features(t.double(), 128, torch.float64)
    half = torch.arange(64, device=dev, dtype=torch.float64)
    ang = (2 * math.pi) * t.double()[:, None] * torch.exp(-math.log(10000.0) * half / 63)[None]
    e_ang = 6 * U * ang.abs()                      # f = expf(c i / 63): 4 u32, a = (2 pi t) f: 2 u32 (:68-69)
    e_emb = torch.cat([e_ang, e_ang], 1) + 4 * U   # cosf / sinf (:70)
    h, eh = silu(*lin("time_mlp.0", emb, e_emb))
    te, ete = lin("time_mlp.2", h, eh)
    tmap, etmap = lin("to_time_map", te, ete)
    y = yk.double().clone()
    s = torch.sin(y[:, 1])
    y[:, 1] = s
    y[:, 2] = torch.cos(s)
    ey = torch.zeros_like(y)
    ey[:, 1] = 4 * U
    ey[:, 2] = 8 * U
    h0, eh0 = silu(*lin("cond_emb.cont_mlp.0", y, ey))
    zc, ezc = silu(*lin("cond_emb.cont_mlp.2", h0, eh0))
    za, eza = silu(W("cond_emb.cat_emb.weight")[yc.clamp(0, 4)], torch.zeros((yc.shape[0], 128), device=dev, dtype=torch.float64))
    ce, ece = lin("cond_emb.out.1", torch.cat([za, zc], 1), torch.cat([eza, ezc], 1))
    cmap, ecmap = lin("to_cond_map", ce, ece)
    # wsum[c][j] = fp32 sum of the 9 taps of the constant map j (tcs_api.cu:934-940): 9 u32 of the sum of |taps|
    w0 = W("down1.net.0.weight")
    wsum, wabs = w0[:, 1:].sum((2, 3)), w0[:, 1:].abs().sum((2, 3))
    maps, emaps = torch.cat([tmap, cmap], 1), torch.cat([etmap, ecmap], 1)
    b0 = W("down1.net.0.bias")
    bias = b0 + maps @ wsum.T
    # tvec / cvec: fma chains of 8 terms (:79-82, :51-54), then tvec + cvec (kernels_simt.cu:230)
    e = emaps @ wsum.abs().T + 9 * U * maps.abs() @ wabs.T + 10 * U * (b0.abs() + maps.abs() @ wsum.abs().T) + U * bias.abs()
    return bias, e


def layer_reference(name, sd, inp, x, t_rows, yc_rows, yk_rows, stash, guidance=1.5, uncond=1):
    """fp64 reference and per-element bound of one layer from its input taps (chunk of batch rows)."""
    ins, kind, key, gkey, _, C = LAYERS[name]
    dev = inp[0].device if inp else x.device
    P = lambda k: sd[k].to(dev)
    if kind == "first":
        w0 = P(key + ".weight").double()[:, :1]
        bias, e_b = _embed_with_error(sd, t_rows, yc_rows, yk_rows)
        xx = x.double().reshape(-1, 64, 64, 1)
        if uncond:
            xx = xx.repeat_interleave(2, 0)
        v = lb.conv64(xx, w0, None, 3, 1) + bias[:, None, None, :]
        # the 9-tap fp32 FFMA sum (kernels_simt.cu:249-...), the bias as above; statistics in fp64 (:164-222)
        e_t = 10 * U * lb.conv64(xx.abs(), w0.abs(), None, 3, 1) + e_b[:, None, None, :]
        return lb.gn_silu_with_bound(v, e_t, P(gkey + ".weight"), P(gkey + ".bias"), stash=None, stats_u=2.0 ** -53)
    if kind == "attn":
        pu = _pu()
        bfw = lambda k: P(k).bfloat16().float()
        r, _ = pu.attn_block_reference(inp[0], P("attn.norm.weight"), P("attn.norm.bias"), bfw("attn.qkv.weight"),
                                       P("attn.qkv.bias"), bfw("attn.proj.weight"), P("attn.proj.bias"))
        return r, None
    if kind == "ups":
        up, d = lb.upsample_rounding(inp[0].double())
        r, e = lb.conv_with_error(up, P(key + ".weight"), P(key + ".bias"), 3, 1, dx=d)
        return r, lb.bf16_output(r, e)
    xin = torch.cat([i.double() for i in inp], dim=-1)
    k, s = (4, 2) if kind == "conv" else (3, 1)
    if kind == "eps":
        if uncond:
            r, bound = lb.eps_cfg_with_bound(xin, P(key + ".weight"), P(key + ".bias"), guidance)
        else:
            r, bound = lb.conv_with_error(xin, P(key + ".weight"), P(key + ".bias"), 3, 1)
        return r, bound
    r, e = lb.conv_with_error(xin, P(key + ".weight"), P(key + ".bias"), k, s)
    if kind == "conv":
        return r, lb.bf16_output(r, e)
    return lb.gn_silu_with_bound(r, e, P(gkey + ".weight"), P(gkey + ".bias"), stash=stash, bias=P(key + ".bias"))


def chain(m, sd, x, t, yc, yk, uncond, layers=None, stash="fused", gate=True, report=None, taps=None):
    """Check each layer against its fp64 reference from the pass's own input taps.  Returns {layer: result}."""
    taps = {} if taps is None else taps
    def get(nm):
        if nm not in taps:
            taps[nm] = tap(m, nm, x, t, yc, yk, uncond)
        return taps[nm]
    yc_r, yk_r, t_r = _rows(x.shape[0], uncond, yc, yk, t)
    out = {}
    for name in layers or LAYERS:
        t0 = time.time()
        ins, kind, key, gkey, tile, C = LAYERS[name]
        got = get(name)
        inputs = [get(i) for i in ins]
        step = CHUNK_IMAGES * (2 if uncond else 1)
        res = {"worst": 0.0, "worst_img_rel": 0.0, "nbad": 0, "tiles": [], "msg": None}
        nrows = got.shape[0] * (2 if kind == "eps" and uncond else 1)
        for b0 in range(0, nrows, step):
            sl = slice(b0, b0 + step)
            esl = slice(b0 // 2, (b0 + step) // 2) if (kind == "eps" and uncond) else sl
            xs = x[b0 // (2 if uncond else 1):(b0 + step) // (2 if uncond else 1)]
            ref, bound = layer_reference(name, sd, [i[sl] for i in inputs], xs, t_r[sl], yc_r[sl], yk_r[sl], stash,
                                         uncond=uncond)
            g = got[esl].double()
            rows = "cfg" if (uncond and kind != "eps") else None
            if kind == "attn":
                r = lb.check_branch(name, g, ref, inputs[0][sl].double(), C_ATTN, ATTN_BRANCH_GATE, rows=rows, b0=b0)
            else:
                r = lb.check_layer(name, g, ref, bound, tile, max(C // 8, 1), rows=rows, gate=False,
                                   b0=esl.start)
            res["worst"] = max(res["worst"], r["worst"])
            res["worst_img_rel"] = max(res["worst_img_rel"], r["worst_img_rel"])
            res["nbad"] += r["nbad"]
            res["tiles"] += r["tiles"]
            if r.get("msg") and res["msg"] is None:
                res["msg"] = r["msg"]
        torch.cuda.synchronize()
        res["time"] = time.time() - t0
        out[name] = res
        line = (f"{name:16s} worst err/bound {res['worst']:.3f}  worst image rel-L2 {res['worst_img_rel']:.2e}  "
                f"{res['time']:.1f} s")
        if report is not None:
            report.append(line)
        print(line)
        if gate:
            assert res["nbad"] == 0, res["msg"]
    return out


def _inputs(n, scale, tval, seed=21):
    import toycrystals_oracle as orc
    yc, yk = orc.condition_grid(n, 4, 4)
    g = torch.Generator().manual_seed(seed)
    x = torch.randn((n, 1, 64, 64), generator=g) * scale
    return x.cuda(), torch.full((n,), tval).cuda(), yc.cuda(), yk.cuda()


# ---- A: the production pass, n = 1024 with CFG = 2048 images ---------------------------------------------------
@pytest.mark.parametrize("scale,tval", [(1.0, 1.0), (900.0, 0.005)])
def test_production_pass_layer_by_layer(scale, tval):
    pu = _pu()
    import toycrystals_oracle as orc
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    m = pu.model("bf16", "tcgen05", seed=1, chunk=2048)
    sd = orc.default_init_state_dict(1)
    x, t, yc, yk = _inputs(1024, scale, tval)
    taps = {}
    t0 = time.time()
    chain(m, sd, x, t, yc, yk, 1, taps=taps)
    # the facts the chain relies on: taps are bf16 values, and a tap is the same tensor in every pass
    for nm, v in taps.items():
        if nm != "eps":
            assert torch.equal(v, v.bfloat16().float()), nm
    again = tap(m, "down2.net.3.act", x, t, yc, yk, 1)
    assert torch.equal(again, taps["down2.net.3.act"])
    # the checker names a planted fault: one 16 x 16 tile of image 700's unconditional row taken from image 701
    bad = taps["down1.net.3.act"].clone()
    bad[1401, 16:32, 32:48] = bad[1403, 16:32, 32:48]
    yc_r, yk_r, t_r = _rows(1024, 1, yc, yk, t)
    ref, bound = layer_reference("down1.net.3.act", sd, [taps["down1.net.0.act"][1400:1404]], None, t_r[1400:1404],
                                 yc_r[1400:1404], yk_r[1400:1404], "fused")
    r = lb.check_layer("down1.net.3.act", bad[1400:1404].double(), ref, bound, (16, 16), 12, rows="cfg", gate=False, b0=1400)
    assert r["tiles"] == [(1401, 1, 2)], r
    assert "image 700 (unconditional row 1401), tile (1,2)" in r["msg"], r["msg"]
    print(f"chain wall time {time.time() - t0:.1f} s")


# ---- B: the same chain under other grids: bit-identical outputs ---------------------------------------------------
def _fresh_model(sd, chunk, precision="bf16", engine="auto"):
    from toycrystals_b200.models.sde_score_model import CondUNetTiny
    pu = _pu()
    m = CondUNetTiny(**pu.CFG, precision=precision, engine=engine, chunk=chunk)
    m.load_state_dict(sd)
    return m.cuda().eval()


@pytest.mark.parametrize("n,uncond", [(75, 1), (149, 0)])
def test_chain_is_grid_invariant(monkeypatch, n, uncond):
    """B = 150 (CFG rows) and B = 149 (odd) on the default grid (bounds of A), then with TCS_MAX_CTAS = 40 / 36 (images
    straddle waves, CTAs loop over many tiles) and 18 (the 64x64 fused-GroupNorm layers fall back to one whole image
    group): every activation tap and eps must be bit-identical, the exchange being indexed by tile and summed in a
    fixed order.  The cap is only ever lowered below the device's residency."""
    from toycrystals_b200 import _cabi
    import toycrystals_oracle as orc
    sd = orc.default_init_state_dict(1)
    x, t, yc, yk = _inputs(n, 37.0, 0.37, seed=5)
    monkeypatch.delenv("TCS_MAX_CTAS", raising=False)
    m = _fresh_model(sd, 256)
    resident = int(_cabi.lib().tcs_launch_mode(m.engine_handle())) >> 8
    base = {}
    chain(m, sd, x, t, yc, yk, uncond, taps=base)
    del m
    names = [k for k in LAYERS if k.endswith(".act") or k in ("ds1", "ds2", "attn", "us2_conv", "us1_conv", "eps")]
    ran = []
    for cap in (40, 36, 18):
        if cap >= resident:
            continue
        monkeypatch.setenv("TCS_MAX_CTAS", str(cap))
        m = _fresh_model(sd, 256)
        for nm in names:
            got = tap(m, nm, x, t, yc, yk, uncond)
            assert torch.equal(got, base[nm]), f"TCS_MAX_CTAS={cap}: {nm} differs from the default grid " \
                f"(max |diff| {float((got - base[nm]).abs().max()):.3g})"
        ran.append(cap)
        del m
    print(f"resident CTAs {resident}; grids checked {ran}")
    assert ran, "no CTA cap below the device's residency"


# ---- C: GroupNorm shift invariance ----------------------------------------------------------------------------
def _median_sigma(sd, taps, x, t, yc, yk, uncond, name):
    ins, kind, key, gkey, _, C = LAYERS[name]
    yc_r, yk_r, t_r = _rows(x.shape[0], uncond, yc, yk, t)
    if kind == "first":
        w0 = sd[key + ".weight"].cuda().double()[:, :1]
        bias, _ = _embed_with_error(sd, t_r, yc_r, yk_r)
        xx = x.double().reshape(-1, 64, 64, 1).repeat_interleave(2 if uncond else 1, 0)
        v = lb.conv64(xx, w0, None, 3, 1) + bias[:, None, None, :]
    else:
        xin = torch.cat([taps[i].double() for i in ins], -1)
        v, _ = lb.conv_with_error(xin, sd[key + ".weight"].cuda(), sd[key + ".bias"].cuda(), 3, 1)
    return float(lb.group_stats(v)[3].median())


def _shifted(sd, sig, r):
    out = {k: v.clone() for k, v in sd.items()}
    for name in GN_LAYERS:
        key = LAYERS[name][2]
        out[key + ".bias"] += r * sig[name]
    return out


@pytest.mark.parametrize("fused", [True, False])
def test_groupnorm_is_shift_invariant(fused):
    """Add r sigma_g to every bias of each conv followed by GroupNorm (the nine fused ones and the first conv); r <= 16
    must keep the bound of A with the stash rounding written as 2^-11 (|v - mu_g| + sigma_g), and each layer's worst
    per-image rel-L2 within SAFETY times the unshifted one; r = 64 is reported only.
    The fp16 range guard must stay silent.  fused=False: conv -> raw fp32 -> gn_apply (the first conv stays fused)."""
    from toycrystals_b200 import _cabi
    import toycrystals_oracle as orc
    sd = orc.default_init_state_dict(1)
    n, uncond = 16, 1
    x, t, yc, yk = _inputs(n, 1.0, 0.6, seed=3)
    m0 = _fresh_model(sd, 64)
    taps0 = {}
    for nm in GN_LAYERS:
        for i in LAYERS[nm][0]:
            taps0.setdefault(i, tap(m0, i, x, t, yc, yk, uncond))
    sig = {nm: _median_sigma(sd, taps0, x, t, yc, yk, uncond, nm) for nm in GN_LAYERS}
    del m0
    report = []
    for r in (0, 4, 16, 64):
        sd_r = _shifted(sd, sig, r)
        m = _fresh_model(sd_r, 64)
        m._fuse_gn = fused
        h = m.engine_handle()
        res = chain(m, sd_r, x, t, yc, yk, uncond, layers=GN_LAYERS, stash="robust" if fused else None,
                    gate=False, report=report)
        assert int(_cabi.lib().tcs_check(h)) & 1 == 0, f"r={r}: the fp16 range guard fired"
        worst = max(v["worst"] for v in res.values())
        print(f"{'fused' if fused else 'unfused'} r={r}: worst err/bound {worst:.3f}")
        if r == 0:
            base = {nm: v["worst_img_rel"] for nm, v in res.items()}
        if r <= 16:
            for nm, v in res.items():
                assert v["nbad"] == 0, f"r={r}: {v['msg']}"
                # the shift must not cost accuracy in bulk either (an fp16 stash of v + bias: 2.4x at r = 16, 8x at 64)
                assert v["worst_img_rel"] <= lb.SAFETY * base[nm], \
                    f"r={r}: {nm} worst per-image rel-L2 {v['worst_img_rel']:.3e}, unshifted {base[nm]:.3e}"
        del m


def test_groupnorm_shift_at_the_production_batch():
    """r = 16 once at B = 2048 on the fused path."""
    import toycrystals_oracle as orc
    sd = orc.default_init_state_dict(1)
    x, t, yc, yk = _inputs(1024, 1.0, 0.6, seed=3)
    m0 = _fresh_model(sd, 2048)
    taps0 = {}
    for nm in GN_LAYERS:
        for i in LAYERS[nm][0]:
            taps0.setdefault(i, tap(m0, i, x[:64], t[:64], yc[:64], yk[:64], 1))
    sig = {nm: _median_sigma(sd, taps0, x[:64], t[:64], yc[:64], yk[:64], 1, nm) for nm in GN_LAYERS}
    del m0
    sd_r = _shifted(sd, sig, 16)
    m = _fresh_model(sd_r, 2048)
    chain(m, sd_r, x, t, yc, yk, 1, layers=GN_LAYERS, stash="robust")
