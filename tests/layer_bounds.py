"""Per-element error bounds of the layers of the bf16 score pass, and the localisation of a violation.

Each bound is the sum of the roundings the kernel performs, evaluated on an fp64 reference of the layer computed from the
very bf16 values the kernel read, so errors never compound from layer to layer.  Unit roundoffs: bf16 2^-8, fp16 2^-11,
fp32 2^-24.  The only free constant is SAFETY, applied once to the whole bound.  Line numbers refer to csrc/.

Works on CPU or CUDA tensors (the GPU chain test runs it on the device in float64)."""
from __future__ import annotations

import torch
import torch.nn.functional as F

U_BF16, U_F16, U_F32 = 2.0 ** -8, 2.0 ** -11, 2.0 ** -24
U_TANH = 2.0 ** -10.987     # tanh.approx.f32: maximum relative error stated by the PTX ISA
GN_EPS = 1e-5
SAFETY = 2.0
SILU_SLOPE = 1.1            # max |d silu / dy| = 1.0998
# depth of the fp32 GroupNorm summation trees, beyond the channels of a group that one lane adds (conv_tc.cu:915-918):
# 5 butterfly levels (:944-957), 8 epilogue warps (:971), ceil(G / 2) <= 8 exchange words per lane (:999) and one
# shuffle (:1002); the unfused EPI_RAW_STATS path (:1094-1105) stops after the butterflies and combines in fp64
GN_TREE_EXTRA = 5 + 8 + 8 + 1


def conv64(x, w, b, k, s):
    """Circular conv (pad 1 for 3x3 and 4x4/s2, none for 1x1) on NHWC float64."""
    x = x.permute(0, 3, 1, 2)
    if k > 1:
        x = F.pad(x, (1, 1, 1, 1), mode="circular")
    return F.conv2d(x, w, b, stride=s).permute(0, 2, 3, 1)


def conv_with_error(x, w, b, k, s, dx=None):
    """Reference of a tcgen05 conv with its pre-rounding error bound.  x: the bf16 activations the kernel read (float64),
    w / b: fp32 parameters; the weights are packed as bf16, the bias is read in fp32.  bf16 x bf16 products are exact in
    fp32, the K = cin k^2 products and the bias are summed in fp32: |err| <= K u32 S with S = conv(|x|, |w|) + |b|.
    dx: optional elementwise bound of an error already in x (propagated through |w|)."""
    wq = w.to(x.device).bfloat16().double()
    bd = b.to(x.device).double()
    r = conv64(x, wq, bd, k, s)
    S = conv64(x.abs(), wq.abs(), bd.abs(), k, s)
    e = (w.shape[1] * k * k + 1) * U_F32 * S
    if dx is not None:
        e = e + conv64(dx, wq.abs(), None, k, s)
    return r, e


def bf16_output(r, e):
    """One rounding to bf16 of a value within e of r."""
    return U_BF16 * r.abs() + (1.0 + U_BF16) * e


def group_stats(t):
    """Per (image, group) mean and std (biased, + eps) of an NHWC tensor, expanded to [B, 1, 1, C]."""
    B, H, W, C = t.shape
    tg = t.reshape(B, H * W, 8, C // 8)
    mu = tg.mean(dim=(1, 3))
    var = tg.var(dim=(1, 3), unbiased=False)
    ex = lambda g: g[:, None, None, :, None].expand(B, 1, 1, 8, C // 8).reshape(B, 1, 1, C)
    return ex(mu), ex(torch.sqrt(var + GN_EPS)), mu, torch.sqrt(var)


def group_mean(a, C):
    """Mean over the pixels and channels of each (image, group), expanded like group_stats."""
    B = a.shape[0]
    g = a.reshape(B, -1, 8, C // 8).mean(dim=(1, 3))
    return g[:, None, None, :, None].expand(B, 1, 1, 8, C // 8).reshape(B, 1, 1, C)


def gn_silu_with_bound(t, e_t, gamma, beta, stash="fused", bias=None, stats_u=U_F32):
    """GroupNorm(8) + SiLU of the pre-norm values t (fp64, NHWC) whose computed form is within e_t of t.

    stash = "fused": the fused epilogue stores t - K_g as fp16 (conv_tc.cu:919-920), K_g = the mean of the group's conv
    biases (:291-305); "robust": the same with the rounding written as 2^-11 (|t - mu_g| + sigma_g), i.e. what a stash
    independent of the group mean achieves; None: the pre-norm values stay fp32 (unfused path, first conv).
    stats_u: unit roundoff of the statistics sums (fp32 in conv_tc / gn_finalize; the first conv's are fp64).
    Returns (r, bound) with r the fp64 SiLU output and bound the bf16 output bound."""
    B, H, W, C = t.shape
    cpg = C // 8
    ga = gamma.to(t.device).double().reshape(1, 1, 1, C)
    be = beta.to(t.device).double().reshape(1, 1, 1, C)
    mu, sig, _, _ = group_stats(t)
    y = (t - mu) / sig * ga + be
    r = F.silu(y)
    if stash == "fused":
        kg = bias.to(t.device).double().reshape(8, cpg).mean(dim=1).repeat_interleave(cpg).reshape(1, 1, 1, C)
        e_st = U_F16 * (t - kg).abs()
    elif stash == "robust":
        kg = mu
        e_st = U_F16 * ((t - mu).abs() + sig)
    else:
        kg = torch.zeros_like(mu)
        e_st = torch.zeros_like(t)
    # statistics: fp32 sums of (t - K_g) and (t - K_g)^2 over H W cpg terms through a tree of depth cpg + GN_TREE_EXTRA
    # (conv_tc.cu:915-918, 944-1002; kernels_simt.cu:362-383), then var = E[v^2] - mean^2 (conv_tc.cu:1007-1008), plus
    # what the accumulation error of t itself moves them
    D = cpg + GN_TREE_EXTRA
    a = (t - kg).abs()
    d_mu = D * stats_u * group_mean(a, C) + group_mean(e_t, C)
    d_var = D * stats_u * group_mean(a * a, C) + 2.0 * (mu - kg).abs() * d_mu + 2.0 * group_mean((t - mu).abs() * e_t, C)
    sc = ga.abs() / sig
    e_y = sc * (e_t + e_st + d_mu + (t - mu).abs() * d_var / (2.0 * sig * sig))
    # fp32 affine table and application (conv_tc.cu:1015-1018, 1052-1053; kernels_simt.cu:444): scale = rstd gamma,
    # shift = beta - mean scale, v scale + shift, rsqrtf (2 ulp)
    e_y = e_y + 4.0 * U_F32 * (sc * (a + (mu - kg).abs()) + be.abs()) + 2.0 ** -22 * (y - be).abs()
    # SiLU = h + h tanh.approx(h), h = y / 2 (conv_tc.cu:1054-1055; kernels_simt.cu:385-391): |h tanh h| <= |y| / 2
    e = SILU_SLOPE * e_y + 0.5 * y.abs() * U_TANH + 2.0 * U_F32 * (r.abs() + y.abs())
    return r, bf16_output(r, e)


def upsample_rounding(x):
    """nn.Upsample(x2, bilinear) of the bf16 tensor x (fp64, NHWC) as the UPS conv forms it: a four-term fp32 blend
    rounded once to bf16 (conv_tc.cu, UPS blending warps).  Returns (up, d): up = bf16(fp64 blend), d = an elementwise
    bound of |kernel value - up|: nonzero only where the fp32 blend error (4 u32 of the blend of |x|) may cross a bf16
    rounding boundary, and then one bf16 spacing."""
    up64 = F.interpolate(x.permute(0, 3, 1, 2), scale_factor=2, mode="bilinear", align_corners=False)
    upa = F.interpolate(x.abs().permute(0, 3, 1, 2), scale_factor=2, mode="bilinear", align_corners=False)
    lo, hi = up64 - 4 * U_F32 * upa, up64 + 4 * U_F32 * upa
    up = up64.float().bfloat16().double()
    straddle = lo.float().bfloat16() != hi.float().bfloat16()
    d = torch.where(straddle, 2.0 * U_BF16 * upa + 8 * U_F32 * upa, torch.zeros_like(up))
    return up.permute(0, 2, 3, 1), d.permute(0, 2, 3, 1)


def eps_cfg_with_bound(x, w, b, guidance):
    """The 96 -> 1 output conv in pair mode: conditional row 2i, unconditional row 2i+1, combined in fp32 as
    e_u + g (e_c - e_u) (conv_tc.cu:854).  Returns (eps [n,64,64,1] fp64, bound)."""
    r, e = conv_with_error(x, w, b, 3, 1)
    rc, ru, ec, eu = r[0::2], r[1::2], e[0::2], e[1::2]
    out = ru + guidance * (rc - ru)
    bound = (1 + guidance) * ec + guidance * eu + \
        U_F32 * (rc - ru).abs() * (1 + guidance) + 2.0 * U_F32 * (out.abs() + (guidance * (rc - ru)).abs())
    return out, bound


# ---- localisation ------------------------------------------------------------------------------------------------
def check_layer(name, got, ref, bound, tile, cpg, rows=None, safety=SAFETY, gate=True, b0=0):
    """Compare got with ref element by element against safety * bound (all NHWC).  tile = (rows, cols) of the CTA tile of
    the kernel that wrote the layer; cpg = channels per GroupNorm group (or per reported channel block); rows = "cfg"
    when batch rows alternate conditional / unconditional.  Returns a dict of the worst err / bound, the worst per-image
    rel-L2 and the violating (image row, tile) set; raises AssertionError naming them when gate is set.  b0: batch row of
    got[0] (the tensors may be a chunk of the batch)."""
    err = (got.double() - ref).abs()
    q = err / (safety * bound).clamp_min(1e-300)
    B, H, W, C = ref.shape
    bad = q > 1.0
    per_img = (err.flatten(1).norm(dim=1) / ref.flatten(1).norm(dim=1).clamp_min(1e-300))
    res = {"worst": float(q.max()), "worst_img_rel": float(per_img.max()), "nbad": int(bad.sum()), "tiles": [],
           "groups": []}
    if res["nbad"] == 0:
        return res
    th, tw = tile
    idx = bad.nonzero()
    tiles = torch.stack([idx[:, 0] + b0, idx[:, 1] // th, idx[:, 2] // tw], dim=1).unique(dim=0).tolist()
    res["tiles"] = [tuple(t) for t in tiles]
    res["groups"] = sorted(set((idx[:, 3] // cpg).tolist()))
    flat = int(q.flatten().argmax())
    b, rem = divmod(flat, H * W * C)
    y, rem = divmod(rem, W * C)
    x, c = divmod(rem, C)
    b += b0
    res["at"] = (b, y, x, c)
    if rows == "cfg":
        who = f"image {b // 2} ({'unconditional' if b % 2 else 'conditional'} row {b})"
    else:
        who = f"image {b}"
    shown = ", ".join(f"b{t[0]}:({t[1]},{t[2]})" for t in res["tiles"][:8])
    msg = (f"{name}: {res['nbad']} elements over the bound in {len(res['tiles'])} tile(s); worst err/bound "
           f"{res['worst']:.3g} at {who}, tile ({y // th},{x // tw}) = rows {y // th * th}-{y // th * th + th - 1} cols "
           f"{x // tw * tw}-{x // tw * tw + tw - 1} of the {th}x{tw}-pixel CTA tiles, pixel ({y},{x}), channel {c} "
           f"(group {c // cpg}); got {float(got.flatten()[flat]):.6g} want {float(ref.flatten()[flat]):.6g} bound "
           f"{float(safety * bound.flatten()[flat]):.3g}; violating tiles (row:(ty,tx)) {shown}")
    res["msg"] = msg
    if gate:
        raise AssertionError(msg)
    return res


def check_branch(name, got, ref, x, c_elem, rel_gate, rows=None, b0=0):
    """Attention block: per image, the branch (out - x) within rel_gate rel-L2 of the reference branch, and per element
    |got - r| <= 2^-8 |r| + c_elem rms_image(r - x)."""
    br = (ref - x)
    rel = (got.double() - x - br).flatten(1).norm(dim=1) / br.flatten(1).norm(dim=1)
    rms = br.flatten(1).pow(2).mean(dim=1).sqrt().reshape(-1, 1, 1, 1)
    bound = U_BF16 * ref.abs() + c_elem * rms
    worst_rel = float(rel.max())
    assert worst_rel <= rel_gate, f"{name}: batch row {b0 + int(rel.argmax())} branch rel-L2 {worst_rel:.3e} > {rel_gate}"
    res = check_layer(name, got, ref, bound, (16, 16), ref.shape[-1] // 8, rows=rows, safety=1.0, b0=b0)
    res["worst_img_rel"] = worst_rel
    return res
