"""CPU self-tests of the per-element layer bounds and their localisation (tests/layer_bounds.py): an emulation of the
fused conv + GroupNorm + SiLU epilogue that rounds where the kernel rounds must pass, and each planted fault must fail
and be reported at the image, CFG row, tile and group where it was planted."""
import pytest
import torch
import torch.nn.functional as F

import layer_bounds as lb

B, H, CIN, COUT, TILE = 4, 32, 8, 16, (16, 16)   # 4 tiles of 16 x 16 per image, 2 channels per group


def _params(seed=0, shift=0.0):
    g = torch.Generator().manual_seed(seed)
    x = F.silu(torch.randn((B, H, H, CIN), generator=g, dtype=torch.float64)).bfloat16().double()
    w = torch.randn((COUT, CIN, 3, 3), generator=g) / 8.5
    b = 0.3 * torch.randn(COUT, generator=g) + shift
    gamma, beta = 1 + 0.3 * torch.randn(COUT, generator=g), 0.2 * torch.randn(COUT, generator=g)
    return x, w, b, gamma, beta


def _terms(x, w, halo_bug_image=None):
    """The K = cin 9 products of each output, exact (bf16 x bf16 fits fp32): [K, B, H, W, Cout]."""
    xp = F.pad(x.permute(0, 3, 1, 2), (1, 1, 1, 1), mode="circular")
    if halo_bug_image is not None:    # left halo column wraps to W-2 instead of W-1 in one image
        xp[halo_bug_image, :, :, 0] = xp[halo_bug_image, :, :, H - 1]
    wq = w.bfloat16().double()
    out = []
    for ky in range(3):
        for kx in range(3):
            win = xp[:, :, ky:ky + H, kx:kx + H]                      # [B, Cin, H, W]
            for ci in range(CIN):
                out.append(win[:, ci, :, :, None] * wq[None, None, None, :, ci, ky, kx])
    return torch.stack(out)


def _emulate(x, w, b, gamma, beta, drop=None, halo_bug_image=None, stats_from=None, seed=1):
    """fp32 sum of the products in a shuffled order -> + bias -> fp16 stash of v - K_g -> fp32 group sums ->
    mean / var in fp64 -> fp32 affine -> SiLU = h + h tanh(h) in fp32 -> bf16."""
    T = _terms(x, w, halo_bug_image)
    if drop is not None:             # (image, ty, tx, tap): one tap's products missing in one tile
        img, ty, tx, tp = drop
        T[tp * CIN:(tp + 1) * CIN, img, ty * 16:(ty + 1) * 16, tx * 16:(tx + 1) * 16] = 0
    perm = torch.randperm(T.shape[0], generator=torch.Generator().manual_seed(seed))
    acc = torch.zeros(T.shape[1:], dtype=torch.float32)
    for i in perm:
        acc = acc + T[i].float()
    t = acc + b.float()
    kg = b.float().reshape(8, -1).mean(1).repeat_interleave(COUT // 8)
    v = t - kg
    stash = v.half().float()
    vg = v.reshape(B, -1, 8, COUT // 8)
    s1, s2 = vg.sum((1, 3)).double(), (vg * vg).sum((1, 3)).double()
    if stats_from is not None:       # image a normalised with the statistics of image b
        a, bb = stats_from
        s1[a], s2[a] = s1[bb], s2[bb]
    n = H * H * (COUT // 8)
    mean = s1 / n
    rstd = (1.0 / torch.sqrt((s2 / n - mean * mean).clamp_min(0) + lb.GN_EPS)).float()
    ex = lambda z: z[:, None, None, :, None].expand(B, 1, 1, 8, COUT // 8).reshape(B, 1, 1, COUT)
    sc = ex(rstd) * gamma.float()
    sh = beta.float() - ex(mean.float()) * sc
    h = 0.5 * (stash * sc + sh)
    return (h + h * torch.tanh(h)).bfloat16().double()


def _reference(x, w, b, gamma, beta, stash="fused"):
    r, e = lb.conv_with_error(x, w, b, 3, 1)
    return lb.gn_silu_with_bound(r, e, gamma, beta, stash=stash, bias=b)


def _check(got, ref, bound, rows=None):
    return lb.check_layer("emulated", got, ref, bound, TILE, COUT // 8, rows=rows, gate=False)


@pytest.mark.parametrize("shift", [0.0, 20.0])
def test_faithful_emulation_passes(shift):
    """Bias shifts of ~16 group standard deviations included: the shifted stash keeps its bound."""
    p = _params(shift=shift)
    ref, bound = _reference(*p)
    res = _check(_emulate(*p), ref, bound)
    assert res["nbad"] == 0, res.get("msg")
    assert res["worst"] > 1e-3          # the bound is not vacuous
    _, bound_r = _reference(*p, stash="robust")
    assert _check(_emulate(*p), ref, bound_r)["nbad"] == 0


def test_unshifted_stash_fails_the_shift_robust_bound():
    """An fp16 stash of v + bias itself (no K_g) at a shift of 64 sigma: caught by the shift-robust bound."""
    x, w, b, gamma, beta = _params(shift=0.0)
    r0, _ = lb.conv_with_error(x, w, b, 3, 1)
    shift = 64 * float(lb.group_stats(r0)[3].median())
    b = b + shift
    ref, bound = _reference(x, w, b, gamma, beta, stash="robust")
    good = _emulate(x, w, b, gamma, beta)
    assert _check(good, ref, bound)["nbad"] == 0
    r, _ = lb.conv_with_error(x, w, b, 3, 1)
    mu, sig, _, _ = lb.group_stats(r)
    bad = F.silu((r.float().half().double() - mu) / sig * gamma.double() + beta.double()).bfloat16().double()
    assert _check(bad, ref, bound)["nbad"] > 0


def test_dropped_tap_in_one_tile_is_located():
    p = _params()
    ref, bound = _reference(*p)
    res = _check(_emulate(*p, drop=(1, 1, 0, 4)), ref, bound)
    # the missing products also move image 1's group statistics, so its other tiles may fail too; the worst is the tile
    assert {t[0] for t in res["tiles"]} == {1}, res
    assert "image 1, tile (1,0)" in res["msg"], res["msg"]


def test_tile_from_the_neighbouring_image_is_located():
    p = _params()
    ref, bound = _reference(*p)
    got = _emulate(*p)
    got[2, 0:16, 16:32] = got[3, 0:16, 16:32]
    res = _check(got, ref, bound)
    assert res["tiles"] == [(2, 0, 1)], res


def test_halo_off_by_one_at_the_image_edge_is_located():
    p = _params()
    ref, bound = _reference(*p)
    res = _check(_emulate(*p, halo_bug_image=3), ref, bound)
    # the worst element is in the first pixel column, where the halo is read (the statistics spread the rest over image 3)
    assert {t[0] for t in res["tiles"]} == {3} and res["at"][2] == 0, res


def test_neighbour_statistics_are_located():
    p = _params()
    ref, bound = _reference(*p)
    res = _check(_emulate(*p, stats_from=(2, 1)), ref, bound)
    assert res["nbad"] > 0 and {t[0] for t in res["tiles"]} == {2}, res


def test_swapped_group_affine_is_located():
    x, w, b, gamma, beta = _params()
    ref, bound = _reference(x, w, b, gamma, beta)
    perm = torch.arange(COUT)
    perm[6:8], perm[10:12] = torch.arange(10, 12), torch.arange(6, 8)     # groups 3 and 5
    res = _check(_emulate(x, w, b, gamma[perm], beta[perm]), ref, bound)
    assert res["nbad"] > 0 and set(res["groups"]) <= {3, 5}, res
    assert "(group 3)" in res["msg"] or "(group 5)" in res["msg"]


def test_cfg_rows_swapped_are_located():
    """The output conv in pair mode: rows 2i (conditional) and 2i+1 (unconditional) swapped for image 1."""
    g = torch.Generator().manual_seed(4)
    x = torch.randn((2 * B, H, H, COUT), generator=g, dtype=torch.float64).bfloat16().double()
    w, b = torch.randn((1, COUT, 3, 3), generator=g) / 12, torch.tensor([0.1])
    ref, bound = lb.eps_cfg_with_bound(x, w, b, 1.5)
    e = lb.conv64(x, w.bfloat16().double(), b.double(), 3, 1).float()
    got = (e[1::2] + 1.5 * (e[0::2] - e[1::2])).double()
    assert lb.check_layer("eps", got, ref, bound, (2, 64), 1, gate=False)["nbad"] == 0
    got[1] = (e[2] + 1.5 * (e[3] - e[2])).double()
    res = lb.check_layer("eps", got, ref, bound, (2, 64), 1, gate=False)
    assert res["nbad"] > 0 and {t[0] for t in res["tiles"]} == {1}, res
    with pytest.raises(AssertionError, match=r"eps: .* at image 1, tile"):
        lb.check_layer("eps", got, ref, bound, (2, 64), 1)
