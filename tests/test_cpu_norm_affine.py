"""The norm-affine tests have power: every deliberate fault of tests/norm_affine.py moves what the GPU tests compare by
far more than the gate that compares it.  fp64 oracles on the CPU; run with -s for the table of effects and gates.

- Score network: the mutated layer's activation (the first mutated layer in network order, whose input is still the
  unmutated network's) moves by >= 10x the bf16 per-layer gate of test_layers_against_oracle (1.5e-2 rel-L2), in every
  image.  The fp32 gates (2e-5 / 5e-5) are 300x smaller still.
- Prior: eps moves by >= 100x the fp32 gate (1e-4 rel-L2).  Only some faults also clear 10x the bf16 gate (2e-2); the
  test pins which, so that the bf16 prior tests are known to witness those and only those at that margin."""
import os

import pytest
import torch

import latent_prior_oracle as po
import norm_affine as na
import toycrystals_oracle as orc

torch.set_num_threads(max(1, min(8, os.cpu_count() or 1)))
SEED = 7
SCORE_GATE_BF16 = 1.5e-2
PRIOR_GATE = {"fp32": 1e-4, "bf16": 2e-2}
# the prior faults whose eps effect clears 10x the bf16 gate on the inputs below (the others: 0.11 each)
PRIOR_BF16_WITNESSED = {"swap blocks.2.norm <-> blocks.5.norm", "weight <-> bias of out_norm"}


def _sds():
    return {"score": orc.default_init_state_dict(1), "prior": po.prior_default_init(0)}


@pytest.mark.parametrize("net", ["score", "prior"])
def test_affine_state_dict_changes_only_the_norm_layers(net):
    sd = _sds()[net]
    keep = {k: v.clone() for k, v in sd.items()}
    a = na.affine_state_dict(sd, SEED)
    assert list(a) == list(sd)
    assert all(torch.equal(sd[k], keep[k]) for k in sd), "the input state dict was modified"
    layers = na.norm_layers(sd)
    assert len(layers) == (11 if net == "score" else 9)
    nk = set(na.norm_keys(sd))
    for k, v in sd.items():
        assert a[k].dtype == v.dtype and a[k].shape == v.shape, k
        if k not in nk:
            assert torch.equal(a[k].view(torch.uint8), v.view(torch.uint8)), f"{k} is not bit-identical"
    for layer in layers:
        gam, bet = a[layer + ".weight"], a[layer + ".bias"]
        assert torch.equal(sd[layer + ".weight"], torch.ones_like(gam)) and not sd[layer + ".bias"].any()   # PyTorch's init
        # per-channel values that differ from each other, and the three edge channels
        assert gam.unique().numel() >= gam.numel() - 2 and bet.unique().numel() >= bet.numel() - 2, layer
        assert (gam == 0).sum() == 1 and (gam == -1.5).sum() == 1 and (bet.abs() == 2.0).sum() == 1, layer
        assert float(gam.std()) > 0.3 and float(bet.std()) > 0.3, layer
    # no two layers share values, the draw is seeded, and another seed draws other values
    firsts = [tuple(a[layer + ".weight"][:4].tolist()) for layer in layers]
    assert len(set(firsts)) == len(firsts)
    b = na.affine_state_dict(sd, SEED)
    assert all(torch.equal(a[k], b[k]) for k in a)
    c = na.affine_state_dict(sd, SEED + 1)
    assert all(not torch.equal(a[k], c[k]) for k in nk)


@pytest.mark.parametrize("net", ["score", "prior"])
def test_each_mutation_changes_exactly_its_layers(net):
    a = na.affine_state_dict(_sds()[net], SEED)
    names = []
    for name, layers, m in na.mutations(a):
        names.append(name)
        changed = {k.rsplit(".", 1)[0] for k in a if not torch.equal(a[k], m[k])}
        assert changed == set(layers), (name, changed)
        assert list(m) == list(a)
    assert len(names) == (6 if net == "score" else 4) and len(set(names)) == len(names)


def _per_image_rel(a, b):
    return (a - b).flatten(1).norm(dim=1) / b.flatten(1).norm(dim=1)


def test_score_mutations_move_their_layer_beyond_the_bf16_gate():
    sd = na.affine_state_dict(orc.default_init_state_dict(1), SEED)
    g = torch.Generator().manual_seed(21)
    # conditional and unconditional rows at t = 1 (the production chain's time) and t = 0.37
    x = torch.randn((4, 1, 64, 64), generator=g, dtype=torch.float64)
    t = torch.tensor([1.0, 1.0, 0.37, 0.37], dtype=torch.float64)
    yc = torch.tensor([0, 4, 2, 4])
    yk = torch.zeros((4, 4), dtype=torch.float64)
    yk[0, 1], yk[2, 1] = 0.5, 1.0

    def taps_of(s):
        taps = {}
        with torch.no_grad():
            taps["eps"] = orc.score_net(s, orc.DEFAULT_CFG, x, t, yc, yk, taps)
        return taps

    base = taps_of(sd)
    print(f"\n{'score-network fault':58s} {'layer':16s} min image rel-L2  (gate {SCORE_GATE_BF16:g} bf16)  eps")
    for name, layers, m in na.mutations(sd):
        got = taps_of(m)
        nm = na.tap_of(layers[0])
        eff = float(_per_image_rel(got[nm], base[nm]).min())
        eps = float(_per_image_rel(got["eps"], base["eps"]).min())
        print(f"{name:58s} {nm:16s} {eff:.3f} = {eff / SCORE_GATE_BF16:5.1f}x gate          {eps:.3f}")
        assert eff >= 10 * SCORE_GATE_BF16, (name, nm, eff)
        # every layer before the first mutated one is untouched, so the GPU chain's message names that layer
        for other in na.SCORE_NORMS[:na.SCORE_NORMS.index(layers[0])]:
            assert torch.equal(got[na.tap_of(other)], base[na.tap_of(other)]), (name, other)


def test_prior_mutations_move_eps_beyond_the_fp32_gate():
    sd = na.affine_state_dict(po.prior_default_init(0), SEED)
    g = torch.Generator().manual_seed(21)
    n = 64
    z = torch.randn((n, 32), generator=g, dtype=torch.float64) * 2.0
    t = torch.randint(0, 1000, (n,), generator=g)
    yc, yk = orc.condition_grid(n, 4, 4)
    base = po.film_prior(sd, po.PRIOR_CFG, z, t, yc, yk.double())
    assert orc.rel_l2(base, po.film_prior(po.prior_default_init(0), po.PRIOR_CFG, z, t, yc, yk.double())) > 0.1
    witnessed = set()
    print(f"\n{'prior fault':44s} eps rel-L2   x fp32 gate   x bf16 gate")
    for name, layers, m in na.mutations(sd):
        eff = orc.rel_l2(po.film_prior(m, po.PRIOR_CFG, z, t, yc, yk.double()), base)
        print(f"{name:44s} {eff:.3f}      {eff / PRIOR_GATE['fp32']:8.0f}      {eff / PRIOR_GATE['bf16']:6.1f}")
        assert eff >= 100 * PRIOR_GATE["fp32"], (name, eff)
        if eff >= 10 * PRIOR_GATE["bf16"]:
            witnessed.add(name)
    assert witnessed == PRIOR_BF16_WITNESSED, witnessed
