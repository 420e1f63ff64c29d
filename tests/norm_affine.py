"""Per-channel GroupNorm / LayerNorm affines for the tests, and deliberately wrong variants of them.

PyTorch initialises every norm layer with weight = 1 and bias = 0, so under the default inits a gamma or beta read at the
wrong channel, swapped with another layer's or dropped entirely gives exactly the right answer.  affine_state_dict()
replaces every norm layer's weight / bias by seeded per-channel values; mutations() yields the faults such values expose.
Works for the score network's and the prior's state dicts."""
from __future__ import annotations

import torch

SCORE_NORMS = ["down1.net.1", "down1.net.4", "down2.net.1", "down2.net.4", "mid.net.1", "mid.net.4", "attn.norm",
               "up2.net.1", "up2.net.4", "up1.net.1", "up1.net.4"]
GROUPS = 8   # GroupNorm(8, C) in every score-network norm layer


def prior_norms(n_blocks: int = 8):
    return [f"blocks.{i}.norm" for i in range(n_blocks)] + ["out_norm"]


def norm_layers(sd):
    """The norm layers of sd in network order (score network or prior)."""
    if "down1.net.1.weight" in sd:
        return list(SCORE_NORMS)
    n = sum(1 for k in sd if k.startswith("blocks.") and k.endswith(".norm.weight"))
    assert n > 0 and "out_norm.weight" in sd, "neither the score network's nor the prior's state dict"
    return prior_norms(n)


def norm_keys(sd):
    return [f"{layer}.{p}" for layer in norm_layers(sd) for p in ("weight", "bias")]


def tap_of(layer):
    """The score-network activation tap (parity_utils.LAYERS / tcs_debug_layer name) that a norm layer writes."""
    if layer == "attn.norm":
        return "attn"
    block, _, idx = layer.rpartition(".")
    return f"{block}.{int(idx) - 1}.act"


def affine_state_dict(sd, seed):
    """A copy of sd whose norm layers carry gamma = 1 + 0.5 N(0,1), beta = 0.5 N(0,1), one draw per layer, with three edge
    channels forced in every layer: gamma = 0 (the output is SiLU(beta), a constant), gamma = -1.5 and |beta| = 2.
    Every other tensor keeps its values bit for bit."""
    g = torch.Generator().manual_seed(seed)
    out = {k: v.clone() for k, v in sd.items()}
    for layer in norm_layers(sd):
        w = sd[layer + ".weight"]
        C = w.shape[0]
        gamma = 1.0 + 0.5 * torch.randn(C, generator=g, dtype=torch.float64)
        beta = 0.5 * torch.randn(C, generator=g, dtype=torch.float64)
        c0, c1, c2 = torch.randperm(C, generator=g)[:3].tolist()
        gamma[c0] = 0.0
        gamma[c1] = -1.5
        beta[c2] = 2.0 if float(torch.rand(1, generator=g)) < 0.5 else -2.0
        out[layer + ".weight"] = gamma.to(w.dtype)
        out[layer + ".bias"] = beta.to(w.dtype)
    return out


def _copy(sd):
    return {k: v.clone() for k, v in sd.items()}


def _swap(sd, a, b):
    out = _copy(sd)
    for p in ("weight", "bias"):
        out[f"{a}.{p}"], out[f"{b}.{p}"] = sd[f"{b}.{p}"].clone(), sd[f"{a}.{p}"].clone()
    return out


def mutations(sd_affine):
    """Yield (name, mutated layers in network order, state dict) for each deliberate fault of a norm affine:
    (a) two same-width layers' affines swapped, (b) one layer's gamma rolled by one channel (score network: within one
    group, and across every group boundary), (c) weight and bias swapped in one layer, (d) one layer reset to the identity."""
    layers = norm_layers(sd_affine)
    order = {k: i for i, k in enumerate(layers)}
    ordered = lambda *ls: sorted(ls, key=order.__getitem__)
    if layers == SCORE_NORMS:
        swaps = [("down1.net.1", "up1.net.4"), ("mid.net.4", "attn.norm")]
        roll_in, roll_across, wb, ident = "up2.net.1", "down2.net.4", "mid.net.1", "up1.net.1"
    else:
        swaps = [("blocks.2.norm", "blocks.5.norm")]
        roll_in, roll_across, wb, ident = None, "blocks.0.norm", "out_norm", "blocks.3.norm"
    for a, b in swaps:
        assert sd_affine[a + ".weight"].shape == sd_affine[b + ".weight"].shape
        yield f"swap {a} <-> {b}", ordered(a, b), _swap(sd_affine, a, b)
    if roll_in is not None:
        out = _copy(sd_affine)
        w = out[roll_in + ".weight"]
        cpg = w.shape[0] // GROUPS
        g = 3
        w[g * cpg:(g + 1) * cpg] = torch.roll(w[g * cpg:(g + 1) * cpg].clone(), 1)
        yield f"roll gamma by one channel within group {g} of {roll_in}", [roll_in], out
    out = _copy(sd_affine)
    out[roll_across + ".weight"] = torch.roll(sd_affine[roll_across + ".weight"], 1)
    what = "across every group boundary" if layers == SCORE_NORMS else "by one channel"
    yield f"roll gamma {what} of {roll_across}", [roll_across], out
    out = _copy(sd_affine)
    out[wb + ".weight"], out[wb + ".bias"] = sd_affine[wb + ".bias"].clone(), sd_affine[wb + ".weight"].clone()
    yield f"weight <-> bias of {wb}", [wb], out
    out = _copy(sd_affine)
    out[ident + ".weight"] = torch.ones_like(sd_affine[ident + ".weight"])
    out[ident + ".bias"] = torch.zeros_like(sd_affine[ident + ".bias"])
    yield f"identity affine in {ident}", [ident], out
