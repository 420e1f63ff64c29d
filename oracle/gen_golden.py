#!/usr/bin/env python3
"""Generate tests/golden/*.pt from the UNMODIFIED reference, and pin the oracle to it.

Runs only in the build container (needs /root/reference, read-only).  The reference module
imports matplotlib at module scope, which is not installed, so ``oracle/_stubs`` is put on
sys.path first.  For every vector the script asserts that ``oracle/toycrystals_oracle.py``
agrees with the reference BIT-EXACTLY in fp32 on CPU before writing it.

    python oracle/gen_golden.py            # rewrites tests/golden/
"""
from __future__ import annotations

import math
import os
import sys

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, os.path.join(HERE, "_stubs"))
sys.path.insert(0, "/root/reference/src")
sys.path.insert(0, HERE)

import toycrystals.models.sde_score_model as ref  # noqa: E402  (the reference, read-only)
import toycrystals_oracle as orc  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")
CFG = dict(orc.DEFAULT_CFG)
torch.set_num_threads(8)


class _Tape:
    """Replays pre-drawn tensors in place of torch.randn / torch.randn_like."""

    def __init__(self, tensors):
        self.q = list(tensors)

    def randn(self, *a, **k):
        return self.q.pop(0).clone()

    def randn_like(self, x, *a, **k):
        return self.q.pop(0).clone()


def _ref_model(seed):
    torch.manual_seed(seed)
    m = ref.CondUNetTiny(**CFG).eval()
    return m


def _summ(x):
    x = x.detach()
    return dict(shape=list(x.shape), mean=float(x.double().mean()), std=float(x.double().std()),
                absmax=float(x.abs().max()), head=x.flatten()[:8].clone())


def main():
    os.makedirs(OUT, exist_ok=True)
    gen = torch.Generator().manual_seed(1234)

    # ---- weights: oracle's layer-order init == reference default init ------------------
    m0, m1 = _ref_model(0), _ref_model(1)
    sd0, sd1 = orc.default_init_state_dict(0), orc.default_init_state_dict(1)
    for sd, m in ((sd0, m0), (sd1, m1)):
        rsd = m.state_dict()
        assert list(rsd.keys()) == list(sd.keys()), "state-dict key order differs"
        for k in rsd:
            assert torch.equal(rsd[k], sd[k]), k
    wsum = {k: float(v.double().sum()) for k, v in sd0.items()}
    print("weights: oracle init == reference init (seeds 0,1), %d tensors, %d params"
          % (len(sd0), sum(v.numel() for v in sd0.values())))

    # ---- known answers ------------------------------------------------------------------
    sde = ref.VPSDE(0.1, 30.0)
    sch = orc.Schedule(0.1, 30.0)
    tt = torch.tensor([1.0, 0.5, 0.005])
    for f in ("beta", "int_beta", "alpha", "sigma"):
        assert torch.equal(getattr(sde, f)(tt), getattr(sch, f)(tt)), f
    ts = orc.time_grid(300, 0.005)
    th = torch.tensor([[0.0, 0.7, 0.0, 0.0]])
    yq = th.clone(); v = yq[:, 1]; yq[:, 1] = torch.sin(v); yq[:, 2] = torch.cos(v)  # aliasing as in the reference
    kat = dict(
        t=tt, beta=sde.beta(tt), int_beta=sde.int_beta(tt), alpha=sde.alpha(tt), sigma=sde.sigma(tt),
        grid300=ts.clone(), theta_quirk=yq.clone(),
        temb=ref.timestep_embedding(tt, 128), weight_sums=wsum,
    )
    assert torch.equal(kat["temb"], orc.time_features(tt, 128))
    m0c = m0.cond_emb(torch.tensor([2, 4, 0]), torch.tensor([[0, .7, 0, 0], [0, 0, 0, 0], [0, 1.0, 0, 0.]]))
    oc = orc.condition_vector(sd0, CFG, torch.tensor([2, 4, 0]),
                              torch.tensor([[0, .7, 0, 0], [0, 0, 0, 0], [0, 1.0, 0, 0.]]))
    assert torch.equal(m0c, oc)
    kat["cond_vec"] = m0c.detach().clone()
    torch.save(kat, os.path.join(OUT, "kat.pt"))

    # ---- single forwards, with per-layer hooks -------------------------------------------
    n = 3
    x = torch.randn((n, 1, 64, 64), generator=gen)
    y_cat, y_cont = orc.condition_grid(n, 4, 4)
    ry_cat = torch.tensor([i % m0.n_types for i in range(n)], dtype=torch.int64)
    assert torch.equal(ry_cat, y_cat)
    fwd = dict(x=x, y_cat=y_cat, y_cont=y_cont, cases=[])
    for scale, tval in ((1.0, 1.0), (37.0, 0.37), (900.0, 0.005)):
        xs = x * scale  # the random-weight trajectory grows to |x|~1e3; cover that range
        t = torch.full((n,), tval)
        rec = {}
        hooks = []
        for name, mod in m0.named_modules():
            if isinstance(mod, (torch.nn.Conv2d, ref.SelfAttention2d)) and name not in ("attn.qkv", "attn.proj"):
                hooks.append(mod.register_forward_hook(lambda _m, _i, o, name=name: rec.__setitem__(name, o.detach())))
        with torch.no_grad():
            e_c = m0(xs, t, y_cat, y_cont)
            e_u = m0(xs, t, torch.full_like(y_cat, 4), torch.zeros_like(y_cont))
            e_g = ref.predict_eps_cfg(m0, xs, t, y_cat, y_cont, 1.5)
        for h in hooks:
            h.remove()
        taps = {}
        with torch.no_grad():
            o_u = orc.score_net(sd0, CFG, xs, t, torch.full_like(y_cat, 4), torch.zeros_like(y_cont), taps)
            o_c = orc.score_net(sd0, CFG, xs, t, y_cat, y_cont)
            o_g = orc.eps_cfg(sd0, CFG, xs, t, y_cat, y_cont, 1.5)
        assert torch.equal(e_c, o_c) and torch.equal(e_u, o_u) and torch.equal(e_g, o_g), "oracle != reference"
        # the hooks saw the *last* call = unconditional branch inside predict_eps_cfg? no: order is
        # cond call, uncond call, then predict_eps_cfg (uncond, cond) -> last recorded = cond branch.
        taps_c = {}
        with torch.no_grad():
            orc.score_net(sd0, CFG, xs, t, y_cat, y_cont, taps_c)
        lay = {}
        for name, o in rec.items():
            key = {"attn": "attn"}.get(name, name + ".raw" if ".net." in name else name)
            if key == "out":
                continue
            assert torch.equal(o, taps_c[key]), f"tap {name}"
            lay[key] = _summ(o)
        fwd["cases"].append(dict(scale=scale, t=tval, eps_c=e_c, eps_u=e_u, eps_cfg15=e_g, layers=lay))
        print(f"forward t={tval}: oracle == reference bit-exact; |eps| max {float(e_g.abs().max()):.3e}")
    torch.save(fwd, os.path.join(OUT, "score_fwd.pt"))

    # ---- samplers (EMA weights = seed-1 instance), injected noise ---------------------------
    n = 2
    y_cat, y_cont = orc.condition_grid(n, 4, 4)
    out = {}
    for sampler, steps, cfg_s in (("ode", 3, 1.5), ("sde", 4, 1.5), ("sde", 3, 0.0)):
        x_init = torch.randn((n, 1, 64, 64), generator=gen)
        noise = [torch.randn((n, 1, 64, 64), generator=gen) for _ in range(steps)] if sampler == "sde" else []
        tape = _Tape([x_init] + noise)
        real_randn, real_like = torch.randn, torch.randn_like
        eps_log = []
        real_pred = ref.predict_eps_cfg

        def logged(model, x_t, t, yc, yk, guidance_scale):
            e = real_pred(model, x_t, t, yc, yk, guidance_scale)
            eps_log.append(e.clone())
            return e

        torch.randn, torch.randn_like, ref.predict_eps_cfg = tape.randn, tape.randn_like, logged
        try:
            fn = ref.sample_probability_flow_ode if sampler == "ode" else ref.sample_reverse_sde_euler_maruyama
            img = fn(model=m1, sde=sde, y_cat=y_cat, y_cont=y_cont, img_shape=(n, 1, 64, 64),
                     n_steps=steps, guidance_scale=cfg_s, t_end=0.005)
        finally:
            torch.randn, torch.randn_like, ref.predict_eps_cfg = real_randn, real_like, real_pred
        assert not tape.q, "reference consumed a different number of random draws than expected"
        tr = orc.sample(sd1, CFG, sch, y_cat, y_cont, x_init, sampler, steps, cfg_s, 0.005, noise)
        assert torch.equal(tr.image, img), f"{sampler}: oracle image != reference"
        assert len(tr.eps) == len(eps_log) and all(torch.equal(a, b) for a, b in zip(tr.eps, eps_log))
        nfe = (2 * steps + 1) if sampler == "ode" else (steps + 1)
        assert len(eps_log) == nfe
        key = f"{sampler}_s{steps}_cfg{cfg_s}"
        # the image is ((x0_hat + 1) / 2).clamp(0, 1) (tests/parity_utils.image_of); the teacher-forcing traces keep the
        # first sample only, so that the file stays under 1 MB
        out[key] = dict(sampler=sampler, steps=steps, cfg=cfg_s, t_end=0.005, y_cat=y_cat, y_cont=y_cont,
                        x_init=x_init, noise=noise, x0_hat=tr.x0_hat, eps=[e[:1].clone() for e in eps_log],
                        x_in=[x[:1].clone() for x in tr.x_in], t_in=tr.t_in)
        print(f"{key}: oracle == reference bit-exact; NFE={nfe}; |x0_hat| max {float(tr.x0_hat.abs().max()):.3e}; "
              f"image zeros/ones {(img == 0).float().mean():.2f}/{(img == 1).float().mean():.2f}")
    torch.save(out, os.path.join(OUT, "samplers.pt"))
    for f in sorted(os.listdir(OUT)):
        print(f, os.path.getsize(os.path.join(OUT, f)), "bytes")


if __name__ == "__main__":
    main()
