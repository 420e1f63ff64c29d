"""CPU suite (-m "not gpu"): the oracle against the committed golden vectors and known answers,
host logic of the shim, and the C-ABI library surface (no compute calls)."""
import ctypes as C
import math
import os
import re

import numpy as np
import pytest
import torch

import toycrystals_oracle as orc
import philox_ref
from toycrystals_b200 import _cabi
from toycrystals_b200.models import sde_score_model as shim

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
torch.set_num_threads(max(1, min(8, os.cpu_count() or 1)))


def _load(golden_dir, name):
    return torch.load(os.path.join(golden_dir, name), weights_only=False)


# ---- known answers (SURVEY section 4) -------------------------------------------------------------
def test_schedule_known_answers(golden_dir):
    kat = _load(golden_dir, "kat.pt")
    s = orc.Schedule(0.1, 30.0)
    for f in ("beta", "int_beta", "alpha", "sigma"):
        assert torch.equal(getattr(s, f)(kat["t"]), kat[f])
    assert float(s.beta(torch.tensor(1.0))) == pytest.approx(30.0)
    assert float(s.alpha(torch.tensor(1.0))) == pytest.approx(5.394e-4, rel=1e-3)
    assert float(s.sigma(torch.tensor(0.005))) == pytest.approx(0.029553, rel=1e-4)


def test_time_grid_known_answers(golden_dir):
    kat = _load(golden_dir, "kat.pt")
    ts = orc.time_grid(300, 0.005)
    assert torch.equal(ts, kat["grid300"])
    assert float(ts[0]) == 1.0 and float(ts[-1]) == pytest.approx(0.005)
    assert float(ts[1]) == pytest.approx(0.99337769, abs=1e-7)
    assert float(ts[-1] - ts[-2]) == pytest.approx(-1.1056e-5, rel=1e-3)


def test_theta_aliasing_quirk(golden_dir):
    kat = _load(golden_dir, "kat.pt")
    q = kat["theta_quirk"][0]
    assert q[1] == pytest.approx(math.sin(0.7)) and q[2] == pytest.approx(math.cos(math.sin(0.7)))
    assert abs(float(q[2]) - math.cos(0.7)) > 1e-2  # NOT cos(theta)
    sd = orc.default_init_state_dict(0)
    out = orc.condition_vector(sd, orc.DEFAULT_CFG, torch.tensor([2, 4, 0]),
                               torch.tensor([[0, .7, 0, 0], [0, 0, 0, 0], [0, 1.0, 0, 0.]]))
    assert torch.equal(out, kat["cond_vec"])
    assert torch.equal(orc.time_features(kat["t"], 128), kat["temb"])


def test_default_init_matches_golden_weight_sums(golden_dir):
    kat = _load(golden_dir, "kat.pt")
    sd = orc.default_init_state_dict(0)
    assert len(sd) == 71 and sum(v.numel() for v in sd.values()) == 3_314_257
    for k, v in sd.items():
        assert float(v.double().sum()) == pytest.approx(kat["weight_sums"][k], rel=1e-12, abs=1e-12)
    # the shim's parameter container initialises identically and has the same layout
    torch.manual_seed(0)
    m = shim.CondUNetTiny(**orc.DEFAULT_CFG)
    msd = m.state_dict()
    assert list(msd.keys()) == list(sd.keys())
    assert all(torch.equal(msd[k], sd[k]) for k in sd)


# ---- oracle vs golden vectors generated from the reference ------------------------------------------
def test_oracle_forward_matches_reference_golden(golden_dir):
    g = _load(golden_dir, "score_fwd.pt")
    sd = orc.default_init_state_dict(0)
    case = g["cases"][0]
    x = g["x"] * case["scale"]
    t = torch.full((x.shape[0],), case["t"])
    with torch.no_grad():
        e = orc.eps_cfg(sd, orc.DEFAULT_CFG, x, t, g["y_cat"], g["y_cont"], 1.5)
    assert orc.rel_l2(e, case["eps_cfg15"]) < 1e-6


def test_oracle_sampler_matches_reference_golden(golden_dir):
    sd = orc.default_init_state_dict(1)
    for key, g in _load(golden_dir, "samplers.pt").items():
        tr = orc.sample(sd, orc.DEFAULT_CFG, orc.Schedule(0.1, 30.0), g["y_cat"], g["y_cont"], g["x_init"], g["sampler"],
                        g["steps"], g["cfg"], g["t_end"], g["noise"])
        assert orc.rel_l2(tr.x0_hat, g["x0_hat"]) < 1e-5, key
        assert len(tr.eps) == len(g["eps"]) == (2 * g["steps"] + 1 if g["sampler"] == "ode" else g["steps"] + 1), key
        k = g["eps"][0].shape[0]          # the stored traces hold the first k samples of the run
        for e, e_ref in zip(tr.eps, g["eps"]):
            assert orc.rel_l2(e[:k], e_ref) < 1e-5, key


def test_oracle_zero_out_conv_is_linear_recurrence():
    """With the out conv zeroed eps == 0 and the samplers reduce to a scalar recurrence in x."""
    sd = orc.default_init_state_dict(0)
    sd["out.weight"].zero_(); sd["out.bias"].zero_()
    n, steps = 1, 5
    y_cat, y_cont = orc.condition_grid(n, 4, 4)
    x0 = torch.randn((n, 1, 64, 64), generator=torch.Generator().manual_seed(3))
    sch = orc.Schedule(0.1, 30.0)
    tr = orc.sample(sd, orc.DEFAULT_CFG, sch, y_cat, y_cont, x0, "ode", steps, 1.5, 0.005)
    ts = orc.time_grid(steps, 0.005).double()
    f = 1.0
    for i in range(steps):
        b0, b1, dt = float(sch.beta(ts[i])), float(sch.beta(ts[i + 1])), float(ts[i + 1] - ts[i])
        d0 = -0.5 * b0
        d1 = -0.5 * b1 * (1 + d0 * dt)
        f = f * (1 + 0.5 * (d0 + d1 / 1.0) * dt) if False else f + 0.5 * (d0 * f + d1 * f) * dt
    a = float(sch.alpha(ts[-1]))
    assert orc.rel_l2(tr.x0_hat, x0 * (f / a)) < 1e-4


def test_condition_grid_and_validation():
    y_cat, y_cont = orc.condition_grid(36, 4, 4)
    assert y_cat.tolist() == [i % 4 for i in range(36)]
    assert torch.equal(y_cont[:, 1], torch.linspace(0.0, math.pi / 3.0, 36))
    assert float(y_cont[:, [0, 2, 3]].abs().max()) == 0.0
    sd = orc.default_init_state_dict(0)
    with pytest.raises(ValueError):
        orc.sample(sd, orc.DEFAULT_CFG, orc.Schedule(), y_cat[:1], y_cont[:1], torch.zeros(1, 1, 64, 64), "ode", 1, 0.0, 1.5)
    with pytest.raises(ValueError):
        orc.sample(sd, orc.DEFAULT_CFG, orc.Schedule(), y_cat[:1], y_cont[:1], torch.zeros(1, 1, 64, 64), "xx", 1, 0.0, 0.1)


def test_philox_known_answer_vectors():
    # Random123 kat_vectors, philox4x32-10
    r = philox_ref.philox4x32_10([0], [0], [0], [0], 0, 0)
    assert [int(v[0]) for v in r] == [0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8]
    r = philox_ref.philox4x32_10([0xffffffff], [0xffffffff], [0xffffffff], [0xffffffff], 0xffffffff, 0xffffffff)
    assert [int(v[0]) for v in r] == [0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd]
    r = philox_ref.philox4x32_10([0x243f6a88], [0x85a308d3], [0x13198a2e], [0x03707344], 0xa4093822, 0x299f31d0)
    assert [int(v[0]) for v in r] == [0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1]
    z = philox_ref.normal_image(1234, 7, 0)
    assert abs(z.mean()) < 0.06 and abs(z.std() - 1.0) < 0.04


# ---- C-ABI surface ---------------------------------------------------------------------------------
def test_library_exports_every_declared_symbol():
    hdr = "".join(re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", f)).read(), flags=re.S)
                  for f in ("tcs.h", "tcs_prior.h"))
    declared = set(re.findall(r"\b(tcs_[a-z0-9_]+)\s*\(", hdr))
    assert declared, "no declarations parsed"
    L = _cabi.lib()
    for name in declared:
        assert hasattr(L, name), f"libtcs.so does not export {name}"
    assert declared == set(_cabi.SIGNATURES), (declared ^ set(_cabi.SIGNATURES))
    assert b"sm_100a" in L.tcs_build_info()


def test_host_schedule_matches_torch_fp32():
    L = _cabi.lib()
    for steps, t_end in ((300, 0.005), (3, 0.005), (4, 0.005), (200, 1e-3), (7, 0.3)):
        buf = (C.c_float * (steps + 1))()
        assert L.tcs_time_grid_host(steps, t_end, buf) == 0
        ts = orc.time_grid(steps, t_end)
        mine = np.frombuffer(buf, dtype=np.float32)
        # torch's CPU linspace is vectorised per SIMD width (base + lane*step in the second half), its
        # CUDA linspace is the scalar formula libtcs uses: they agree to 1 ulp of u, not bit for bit.
        np.testing.assert_allclose(mine, ts.numpy(), rtol=2e-6, atol=0)
        assert mine[0] == ts.numpy()[0] and mine[-1] == ts.numpy()[-1]
        s = orc.Schedule(0.1, 30.0)
        for i in (0, steps // 2, steps):
            b, a, g = C.c_float(), C.c_float(), C.c_float()
            L.tcs_schedule_host(0.1, 30.0, float(ts[i]), C.byref(b), C.byref(a), C.byref(g))
            assert b.value == float(s.beta(ts[i]))
            assert a.value == pytest.approx(float(s.alpha(ts[i])), rel=3e-7)
            assert g.value == pytest.approx(float(s.sigma(ts[i])), rel=3e-7)
    assert L.tcs_nfe(_cabi.SAMPLER_ODE, 300) == 601 and L.tcs_nfe(_cabi.SAMPLER_SDE, 300) == 301


def test_create_fails_loudly_without_gpu_or_on_bad_config():
    L = _cabi.lib()
    cfg = _cabi.TcsConfig()
    L.tcs_default_config(C.byref(cfg))
    assert (cfg.n_types, cfg.base_ch, cfg.beta_max) == (4, 96, 30.0)
    h = C.c_void_p()
    cfg.base_ch = 32
    assert L.tcs_create(C.byref(h), C.byref(cfg)) == _cabi.ERR_UNSUPPORTED
    assert b"base_ch=96" in L.tcs_last_error()
    if not torch.cuda.is_available():
        cfg.base_ch = 96
        assert L.tcs_create(C.byref(h), C.byref(cfg)) == _cabi.ERR_CUDA
        assert b"no CPU fallback" in L.tcs_last_error()


def test_shim_has_no_cpu_path_and_keeps_reference_errors():
    m = shim.CondUNetTiny(**orc.DEFAULT_CFG)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m(torch.zeros(1, 1, 64, 64), torch.zeros(1), torch.zeros(1, dtype=torch.long), torch.zeros(1, 4))
    y_cat, y_cont = orc.condition_grid(2, 4, 4)
    with pytest.raises(ValueError, match=r"t_end must be in \(0,1\)"):
        shim.sample_probability_flow_ode(m, shim.VPSDE(), y_cat, y_cont, (2, 1, 64, 64), t_end=1.0)
    with pytest.raises(ValueError, match="requires y_cont_dim >= 3"):
        shim.CondUNetTiny(4, 2)
    with pytest.raises(ValueError, match="Unknown sampler"):
        shim.save_sde_samples(m, shim.VPSDE(), "/tmp/x.png", torch.device("cpu"), sampler="heun")
    s, o = shim.VPSDE(0.1, 30.0), orc.Schedule(0.1, 30.0)
    t = torch.tensor([1.0, 0.3, 0.005])
    for f in ("beta", "int_beta", "alpha", "sigma"):
        assert torch.equal(getattr(s, f)(t), getattr(o, f)(t))
    assert shim.VPSDE().beta_max == 20.0


def test_cli_checkpoint_errors(tmp_path):
    import importlib.util
    spec = importlib.util.spec_from_file_location(
        "tcs_cli", os.path.join(ROOT, "vae-diffusion-toy-crystals_b200", "scripts", "sample_sde_score_model.py"))
    cli = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(cli)
    assert cli._infer_ckpt_path("o", "last").endswith("o/checkpoints/sde_score_model_last.pt")
    assert cli._infer_ckpt_path("o", "x/y.pt") == "x/y.pt"
    with pytest.raises(ValueError):
        cli._infer_ckpt_path("o", "newest")
    with pytest.raises(FileNotFoundError, match="Checkpoint not found"):
        cli.main(["--out-dir", str(tmp_path), "--device", "cuda"])
    ck = orc.make_checkpoint()
    assert set(ck) == {"epoch_next", "model", "opt", "loss_hist", "config", "ema"}
    assert ck["config"]["beta_max"] == 30.0 and len(ck["model"]) == 71


def test_adopt_accepts_any_module_with_the_reference_state_dict():
    class Foreign(torch.nn.Module):     # stands in for the training script's reference model / ema_model
        def __init__(self, sd):
            super().__init__()
            self.inner = shim.CondUNetTiny(**orc.DEFAULT_CFG)
            self.inner.load_state_dict(sd)

        def state_dict(self, *a, **k):
            return self.inner.state_dict(*a, **k)

    sd = orc.default_init_state_dict(1)
    f = Foreign(sd)
    fast = shim.adopt(f)
    assert isinstance(fast, shim.CondUNetTiny) and fast._arch == {**orc.DEFAULT_CFG}
    assert all(torch.equal(v, sd[k]) for k, v in fast.state_dict().items())
    assert shim.adopt(f) is fast            # cached while the parameters are unchanged
    with torch.no_grad():
        f.inner.out.bias.add_(1.0)          # an optimiser / EMA step
    again = shim.adopt(f)
    assert float(again.state_dict()["out.bias"]) == pytest.approx(float(sd["out.bias"]) + 1.0, rel=1e-6)
    with pytest.raises(TypeError, match="does not carry"):
        shim.adopt(torch.nn.Linear(2, 2))


# ---- round 2: build freshness and the staged reference ------------------------------------------------
def test_library_carries_the_hash_of_the_sources_in_the_tree():
    """A prebuilt libtcs.so that does not match csrc/ + include/ must never be used silently (round-1 review #11)."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("tcs_build", os.path.join(ROOT, "vae-diffusion-toy-crystals_b200", "build.py"))
    bm = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bm)
    info = _cabi.lib().tcs_build_info().decode()
    assert f"TCS_SRC_HASH={bm.source_hash()}" in info, f"stale libtcs.so: {info}; run python __graft_entry__.py build"
    assert bm.lib_hash() == bm.source_hash()


def test_staged_reference_is_the_unmodified_module_and_runs():
    """bench.py's reference arm drives the reference's own module from oracle/_ref (oracle/stage_ref.py)."""
    import hashlib
    import bench
    staged = bench._reference_module()
    if staged is None:
        pytest.skip("oracle/_ref not staged (run python oracle/stage_ref.py in the build container)")
    ref, man = staged
    src = "/root/reference/src/toycrystals/models/sde_score_model.py"
    if os.path.exists(src):
        assert hashlib.sha256(open(src, "rb").read()).hexdigest() == man["files"]["toycrystals/models/sde_score_model.py"]
    img = bench._reference_job(ref, torch.device("cpu"), 2, 1)()
    assert img.shape == (2, 1, 64, 64) and float(img.min()) >= 0.0 and float(img.max()) <= 1.0
    # the same run through the oracle port with the same random draws: bit-identical (the pin of the oracle).
    # _reference_job seeds torch with 1, builds the model, and the sampler then draws x_T and one z per step.
    torch.manual_seed(1)
    sd = {k: v.clone() for k, v in ref.CondUNetTiny(4, 4, 96, 128, 8, 8).state_dict().items()}
    x0 = torch.randn((2, 1, 64, 64))
    z = torch.randn((2, 1, 64, 64))
    y_cat, y_cont = orc.condition_grid(2, 4, 4)
    with torch.no_grad():
        tr = orc.sample(sd, orc.DEFAULT_CFG, orc.Schedule(0.1, 30.0), y_cat, y_cont, x0, "sde", 1, 1.5, 0.005, [z])
    assert torch.equal(img, tr.image)


def test_attention_weight_image_layout():
    """Host logic of the fused attention block (csrc/attn_tc.cu): the byte image the kernel bulk-copies into shared memory.
    Per head [3 blocks of 64 input channels][144 rows = q | k | v rows of that head][128 B], then the projection
    [3][192 rows][128 B]; bf16; the 16-byte chunk c of row r sits at chunk position c ^ (r & 7) (SWIZZLE_128B, which the UMMA
    descriptors of the kernel assume).  Rows follow torch.chunk(qkv, 3) and the head split of SelfAttention2d.forward
    (sde_score_model.py:149-155).  No GPU needed."""
    L = _cabi.lib()
    g = torch.Generator().manual_seed(3)
    qkv_w = torch.randn((576, 192), generator=g)
    proj_w = torch.randn((192, 192), generator=g)
    need = int(L.tcs_debug_attn_pack(None, None, None, 0))
    assert need == 4 * 3 * 144 * 128 + 3 * 192 * 128
    buf = np.zeros(need, dtype=np.uint8)
    got = L.tcs_debug_attn_pack(qkv_w.numpy().ctypes.data, proj_w.numpy().ctypes.data, buf.ctypes.data, need)
    assert got == need
    words = torch.from_numpy(buf.view(np.int16).copy()).view(torch.bfloat16).float()

    def unpack(base_bytes, rows):   # [3 blocks][rows][64] -> [rows, 192]
        out = torch.empty((rows, 192))
        blk = words[base_bytes // 2: base_bytes // 2 + 3 * rows * 64].reshape(3, rows, 8, 8)   # [block][row][chunk position][8]
        for r in range(rows):
            pos = torch.tensor([c ^ (r & 7) for c in range(8)])
            out[r] = blk[:, r, pos, :].reshape(192)
        return out

    for h in range(4):
        w = unpack(h * 3 * 144 * 128, 144)
        for kind in range(3):   # q, k, v rows of head h
            want = qkv_w[kind * 192 + h * 48: kind * 192 + (h + 1) * 48].bfloat16().float()
            assert torch.equal(w[kind * 48:(kind + 1) * 48], want), (h, kind)
    assert torch.equal(unpack(4 * 3 * 144 * 128, 192), proj_w.bfloat16().float())
