"""Drop-in for the sampling surface of the reference module
``src/toycrystals/models/sde_score_model.py`` — same names, argument meaning, defaults and
error behaviour — with every computation done by libtcs.so (hand-written sm_100a kernels).

    CondUNetTiny                       (reference :170-266)  parameter container + tcs_score
    VPSDE                              (:273-298)
    predict_eps_cfg                    (:402-423)  -> tcs_score, CFG as ONE doubled batch
    sample_probability_flow_ode        (:452-504)  -> tcs_sample (Heun)
    sample_reverse_sde_euler_maruyama  (:507-569)  -> tcs_sample (Euler-Maruyama)
    sample_dpmpp_2m                    (addition)  -> tcs_sample (DPM-Solver++(2M), one evaluation per step)
    save_sde_samples                   (:301-355)  condition grid + sampler + 6x6 PNG

PyTorch is used for device memory, streams and the state-dict container only.  There is no CPU
path: a model whose parameters are not on a CUDA (B200) device raises.
"""
from __future__ import annotations

import ctypes as C
import math
import os
import warnings
import weakref
from dataclasses import dataclass
from typing import Dict, List, Optional, Tuple

import torch
import torch.nn as nn

from .. import _cabi

_PRECISIONS = {"fp32": _cabi.FP32, "bf16": _cabi.BF16}
_ENGINES = {"auto": _cabi.ENGINE_AUTO, "simt": _cabi.ENGINE_SIMT, "tcgen05": _cabi.ENGINE_TCGEN05}


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _stream_ptr(device: torch.device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def _as_f32(t: torch.Tensor, device) -> torch.Tensor:
    return t.to(device=device, dtype=torch.float32).contiguous()


# ------------------------------------------------------------------------------------------------
# parameter container with the reference's state-dict layout (SURVEY 8a-W)
# ------------------------------------------------------------------------------------------------
def _gn_groups(ch: int, max_groups: int = 8) -> int:
    """Largest group count <= max_groups that divides ch (reference :89-94)."""
    g = min(max_groups, ch)
    while g > 1 and ch % g:
        g -= 1
    return g


_SUPPORTED_ARCH = dict(base_ch=96, emb_dim=128, cond_ch=8, time_ch=8)


def _parameter_plan(n_types, y_cont_dim, base_ch, emb_dim, cond_ch, time_ch) -> List[Tuple[str, nn.Module]]:
    """(dotted state-dict prefix, torch layer) in the order the reference constructor creates them,
    so that default initialisation under a given torch seed is identical."""
    e, b = emb_dim, base_ch
    plan: List[Tuple[str, object]] = [
        ("cond_emb.cat_emb", lambda: nn.Embedding(n_types + 1, e)),
        ("cond_emb.cont_mlp.0", lambda: nn.Linear(y_cont_dim, e)),
        ("cond_emb.cont_mlp.2", lambda: nn.Linear(e, e)),
        ("cond_emb.out.1", lambda: nn.Linear(2 * e, e)),
        ("time_mlp.0", lambda: nn.Linear(e, e)),
        ("time_mlp.2", lambda: nn.Linear(e, e)),
        ("to_cond_map", lambda: nn.Linear(e, cond_ch)),
        ("to_time_map", lambda: nn.Linear(e, time_ch)),
    ]

    def conv(name, i, o, k):
        plan.append((name, lambda: nn.Conv2d(i, o, kernel_size=k)))

    def block(name, i, o):
        conv(f"{name}.net.0", i, o, 3)
        plan.append((f"{name}.net.1", lambda: nn.GroupNorm(_gn_groups(o), o)))
        conv(f"{name}.net.3", o, o, 3)
        plan.append((f"{name}.net.4", lambda: nn.GroupNorm(_gn_groups(o), o)))

    block("down1", 1 + cond_ch + time_ch, b)
    conv("ds1", b, b, 4)
    block("down2", b, 2 * b)
    conv("ds2", 2 * b, 2 * b, 4)
    block("mid", 2 * b, 2 * b)
    plan.append(("attn.norm", lambda: nn.GroupNorm(_gn_groups(2 * b), 2 * b)))
    conv("attn.qkv", 2 * b, 6 * b, 1)
    conv("attn.proj", 2 * b, 2 * b, 1)
    conv("us2_conv", 2 * b, 2 * b, 3)
    block("up2", 4 * b, b)
    conv("us1_conv", b, b, 3)
    block("up1", 2 * b, b)
    conv("out", b, 1, 3)
    return plan


class CondUNetTiny(nn.Module):
    """eps_hat = CondUNetTiny(x_t, t, y_cat, y_cont) evaluated by libtcs.

    Constructor arguments and ``state_dict()`` keys/shapes are the reference's.  Extra keyword
    arguments select the arithmetic: ``precision`` "bf16" (tcgen05 tensor cores, default) or
    "fp32" (FFMA kernels, the 1e-4 parity mode); ``engine``/``chunk``/``use_graph`` are tuning knobs.
    The environment variables TCS_PRECISION / TCS_ENGINE / TCS_CHUNK override the defaults.
    """

    def __init__(self, n_types: int, y_cont_dim: int, base_ch: int = 32, emb_dim: int = 128, cond_ch: int = 8,
                 time_ch: int = 8, *, precision: Optional[str] = None, engine: Optional[str] = None,
                 chunk: Optional[int] = None, use_graph: bool = True) -> None:
        super().__init__()
        self.n_types = int(n_types)
        self.y_cont_dim = int(y_cont_dim)
        if self.y_cont_dim < 3:
            raise ValueError("theta_sincos requires y_cont_dim >= 3 (needs indices 1 and 2).")
        if (2 * int(base_ch)) % 4 != 0:
            raise ValueError(f"ch ({2 * int(base_ch)}) must be divisible by num_heads (4)")
        self._arch = dict(n_types=self.n_types, y_cont_dim=self.y_cont_dim, base_ch=int(base_ch), emb_dim=int(emb_dim),
                          cond_ch=int(cond_ch), time_ch=int(time_ch))
        bad = {k: self._arch[k] for k, v in _SUPPORTED_ARCH.items() if self._arch[k] != v}
        if bad:   # fail at construction, not at the first forward (the reference's own default base_ch=32 is one of these)
            raise NotImplementedError(
                f"libtcs is built for the CLI/README architecture base_ch=96, emb_dim=128, cond_ch=8, time_ch=8 only; "
                f"got {bad}. Pass base_ch=96 explicitly (the reference constructor defaults to 32).")
        for path, make in _parameter_plan(**self._arch):
            parent: nn.Module = self
            parts = path.split(".")
            for p in parts[:-1]:
                if not hasattr(parent, p):
                    parent.add_module(p, nn.Module())
                parent = getattr(parent, p)
            parent.add_module(parts[-1], make())
        self.precision = (precision or os.environ.get("TCS_PRECISION", "bf16")).lower()
        self.engine = (engine or os.environ.get("TCS_ENGINE", "auto")).lower()
        self.chunk = int(chunk if chunk is not None else os.environ.get("TCS_CHUNK", "0"))
        self.use_graph = bool(use_graph)
        if self.precision not in _PRECISIONS:
            raise ValueError(f"precision must be one of {sorted(_PRECISIONS)}, got {self.precision!r}")
        if self.engine not in _ENGINES:
            raise ValueError(f"engine must be one of {sorted(_ENGINES)}, got {self.engine!r}")
        self._handle: Optional[C.c_void_p] = None
        self._handle_key = None
        self._checksum = None
        self._key_by_checksum = False
        self._fuse_gn = True   # cleared (sticky) when a fused GroupNorm layer reports values beyond its fp16 staging range
        # VPSDE constants baked into the handle: used by the tcs_sde_update / tcs_ode_update test hooks only; the
        # samplers pass their `sde` per call (tcs_sample_args.beta_min/beta_max), so a different VPSDE does not
        # rebuild the handle
        self._sde_key: Tuple[float, float] = (0.1, 30.0)

    # -- engine management --------------------------------------------------------------------
    def _weights_key(self):
        ps = list(self.parameters())
        # adopted (foreign) modules are re-copied on every call, which bumps _version without changing a bit: for them
        # the checksum alone decides
        ver = None if self._key_by_checksum else tuple((p.data_ptr(), p._version) for p in ps)
        return (ps[0].device, self.precision, self.engine, self.chunk, self.use_graph, self._sde_key, ver, self._checksum,
                self._fuse_gn)

    def weights_checksum(self) -> Tuple[int, float]:
        """Device-side checksum of all parameters: catches in-place updates made through ``.data`` (the training loop's
        EMA update, scripts/train_sde_score_model.py:239-240), which do not bump ``_version``.  One small reduction and a
        host read."""
        return params_checksum(self)

    def refresh(self) -> "CondUNetTiny":
        """Re-read the parameters on the next call if they changed behind autograd's back (``p.data.mul_(...)``).
        The samplers call this themselves (a sampling job costs far more than the check); ``forward`` /
        ``predict_eps_cfg`` do not (they may sit in a per-step loop), so call it after editing ``.data`` by hand."""
        if next(self.parameters()).device.type == "cuda":
            self._checksum = self.weights_checksum()
        return self

    def _release(self):
        if self._handle is not None:
            _cabi.lib().tcs_destroy(self._handle)
            self._handle = None
            self._handle_key = None

    def __del__(self):
        try:
            self._release()
        except Exception:
            pass

    def set_precision(self, precision: str, engine: str = "auto") -> "CondUNetTiny":
        self.precision, self.engine = precision.lower(), engine.lower()
        return self

    def engine_handle(self, sde: Optional["VPSDE"] = None) -> C.c_void_p:
        """Create / refresh the libtcs handle for the current parameters (lazy, cached)."""
        if sde is not None:
            self._sde_key = (float(sde.beta_min), float(sde.beta_max))
        dev = next(self.parameters()).device
        if dev.type != "cuda":
            raise RuntimeError("toycrystals_b200 runs on a CUDA (B200, sm_100a) device only; move the model with "
                               ".to('cuda') — there is no CPU fallback (use the reference package for --device cpu)")
        key = self._weights_key()
        if self._handle is not None and key == self._handle_key:
            return self._handle
        self._release()
        L = _cabi.lib()
        cfg = _cabi.TcsConfig()
        L.tcs_default_config(C.byref(cfg))
        for k, v in self._arch.items():
            setattr(cfg, k, v)
        cfg.beta_min, cfg.beta_max = self._sde_key
        cfg.precision = _PRECISIONS[self.precision]
        cfg.engine = _ENGINES[self.engine]
        cfg.device = dev.index if dev.index is not None else torch.cuda.current_device()
        cfg.chunk = self.chunk
        cfg.use_graph = 1 if self.use_graph else 0
        cfg.fuse_gn = 1 if self._fuse_gn else 0
        h = C.c_void_p()
        _cabi.check(L.tcs_create(C.byref(h), C.byref(cfg)))
        try:
            torch.cuda.synchronize(dev)
            for name, t in self.state_dict().items():
                w = t.detach().to(torch.float32).contiguous()
                shape = (C.c_int64 * w.dim())(*w.shape)
                _cabi.check(L.tcs_set_weight(h, name.encode(), w.data_ptr(), shape, w.dim()))
            _cabi.check(L.tcs_finalize_weights(h))
        except Exception:
            L.tcs_destroy(h)
            raise
        self._handle, self._handle_key = h, key
        return h

    def launch_count(self) -> int:
        return 0 if self._handle is None else int(_cabi.lib().tcs_launch_count(self._handle))

    # -- reference surface --------------------------------------------------------------------------
    def forward(self, x_t: torch.Tensor, t: torch.Tensor, y_cat: torch.Tensor, y_cont: torch.Tensor) -> torch.Tensor:
        return _score(self, x_t, t, y_cat, y_cont, 0.0)


def params_checksum(module: nn.Module) -> Tuple[int, float]:
    """Bit pattern sum + sum of squares of all of a module's (fp32) parameters, computed on their device."""
    flat = torch.cat([p.detach().reshape(-1) for p in module.parameters()])
    a = flat.view(torch.int32).sum(dtype=torch.int64)
    b = (flat.double() ** 2).sum()
    return int(a.item()), float(b.item())


_adopted: "Dict[int, Tuple[object, CondUNetTiny]]" = {}


def adopt(model: nn.Module, precision: Optional[str] = None) -> CondUNetTiny:
    """Accept ANY module that carries the reference ``CondUNetTiny`` state dict (e.g. the training script's ``model`` /
    ``ema_model``, scripts/train_sde_score_model.py:263-279) and return the libtcs-backed equivalent, so the training-time
    sampling hook ``save_sde_samples(model=sample_model, ...)`` runs on the fast path unchanged.  The architecture is read
    off the tensor shapes; the weights are copied on every call and re-packed whenever their checksum changed (the EMA
    update writes through ``.data``, which autograd's version counter does not record)."""
    if isinstance(model, CondUNetTiny):
        return model
    sd = model.state_dict()
    try:
        arch = dict(n_types=int(sd["cond_emb.cat_emb.weight"].shape[0]) - 1,
                    y_cont_dim=int(sd["cond_emb.cont_mlp.0.weight"].shape[1]),
                    base_ch=int(sd["down1.net.3.weight"].shape[0]), emb_dim=int(sd["time_mlp.0.weight"].shape[0]),
                    cond_ch=int(sd["to_cond_map.weight"].shape[0]), time_ch=int(sd["to_time_map.weight"].shape[0]))
    except KeyError as e:
        raise TypeError(f"model does not carry the CondUNetTiny state dict (missing {e})") from None
    # A foreign module's parameters may be updated through `.data` (the reference's EMA loop), which `_version` does not
    # see: always copy the state dict (device-to-device, 13 MB) and let the checksum decide whether libtcs re-packs.
    hit = _adopted.get(id(model))
    fast = hit[1] if hit is not None and hit[0] == tuple(sorted(arch.items())) else CondUNetTiny(**arch, precision=precision)
    with torch.no_grad():
        fast.load_state_dict(sd)
    fast = fast.to(next(iter(sd.values())).device).eval()
    fast._key_by_checksum = True
    fast.refresh()
    if hit is None:   # drop the libtcs twin (and its device workspace) together with the module it shadows
        weakref.finalize(model, _adopted.pop, id(model), None)
    _adopted[id(model)] = (tuple(sorted(arch.items())), fast)
    return fast


def _run_checked(model: CondUNetTiny, enqueue) -> None:
    """enqueue(handle) once; if libtcs then reports that a fused GroupNorm layer saw pre-norm activations beyond the fp16
    staging range (|v| > 65504: possible with untrained / exploding weights, never seen with the README model), switch
    this model to the unfused GroupNorm path for good and run the call again, so that a clipped result is never returned."""
    L = _cabi.lib()
    for attempt in (0, 1):
        h = model.engine_handle()
        enqueue(h)
        bits = int(L.tcs_check(h))
        if bits < 0:
            _cabi.check(bits)
        if not (bits & 1):
            return
        if attempt == 1 or not model._fuse_gn:
            raise _cabi.TcsError("libtcs: activation range error persists on the unfused GroupNorm path")
        warnings.warn("toycrystals_b200: a pre-GroupNorm activation exceeded the fp16 staging range of the fused conv "
                      "epilogue; re-running on the unfused GroupNorm path (kept for this model from now on)")
        model._fuse_gn = False


def _score(model: CondUNetTiny, x_t, t, y_cat, y_cont, guidance: float) -> torch.Tensor:
    model = adopt(model)
    dev = next(model.parameters()).device
    if dev.type != "cuda":
        model.engine_handle()   # raises: no CPU fallback
    B, Cc, H, W = x_t.shape
    if Cc != 1 or H != 64 or W != 64:
        raise NotImplementedError(f"libtcs evaluates [B,1,64,64] images only (got {tuple(x_t.shape)})")
    x = _as_f32(x_t, dev)
    tt = _as_f32(t, dev).reshape(-1)
    if tt.numel() == 1 and B > 1:
        tt = tt.expand(B).contiguous()
    yc = y_cat.to(device=dev, dtype=torch.int64).contiguous()
    yk = _as_f32(y_cont, dev)
    out = torch.empty((B, 1, 64, 64), device=dev, dtype=torch.float32)
    with torch.cuda.device(dev):
        _run_checked(model, lambda h: _cabi.check(_cabi.lib().tcs_score(
            h, x.data_ptr(), tt.data_ptr(), yc.data_ptr(), yk.data_ptr(), B, float(guidance), out.data_ptr(),
            _stream_ptr(dev))))
    return out


@dataclass(frozen=True)
class VPSDE:
    """VP SDE with linear beta(t) on [0,1]; tensor-in tensor-out like the reference (:273-298)."""
    beta_min: float = 0.1
    beta_max: float = 20.0

    def beta(self, t: torch.Tensor) -> torch.Tensor:
        return self.beta_min + t * (self.beta_max - self.beta_min)

    def int_beta(self, t: torch.Tensor) -> torch.Tensor:
        return self.beta_min * t + 0.5 * (self.beta_max - self.beta_min) * (t ** 2)

    def alpha(self, t: torch.Tensor) -> torch.Tensor:
        return torch.exp(-0.5 * self.int_beta(t))

    def sigma(self, t: torch.Tensor) -> torch.Tensor:
        a = self.alpha(t)
        return torch.sqrt(torch.clamp(1.0 - a * a, min=1e-8))


@torch.no_grad()
def predict_eps_cfg(model: CondUNetTiny, x_t: torch.Tensor, t: torch.Tensor, y_cat: torch.Tensor,
                    y_cont: torch.Tensor, guidance_scale: float) -> torch.Tensor:
    """eps = eps_u + s (eps_c - eps_u); s <= 0 -> a single conditional evaluation."""
    return _score(model, x_t, t, y_cat, y_cont, float(guidance_scale))


@dataclass
class SamplerTrace:
    eps: torch.Tensor      # [nfe, n, 1, 64, 64] CFG-combined eps of every network evaluation
    x_in: torch.Tensor     # [nfe, n, 1, 64, 64] the x_t each evaluation saw
    x0_hat: torch.Tensor   # [n, 1, 64, 64] projection before the [0,1] map and clamp


def _sample(model: CondUNetTiny, sde: VPSDE, y_cat, y_cont, img_shape, n_steps, guidance_scale, t_end, sampler: int,
            x_init=None, noise=None, seed=None, global_index_offset=0, return_trace=False):
    model = adopt(model)
    device = y_cat.device
    B, Cc, H, W = img_shape
    assert Cc == 1
    t_end = float(t_end)
    if not (0.0 < t_end < 1.0):
        raise ValueError(f"t_end must be in (0,1), got {t_end}")
    if device.type != "cuda":
        raise RuntimeError("toycrystals_b200 samples on a CUDA (B200) device only: y_cat/y_cont must live on the "
                           "GPU (no CPU fallback)")
    if H != 64 or W != 64:
        raise NotImplementedError(f"libtcs samples 64x64 images only (got {H}x{W})")
    model.refresh()
    L = _cabi.lib()
    n_steps = int(n_steps)
    yc = y_cat.to(torch.int64).contiguous()
    yk = _as_f32(y_cont, device)
    if x_init is None and seed is None:
        # same draw as the reference: one torch.randn from the device's global generator
        x_init = torch.randn((B, Cc, H, W), device=device)
    # x_init None with a seed: the kernel draws x_T from Philox keyed (seed, global_index_offset + i), so `seed=` alone
    # reproduces a run and a sharded job equals the unsharded one
    x_init = None if x_init is None else _as_f32(x_init, device)
    noise_t = None
    if sampler == _cabi.SAMPLER_SDE:
        if isinstance(noise, str) and noise == "torch":
            # reference-identical consumption of the global generator: one randn_like per step
            noise_t = (torch.stack([torch.randn((B, 1, 64, 64), device=device) for _ in range(n_steps)])
                       if n_steps else None)
        elif torch.is_tensor(noise):
            noise_t = _as_f32(noise, device)
            if noise_t.shape[0] != n_steps or noise_t[0].numel() != B * 4096:
                raise ValueError("noise must be [n_steps, B, 1, 64, 64]")
    if seed is None:
        seed = int(torch.randint(0, 2 ** 62, (1,)).item())  # torch.manual_seed controls the Philox stream
    out = torch.empty((B, 1, 64, 64), device=device, dtype=torch.float32)
    nfe = L.tcs_nfe(sampler, n_steps)
    tr_eps = tr_x = x0h = None
    if return_trace:
        tr_eps = torch.empty((nfe, B, 1, 64, 64), device=device, dtype=torch.float32)
        tr_x = torch.empty_like(tr_eps)
        x0h = torch.empty_like(out)
    a = _cabi.TcsSampleArgs()
    a.sampler, a.n, a.steps = sampler, B, n_steps
    a.guidance, a.t_end = float(guidance_scale), t_end
    a.y_cat, a.y_cont = yc.data_ptr(), yk.data_ptr()
    a.x_init, a.noise = _ptr(x_init), _ptr(noise_t)
    a.beta_min, a.beta_max = float(sde.beta_min), float(sde.beta_max)
    a.seed, a.global_index_offset = int(seed) & (2 ** 64 - 1), int(global_index_offset)
    a.x_out, a.trace_eps, a.trace_x, a.x0_hat = out.data_ptr(), _ptr(tr_eps), _ptr(tr_x), _ptr(x0h)
    with torch.cuda.device(device):
        _run_checked(model, lambda h: _cabi.check(L.tcs_sample(h, C.byref(a), _stream_ptr(device))))
    if noise_t is not None:
        noise_t.record_stream(torch.cuda.current_stream(device))
    if return_trace:
        return out, SamplerTrace(tr_eps, tr_x, x0h)
    return out


@torch.no_grad()
def sample_probability_flow_ode(model: CondUNetTiny, sde: VPSDE, y_cat: torch.Tensor, y_cont: torch.Tensor,
                                img_shape: Tuple[int, int, int, int], n_steps: int = 200,
                                guidance_scale: float = 0.0, t_end: float = 1e-3, *, x_init=None, seed=None,
                                global_index_offset: int = 0, return_trace: bool = False):
    """Deterministic sampler: probability-flow ODE, Heun (2nd order), quadratic time grid, final
    x0 projection; returns [B,1,64,64] in [0,1].  Keyword-only extras are additions."""
    return _sample(model, sde, y_cat, y_cont, img_shape, n_steps, guidance_scale, t_end, _cabi.SAMPLER_ODE,
                   x_init=x_init, seed=seed, global_index_offset=global_index_offset, return_trace=return_trace)


@torch.no_grad()
def sample_reverse_sde_euler_maruyama(model: CondUNetTiny, sde: VPSDE, y_cat: torch.Tensor, y_cont: torch.Tensor,
                                      img_shape: Tuple[int, int, int, int], n_steps: int = 200,
                                      guidance_scale: float = 0.0, t_end: float = 1e-3, *, x_init=None, noise=None,
                                      seed=None, global_index_offset: int = 0, return_trace: bool = False):
    """Stochastic sampler: reverse-time VP-SDE, Euler-Maruyama (noise on every step, the last
    included).  ``noise``: None = in-kernel Philox4x32-10 keyed (seed, global sample index, step);
    "torch" = one torch.randn_like per step exactly like the reference; a tensor
    [n_steps,B,1,64,64] = injected."""
    return _sample(model, sde, y_cat, y_cont, img_shape, n_steps, guidance_scale, t_end, _cabi.SAMPLER_SDE,
                   x_init=x_init, noise=noise, seed=seed, global_index_offset=global_index_offset,
                   return_trace=return_trace)


@torch.no_grad()
def sample_dpmpp_2m(model: CondUNetTiny, sde: VPSDE, y_cat: torch.Tensor, y_cont: torch.Tensor,
                    img_shape: Tuple[int, int, int, int], n_steps: int = 20, guidance_scale: float = 0.0,
                    t_end: float = 1e-3, *, x_init=None, seed=None, global_index_offset: int = 0,
                    return_trace: bool = False):
    """Deterministic sampler: DPM-Solver++(2M) (Lu et al. 2022, Algorithm 2) on the probability-flow ODE, times
    uniform in log-SNR from t = 1 to t_end, first-order first step (and last step when n_steps < 15), one network
    evaluation per step, final x0 projection; returns [B,1,64,64] in [0,1].  n_steps + 1 evaluations in all, against
    2 n_steps + 1 for the Heun ODE sampler.  ``x_init`` / ``seed`` / ``global_index_offset`` / ``return_trace`` as for
    the other samplers; the trace has the SDE sampler's layout."""
    return _sample(model, sde, y_cat, y_cont, img_shape, n_steps, guidance_scale, t_end, _cabi.SAMPLER_DPMPP_2M,
                   x_init=x_init, seed=seed, global_index_offset=global_index_offset, return_trace=return_trace)


_SAMPLERS = {"ode": sample_probability_flow_ode, "sde": sample_reverse_sde_euler_maruyama, "dpm++2m": sample_dpmpp_2m}


def condition_grid(model: CondUNetTiny, n: int, theta_max: float, device, offset: int = 0, n_total: Optional[int] = None):
    """y_cat[i] = i % n_types, y_cont[i] = [0, linspace(0, theta_max, n)[i], 0, ...] (reference :317-321),
    generated on the device by libtcs; (offset, n_total) select a shard of a larger grid."""
    device = torch.device(device)
    model = adopt(model)
    h = model.engine_handle()
    n_total = n if n_total is None else n_total
    y_cat = torch.empty((n,), device=device, dtype=torch.int64)
    y_cont = torch.empty((n, model.y_cont_dim), device=device, dtype=torch.float32)
    with torch.cuda.device(device):
        _cabi.check(_cabi.lib().tcs_condition_grid(h, n, offset, n_total, float(theta_max), y_cat.data_ptr(),
                                                   y_cont.data_ptr(), _stream_ptr(device)))
    return y_cat, y_cont


def _write_grid_png(x: torch.Tensor, out_path: str, title: str) -> None:
    """6x6 grey-scale grid of the first 36 images (the reference plots the same subset, :348-355)."""
    from PIL import Image, ImageDraw

    k = min(36, x.shape[0])
    imgs = (x[:k, 0].detach().float().clamp(0, 1) * 255.0).round().to(torch.uint8).cpu().numpy()
    cell, gap, top = 64 * 3, 6, 22
    canvas = Image.new("L", (6 * cell + 7 * gap, top + 6 * cell + 7 * gap), 255)
    for i in range(k):
        r, c = divmod(i, 6)
        tile = Image.fromarray(imgs[i], mode="L").resize((cell, cell), Image.NEAREST)
        canvas.paste(tile, (gap + c * (cell + gap), top + gap + r * (cell + gap)))
    ImageDraw.Draw(canvas).text((gap, 4), title, fill=0)
    canvas.save(out_path)


@torch.no_grad()
def save_sde_samples(model: CondUNetTiny, sde: VPSDE, out_path: str, device: torch.device, n: int = 36,
                     theta_max: float = math.pi / 3.0, steps: int = 200, cfg: float = 0.0, t_end: float = 1e-3,
                     sampler: str = "ode") -> None:
    """Save a 6x6 grid: cycle lattice types, sweep theta in [0, theta_max].  ``model`` may be the libtcs-backed
    CondUNetTiny or any module with the reference state dict (the training script's hook passes its own)."""
    model.eval()
    device = torch.device(device)
    if sampler not in _SAMPLERS:
        raise ValueError(f"Unknown sampler='{sampler}'. Use 'ode', 'sde' or 'dpm++2m'.")
    model = adopt(model)
    y_cat, y_cont = condition_grid(model, n, theta_max, device)
    fn = _SAMPLERS[sampler]
    x = fn(model=model, sde=sde, y_cat=y_cat, y_cont=y_cont, img_shape=(n, 1, 64, 64), n_steps=steps,
           guidance_scale=cfg, t_end=t_end)
    _write_grid_png(x, out_path, f"{sampler} | steps={steps} | cfg={cfg:.2f} | t_end={t_end:g}")
