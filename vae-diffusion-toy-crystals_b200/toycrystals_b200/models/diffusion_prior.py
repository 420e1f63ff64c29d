"""Drop-in for the sampling surface of the reference module ``src/toycrystals/models/diffusion_prior.py`` (and of
``save_diffusion_samples`` in ``scripts/train_diffusion_prior.py``) — BASELINE configs[3], SURVEY 8(f) row 1.

    DiffusionPriorFiLM            (reference :57-127)   parameter container + tcs_prior_eps
    DiffusionSchedule.linear      (:177-188)
    DiffusionSchedule.ddim_sample (:200-252)            -> tcs_prior_ddim_sample (eta = 0)
    save_diffusion_samples        (scripts/train_diffusion_prior.py:61-106)  DDIM -> un-standardise -> CondVAE.decode

Same names, argument meaning, defaults and error behaviour; every computation is done by libtcs.so (tcgen05 GEMMs for
the FiLM blocks, CUDA-core kernels for the rest).  PyTorch holds the parameters and the device memory only; there is no
CPU path.  Training-time members of the reference module (DiffusionPrior, q_sample) are out of scope.
"""
from __future__ import annotations

import ctypes as C
import math
import os
from dataclasses import dataclass
from typing import Optional

import torch
import torch.nn as nn

from .. import _cabi
from .sde_score_model import _as_f32, _ptr, _stream_ptr, _write_grid_png, params_checksum

_PRECISIONS = {"fp32": _cabi.FP32, "bf16": _cabi.BF16}


class FiLMResBlock(nn.Module):
    """Parameter container of one block (reference :39-54); evaluated inside libtcs."""

    def __init__(self, width: int, cond_dim: int, mult: int = 4) -> None:
        super().__init__()
        self.norm = nn.LayerNorm(width)
        self.fc1 = nn.Linear(width, mult * width)
        self.fc2 = nn.Linear(mult * width, width)
        self.cond = nn.Linear(cond_dim, 2 * width)


class DiffusionPriorFiLM(nn.Module):
    """eps_hat = DiffusionPriorFiLM(z_t, t, y_cat, y_cont) evaluated by libtcs.

    Constructor arguments, construction order (hence default initialisation under a torch seed) and ``state_dict()``
    keys/shapes are the reference's.  ``precision``: "bf16" (tcgen05 GEMMs, fp32 accumulation and residual stream;
    default) or "fp32" (FFMA GEMMs, the parity mode).  TCS_PRECISION overrides the default.
    """

    def __init__(self, z_dim: int, n_types: int, y_cont_dim: int, t_emb_dim: int = 64, width: int = 256, n_blocks: int = 6,
                 y_cat_emb_dim: int = 64, *, precision: Optional[str] = None, use_graph: bool = True) -> None:
        super().__init__()
        self.z_dim = int(z_dim)
        self.n_types = int(n_types)
        self.y_cont_dim = int(y_cont_dim)
        self.t_emb_dim = int(t_emb_dim)
        self.y_cat_emb = nn.Embedding(self.n_types, y_cat_emb_dim)
        self.y_cont_mlp = nn.Sequential(nn.Linear(self.y_cont_dim, y_cat_emb_dim), nn.SiLU(),
                                        nn.Linear(y_cat_emb_dim, y_cat_emb_dim))
        self.y_fuse = nn.Sequential(nn.Linear(2 * y_cat_emb_dim, width), nn.SiLU(), nn.Linear(width, width))
        self.t_mlp = nn.Sequential(nn.Linear(self.t_emb_dim, width), nn.SiLU(), nn.Linear(width, width))
        self.in_proj = nn.Linear(self.z_dim, width)
        self.blocks = nn.ModuleList([FiLMResBlock(width, 2 * width) for _ in range(n_blocks)])
        self.out_norm = nn.LayerNorm(width)
        self.out_proj = nn.Linear(width, self.z_dim)
        self._arch = dict(z_dim=self.z_dim, n_types=self.n_types, y_cont_dim=self.y_cont_dim, t_emb_dim=self.t_emb_dim,
                          width=int(width), n_blocks=int(n_blocks), y_cat_emb_dim=int(y_cat_emb_dim))
        self.precision = (precision or os.environ.get("TCS_PRECISION", "bf16")).lower()
        if self.precision not in _PRECISIONS:
            raise ValueError(f"precision must be one of {sorted(_PRECISIONS)}, got {self.precision!r}")
        self.use_graph = bool(use_graph)
        self._handle: Optional[C.c_void_p] = None
        self._handle_key = None
        self._checksum = None
        self._sched_key = (1000, 1e-4, 0.05)

    def refresh(self) -> "DiffusionPriorFiLM":
        """Re-read the parameters on the next call if they changed behind autograd's back (``p.data.copy_(...)``, an EMA
        update), which ``_version`` does not record.  ``forward`` and ``ddim_sample`` do not check (the checksum reads all
        400 MB of parameters at width 1024), so call this after editing ``.data`` by hand; ``save_diffusion_samples``
        calls it itself."""
        if next(self.parameters()).device.type == "cuda":
            self._checksum = params_checksum(self)
        return self

    def _release(self):
        if self._handle is not None:
            _cabi.lib().tcs_prior_destroy(self._handle)
            self._handle = None
            self._handle_key = None

    def __del__(self):
        try:
            self._release()
        except Exception:
            pass

    def engine_handle(self, sched: Optional["DiffusionSchedule"] = None) -> C.c_void_p:
        """Create / refresh the libtcs handle for the current parameters (lazy, cached)."""
        if sched is not None:
            self._sched_key = sched._linear_key()
        ps = list(self.parameters())
        dev = ps[0].device
        if dev.type != "cuda":
            raise RuntimeError("toycrystals_b200 runs on a CUDA (B200, sm_100a) device only; move the model with "
                               ".to('cuda') — there is no CPU fallback (use the reference package for --device cpu)")
        key = (dev, self.precision, self.use_graph, self._sched_key, tuple((p.data_ptr(), p._version) for p in ps),
               self._checksum)
        if self._handle is not None and key == self._handle_key:
            return self._handle
        self._release()
        L = _cabi.lib()
        cfg = _cabi.TcsPriorConfig()
        L.tcs_prior_default_config(C.byref(cfg))
        for k, v in self._arch.items():
            setattr(cfg, k, v)
        cfg.T, cfg.beta_start, cfg.beta_end = self._sched_key
        cfg.precision = _PRECISIONS[self.precision]
        cfg.device = dev.index if dev.index is not None else torch.cuda.current_device()
        cfg.use_graph = 1 if self.use_graph else 0
        h = C.c_void_p()
        _cabi.check(L.tcs_prior_create(C.byref(h), C.byref(cfg)))
        try:
            torch.cuda.synchronize(dev)
            for name, t in self.state_dict().items():
                w = t.detach().to(torch.float32).contiguous()
                shape = (C.c_int64 * w.dim())(*w.shape)
                _cabi.check(L.tcs_prior_set_weight(h, name.encode(), w.data_ptr(), shape, w.dim()))
            _cabi.check(L.tcs_prior_finalize_weights(h))
        except Exception:
            L.tcs_prior_destroy(h)
            raise
        self._handle, self._handle_key = h, key
        return h

    def launch_count(self) -> int:
        return 0 if self._handle is None else int(_cabi.lib().tcs_prior_launch_count(self._handle))

    def forward(self, z_t: torch.Tensor, t: torch.Tensor, y_cat: torch.Tensor, y_cont: torch.Tensor) -> torch.Tensor:
        h = self.engine_handle()
        dev = next(self.parameters()).device
        B = int(z_t.shape[0])
        z = _as_f32(z_t, dev)
        tt = t.to(device=dev, dtype=torch.int64).contiguous()
        yc = y_cat.to(device=dev, dtype=torch.int64).contiguous()
        yk = _as_f32(y_cont, dev)
        out = torch.empty((B, self.z_dim), device=dev, dtype=torch.float32)
        with torch.cuda.device(dev):
            _cabi.check(_cabi.lib().tcs_prior_eps(h, z.data_ptr(), tt.data_ptr(), yc.data_ptr(), yk.data_ptr(), B,
                                                  out.data_ptr(), _stream_ptr(dev)))
        return out


@dataclass
class DdimTrace:
    eps: torch.Tensor     # [steps_run, B, z_dim] eps of every evaluation
    z_in: torch.Tensor    # [steps_run, B, z_dim] the z_t every evaluation saw
    timesteps: torch.Tensor  # [steps_run] int64


@dataclass(frozen=True)
class DiffusionSchedule:
    """DDPM constants of a linear beta schedule (reference :163-188).  The tensors are the reference's; the DDIM loop
    itself recomputes the same fp32 constants inside libtcs from (T, beta_start, beta_end)."""
    betas: torch.Tensor
    alphas: torch.Tensor
    alpha_bars: torch.Tensor
    sqrt_alpha_bars: torch.Tensor
    sqrt_one_minus_alpha_bars: torch.Tensor
    T: int = 0
    beta_start: float = 0.0
    beta_end: float = 0.0

    @staticmethod
    def linear(T: int, beta_start: float, beta_end: float, device: torch.device) -> "DiffusionSchedule":
        betas = torch.linspace(beta_start, beta_end, steps=T, device=device, dtype=torch.float32)
        alphas = 1.0 - betas
        alpha_bars = torch.cumprod(alphas, dim=0)
        return DiffusionSchedule(betas=betas, alphas=alphas, alpha_bars=alpha_bars, sqrt_alpha_bars=torch.sqrt(alpha_bars),
                                 sqrt_one_minus_alpha_bars=torch.sqrt(1.0 - alpha_bars), T=int(T),
                                 beta_start=float(beta_start), beta_end=float(beta_end))

    def _linear_key(self):
        if self.T <= 0:
            raise NotImplementedError("libtcs samples with linear beta schedules only: build the schedule with "
                                      "DiffusionSchedule.linear(T, beta_start, beta_end, device)")
        return (self.T, self.beta_start, self.beta_end)

    @torch.no_grad()
    def ddim_sample(self, model: DiffusionPriorFiLM, y_cat: torch.Tensor, y_cont: torch.Tensor, n_steps: int = 50,
                    eta: float = 0.0, *, z_init: Optional[torch.Tensor] = None, seed: Optional[int] = None,
                    global_index_offset: int = 0, return_trace: bool = False):
        """DDIM sampling (eta=0 -> deterministic); returns z0 [B, z_dim].  Keyword-only extras are additions:
        ``z_init`` injects the initial latent (default: one torch.randn from the device generator, like the reference;
        ``seed`` switches to the in-library Philox stream keyed (seed, global sample index))."""
        model.eval()
        device = self.betas.device
        if eta != 0.0:
            raise NotImplementedError("eta != 0 not implemented in this minimal version")
        if device.type != "cuda":
            raise RuntimeError("toycrystals_b200 samples on a CUDA (B200) device only: build the schedule on the GPU "
                               "(no CPU fallback)")
        B = int(y_cat.shape[0])
        h = model.engine_handle(self)
        L = _cabi.lib()
        yc = y_cat.to(device=device, dtype=torch.int64).contiguous()
        yk = _as_f32(y_cont, device)
        if z_init is None and seed is None:
            z_init = torch.randn((B, model.z_dim), device=device)
        zi = None if z_init is None else _as_f32(z_init, device)
        out = torch.empty((B, model.z_dim), device=device, dtype=torch.float32)
        tr_e = tr_z = ts = None
        if return_trace:
            buf = (C.c_int64 * max(int(n_steps), 1))()
            cnt = C.c_int32()
            _cabi.check(L.tcs_prior_timesteps_host(self.T, int(n_steps), buf, C.byref(cnt)))
            ts = torch.tensor(list(buf[:cnt.value]), dtype=torch.int64)
            tr_e = torch.empty((cnt.value, B, model.z_dim), device=device, dtype=torch.float32)
            tr_z = torch.empty_like(tr_e)
        a = _cabi.TcsDdimArgs()
        a.n, a.n_steps = B, int(n_steps)
        a.y_cat, a.y_cont, a.z_init = yc.data_ptr(), yk.data_ptr(), _ptr(zi)
        a.seed, a.global_index_offset = int(seed or 0) & (2 ** 64 - 1), int(global_index_offset)
        a.z0_out, a.trace_eps, a.trace_z = out.data_ptr(), _ptr(tr_e), _ptr(tr_z)
        with torch.cuda.device(device):
            _cabi.check(L.tcs_prior_ddim_sample(h, C.byref(a), _stream_ptr(device)))
        if return_trace:
            return out, DdimTrace(tr_e, tr_z, ts)
        return out


@torch.no_grad()
def sample_images(vae, prior: DiffusionPriorFiLM, sched: DiffusionSchedule, y_cat: torch.Tensor, y_cont: torch.Tensor,
                  z_mean: torch.Tensor, z_std: torch.Tensor, ddim_steps: int = 50, **ddim_kwargs) -> torch.Tensor:
    """DDIM in the standardised latent space, un-standardise, decode: the tensor part of save_diffusion_samples
    (scripts/train_diffusion_prior.py:84-95).  Returns x [B,1,64,64] in (0,1)."""
    z_norm = sched.ddim_sample(prior, y_cat=y_cat, y_cont=y_cont, n_steps=ddim_steps, eta=0.0, **ddim_kwargs)
    return vae.decode(z_norm, y_cat, y_cont, z_mean=z_mean, z_std=z_std)


@torch.no_grad()
def save_diffusion_samples(vae, prior: DiffusionPriorFiLM, sched: DiffusionSchedule, out_path: str, device: torch.device,
                           z_mean: torch.Tensor, z_std: torch.Tensor, n: int = 36, theta_max: float = math.pi / 3.0,
                           ddim_steps: int = 50) -> None:
    """Make a 6x6 grid, cycling lattice types, sweeping theta in [0, pi/3] (reference signature and conditions)."""
    vae.eval()
    prior.eval().refresh()   # the training loop may have updated the weights through .data
    device = torch.device(device)
    y_cat = torch.tensor([i % vae.n_types for i in range(n)], device=device, dtype=torch.int64)
    thetas = torch.linspace(0.0, theta_max, steps=n, device=device)
    y_cont = torch.zeros((n, vae.y_cont_dim), device=device)
    y_cont[:, 1] = thetas
    x = sample_images(vae, prior, sched, y_cat, y_cont, z_mean, z_std, ddim_steps)
    _write_grid_png(x, out_path, f"latent diffusion prior | ddim_steps={ddim_steps}")
