"""Shared helpers of the parity tests (CUDA path vs oracle)."""
from __future__ import annotations

import ctypes as C
import os

import torch
import torch.nn.functional as F

import toycrystals_oracle as orc
from toycrystals_b200 import _cabi
from toycrystals_b200.models.sde_score_model import CondUNetTiny, VPSDE

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
CFG = dict(orc.DEFAULT_CFG)
_models = {}


def rel_l2(a, b):
    return orc.rel_l2(a, b)


TEST_CHUNK = 128   # images per network pass in the tests; the library default (2048) needs 15-35 GB of workspace per model
MAX_MODELS = 4


def model(precision: str, engine: str = "auto", seed: int = 0, chunk: int = 0, use_graph: bool = True) -> CondUNetTiny:
    """Cached libtcs-backed model.  chunk = 0 -> TEST_CHUNK (pass chunk=2048 for the production pass size); the cache
    keeps the MAX_MODELS most recently used models and frees the others' device workspaces."""
    chunk = chunk or TEST_CHUNK
    key = (precision, engine, seed, chunk, use_graph)
    if key in _models:
        _models[key] = _models.pop(key)          # most recently used last
        return _models[key]
    while len(_models) >= MAX_MODELS:
        old = _models.pop(next(iter(_models)))
        old._release()
        del old
        torch.cuda.empty_cache()
    m = CondUNetTiny(**CFG, precision=precision, engine=engine, chunk=chunk, use_graph=use_graph)
    m.load_state_dict(orc.default_init_state_dict(seed))
    _models[key] = m.to("cuda").eval()
    return _models[key]


def golden(name):
    return torch.load(os.path.join(GOLDEN, name), weights_only=False)


def image_of(x0_hat):
    """The reference's final map from the pre-clamp projection to the [0,1] image (bit-exact in fp32), so that the golden
    files store x0_hat only."""
    return ((x0_hat + 1.0) * 0.5).clamp(0.0, 1.0)


def conv_reference(in0, in1, w, b, ksize, stride, round_bf16=False):
    """torch circular conv on NHWC fp32 inputs; returns NHWC fp32."""
    x = in0 if in1 is None else torch.cat([in0, in1], dim=-1)
    if round_bf16:
        x = x.bfloat16().float()
        w = w.bfloat16().float()
    x = x.permute(0, 3, 1, 2).double()
    if ksize > 1:
        x = F.pad(x, (1, 1, 1, 1), mode="circular")
    y = F.conv2d(x, w.double(), b.double(), stride=stride)
    return y.permute(0, 2, 3, 1).contiguous()


def debug_conv(engine, precision, in0, in1, w, b, ksize, stride, epi):
    """in0/in1 NHWC fp32 CUDA tensors.  Returns (out NHWC fp32, stats [B,8,2] or None)."""
    L = _cabi.lib()
    B, Hin, Win, c0 = in0.shape
    c1 = 0 if in1 is None else in1.shape[-1]
    Ho, Wo = Hin // stride, Win // stride
    cout = w.shape[0]
    out = torch.full((B, Ho, Wo, cout), float("nan"), device="cuda")
    stats = torch.zeros((B, 8, 2), device="cuda") if epi == 0 else None
    torch.cuda.synchronize()
    _cabi.check(L.tcs_debug_conv(_cabi.__dict__["ENGINE_" + engine.upper()], _cabi.__dict__[precision.upper()], B, Ho, Wo,
                                 c0, c1, cout, ksize, stride, in0.data_ptr(), None if in1 is None else in1.data_ptr(),
                                 w.contiguous().data_ptr(), b.data_ptr(), out.data_ptr(),
                                 None if stats is None else stats.data_ptr(), epi, None))
    torch.cuda.synchronize()
    return out, stats


ATTN_DBG_FLOATS = 256 * 192 + 256 * 576 + 256 * 192 + 256 * 4


def debug_attn_block(x, gn_w, gn_b, qkv_w, qkv_b, proj_w, proj_b, want_dbg=False):
    """The fused attention block (csrc/attn_tc.cu) in isolation.  x NHWC fp32 [B,16,16,192] on CUDA, weights in the
    PyTorch layouts.  Returns (out NHWC fp32, dbg dict of image-0 intermediates or None)."""
    L = _cabi.lib()
    B = x.shape[0]
    out = torch.full((B, 16, 16, 192), float("nan"), device="cuda")
    dbg = torch.zeros((ATTN_DBG_FLOATS,), device="cuda") if want_dbg else None
    ts = [t.contiguous().float().cuda() for t in (x, gn_w, gn_b, qkv_w.reshape(576, 192), qkv_b, proj_w.reshape(192, 192), proj_b)]
    torch.cuda.synchronize()
    _cabi.check(L.tcs_debug_attn_block(B, *[t.data_ptr() for t in ts], out.data_ptr(),
                                       None if dbg is None else dbg.data_ptr(), None))
    torch.cuda.synchronize()
    d = None
    if dbg is not None:
        o = [0, 256 * 192, 256 * 192 + 256 * 576, 256 * 192 + 256 * 576 + 256 * 192]
        d = {"xn": dbg[o[0]:o[1]].reshape(256, 192), "qkv": dbg[o[1]:o[2]].reshape(256, 576),
             "y": dbg[o[2]:o[3]].reshape(256, 192), "l": dbg[o[3]:ATTN_DBG_FLOATS].reshape(256, 4)}
    return out, d


def attn_block_reference(x, gn_w, gn_b, qkv_w, qkv_b, proj_w, proj_b):
    """fp64 SelfAttention2d.forward (sde_score_model.py:136-167) on NHWC input; returns NHWC out + the intermediates."""
    B = x.shape[0]
    xd = x.double().permute(0, 3, 1, 2)
    xn = F.group_norm(xd, 8, gn_w.double(), gn_b.double(), eps=1e-5)
    qkv = F.conv2d(xn, qkv_w.double().reshape(576, 192, 1, 1), qkv_b.double())
    q, k, v = torch.chunk(qkv, 3, dim=1)
    sh = lambda t: t.reshape(B, 4, 48, 256).transpose(2, 3)
    y = F.scaled_dot_product_attention(sh(q), sh(k), sh(v))
    y = y.transpose(2, 3).contiguous().reshape(B, 192, 16, 16)
    out = xd + F.conv2d(y, proj_w.double().reshape(192, 192, 1, 1), proj_b.double())
    to_tok = lambda t: t.permute(0, 2, 3, 1).reshape(B, 256, -1)
    return out.permute(0, 2, 3, 1).contiguous(), {"xn": to_tok(xn), "qkv": to_tok(qkv), "y": to_tok(y)}


def debug_conv_ups(in_lo, w, b):
    """conv3x3_circular(bilinear x2 (in_lo)) with the upsample fused into the tcgen05 conv.  in_lo NHWC fp32 CUDA."""
    L = _cabi.lib()
    B, h, wd, cin = in_lo.shape
    cout = w.shape[0]
    out = torch.full((B, 2 * h, 2 * wd, cout), float("nan"), device="cuda")
    torch.cuda.synchronize()
    _cabi.check(L.tcs_debug_conv_ups(B, 2 * h, 2 * wd, cin, cout, in_lo.contiguous().data_ptr(), w.contiguous().data_ptr(),
                                     b.data_ptr(), out.data_ptr(), None))
    torch.cuda.synchronize()
    return out


def debug_layer(m: CondUNetTiny, name, x, t, y_cat, y_cont, C_out, res, uncond=0):
    """One layer's output of a network pass over x (NHWC fp32).  uncond=1 runs the CFG batch: 2n rows alternating
    conditional / unconditional; its "eps" tap is the guided eps (guidance 1.5) of the n samples."""
    h = m.engine_handle()
    n = x.shape[0]
    rows = n * (2 if uncond and name != "eps" else 1)
    out = torch.full((rows, res, res, C_out), float("nan"), device="cuda")
    got = _cabi.lib().tcs_debug_layer(h, name.encode(), x.data_ptr(), t.data_ptr(), y_cat.data_ptr(), y_cont.data_ptr(),
                                      n, 1 if uncond else 0, out.data_ptr(), out.numel(), None)
    if got < 0:
        _cabi.check(int(got))
    torch.cuda.synchronize()
    assert got == out.numel(), (name, got, out.numel())
    return out


# layer name -> (channels, resolution, is post-activation tap)
LAYERS = [
    ("down1.net.0.raw", 96, 64), ("down1.net.0.act", 96, 64), ("down1.net.3.raw", 96, 64), ("down1.net.3.act", 96, 64),
    ("ds1", 96, 32), ("down2.net.0.raw", 192, 32), ("down2.net.0.act", 192, 32), ("down2.net.3.raw", 192, 32),
    ("down2.net.3.act", 192, 32), ("ds2", 192, 16), ("mid.net.0.raw", 192, 16), ("mid.net.0.act", 192, 16),
    ("mid.net.3.raw", 192, 16), ("mid.net.3.act", 192, 16), ("attn", 192, 16), ("us2_conv", 192, 32),
    ("up2.net.0.raw", 96, 32), ("up2.net.0.act", 96, 32), ("up2.net.3.raw", 96, 32), ("up2.net.3.act", 96, 32),
    ("us1_conv", 96, 64), ("up1.net.0.raw", 96, 64), ("up1.net.0.act", 96, 64), ("up1.net.3.raw", 96, 64),
    ("up1.net.3.act", 96, 64),
]
