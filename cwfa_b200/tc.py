"""Tensor-core side: C8 half-precision tensors, packed weights and the tcgen05 convolution wrapper.

C8 layout: [N][Cp/8][H][W][8] bf16 (default) or fp16, Cp = channels rounded up to a multiple of 16.
"""
from __future__ import annotations

from typing import Optional

import torch

from . import _lib
from .ops import _ck, _p, _stream

_DTYPES = {"bf16": (torch.bfloat16, 1), "fp16": (torch.float16, 0)}


def pad16(c: int) -> int:
    return (c + 15) // 16 * 16


class C8:
    """A (N, C, H, W) activation stored as [N][Cp/8][H][W][8] half precision."""

    __slots__ = ("data", "C", "kind")

    def __init__(self, data: torch.Tensor, C: int, kind: str):
        self.data, self.C, self.kind = data, C, kind

    @property
    def N(self): return self.data.shape[0]
    @property
    def Cp(self): return self.data.shape[1] * 8
    @property
    def H(self): return self.data.shape[2]
    @property
    def W(self): return self.data.shape[3]
    @property
    def is_bf16(self): return _DTYPES[self.kind][1]

    @staticmethod
    def empty(N, C, H, W, device, kind="bf16", Cp: Optional[int] = None) -> "C8":
        Cp = pad16(C) if Cp is None else Cp
        return C8(torch.empty((N, Cp // 8, H, W, 8), device=device, dtype=_DTYPES[kind][0]), C, kind)


def to_c8(x: torch.Tensor, kind: str = "bf16", Cp: Optional[int] = None) -> C8:
    x = _ck(x, "x")
    N, C, H, W = x.shape
    out = C8.empty(N, C, H, W, x.device, kind, Cp)
    _lib.call("cwfa_nchw_to_c8", x.data_ptr(), out.data.data_ptr(), N, C, out.Cp, H * W, out.is_bf16, _stream())
    return out


def from_c8(x: C8) -> torch.Tensor:
    y = torch.empty((x.N, x.C, x.H, x.W), device=x.data.device, dtype=torch.float32)
    _lib.call("cwfa_c8_to_nchw", x.data.data_ptr(), y.data_ptr(), x.N, x.C, x.Cp, x.H * x.W, x.is_bf16, _stream())
    return y


def dy_prep(dy: torch.Tensor, y: Optional[torch.Tensor], kind: str, *, want_f32: bool = False, want_bias: bool = False):
    """One pass over a convolution's output cotangent (autograd of ``nn.Conv2d``): ``g = dy * ELU'(y)`` (``y`` given) or ``dy``,
    returned as the C8 tensor the data / weight gradient kernels read, optionally as fp32 NCHW, plus its per-channel sums
    (the bias gradient).  Returns ``(g8, g32 or None, db or None)``."""
    dy = _ck(dy, "dy")
    N, C, H, W = dy.shape
    g8 = C8.empty(N, C, H, W, dy.device, kind)
    g32 = torch.empty_like(dy) if want_f32 else None
    db = ws = None
    if want_bias:
        db = torch.empty(C, device=dy.device, dtype=torch.float32)
        ws = torch.empty(_lib.load().cwfa_dy_prep_workspace_floats(N, g8.Cp), device=dy.device, dtype=torch.float32)
    _lib.call("cwfa_dy_prep", dy.data_ptr(), None if y is None else _ck(y, "y").data_ptr(), g8.data.data_ptr(), _p(g32), _p(db), _p(ws),
              N, C, g8.Cp, H * W, g8.is_bf16, _stream())
    return g8, g32, db


def prelu_c8(x: C8, slope: torch.Tensor) -> C8:
    """PReLU with a scalar slope (read on the device) on a C8 tensor."""
    y = C8(torch.empty_like(x.data), x.C, x.kind)
    _lib.call("cwfa_c8_prelu", x.data.data_ptr(), _ck(slope.detach(), "slope").data_ptr(), y.data.data_ptr(), x.N, x.Cp, x.H * x.W,
              x.is_bf16, _stream())
    return y


def prelu_bwd_c8(dy: C8, pre: C8, slope: torch.Tensor):
    """Adjoint of ``prelu_c8``: ``g = dy * PReLU'(pre)`` (C8) and ``stats`` (2 * Cp,): per-channel ``sum g`` then per-channel
    ``sum dy * min(pre, 0)`` (summed over channels = the slope gradient)."""
    if dy.data.shape != pre.data.shape or dy.kind != pre.kind:
        raise ValueError("prelu_bwd_c8: layout mismatch")
    g = C8(torch.empty_like(dy.data), dy.C, dy.kind)
    stats = torch.empty(2 * dy.Cp, device=dy.data.device, dtype=torch.float32)
    ws = torch.empty(_lib.load().cwfa_c8_stats_workspace_floats(dy.Cp), device=dy.data.device, dtype=torch.float32)
    _lib.call("cwfa_c8_prelu_bwd", dy.data.data_ptr(), pre.data.data_ptr(), _ck(slope.detach(), "slope").data_ptr(), g.data.data_ptr(),
              stats.data_ptr(), ws.data_ptr(), dy.N, dy.Cp, dy.H * dy.W, dy.is_bf16, _stream())
    return g, stats


def elu_bwd_c8(dy: C8, y: C8):
    """ELU adjoint from the activation's output: ``g = dy * (y > 0 ? 1 : y + 1)`` (C8) and ``stats`` whose first Cp entries are
    the per-channel sums of g."""
    if dy.data.shape != y.data.shape or dy.kind != y.kind:
        raise ValueError("elu_bwd_c8: layout mismatch")
    g = C8(torch.empty_like(dy.data), dy.C, dy.kind)
    stats = torch.empty(2 * dy.Cp, device=dy.data.device, dtype=torch.float32)
    ws = torch.empty(_lib.load().cwfa_c8_stats_workspace_floats(dy.Cp), device=dy.data.device, dtype=torch.float32)
    _lib.call("cwfa_c8_elu_bwd", dy.data.data_ptr(), y.data.data_ptr(), g.data.data_ptr(), stats.data_ptr(), ws.data_ptr(),
              dy.N, dy.Cp, dy.H * dy.W, dy.is_bf16, _stream())
    return g, stats


def channel_sums_c8(x: C8) -> torch.Tensor:
    """Per-channel sums over (N, H, W) of a C8 tensor -> (Cp,) fp32 (deterministic two-stage reduction)."""
    stats = torch.empty(2 * x.Cp, device=x.data.device, dtype=torch.float32)
    ws = torch.empty(_lib.load().cwfa_c8_stats_workspace_floats(x.Cp), device=x.data.device, dtype=torch.float32)
    _lib.call("cwfa_c8_channel_stats", x.data.data_ptr(), stats.data_ptr(), ws.data_ptr(), x.N, x.Cp, x.H * x.W, x.is_bf16, _stream())
    return stats[:x.Cp]


def pick_bn(cout_p: int) -> int:
    """Largest legal N tile (multiple of 16, <= 256) that divides the padded output channels."""
    for bn in (256, 128, 96, 64, 48, 32, 16):
        if cout_p % bn == 0:
            return bn
    raise ValueError(cout_p)


class PackedConv:
    """Weights of one Conv2d packed for the streamed B operand, plus padded bias."""

    def __init__(self, weight: torch.Tensor, bias: Optional[torch.Tensor], kind: str = "bf16", bn: Optional[int] = None,
                 cin_p: Optional[int] = None, transposed: bool = False):
        w = _ck(weight.detach(), "weight")
        if transposed:                      # ConvTranspose2d(k=2,s=2): (Cin, Cout, 2, 2) -> 1x1 conv to 4*Cout_p channels
            Cin, Cout = w.shape[0], w.shape[1]
            KH = KW = 1
        else:
            Cout, Cin, KH, KW = w.shape
        self.Cin, self.Cout, self.KH, self.KW, self.kind = Cin, Cout, KH, KW, kind
        self.transposed = transposed
        self.Cin_p = pad16(Cin) if cin_p is None else cin_p
        self.Cout_p = pad16(Cout)
        tot_p = 4 * self.Cout_p if transposed else self.Cout_p
        if bn is None and transposed:
            # transposed convs: an n-block holds both horizontal sub-pixels (BN/2 channels each): BN % 32 == 0, BN | 2*Cout_p
            bn = next(c for c in (256, 192, 128, 96, 64, 32) if (2 * self.Cout_p) % c == 0)
        if bn is None:
            bn = pick_bn(tot_p)
            if self.Cin_p <= 64 and not transposed:
                # small-K convs are epilogue/bandwidth-bound; tile widths measured best on B200 (scripts/sweep_conv_tc.py)
                for cand in (256, 128, 192, 64, 160, 96, 48, 32, 16):
                    if tot_p % cand == 0:
                        bn = cand
                        break
        self.BN = bn
        self.tot_p = tot_p
        lib = _lib.load()
        n = lib.cwfa_tc_packed_weight_elems(self.Cin_p, tot_p, KH, KW, self.BN)
        if n < 0:
            raise ValueError(f"cannot pack conv Cin_p={self.Cin_p} Cout_p={tot_p} BN={self.BN}")
        self.packed = torch.empty(n, device=w.device, dtype=_DTYPES[kind][0])
        _lib.call("cwfa_tc_pack_weights", w.data_ptr(), self.packed.data_ptr(), Cout, Cin, KH, KW, self.Cin_p, self.Cout_p,
                  self.BN, int(transposed), _DTYPES[kind][1], _stream())
        self.bias = None
        if bias is not None:
            b = torch.zeros(tot_p, device=w.device, dtype=torch.float32)
            if transposed:
                # column order of the packed transposed weights: n-block = (row sub-pixel i, channel block of BN/2),
                # columns [j = 0 half | j = 1 half] (see pack_weights_kernel)
                hb = self.BN // 2
                bp = torch.zeros(self.Cout_p, device=w.device, dtype=torch.float32)
                bp[:Cout] = bias.detach().float()
                b.view(2, self.Cout_p // hb, 2, hb)[:] = bp.view(1, self.Cout_p // hb, 1, hb)
            else:
                b[:Cout] = bias.detach().float()
            self.bias = b


def _conv_mb(pc: PackedConv, W: int, mb: Optional[int]) -> int:
    """M-blocks per tile of ``conv_tc``: ``mb`` if given, else the default for the packed tile width and the image width."""
    if mb is not None:
        return mb
    if pc.BN >= 192 and pc.Cin_p <= 64:
        return 1          # small-K, wide-N: 128-pixel tiles keep two CTAs per SM (<= 256 TMEM columns each)
    return 2 if (pc.BN * 2 <= 512 and W > 8) else 1


def conv_tc(x: C8, pc: PackedConv, *, act: int = 0, slope: Optional[torch.Tensor] = None, res=None, res_mode: int = 0,
            out_nchw: bool = False, mb: Optional[int] = None):
    """Implicit-GEMM convolution on the tensor cores.  Returns a C8 tensor (or NCHW fp32 if out_nchw)."""
    if x.Cp != pc.Cin_p or x.kind != pc.kind:
        raise ValueError(f"conv_tc: input has Cp={x.Cp}/{x.kind}, weights expect Cin_p={pc.Cin_p}/{pc.kind}")
    if pc.transposed:
        raise ValueError("use conv_transpose_tc for transposed weights")
    N, H, W = x.N, x.H, x.W
    mb = _conv_mb(pc, W, mb)
    dev = x.data.device
    if out_nchw:
        out = torch.empty((N, pc.Cout, H, W), device=dev, dtype=torch.float32)
        out_ptr, res_ptr = out.data_ptr(), (None if res is None else _ck(res, "res").data_ptr())
    else:
        out = C8.empty(N, pc.Cout, H, W, dev, x.kind, pc.Cout_p)
        out_ptr, res_ptr = out.data.data_ptr(), (None if res is None else res.data.data_ptr())
        if res is not None and (res.Cp != pc.Cout_p or res.kind != x.kind):
            raise ValueError("conv_tc: residual layout mismatch")
    slope_t = None if slope is None else _ck(slope.detach(), "slope")
    _lib.call("cwfa_conv_tc", x.data.data_ptr(), pc.packed.data_ptr(), _p(pc.bias), _p(slope_t), res_ptr, out_ptr,
              N, H, W, pc.Cin_p, pc.Cout, pc.Cout_p, pc.KH, pc.KW, pc.BN, mb, act, res_mode if res is not None else 0,
              1 if out_nchw else 0, x.is_bf16, _stream())
    return out


def conv_tc_plan(x: C8, pc: PackedConv, *, act: int = 0, slope: Optional[torch.Tensor] = None, res_mode: int = 0,
                 out_nchw: bool = False, mb: Optional[int] = None, stats: bool = False, coupling=None) -> dict:
    """The launch plan of ``conv_tc`` (``stats``: of ``conv_tc_bn_stats``' fused-statistics launch) with these arguments, as
    the library computes it; ``coupling = (inverse, external_shift)`` asks for ``conv_tc_coupling(persistent=False)`` instead.
    Keys: ki (kernel index 0-25, see include/cwfa_b200.h), a_stages, b_stages, resident, acc_bufs, wide, grid, items, smem."""
    import ctypes as C
    if coupling is None:
        out_mode, bn, mb = (1 if out_nchw else 0), pc.BN, _conv_mb(pc, x.W, mb)
        inv = ext = 0
    else:
        out_mode, bn, mb = 3, pc.Cout_p, (mb if mb is not None else (2 if x.W > 8 else 1))
        inv, ext = int(bool(coupling[0])), int(bool(coupling[1]))
    v = (C.c_int * 9)()
    _lib.call("cwfa_conv_tc_plan", x.N, x.H, x.W, pc.Cin_p, pc.Cout_p, pc.KH, pc.KW, bn, mb, act, res_mode, out_mode,
              int(slope is not None), int(stats), inv, ext, x.is_bf16, v)
    return dict(zip(("ki", "a_stages", "b_stages", "resident", "acc_bufs", "wide", "grid", "items", "smem"), list(v)))


def conv_tc_bn_stats(x: C8, pc: PackedConv, *, act: int = 0, slope: Optional[torch.Tensor] = None, mb: Optional[int] = None):
    """``conv_tc`` (C8 out, no residual, act none / PReLU) that also accumulates the BatchNorm statistics of its activated
    output in the epilogue.  Returns (out, partial, MB) -- feed ``partial`` to ``batchnorm_c8(..., partial=...)`` -- or
    (out, None, MB) when the shape does not use the wide kernel (the caller then runs the separate statistics pass)."""
    if x.Cp != pc.Cin_p or x.kind != pc.kind or pc.transposed:
        raise ValueError("conv_tc_bn_stats: input / weight layout mismatch")
    N, H, W = x.N, x.H, x.W
    mb = _conv_mb(pc, W, mb)
    if mb * pc.BN <= 256 or pc.Cout_p != pc.Cout:
        return conv_tc(x, pc, act=act, slope=slope, mb=mb), None, mb
    dev = x.data.device
    out = C8.empty(N, pc.Cout, H, W, dev, x.kind, pc.Cout_p)
    part = torch.empty(_lib.load().cwfa_conv_tc_stats_floats(N, H, W, pc.Cout_p, mb), device=dev, dtype=torch.float32)
    slope_t = None if slope is None else _ck(slope.detach(), "slope")
    _lib.call("cwfa_conv_tc_bn", x.data.data_ptr(), pc.packed.data_ptr(), _p(pc.bias), _p(slope_t), out.data.data_ptr(), N, H, W,
              pc.Cin_p, pc.Cout, pc.Cout_p, pc.KH, pc.KW, pc.BN, mb, act, x.is_bf16, part.data_ptr(), _stream())
    return out, part, mb


def conv_transpose_tc(x: C8, pc: PackedConv, skip: Optional[C8] = None, mb: Optional[int] = None) -> C8:
    """ConvTranspose2d(k=2,s=2) (+ skip add) on the tensor cores: 1x1 conv to 4*Cout_p channels whose epilogue
    scatters each channel block to its (i,j) sub-pixel of the (2H,2W) output (unet.py:166,190)."""
    if not pc.transposed:
        raise ValueError("conv_transpose_tc needs weights packed with transposed=True")
    if x.Cp != pc.Cin_p or x.kind != pc.kind:
        raise ValueError("conv_transpose_tc: input layout mismatch")
    N, H, W = x.N, x.H, x.W
    if mb is None:
        mb = 2 if (pc.BN * 2 <= 512 and W > 8) else 1
    out = C8.empty(N, pc.Cout, 2 * H, 2 * W, x.data.device, x.kind, pc.Cout_p)
    if skip is not None and (skip.Cp != pc.Cout_p or skip.H != 2 * H or skip.W != 2 * W):
        raise ValueError("conv_transpose_tc: skip tensor shape mismatch")
    _lib.call("cwfa_conv_tc", x.data.data_ptr(), pc.packed.data_ptr(), _p(pc.bias), None,
              None if skip is None else skip.data.data_ptr(), out.data.data_ptr(),
              N, H, W, pc.Cin_p, pc.Cout, pc.Cout_p, 1, 1, pc.BN, mb, 0, 1 if skip is not None else 0, 2, x.is_bf16, _stream())
    return out


def batchnorm_c8(x: C8, gamma, beta, running_mean, running_var, *, batch_stats: bool, eps: float = 1e-5,
                 pool: bool = False, partial=None):
    """BatchNorm2d on a C8 tensor (batch or running statistics); optionally also returns the 2x2 max-pooled
    tensor (fused).  Channels must not be padded (Cp == C), true for the U-Net widths 256/512/1024.
    ``partial`` = (partial statistics, MB) from ``conv_tc_bn_stats``: the statistics pass over the tensor is skipped."""
    if x.Cp != x.C:
        raise ValueError("batchnorm_c8: padded channel layouts are not supported")
    dev = x.data.device
    Cp, N, H, W = x.Cp, x.N, x.H, x.W
    lib = _lib.load()
    if batch_stats and partial is not None and partial[0] is not None:
        scale = torch.empty(Cp, device=dev, dtype=torch.float32)
        shift = torch.empty(Cp, device=dev, dtype=torch.float32)
        _lib.call("cwfa_bn_partial_finalize", partial[0].data_ptr(), N, H, W, Cp, int(partial[1]), _ck(gamma.detach()).data_ptr(),
                  _ck(beta.detach()).data_ptr(), float(eps), scale.data_ptr(), shift.data_ptr(), None, _stream())
        y = C8.empty(N, x.C, H, W, dev, x.kind, Cp)
        yp = C8.empty(N, x.C, H // 2, W // 2, dev, x.kind, Cp) if pool else None
        _lib.call("cwfa_c8_bn_apply", x.data.data_ptr(), scale.data_ptr(), shift.data_ptr(), y.data.data_ptr(),
                  None if yp is None else yp.data.data_ptr(), N, Cp, H, W, x.is_bf16, _stream())
        return (y, yp) if pool else y
    scale = torch.empty(Cp, device=dev, dtype=torch.float32)
    shift = torch.empty(Cp, device=dev, dtype=torch.float32)
    if batch_stats:                                          # statistics pass + ONE finalize launch straight to scale / shift
        ws = torch.empty(lib.cwfa_c8_stats_workspace_floats(Cp), device=dev, dtype=torch.float32)
        _lib.call("cwfa_c8_bn_batch_scale_shift", x.data.data_ptr(), _ck(gamma.detach()).data_ptr(), _ck(beta.detach()).data_ptr(),
                  float(eps), scale.data_ptr(), shift.data_ptr(), ws.data_ptr(), N, Cp, H * W, x.is_bf16, _stream())
    else:
        rm, rv = _ck(running_mean.detach()), _ck(running_var.detach())
        stats = torch.cat([rm, rv + rm * rm]).contiguous()
        _lib.call("cwfa_bn_finalize_f32", stats.data_ptr(), _ck(gamma.detach()).data_ptr(), _ck(beta.detach()).data_ptr(),
                  scale.data_ptr(), shift.data_ptr(), Cp, 1.0, float(eps), _stream())
    y = C8.empty(N, x.C, H, W, dev, x.kind, Cp)
    yp = C8.empty(N, x.C, H // 2, W // 2, dev, x.kind, Cp) if pool else None
    _lib.call("cwfa_c8_bn_apply", x.data.data_ptr(), scale.data_ptr(), shift.data_ptr(), y.data.data_ptr(),
              None if yp is None else yp.data.data_ptr(), N, Cp, H, W, x.is_bf16, _stream())
    return (y, yp) if pool else y


def layernorm_c8(x: C8, gamma8: C8, beta8: C8, eps: float = 1e-5) -> C8:
    """LayerNorm([C,H,W]) with element-wise affine parameters (networks.py:486-503) on a C8 tensor; ``gamma8`` / ``beta8`` are
    the parameters converted once with ``to_c8(param[None], kind)``."""
    if gamma8.Cp != x.Cp or beta8.Cp != x.Cp or gamma8.H != x.H or gamma8.W != x.W or gamma8.kind != x.kind or beta8.kind != x.kind:
        raise ValueError("layernorm_c8: parameter layout mismatch")
    y = C8.empty(x.N, x.C, x.H, x.W, x.data.device, x.kind, x.Cp)
    ws = torch.empty(_lib.load().cwfa_c8_layernorm_workspace_floats(x.N), device=x.data.device, dtype=torch.float32)
    _lib.call("cwfa_c8_layernorm", x.data.data_ptr(), gamma8.data.data_ptr(), beta8.data.data_ptr(), y.data.data_ptr(),
              ws.data_ptr(), x.N, x.C, x.Cp, x.H * x.W, float(eps), x.is_bf16, _stream())
    return y


def col2im3x3_weights(w: torch.Tensor) -> torch.Tensor:
    """(Cout, Cin, 3, 3) conv weights -> (9 * ceil8(Cout), Cin, 1, 1) weights of the 1x1 convolution whose output
    channel ``(co // 8) * 72 + (ky * 3 + kx) * 8 + co % 8`` is the tap-(ky,kx) partial product of output channel co
    (``col2im3x3_c8`` sums the nine shifted partials)."""
    Cout, Cin = w.shape[0], w.shape[1]
    C8n = (Cout + 7) // 8
    wp = torch.zeros(C8n * 8, Cin, 3, 3, device=w.device, dtype=torch.float32)
    wp[:Cout] = w.detach().float()
    # [chunk, j, Cin, tap] -> [chunk, tap, j, Cin]
    g = wp.view(C8n, 8, Cin, 9).permute(0, 3, 1, 2).reshape(C8n * 72, Cin, 1, 1)
    return g.contiguous()


def col2im3x3_c8(g: C8, bias: Optional[torch.Tensor], C: int) -> C8:
    """Sums the nine shifted tap partials of ``conv_tc(x, PackedConv(col2im3x3_weights(w)))`` into the 3x3 convolution
    output (C channels, zero padding) + bias."""
    Dp = pad16(C)
    if g.Cp < 9 * ((C + 7) // 8) * 8:
        raise ValueError("col2im3x3_c8: partial-product tensor too narrow")
    out = C8.empty(g.N, C, g.H, g.W, g.data.device, g.kind, Dp)
    b = None
    if bias is not None:
        if bias.numel() == Dp and bias.dtype == torch.float32:
            b = _ck(bias.detach(), "bias")          # already padded (hot path: no per-call fill kernels)
        else:
            b = torch.zeros(Dp, device=g.data.device, dtype=torch.float32)
            b[:C] = bias.detach().float()
    _lib.call("cwfa_c8_col2im3x3", g.data.data_ptr(), _p(b), out.data.data_ptr(), g.N, Dp, g.Cp, g.H, g.W, g.is_bf16, _stream())
    return out


class StencilWeights:
    """Operands of ``stencil3d_tc``: the two Conv3d kernels of the conditioning net's depth stencil (networks.py:221-225) packed
    for the fused true-3-D kernel (csrc/stencil_tc.cu; layout in include/cwfa_b200.h)."""

    def __init__(self, w1: torch.Tensor, b1: torch.Tensor, w2: torch.Tensor, b2: torch.Tensor, kind: str = "bf16"):
        w1, b1 = w1.detach().float(), b1.detach().float()           # (Cm, 1, 3, 3, 3) [kh, kw, kd], (Cm)
        w2, b2 = w2.detach().float(), b2.detach().float()           # (1, Cm, 3, 3, 3), (1)
        Cm = w1.shape[0]
        if Cm != 32 or tuple(w1.shape[1:]) != (1, 3, 3, 3) or tuple(w2.shape) != (1, Cm, 3, 3, 3):
            raise ValueError("StencilWeights: needs Conv3d(1, 32, 3) -> Conv3d(32, 1, 3)")
        dt = _DTYPES[kind][0]
        dev = w1.device
        A = torch.zeros(3, Cm, 16, device=dev)                       # [kd][hidden n][k]: k = kh*3+kw < 9
        A[:, :, :9] = w1[:, 0].permute(3, 0, 1, 2).reshape(3, Cm, 9)
        hi = b1.to(dt).float()
        A[1, :, 9], A[1, :, 10] = hi, b1 - hi                        # fp32-accurate bias: [hi | lo] against two 1.0 columns (centre tap)
        W1 = A.view(3, Cm, 2, 8).permute(0, 2, 1, 3)                 # [kd][chunk][n][8]
        B = torch.zeros(3, 16, Cm, device=dev)                       # [kd][n = kh*3+kw][k = c]
        B[:, :9] = w2[0].permute(3, 1, 2, 0).reshape(3, 9, Cm)       # w2[c, kh, kw, kd] -> [kd][kh*3+kw][c]
        W2 = B.view(3, 16, 4, 8).permute(0, 2, 1, 3)                 # [kd][chunk][n][8]
        self.packed = torch.cat([W1.reshape(-1), W2.reshape(-1)]).to(dt).contiguous()
        self.b2 = b2.reshape(1).contiguous()
        self.kind = kind


def stencil3d_tc(x: C8, sw: StencilWeights, slope: torch.Tensor, D: int, rows_max: int = 0) -> C8:
    """Depth stencil of the conditioning net, fused: ``Conv3d(1,32,3) -> PReLU(slope) -> Conv3d(32,1,3)`` over (H, W, depth) of the
    first ``D`` channels of ``x`` (networks.py:239).  ``slope`` is the (1,) PReLU parameter, read on the device."""
    if x.kind != sw.kind or D > x.Cp or slope.numel() != 1:
        raise ValueError("stencil3d_tc: kind / depth mismatch or a per-channel PReLU")
    out = C8.empty(x.N, D, x.H, x.W, x.data.device, x.kind, pad16(D))
    _lib.call("cwfa_stencil3d_tc", x.data.data_ptr(), out.data.data_ptr(), sw.packed.data_ptr(), sw.b2.data_ptr(),
              _ck(slope.detach(), "slope").data_ptr(), x.N, x.H, x.W, D, x.Cp // 8, out.Cp // 8, rows_max, x.is_bf16, _stream())
    return out


def resblock_tc(x: C8, p3: PackedConv, p1: PackedConv, in_chunk_off: int = 0) -> C8:
    """Fused trunk residual block y = ELU(conv1x1(ELU(conv3x3(x))) + x) for 64 channels (one persistent kernel).
    ``x`` may be a wider C8 tensor; ``in_chunk_off`` selects the 64-channel slice (8 chunks) to read."""
    for pc, k in ((p3, 3), (p1, 1)):
        if pc.Cin_p != 64 or pc.Cout_p != 64 or pc.BN != 64 or pc.KH != k or pc.bias is None or pc.kind != x.kind:
            raise ValueError("resblock_tc: needs 64->64 convs (3x3 then 1x1) packed with BN=64 and biases")
    if x.Cp < 64 or in_chunk_off * 8 + 64 > x.Cp:
        raise ValueError("resblock_tc: input slice out of range")
    y = C8.empty(x.N, 64, x.H, x.W, x.data.device, x.kind, 64)
    _lib.call("cwfa_resblock_tc", x.data.data_ptr(), y.data.data_ptr(), p3.packed.data_ptr(), p1.packed.data_ptr(),
              p3.bias.data_ptr(), p1.bias.data_ptr(), x.N, x.H, x.W, x.Cp // 8, in_chunk_off, 8, 0, x.is_bf16, _stream())
    return y


def conv_tc_coupling(b: C8, pc: PackedConv, x: Optional[torch.Tensor], *, ch: int, inverse: bool, clamp: float = 2.0,
                     k_atan: float = 0.636, t_ext: Optional[torch.Tensor] = None, t_scale: float = 1.0,
                     perm: Optional[torch.Tensor] = None, perm_axis: int = 0, logdet: torch.Tensor = None,
                     sumsq: Optional[torch.Tensor] = None, accumulate: bool = True, mb: Optional[int] = None,
                     persistent: Optional[bool] = None, ticket: Optional[torch.Tensor] = None, chunk_off: int = 0) -> torch.Tensor:
    """Last conv of a coupling sub-network with the affine coupling, the log-det partial sums and the preceding
    permutation (as a gather on ``x``) fused into its epilogue.  ``x`` None = zeros (z = 0, inverse only).
    ``logdet`` (B,) is accumulated in place (fixed-order reduction); ``sumsq`` (B,) receives sum(y^2).
    ``ticket``: one zero int32 on the device (the kernel leaves it zero); with it the persistent kernel reduces its partial
    sums itself (last CTA, fixed order) instead of a separate finalize launch."""
    if (b.Cp != pc.Cin_p and not (pc.Cin_p == 64 and chunk_off * 8 + 64 <= b.Cp)) or b.kind != pc.kind:
        raise ValueError("conv_tc_coupling: input layout mismatch")
    need = ch if t_ext is not None else 2 * ch
    if pc.Cout != need or pc.BN != pc.Cout_p:
        raise ValueError(f"conv_tc_coupling: weights give {pc.Cout} channels (BN {pc.BN}), need {need} in one N block")
    N, H, W = b.N, b.H, b.W
    if mb is None:
        mb = 2 if W > 8 else 1
    dev = b.data.device
    y = torch.empty((N, ch, H, W), device=dev, dtype=torch.float32)
    xx = None if x is None else _ck(x, "x")
    tt = None if t_ext is None else _ck(t_ext, "t_ext")
    lib = _lib.load()
    if persistent is None:
        persistent = pc.Cin_p == 64 and pc.KH == 3 and pc.KW == 3 and pc.Cout_p <= 96 and ch <= 48
    if (b.Cp != pc.Cin_p or chunk_off) and not persistent:
        raise ValueError("conv_tc_coupling: a channel slice of a wider tensor needs the persistent kernel")
    if persistent:
        tiles = lib.cwfa_coupling_tc_tiles(H, W)
        ws = torch.empty(2 * N * tiles, device=dev, dtype=torch.float32)
        _lib.call("cwfa_coupling_tc", b.data.data_ptr(), pc.packed.data_ptr(), _p(pc.bias), N, H, W, pc.Cout, pc.Cout_p, _p(xx),
                  y.data_ptr(), _p(tt), float(t_scale), _p(perm), int(perm_axis), ch, float(clamp), float(k_atan), int(inverse),
                  ws.data_ptr(), logdet.data_ptr(), _p(sumsq), int(accumulate), _p(ticket), b.Cp // 8, int(chunk_off), b.is_bf16, _stream())
        if ticket is None:
            _lib.call("cwfa_coupling_finalize", ws.data_ptr(), logdet.data_ptr(), _p(sumsq), N, tiles, int(accumulate), _stream())
        return y
    tiles = lib.cwfa_conv_tc_coupling_tiles(H, W, mb)
    ws = torch.empty(2 * N * tiles, device=dev, dtype=torch.float32)
    _lib.call("cwfa_conv_tc_coupling", b.data.data_ptr(), pc.packed.data_ptr(), _p(pc.bias), N, H, W, pc.Cin_p, pc.Cout,
              pc.Cout_p, pc.KH, pc.KW, mb, _p(xx), y.data_ptr(), _p(tt), float(t_scale), _p(perm), int(perm_axis), ch,
              float(clamp), float(k_atan), int(inverse), ws.data_ptr(), b.is_bf16, _stream())
    _lib.call("cwfa_coupling_finalize", ws.data_ptr(), logdet.data_ptr(), _p(sumsq), N, tiles, int(accumulate), _stream())
    return y


# ---------------------------------------------------------------------------------------------------------------------
# F8: the detail half of a flow level as [N][ceil(ch/8)][H][W][8] fp32 (csrc/coupling_f8.cu) -- the engine's coupling state
# ---------------------------------------------------------------------------------------------------------------------
def ch8(ch: int) -> int:
    return (ch + 7) // 8 * 8


def _i32(t: Optional[torch.Tensor], device) -> Optional[torch.Tensor]:
    return None if t is None else t.to(device=device, dtype=torch.int32).contiguous()


def to_f8(x: torch.Tensor, chan_map: Optional[torch.Tensor] = None) -> torch.Tensor:
    """(N,C,H,W) fp32 -> F8 (N, ceil(C/8), H, W, 8); slot j holds channel ``chan_map[j]`` (identity when None)."""
    x = _ck(x, "x")
    N, C, H, W = x.shape
    y = torch.empty((N, ch8(C) // 8, H, W, 8), device=x.device, dtype=torch.float32)
    _lib.call("cwfa_nchw_to_f8", x.data_ptr(), _p(chan_map), y.data_ptr(), N, C, H * W, _stream())
    return y


def from_f8(x8: torch.Tensor, C: int, chan_map: Optional[torch.Tensor] = None) -> torch.Tensor:
    """F8 -> (N,C,H,W) fp32; channel c reads slot ``chan_map[c]`` (identity when None)."""
    N, G, H, W, _ = x8.shape
    y = torch.empty((N, C, H, W), device=x8.device, dtype=torch.float32)
    _lib.call("cwfa_f8_to_nchw", x8.data_ptr(), _p(chan_map), y.data_ptr(), N, C, H * W, _stream())
    return y


def haar1d_split_f8(x: torch.Tensor):
    """Fused DWT + Split: (B,C,H,W) -> lo (B,C/2,H,W) NCHW and the detail half in F8."""
    x = _ck(x, "x")
    B, C, H, W = x.shape
    h = C // 2
    lo = torch.empty((B, h, H, W), device=x.device, dtype=torch.float32)
    hi = torch.empty((B, ch8(h) // 8, H, W, 8), device=x.device, dtype=torch.float32)
    _lib.call("cwfa_haar1d_fwd_f8", x.data_ptr(), lo.data_ptr(), hi.data_ptr(), B, C, H * W, _stream())
    return lo, hi


def haar1d_merge_f8(lo: torch.Tensor, hi8: torch.Tensor) -> torch.Tensor:
    """Fused Split^-1 + IDWT: lo (B,h,H,W) NCHW + detail half in F8 -> (B,2h,H,W)."""
    lo = _ck(lo, "lo")
    B, h, H, W = lo.shape
    if tuple(hi8.shape) != (B, ch8(h) // 8, H, W, 8):
        raise ValueError(f"haar1d_merge_f8: detail half has shape {tuple(hi8.shape)}, expected {(B, ch8(h) // 8, H, W, 8)}")
    out = torch.empty((B, 2 * h, H, W), device=lo.device, dtype=torch.float32)
    _lib.call("cwfa_haar1d_inv_f8", lo.data_ptr(), hi8.data_ptr(), out.data_ptr(), B, 2 * h, H * W, _stream())
    return out


def coupling_weights_f8(weight: torch.Tensor, bias: torch.Tensor, ch: int, slot_to_chan: torch.Tensor, ext: bool, kind: str) -> "PackedConv":
    """Last conv of a coupling sub-network re-ordered for ``coupling_f8``: output column j (< chp8) = s of storage slot j =
    conv channel ``slot_to_chan[j]``, column chp8 + j = its t (``ext``: s only); padding slots get zero weights and bias."""
    c8 = ch8(ch)
    w, b = weight.detach().float(), bias.detach().float()
    rows = c8 if ext else 2 * c8
    wn = torch.zeros((rows,) + tuple(w.shape[1:]), device=w.device, dtype=torch.float32)
    bn_ = torch.zeros(rows, device=w.device, dtype=torch.float32)
    idx = slot_to_chan.to(w.device).long()
    wn[:ch] = w[idx]
    bn_[:ch] = b[idx]
    if not ext:
        wn[c8:c8 + ch] = w[ch + idx]
        bn_[c8:c8 + ch] = b[ch + idx]
    return PackedConv(wn, bn_, kind, bn=pad16(rows))


def coupling_f8(b: C8, pc: PackedConv, x8: Optional[torch.Tensor], *, ch: int, inverse: bool, clamp: float = 2.0, k_atan: float = 0.636,
                t_ext8: Optional[torch.Tensor] = None, t_scale: float = 1.0, perm: Optional[torch.Tensor] = None, perm_axis: int = 0,
                logdet: torch.Tensor = None, sumsq: Optional[torch.Tensor] = None, accumulate: bool = True,
                ticket: Optional[torch.Tensor] = None, chunk_off: int = 0) -> torch.Tensor:
    """``conv_tc_coupling`` on the F8 detail half (lean epilogue; channel permutations live in ``pc``'s column order).
    ``b`` may be a wider C8 tensor; ``chunk_off`` selects its 64-channel slice (8 chunks)."""
    if chunk_off * 8 + 64 > b.Cp or pc.Cin_p != 64 or pc.KH != 3 or pc.KW != 3 or b.kind != pc.kind or pc.BN != pc.Cout_p:
        raise ValueError("coupling_f8: needs a 3x3 conv from 64 hidden channels packed in one n-block")
    N, H, W = b.N, b.H, b.W
    c8 = ch8(ch)
    y = torch.empty((N, c8 // 8, H, W, 8), device=b.data.device, dtype=torch.float32)
    lib = _lib.load()
    tiles = lib.cwfa_coupling_tc_tiles(H, W)
    ws = torch.empty(2 * N * tiles, device=b.data.device, dtype=torch.float32)
    _lib.call("cwfa_coupling_f8", b.data.data_ptr(), pc.packed.data_ptr(), _p(pc.bias), N, H, W, pc.BN, c8, _p(x8), y.data_ptr(),
              _p(t_ext8), float(t_scale), _p(perm), int(perm_axis), float(clamp), float(k_atan), int(inverse), ws.data_ptr(),
              logdet.data_ptr(), _p(sumsq), int(accumulate), _p(ticket), b.Cp // 8, int(chunk_off), b.is_bf16, _stream())
    if ticket is None:
        _lib.call("cwfa_coupling_finalize", ws.data_ptr(), logdet.data_ptr(), _p(sumsq), N, tiles, int(accumulate), _stream())
    return y


NLL_MAP_FIRST, NLL_MAP_LAST = 1, 2      # cwfa_coupling_f8_map's map_mode bits (include/cwfa_b200.h)


def coupling_f8_map(b: C8, pc: PackedConv, x8: torch.Tensor, nll_map: torch.Tensor, *, ch: int, map_mode: int,
                    row_src: Optional[torch.Tensor] = None, col_src: Optional[torch.Tensor] = None, clamp: float = 2.0,
                    k_atan: float = 0.636, t_ext8: Optional[torch.Tensor] = None, t_scale: float = 1.0,
                    perm: Optional[torch.Tensor] = None, perm_axis: int = 0, logdet: torch.Tensor = None,
                    sumsq: Optional[torch.Tensor] = None, accumulate: bool = True, ticket: Optional[torch.Tensor] = None,
                    chunk_off: int = 0) -> torch.Tensor:
    """Forward ``coupling_f8`` that also accumulates each element's NLL term into ``nll_map`` (F8, the shape of ``x8``), at the
    element's coordinate at the level's input: ``(row_src[h], col_src[w])`` for the element written at ``(h, w)`` (int32 device
    tables, None = identity).  ``map_mode``: ``NLL_MAP_FIRST`` writes -s without reading the map, 0 adds -s, ``NLL_MAP_LAST``
    also adds 0.5 y^2.  The output, log-det and sumsq are bitwise ``coupling_f8``'s."""
    if chunk_off * 8 + 64 > b.Cp or pc.Cin_p != 64 or pc.KH != 3 or pc.KW != 3 or b.kind != pc.kind or pc.BN != pc.Cout_p:
        raise ValueError("coupling_f8_map: needs a 3x3 conv from 64 hidden channels packed in one n-block")
    N, H, W = b.N, b.H, b.W
    c8 = ch8(ch)
    shape = (N, c8 // 8, H, W, 8)
    if x8 is None or tuple(x8.shape) != shape or tuple(nll_map.shape) != shape or nll_map.dtype != torch.float32:
        raise ValueError(f"coupling_f8_map: x8 and nll_map must be fp32 F8 tensors of shape {shape}")
    for name, t, n_ in (("row_src", row_src, H), ("col_src", col_src, W)):
        if t is not None and (t.dtype != torch.int32 or t.numel() != n_ or not t.is_cuda or not t.is_contiguous()):
            raise ValueError(f"coupling_f8_map: {name} must be a contiguous int32 device tensor of {n_} entries")
    y = torch.empty(shape, device=b.data.device, dtype=torch.float32)
    tiles = _lib.load().cwfa_coupling_tc_tiles(H, W)
    ws = torch.empty(2 * N * tiles, device=b.data.device, dtype=torch.float32)
    _lib.call("cwfa_coupling_f8_map", b.data.data_ptr(), pc.packed.data_ptr(), _p(pc.bias), N, H, W, pc.BN, c8, x8.data_ptr(),
              y.data_ptr(), _p(t_ext8), float(t_scale), _p(perm), int(perm_axis), float(clamp), float(k_atan), 0, ws.data_ptr(),
              logdet.data_ptr(), _p(sumsq), int(accumulate), _p(ticket), b.Cp // 8, int(chunk_off), b.is_bf16, _stream(),
              nll_map.data_ptr(), _p(row_src), _p(col_src), int(map_mode))
    if ticket is None:
        _lib.call("cwfa_coupling_finalize", ws.data_ptr(), logdet.data_ptr(), _p(sumsq), N, tiles, int(accumulate), _stream())
    return y


def coupling_f8_samples(b: C8, pc: PackedConv, x8: torch.Tensor, samples: int, *, ch: int, clamp: float = 2.0, k_atan: float = 0.636,
                        t_ext8: Optional[torch.Tensor] = None, t_scale: float = 1.0, perm: Optional[torch.Tensor] = None,
                        perm_axis: int = 0, logdet: torch.Tensor = None, accumulate: bool = True,
                        ticket: Optional[torch.Tensor] = None, chunk_off: int = 0) -> torch.Tensor:
    """Inverse ``coupling_f8`` for ``samples`` latent samples of each of the ``b.N`` condition images: ``x8`` has
    ``b.N * samples`` F8 rows (row n * samples + k = sample k of image n).  s and t are evaluated once per tile for all samples;
    sample k's output is bitwise ``coupling_f8`` on row k.  ``t_ext8`` and ``logdet`` are per condition image."""
    if chunk_off * 8 + 64 > b.Cp or pc.Cin_p != 64 or pc.KH != 3 or pc.KW != 3 or b.kind != pc.kind or pc.BN != pc.Cout_p:
        raise ValueError("coupling_f8_samples: needs a 3x3 conv from 64 hidden channels packed in one n-block")
    N, H, W = b.N, b.H, b.W
    c8 = ch8(ch)
    if tuple(x8.shape) != (N * samples, c8 // 8, H, W, 8):
        raise ValueError(f"coupling_f8_samples: x8 has shape {tuple(x8.shape)}, expected {(N * samples, c8 // 8, H, W, 8)}")
    y = torch.empty_like(x8)
    tiles = _lib.load().cwfa_coupling_tc_tiles(H, W)
    ws = torch.empty(2 * N * tiles, device=b.data.device, dtype=torch.float32)
    _lib.call("cwfa_coupling_f8_samples", b.data.data_ptr(), pc.packed.data_ptr(), _p(pc.bias), N, int(samples), H, W, pc.BN, c8,
              x8.data_ptr(), y.data_ptr(), _p(t_ext8), float(t_scale), _p(perm), int(perm_axis), float(clamp), float(k_atan), 1,
              ws.data_ptr(), logdet.data_ptr(), None, int(accumulate), _p(ticket), b.Cp // 8, int(chunk_off), b.is_bf16, _stream())
    if ticket is None:
        _lib.call("cwfa_coupling_finalize", ws.data_ptr(), logdet.data_ptr(), None, N, tiles, int(accumulate), _stream())
    return y


def haar1d_merge_stats(lo: torch.Tensor, hi: torch.Tensor):
    """Split^-1 + IDWT of K >= 2 latent samples with only their statistics written: ``lo`` (K or 1, h, H, W) -- one row is
    shared by every sample -- and the K-row detail half ``hi`` in F8 (K, ceil(h/8), H, W, 8) or NCHW (K, h, H, W).  Returns
    the per-voxel mean and unbiased standard deviation of the K merged (1, 2h, H, W) volumes."""
    lo = _ck(lo, "lo")
    hi = _ck(hi, "hi")
    L, h, H, W = lo.shape
    K = hi.shape[0]
    f8 = hi.dim() == 5
    want = (K, ch8(h) // 8, H, W, 8) if f8 else (K, h, H, W)
    if tuple(hi.shape) != want or L not in (1, K):
        raise ValueError(f"haar1d_merge_stats: lo {tuple(lo.shape)} and detail half {tuple(hi.shape)} do not match")
    mean = torch.empty((1, 2 * h, H, W), device=lo.device, dtype=torch.float32)
    std = torch.empty_like(mean)
    _lib.call("cwfa_haar1d_inv_stats", lo.data_ptr(), int(L == 1), hi.data_ptr(), int(f8), mean.data_ptr(), std.data_ptr(), K, 2 * h,
              H * W, _stream())
    return mean, std


def resblock_tc_batched(x: C8, sets, in_chunk_offs=None) -> C8:
    """The fused trunk block (``resblock_tc``) for several INDEPENDENT sub-networks in one launch: ``sets`` = [(p3, p1), ...]
    (<= 5); set k reads the 64-channel slice at chunk ``in_chunk_offs[k]`` (default 8 k) of ``x`` and writes slice k of the
    returned tensor (64 * len(sets) channels)."""
    import ctypes as C
    n = len(sets)
    if not 1 <= n <= 5:
        raise ValueError("resblock_tc_batched: 1..5 weight sets")
    for p3, p1 in sets:
        for pc, k in ((p3, 3), (p1, 1)):
            if pc.Cin_p != 64 or pc.Cout_p != 64 or pc.BN != 64 or pc.KH != k or pc.bias is None or pc.kind != x.kind:
                raise ValueError("resblock_tc_batched: needs 64->64 convs (3x3 then 1x1) packed with BN=64 and biases")
    offs = [8 * k for k in range(n)] if in_chunk_offs is None else list(in_chunk_offs)
    if any(o * 8 + 64 > x.Cp for o in offs):
        raise ValueError("resblock_tc_batched: input slice out of range")
    y = C8.empty(x.N, 64 * n, x.H, x.W, x.data.device, x.kind, 64 * n)
    vps = lambda vals: (C.c_void_p * n)(*vals)
    w3, w1 = vps([s_[0].packed.data_ptr() for s_ in sets]), vps([s_[1].packed.data_ptr() for s_ in sets])
    b3, b1 = vps([s_[0].bias.data_ptr() for s_ in sets]), vps([s_[1].bias.data_ptr() for s_ in sets])
    io, oo = (C.c_int * n)(*offs), (C.c_int * n)(*[8 * k for k in range(n)])
    _lib.call("cwfa_resblock_tc_batched", x.data.data_ptr(), y.data.data_ptr(), n, w3, w1, b3, b1, x.N, x.H, x.W, x.Cp // 8, io,
              n * 8, oo, None, None, 0, x.is_bf16, _stream())
    return y


class PackedEntry:
    """The first block of a sub-network trunk folded onto the trunk's 1x1 input conv ``b = Win * lf + bin`` (no activation
    between them, networks.py:60-87), for ``resblock_tc_entry_batched``: ``W3 (*) b = (W3_tap Win) (*) lf + W3 (*) bin``.
    Composed once in fp64, then rounded to ``kind``: the 3x3 conv W3' from the Cin condition channels, the interior bias
    ``b3 + sum_tap W3_tap bin``, the acc2 bias ``b1 + bin`` and the per-edge-class sums of ``W3_tap bin`` over the taps that fall
    outside the image (the network zero-pads b, not lf)."""

    def __init__(self, w_in: torch.Tensor, b_in: torch.Tensor, w3: torch.Tensor, b3: torch.Tensor, p1: PackedConv, kind: str):
        wi, bi = w_in.detach().double(), b_in.detach().double()
        w3d = w3.detach().double()
        if wi.shape[0] != 64 or wi.shape[2:] != (1, 1) or wi.shape[1] > 64 or tuple(w3d.shape) != (64, 64, 3, 3):
            raise ValueError("PackedEntry: needs a 1x1 conv Cin (<= 64) -> 64 followed by a 3x3 conv 64 -> 64")
        if p1.Cin_p != 64 or p1.Cout_p != 64 or p1.BN != 64 or p1.KH != 1 or p1.bias is None or p1.kind != kind:
            raise ValueError("PackedEntry: needs the block's 1x1 conv 64 -> 64 packed with BN=64 and a bias")
        comp = torch.einsum("omhw,mc->ochw", w3d, wi[:, :, 0, 0])
        ctap = torch.einsum("omhw,m->hwo", w3d, bi)                           # W3_tap bin, (3, 3, 64)
        edge = torch.zeros(4, 4, 64, device=ctap.device, dtype=torch.float64)
        for r in range(4):                  # row class: bit 0 = first image row (kh = 0 out), bit 1 = last row (kh = 2 out)
            for c in range(4):              # column class: bit 0 = first column (kw = 0 out), bit 1 = last column (kw = 2 out)
                for kh in range(3):
                    for kw in range(3):
                        if (kh == 0 and r & 1) or (kh == 2 and r & 2) or (kw == 0 and c & 1) or (kw == 2 and c & 2):
                            edge[r, c] += ctap[kh, kw]
        self.kind, self.Cin = kind, wi.shape[1]
        self.p3 = PackedConv(comp.float(), None, kind, bn=64)
        self.pin = PackedConv(w_in, None, kind, bn=64)
        self.p1 = p1
        self.b3 = (b3.detach().double() + ctap.sum((0, 1))).float().contiguous()
        self.b1 = (p1.bias.double() + bi).float().contiguous()
        self.edge = edge.reshape(16, 64).float().contiguous()


def resblock_tc_entry_batched(lf: C8, entries) -> C8:
    """``ELU(W1 ELU(W3 (*) b + b3) + b1 + b)`` with ``b = Win lf + bin`` (zero-padded) for several sub-networks reading the same
    LF condition ``lf``, in one ``cwfa_resblock_tc_batched`` launch of the entry form: ``entries`` = [PackedEntry, ...] (<= 5);
    set k writes slice k of the returned tensor (64 * len(entries) channels).  b is never written."""
    import ctypes as C
    n = len(entries)
    if not 1 <= n <= 5:
        raise ValueError("resblock_tc_entry_batched: 1..5 weight sets")
    if lf.Cp > 64 or any(e.p3.Cin_p != lf.Cp or e.kind != lf.kind for e in entries):
        raise ValueError(f"resblock_tc_entry_batched: condition has Cp={lf.Cp}/{lf.kind}, the entry blocks expect another layout")
    y = C8.empty(lf.N, 64 * n, lf.H, lf.W, lf.data.device, lf.kind, 64 * n)
    vps = lambda vals: (C.c_void_p * n)(*vals)
    w3, w1, win = (vps([e.p3.packed.data_ptr() for e in entries]), vps([e.p1.packed.data_ptr() for e in entries]),
                   vps([e.pin.packed.data_ptr() for e in entries]))
    b3, b1, edge = (vps([e.b3.data_ptr() for e in entries]), vps([e.b1.data_ptr() for e in entries]),
                    vps([e.edge.data_ptr() for e in entries]))
    io, oo = (C.c_int * n)(*([0] * n)), (C.c_int * n)(*[8 * k for k in range(n)])
    _lib.call("cwfa_resblock_tc_batched", lf.data.data_ptr(), y.data.data_ptr(), n, w3, w1, b3, b1, lf.N, lf.H, lf.W, lf.Cp // 8, io,
              n * 8, oo, win, edge, lf.Cp // 8, lf.is_bf16, _stream())
    return y
