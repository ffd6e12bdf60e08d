"""Every conv_tc kernel the dispatcher can select, against F.conv2d in float64 on operands rounded to the same half-precision
grid.  ``cwfa_conv_tc_plan`` reports which of the 26 compiled variants (and which shared-memory plan, grid and item count) a
launch uses, so each case asserts the plan it was written for and the coverage test asserts that the cases reach all 26.

The resident-weights cases run at N=4, 263x270: 1156 (MB=2) or 2312 (MB=1) work items on a 296-CTA grid, so every CTA walks
several items (A-ring parity across items, both TMEM accumulator buffers), several k-blocks (the k-block offset into the resident
weight block) and an all-zero k-block that producer and issuer both skip.  Outputs go to NaN-filled buffers through the raw ABI:
a work item the kernel skipped cannot pass on stale memory."""
import ctypes
import functools

import pytest
import torch
import torch.nn.functional as F

from conftest import rel_l2
from oracle.weights import seeded_randn

DEV = "cuda:0"
ACT = {"none": 0, "prelu": 2, "nchw": 0, "elu_res": 1}      # ops.ACT_NONE / ACT_PRELU / ACT_ELU
SLOPE = 0.2
SIZES = {"res": (4, 263, 270), "ring": (2, 263, 270), "wide": (1, 40, 72)}


def _pad16(c):
    return (c + 15) // 16 * 16


# (kind, cin, cout, k, size, bn, mb, epilogue, plan, twin bn, zero k-block)
#   plan "res2" = resident weights, two TMEM buffers, several items per CTA; "res1" = the same with one buffer;
#   "ring" = streamed weights, several items per CTA; "wide" = the 576-thread kernel (> 256 TMEM columns).
#   epilogue: "none" / "prelu" = lean (C8 out, no residual); "nchw" = generic, fp32 NCHW out; "elu_res" = generic, C8 out,
#   ELU after a pre-activation residual.  twin bn: the same convolution packed with more n-blocks takes the ring path.
CASES = [
    ("bf16", 6, 6, 3, "res", 16, 2, "none", "res2", None, False),
    ("bf16", 29, 6, 3, "res", 16, 2, "prelu", "res2", None, False),
    ("bf16", 48, 48, 3, "res", 48, 2, "none", "res2", 16, False),
    ("bf16", 6, 6, 7, "res", 16, 2, "prelu", "res2", None, False),       # the LRNN's 7x7 6->6 conv
    ("bf16", 6, 192, 3, "res", 192, 1, "none", "res1", 64, False),       # MB * BN = 192: one accumulator buffer
    ("bf16", 80, 16, 3, "res", 16, 2, "none", "res2", None, False),      # 5 k-blocks of 16 channels
    ("bf16", 96, 16, 3, "res", 16, 2, "prelu", "res2", None, False),     # 2 k-blocks of 48
    ("bf16", 112, 16, 3, "res", 16, 1, "none", "res2", None, False),     # 7 k-blocks, MB = 1
    ("bf16", 96, 16, 3, "res", 16, 2, "none", "res2", None, True),       # second k-block all zero: skipped
    ("bf16", 48, 48, 3, "res", 48, 2, "nchw", "res2", 16, False),
    ("bf16", 29, 6, 3, "res", 16, 2, "elu_res", "res2", None, False),
    ("bf16", 64, 64, 3, "ring", 64, 2, "nchw", "ring", None, False),
    ("bf16", 64, 64, 3, "ring", 64, 2, "elu_res", "ring", None, False),
    ("bf16", 64, 64, 3, "ring", 64, 2, "none", "ring", None, False),
    ("bf16", 64, 64, 3, "ring", 64, 2, "prelu", "ring", None, False),
    ("bf16", 256, 256, 3, "wide", 256, 2, "nchw", "wide", None, False),
    ("bf16", 256, 256, 3, "wide", 256, 2, "none", "wide", None, False),
    ("bf16", 256, 256, 3, "wide", 256, 2, "prelu", "wide", None, False),
    ("fp16", 6, 6, 3, "res", 16, 2, "none", "res2", None, False),
    ("fp16", 48, 48, 3, "res", 48, 2, "prelu", "res2", 16, False),
    ("fp16", 29, 6, 3, "res", 16, 2, "elu_res", "res2", None, False),
    ("fp16", 96, 16, 3, "res", 16, 2, "none", "res2", None, True),
    ("fp16", 64, 64, 3, "ring", 64, 2, "nchw", "ring", None, False),
    ("fp16", 64, 64, 3, "ring", 64, 2, "none", "ring", None, False),
    ("fp16", 64, 64, 3, "ring", 64, 2, "prelu", "ring", None, False),
    ("fp16", 256, 256, 3, "wide", 256, 2, "nchw", "wide", None, False),
    ("fp16", 256, 256, 3, "wide", 256, 2, "none", "wide", None, False),
    ("fp16", 256, 256, 3, "wide", 256, 2, "prelu", "wide", None, False),
]
# conv_tc_coupling(persistent=False): the fused coupling epilogue, (kind, inverse, external shift)
COUPLING_CASES = [(kind, inv, ext) for kind in ("bf16", "fp16") for inv in (False, True) for ext in (False, True)]
CPL_SIZE, CPL_CH = (2, 37, 45), 13


def _raw_plan(N, H, W, cin, cout, k, bn, mb, act=0, res_mode=0, out_mode=0, slope=0, inv=0, ext=0, kind="bf16"):
    from cwfa_b200 import _lib
    v = (ctypes.c_int * 9)()
    _lib.call("cwfa_conv_tc_plan", N, H, W, _pad16(cin), _pad16(cout), k, k, bn, mb, act, res_mode, out_mode, slope, 0, inv, ext,
              int(kind == "bf16"), v)
    return list(v)


def _case_plan(case, bn=None):
    kind, cin, cout, k, size, bn0, mb, epi = case[:8]
    N, H, W = SIZES[size]
    return _raw_plan(N, H, W, cin, cout, k, bn or bn0, mb, act=ACT[epi], res_mode=1 if epi == "elu_res" else 0,
                     out_mode=1 if epi == "nchw" else 0, slope=int(epi == "prelu"), kind=kind)


def test_cases_cover_every_conv_tc_kernel():
    """The cases above reach all 26 compiled conv_tc variants (kernel index from the library's own plan): a variant the
    dispatcher gains without a case fails here.  Host-side query only, no GPU needed."""
    seen = {_case_plan(c)[0] for c in CASES}
    N, H, W = CPL_SIZE
    cout = lambda ext: CPL_CH if ext else 2 * CPL_CH
    seen |= {_raw_plan(N, H, W, 64, cout(ext), 3, _pad16(cout(ext)), 2, out_mode=3, inv=int(inv), ext=int(ext), kind=kind)[0]
             for kind, inv, ext in COUPLING_CASES}
    assert seen == set(range(26)), sorted(set(range(26)) - seen)


def _round(t, kind):
    return t.to(torch.bfloat16 if kind == "bf16" else torch.float16).float()


@functools.lru_cache(maxsize=3)
def _operands(kind, cin, cout, k, size, zero_kb):
    """x, w (half grid), bias and the float64 convolution, shared by the cases that differ only in the epilogue."""
    N, H, W = SIZES[size]
    x = _round(seeded_randn((N, cin, H, W), 601), kind)
    w = _round(seeded_randn((cout, cin, k, k), 602, (1.0 / (cin * k * k)) ** 0.5), kind)
    if zero_kb:
        w[:, 48:96] = 0.0
    b = seeded_randn((cout,), 603)
    return x, w, b, F.conv2d(x.double(), w.double(), b.double(), padding=k // 2)


def _c8_raw(data):
    N, G, H, W, _ = data.shape
    return data.float().permute(0, 1, 4, 2, 3).reshape(N, G * 8, H, W)


def _run(xc, pc, epi, res, mb):
    """cwfa_conv_tc into a NaN-filled output; returns the raw output tensor."""
    from cwfa_b200 import _lib, ops
    N, H, W = xc.N, xc.H, xc.W
    if epi == "nchw":
        out = torch.full((N, pc.Cout, H, W), float("nan"), device=DEV)
    else:
        out = torch.full((N, pc.Cout_p // 8, H, W, 8), float("nan"), device=DEV, dtype=xc.data.dtype)
    slope = torch.full((1,), SLOPE, device=DEV) if epi == "prelu" else None
    _lib.call("cwfa_conv_tc", xc.data.data_ptr(), pc.packed.data_ptr(), ops._p(pc.bias), ops._p(slope),
              None if res is None else res.data.data_ptr(), out.data_ptr(), N, H, W, pc.Cin_p, pc.Cout, pc.Cout_p, pc.KH, pc.KW,
              pc.BN, mb, ACT[epi], 1 if res is not None else 0, 1 if epi == "nchw" else 0, xc.is_bf16, ops._stream())
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=lambda c: f"{c[0]}-{c[1]}to{c[2]}-k{c[3]}-{c[4]}-bn{c[5]}-mb{c[6]}-{c[7]}" + ("-zkb" if c[10] else ""))
def test_conv_tc_variant_vs_fp64(case):
    from cwfa_b200 import tc
    kind, cin, cout, k, size, bn, mb, epi, want, twin_bn, zero_kb = case
    x, w, b, ref = _operands(kind, cin, cout, k, size, zero_kb)
    N, H, W = x.shape[0], x.shape[2], x.shape[3]
    xc = tc.to_c8(x.to(DEV), kind)
    pc = tc.PackedConv(w.to(DEV), b.to(DEV), kind, bn=bn)
    res = None
    if epi == "prelu":
        ref = torch.where(ref >= 0, ref, SLOPE * ref)
    elif epi == "elu_res":
        r = _round(seeded_randn((N, cout, H, W), 604), kind)
        res = tc.to_c8(r.to(DEV), kind)
        ref = F.elu(ref + r.double())
    plan = tc.conv_tc_plan(xc, pc, act=ACT[epi], slope=torch.ones(1) if epi == "prelu" else None,
                           res_mode=1 if res is not None else 0, out_nchw=epi == "nchw", mb=mb)
    assert list(plan.values()) == _case_plan(case)
    multi = plan["items"] > plan["grid"]
    assert {"res2": plan["resident"] == 1 and plan["acc_bufs"] == 2 and multi,
            "res1": plan["resident"] == 1 and plan["acc_bufs"] == 1 and multi,
            "ring": plan["resident"] == 0 and plan["wide"] == 0 and multi,
            "wide": plan["wide"] == 1}[want], plan
    out = _run(xc, pc, epi, res, mb)
    torch.cuda.synchronize()
    if epi == "nchw":
        y = out.cpu()
    else:
        raw = _c8_raw(out.cpu())
        assert torch.equal(raw[:, cout:], torch.zeros_like(raw[:, cout:])), "padded output channels must be exactly 0"
        y = raw[:, :cout]
    assert torch.isfinite(y).all(), f"{int((~torch.isfinite(y)).sum())} outputs never written"
    d = (y.double() - ref).abs()
    rms = float(ref.pow(2).mean().sqrt())
    # fp32 output: accumulation order only.  Half output: the store's rounding (<= 1 ulp of the value) on top.
    ulp = 0.0 if epi == "nchw" else (2.0 ** -7 if kind == "bf16" else 2.0 ** -10)
    bound = ulp * ref.abs() + 2e-4 * rms
    bad = d > bound
    err = rel_l2(y, ref)
    print(f"conv_tc {kind} {cin}->{cout} k{k} {N}x{H}x{W} bn{bn} mb{mb} {epi}{' zero-kb' if zero_kb else ''}: plan {plan}  "
          f"rel_l2 {err:.2e}  max_abs {float(d.max()):.2e}")
    if bad.any():
        n, c, h, w_ = [int(v) for v in bad.nonzero()[0]]
        raise AssertionError(f"{int(bad.sum())} elements off; first at (n={n}, c={c}, h={h}, w={w_}), tile (row {h // 16}, "
                             f"col {w_ // (8 * mb)}): got {float(y[n, c, h, w_]):.6g}, want {float(ref[n, c, h, w_]):.6g}")
    assert err < (2e-5 if epi == "nchw" else 6e-3 if kind == "bf16" else 8e-4)
    if twin_bn:
        pc2 = tc.PackedConv(w.to(DEV), b.to(DEV), kind, bn=twin_bn)
        plan2 = tc.conv_tc_plan(xc, pc2, act=ACT[epi], slope=torch.ones(1) if epi == "prelu" else None,
                                res_mode=1 if res is not None else 0, out_nchw=True, mb=mb)
        plan1 = tc.conv_tc_plan(xc, pc, act=ACT[epi], slope=torch.ones(1) if epi == "prelu" else None,
                                res_mode=1 if res is not None else 0, out_nchw=True, mb=mb)
        assert plan1["resident"] == 1 and plan2["resident"] == 0
        y1, y2 = _run(xc, pc, "nchw", None, mb).cpu(), _run(xc, pc2, "nchw", None, mb).cpu()
        e2 = rel_l2(y1, y2)
        print(f"  ring-path twin bn{twin_bn}: plan {plan2}  rel_l2 vs resident {e2:.2e}")
        assert e2 < 1e-6                    # observed: 0 (the two plans issue the same MMAs in the same order)


@pytest.mark.gpu
@pytest.mark.parametrize("kind,inverse,ext", COUPLING_CASES)
def test_conv_tc_coupling_variant_vs_fp64(kind, inverse, ext):
    """conv_tc_kernel<*, 1-4> (conv_tc_coupling with persistent=False) against the float64 coupling reference (same limits as
    test_gpu_coupling.py; observed on a B200: y <= 6.7e-6, log-det <= 3.5e-8, sum y^2 <= 9.1e-7)."""
    from test_gpu_coupling import TOL_LOGDET, TOL_SUMSQ, TOL_Y
    from cwfa_b200 import tc
    from test_gpu_coupling import _coupling_reference
    N, H, W = CPL_SIZE
    ch = CPL_CH
    cout = ch if ext else 2 * ch
    b = _round(seeded_randn((N, 64, H, W), 611), kind)
    w = _round(seeded_randn((cout, 64, 3, 3), 612, 0.04), kind)
    bias = seeded_randn((cout,), 613, 0.5)
    a = F.conv2d(b.double(), w.double(), bias.double(), padding=1)
    x = seeded_randn((N, ch, H, W), 614)
    t_ext = seeded_randn((N, ch, H, W), 615, 0.3) if ext else None
    t_scale = -0.5 ** 0.5 if ext else 1.0
    y_ref, j_ref, sabs = _coupling_reference(a, x.double(), None if t_ext is None else t_ext.double(), t_scale, ch, inverse)
    bc = tc.to_c8(b.to(DEV), kind)
    pc = tc.PackedConv(w.to(DEV), bias.to(DEV), kind, bn=tc.pad16(cout))
    plan = tc.conv_tc_plan(bc, pc, coupling=(inverse, ext))
    assert plan["ki"] == 12 + (4 if kind == "bf16" else 0) + (2 if ext else 0) + (1 if inverse else 0), plan
    logdet = torch.full((N,), 3.0, device=DEV)
    sumsq = torch.full((N,), float("nan"), device=DEV)
    y = tc.conv_tc_coupling(bc, pc, x.to(DEV), ch=ch, inverse=inverse, t_ext=None if t_ext is None else t_ext.to(DEV),
                            t_scale=t_scale, logdet=logdet, sumsq=sumsq, persistent=False).cpu()
    torch.cuda.synchronize()
    err = float(((y.double() - y_ref).abs() / (1.0 + y_ref.abs())).max())
    ld_err = float(((logdet.cpu().double() - 3.0 - j_ref).abs() / sabs).max())
    q_ref = (y_ref ** 2).sum(dim=(1, 2, 3))
    q_err = float(((sumsq.cpu().double() - q_ref).abs() / q_ref).max())
    print(f"conv_tc coupling {kind} inv={int(inverse)} ext={int(ext)}: plan {plan}  y {err:.2e}  logdet {ld_err:.2e}  sumsq {q_err:.2e}")
    assert err < TOL_Y and ld_err < TOL_LOGDET and q_err < TOL_SUMSQ
