"""GPU: the entry form of the trunk block (``cwfa_resblock_tc_batched`` with input-conv weights, ``tc.resblock_tc_entry_batched``),
which folds a sub-network's 1x1 input conv into its first trunk block, against an fp64 CPU reference of the UNCOMPOSED block
``ELU(W1 ELU(W3 (*) b + b3) + b1 + b)``, ``b = Win lf + bin`` zero-padded; and the engine with the composed entry on and off."""
import ctypes as C

import pytest
import torch
import torch.nn.functional as F

from conftest import max_abs, rel_l2
from oracle.weights import seeded_randn

pytestmark = pytest.mark.gpu
DEV = "cuda:0"

# rel-L2 / max-abs limits against the fp64 reference: about 4x the worst values measured on a B200 (1000 W power limit) over the
# cases below (bf16 rel 2.27e-3, abs 2.34e-2; fp16 rel 2.83e-4, abs 3.56e-3)
TOL = {"bf16": (1e-2, 0.1), "fp16": (1.2e-3, 1.5e-2)}


def _round(t, kind):
    return t.to(torch.bfloat16 if kind == "bf16" else torch.float16).float()


def _weights(cin, seed, kind):
    """Input conv, 3x3 and 1x1 of one trunk's first block, the half-precision operands of the kernels pre-rounded."""
    win = _round(seeded_randn((64, cin, 1, 1), seed, (1.0 / cin) ** 0.5), kind)
    w3 = _round(seeded_randn((64, 64, 3, 3), seed + 1, (1.0 / 576) ** 0.5), kind)
    w1 = _round(seeded_randn((64, 64, 1, 1), seed + 2, (1.0 / 64) ** 0.5), kind)
    bin_, b3, b1 = (seeded_randn((64,), seed + 3 + i, 0.3) for i in range(3))
    return win, bin_, w3, b3, w1, b1


def _reference(lf, ws, kind):
    """The uncomposed block in fp64; t is rounded to the half type as the kernel stores it for GEMM2."""
    win, bin_, w3, b3, w1, b1 = (t.double() for t in ws)
    b = F.conv2d(lf.double(), win, bin_)
    t = _round(F.elu(F.conv2d(b, w3, b3, padding=1)).float(), kind).double()
    return F.elu(F.conv2d(t, w1, b1) + b).float()


def _entry(ws, kind):
    from cwfa_b200 import tc
    win, bin_, w3, b3, w1, b1 = (t.to(DEV) for t in ws)
    return tc.PackedEntry(win, bin_, w3, b3, tc.PackedConv(w1, b1, kind, bn=64), kind)


def _launch(lf8, entries, y8, out_off):
    """The C entry point with a caller-provided (NaN-filled) output tensor."""
    from cwfa_b200 import _lib, ops
    n = len(entries)
    vps = lambda vals: (C.c_void_p * n)(*vals)
    _lib.call("cwfa_resblock_tc_batched", lf8.data.data_ptr(), y8.data.data_ptr(), n, vps([e.p3.packed.data_ptr() for e in entries]),
              vps([e.p1.packed.data_ptr() for e in entries]), vps([e.b3.data_ptr() for e in entries]),
              vps([e.b1.data_ptr() for e in entries]), lf8.N, lf8.H, lf8.W, lf8.Cp // 8, (C.c_int * n)(*([0] * n)), y8.Cp // 8,
              (C.c_int * n)(*[8 * (out_off + k) for k in range(n)]), vps([e.pin.packed.data_ptr() for e in entries]),
              vps([e.edge.data_ptr() for e in entries]), lf8.Cp // 8, lf8.is_bf16, ops._stream())


def _nan_c8(N, C_, H, W, kind):
    from cwfa_b200 import tc
    y8 = tc.C8.empty(N, C_, H, W, DEV, kind, C_)
    y8.data.fill_(float("nan"))
    return y8


CASES = [
    # kind, cin, N, H, W, n_sets, zero input
    ("bf16", 48, 1, 48, 80, 5, False),
    ("fp16", 48, 2, 33, 19, 5, False),
    ("bf16", 24, 2, 33, 19, 3, False),
    ("fp16", 24, 1, 48, 80, 2, False),
    ("bf16", 12, 3, 40, 24, 4, False),
    ("fp16", 12, 1, 1, 45, 2, False),
    ("bf16", 6, 1, 37, 1, 1, False),
    ("fp16", 6, 3, 64, 64, 5, False),
    ("bf16", 64, 1, 40, 24, 3, False),      # Cin_p = 64: four K-steps, two A slots
    ("fp16", 64, 2, 17, 33, 1, False),
    ("bf16", 6, 1, 1, 1, 1, False),
    ("bf16", 48, 1, 20, 35, 3, True),       # lf = 0: the output is the bias path alone, every edge and corner class
    ("fp16", 12, 1, 1, 17, 2, True),
    ("fp16", 24, 2, 18, 1, 1, True),
    ("bf16", 64, 1, 31, 18, 2, True),
]


@pytest.mark.parametrize("kind,cin,N,H,W,nsets,zero", CASES)
def test_entry_block_vs_fp64_reference(kind, cin, N, H, W, nsets, zero):
    from cwfa_b200 import tc
    lf = torch.zeros(N, cin, H, W) if zero else _round(seeded_randn((N, cin, H, W), 31), kind)
    lf8 = tc.to_c8(lf.to(DEV), kind)
    wsets = [_weights(cin, 40 + 10 * k, kind) for k in range(nsets)]
    entries = [_entry(ws, kind) for ws in wsets]
    y8 = _nan_c8(N, 64 * nsets, H, W, kind)
    _launch(lf8, entries, y8, 0)
    y = tc.from_c8(y8).cpu()
    rel_lim, abs_lim = TOL[kind]
    for k, ws in enumerate(wsets):
        ref = _reference(lf, ws, kind)
        yk = y[:, 64 * k:64 * (k + 1)]
        assert torch.isfinite(yk).all(), k
        r, a = rel_l2(yk, ref), max_abs(yk, ref)
        print(f"entry {kind} cin={cin} {N}x{H}x{W} set {k}/{nsets}{' zero' if zero else ''}: rel {r:.2e} abs {a:.2e}")
        assert r < rel_lim and a < abs_lim, (k, r, a)
    # the Python wrapper launches the same thing
    assert torch.equal(tc.from_c8(tc.resblock_tc_entry_batched(lf8, entries)).cpu(), y)


@pytest.mark.parametrize("kind,cin,N,H,W,nsets", [("bf16", 48, 1, 48, 80, 5), ("fp16", 24, 2, 33, 19, 3), ("bf16", 12, 3, 64, 64, 5),
                                                  ("fp16", 64, 1, 40, 24, 2), ("bf16", 6, 1, 1, 50, 4)])
def test_batched_entry_equals_per_set_launches(kind, cin, N, H, W, nsets):
    """One launch over several sets (contiguous tile ranges, weight switches inside a CTA's range) == one launch per set, bit
    for bit."""
    from cwfa_b200 import tc
    lf8 = tc.to_c8(_round(seeded_randn((N, cin, H, W), 51), kind).to(DEV), kind)
    entries = [_entry(_weights(cin, 60 + 10 * k, kind), kind) for k in range(nsets)]
    y8 = _nan_c8(N, 64 * nsets, H, W, kind)
    _launch(lf8, entries, y8, 0)
    y = tc.from_c8(y8)
    for k, e in enumerate(entries):
        yk8 = _nan_c8(N, 64, H, W, kind)
        _launch(lf8, [e], yk8, 0)
        assert torch.equal(y[:, 64 * k:64 * (k + 1)], tc.from_c8(yk8)), k


def test_entry_rejects_bad_arguments():
    from cwfa_b200 import _lib, tc
    kind = "bf16"
    lf8 = tc.to_c8(torch.zeros(1, 24, 16, 16, device=DEV), kind)
    e = _entry(_weights(24, 70, kind), kind)
    with pytest.raises(ValueError):
        tc.resblock_tc_entry_batched(tc.to_c8(torch.zeros(1, 48, 16, 16, device=DEV), kind), [e])      # Cin_p mismatch
    with pytest.raises(ValueError):
        tc.resblock_tc_entry_batched(lf8, [e] * 6)
    y8 = _nan_c8(1, 64, 16, 16, kind)
    n = 1
    vp = lambda v: (C.c_void_p * n)(v)
    with pytest.raises(_lib.CwfaError):       # odd chunk count
        _lib.call("cwfa_resblock_tc_batched", lf8.data.data_ptr(), y8.data.data_ptr(), 1, vp(e.p3.packed.data_ptr()),
                  vp(e.p1.packed.data_ptr()), vp(e.b3.data_ptr()), vp(e.b1.data_ptr()), 1, 16, 16, 4, (C.c_int * 1)(0), 8,
                  (C.c_int * 1)(0), vp(e.pin.packed.data_ptr()), vp(e.edge.data_ptr()), 3, 1, None)
    with pytest.raises(_lib.CwfaError):       # missing edge tables
        _lib.call("cwfa_resblock_tc_batched", lf8.data.data_ptr(), y8.data.data_ptr(), 1, vp(e.p3.packed.data_ptr()),
                  vp(e.p1.packed.data_ptr()), vp(e.b3.data_ptr()), vp(e.b1.data_ptr()), 1, 16, 16, 4, (C.c_int * 1)(0), 8,
                  (C.c_int * 1)(0), vp(e.pin.packed.data_ptr()), None, 4, 1, None)


# ---- engine: composed entry on vs off ---------------------------------------------------------------------------------
def _level_trunks(eng, views, n):
    from cwfa_b200 import tc
    lf8 = eng.levels[n]["cond"](eng._views_c8(views, None))
    return [tc.from_c8(it[3])[:, it[4] * 8:it[4] * 8 + 64] for it in eng._trunks(n, lf8) if it[0] == "cat"]


# Composed vs separate input conv (bf16; the fp16 engine keeps the separate input conv, engine.py ``_plan_entry``), limits = the
# engine's stated bf16 tolerance.  Measured on a B200 (1000 W): trunk outputs per level 5.4e-3, volume 9.3e-3 (full config) /
# 8.8e-3 (tiny).  The composed form rounds once less (b is no longer stored in half precision) and rounds W3' = W3_tap Win instead
# of W3.
def _compare_engine(model, views, mv, kind, label):
    from cwfa_b200.engine import CWFAEngine
    eng = CWFAEngine(model, kind)
    assert all(lv["entry"] is not None for lv in eng.levels)
    out = {}
    for on in (True, False):
        eng.composed_entry = on
        out[on] = ([_level_trunks(eng, views, n) for n in range(len(eng.levels))], eng.reconstruct(views, mv))
    worst = 0.0
    for n in range(len(eng.levels)):
        r = max(rel_l2(a, b) for a, b in zip(out[True][0][n], out[False][0][n]))
        worst = max(worst, r)
        print(f"engine {label} {kind} level {n}: trunk output rel-L2 composed vs input conv + block {r:.2e}")
    rv = rel_l2(out[True][1], out[False][1])
    print(f"engine {label} {kind}: volume rel-L2 composed vs input conv + block {rv:.2e}")
    return eng, out[True][1], worst, rv


def test_engine_composed_entry_tiny(golden_tiny):
    from cwfa_b200.engine import CWFAEngine
    from helpers import build_tiny_model, tiny_inputs
    model = build_tiny_model(golden_tiny, DEV)
    views, mvs = tiny_inputs(golden_tiny)
    views, mvs = views.to(DEV), [t.to(DEV) for t in mvs]
    eng, vol, worst, rv = _compare_engine(model, views, mvs, "bf16", "tiny")
    assert worst < 2e-2 and rv < 2e-2
    eng.composed_entry = True
    assert torch.equal(eng.reconstruct_graphed(views, mvs), vol)          # graph replay == eager, bitwise
    assert all(lv["entry"] is None for lv in CWFAEngine(model, "fp16").levels)


def test_engine_composed_entry_full():
    import os
    from conftest import GOLDEN
    from helpers import build_full_model, full_inputs
    fx = torch.load(os.path.join(GOLDEN, "r2_full.pt"), weights_only=False)
    model = build_full_model(fx, DEV)
    views, mvs = full_inputs(fx)
    views, mvs = views.to(DEV), [t.to(DEV) for t in mvs]
    _, _, worst, rv = _compare_engine(model, views, mvs, "bf16", "full")
    assert worst < 2e-2 and rv < 2e-2
