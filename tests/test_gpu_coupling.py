"""GPU: the two persistent coupling kernels (coupling_f8 on the F8 detail half, coupling_tc on NCHW) against a float64 CPU
reference of the same operation: the last 3x3 conv of a coupling sub-network (64 hidden channels, operands on the half grid),
the affine coupling of coupling_layers.py:490-500, the preceding permutation as a gather on x, and the per-sample
log-det / sum of y^2.

Every output buffer is filled with NaN before the call (the caching allocator could otherwise hand back the correct result of
an identical earlier call, and a tile the kernel skipped would pass), and every element is checked on its own: one wrong pixel
row among 100k elements fails.  Shapes: a ragged one (no dimension a multiple of 16, one below 16) and a multi-tile one
(N=3 at 230x230: 675 tiles on the 148-CTA grid, so every CTA walks 4-5 tiles through both TMEM accumulator buffers and
around the A ring)."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from conftest import rel_l2
from oracle.weights import seeded_randn

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
CLAMP, K_ATAN = 2.0, 0.636
T_SCALE = -0.5 ** 0.5
SHAPES = {"ragged": (2, 37, 13), "multi": (3, 230, 230)}
BIG = 1.0e3            # the channel slices of the 192-channel input that the kernel must not read

# Limits at ~4x the worst error observed over the cases below on a B200 (1000 W power limit):
#   y, per element |y - ref| / (1 + |ref|):  coupling_f8 1.6e-5 (bf16) / 8.6e-6 (fp16), coupling_tc 4.5e-6 / 1.2e-5
#   log-det, |logdet - ref| / sum |s|:      1.2e-6 (coupling_f8, ch = 1), else <= 2.5e-7
#   sum y^2, relative:                       2.2e-6
# (fp32 accumulation order, the hi + lo split of the bias in coupling_f8, atan_fast and ex2.approx; dropping the lo half of the
# bias alone gives 1.4e-2.)
TOL_Y = 6e-5
TOL_LOGDET = 5e-6
TOL_SUMSQ = 1e-5


def _round(t, kind):
    return t.to(torch.bfloat16 if kind == "bf16" else torch.float16).float()


def _coupling_reference(a, x, t_ext, t_scale, ch, inverse, clamp=CLAMP, k=K_ATAN):
    """coupling_layers.py:490-500 on the conv output a = [s_raw | t] (or t = t_scale * t_ext)."""
    s = clamp * k * torch.atan(a[:, :ch])
    t = t_scale * t_ext if t_ext is not None else a[:, ch:2 * ch]
    if inverse:
        y = (x - t) * torch.exp(-s)
        j = -s.sum(dim=(1, 2, 3))
    else:
        y = torch.exp(s) * x + t
        j = s.sum(dim=(1, 2, 3))
    return y, j, s.abs().sum(dim=(1, 2, 3))


@pytest.fixture(scope="module")
def conv_ref():
    """(shape, kind) -> b (N,64,H,W), 96 output rows of 3x3 weights + bias on the half grid, and a = conv(b) in float64.
    A coupling of ch channels uses rows [0, ch) as s and rows [48, 48 + ch) as t, so one fp64 convolution per (shape, kind)
    serves every case."""
    cache = {}

    def get(shape, kind):
        key = (shape, kind)
        if key not in cache:
            N, H, W = SHAPES[shape]
            b = _round(seeded_randn((N, 64, H, W), 501), kind)
            w = _round(seeded_randn((96, 64, 3, 3), 502, 0.04), kind)
            bias = seeded_randn((96,), 503, 0.5)          # large enough that the bias's lo half matters at the tolerance
            a = F.conv2d(b.double(), w.double(), bias.double(), padding=1)
            cache[key] = (b, w, bias, a)
        return cache[key]
    return get


def _rows(ch, ext):
    return list(range(ch)) + ([] if ext else list(range(48, 48 + ch)))


def _c8_slice(b, kind, chunk_off):
    """b (N,64,H,W) as the 8-chunk slice at chunk_off of a 192-channel C8 tensor [N][24][H][W][8] whose other slices hold
    large values (built in torch, not with the library's converters)."""
    N, _, H, W = b.shape
    full = _round(BIG * (1.0 + seeded_randn((N, 192, H, W), 504).abs()), kind)
    full[:, 8 * chunk_off:8 * chunk_off + 64] = b
    dt = torch.bfloat16 if kind == "bf16" else torch.float16
    return full.view(N, 24, 8, H, W).permute(0, 1, 3, 4, 2).contiguous().to(dt).to(DEV)


def _to_f8(x, c8):
    N, C, H, W = x.shape
    xp = torch.zeros(N, c8, H, W, dtype=x.dtype)
    xp[:, :C] = x
    return xp.view(N, c8 // 8, 8, H, W).permute(0, 1, 3, 4, 2).contiguous()


def _from_f8(y8):
    N, G, H, W, _ = y8.shape
    return y8.permute(0, 1, 4, 2, 3).reshape(N, G * 8, H, W)


def _nan(*shape):
    return torch.full(shape, float("nan"), device=DEV)


def _check_elements(y, ref, tol, what):
    """Every element within tol * (1 + |ref|); on failure name the first bad (n, c, h, w) and its 16x16 tile."""
    y, ref = y.double().cpu(), ref.double().cpu()
    assert torch.isfinite(y).all(), f"{what}: {int((~torch.isfinite(y)).sum())} non-finite outputs (a tile not written?)"
    err = (y - ref).abs() / (1.0 + ref.abs())
    worst = float(err.max())
    if worst > tol:
        n, c, h, w = [int(v) for v in (err > tol).nonzero()[0]]
        raise AssertionError(f"{what}: {int((err > tol).sum())} elements off, worst {worst:.2e} > {tol:.1e}; first at "
                             f"(n={n}, c={c}, h={h}, w={w}) tile (row {h // 16}, col {w // 16}): got {float(y[n, c, h, w]):.6g}, "
                             f"want {float(ref[n, c, h, w]):.6g}")
    return worst


def _check_reductions(logdet, sumsq, j_ref, sabs, y_ref, base, what):
    ld_err = ((logdet.double().cpu() - base - j_ref).abs() / sabs).max().item()
    q_ref = (y_ref ** 2).sum(dim=(1, 2, 3))
    q_err = ((sumsq.double().cpu() - q_ref).abs() / q_ref).max().item()
    assert ld_err < TOL_LOGDET, f"{what}: log-det off by {ld_err:.2e} of sum |s|"
    assert q_err < TOL_SUMSQ, f"{what}: sum y^2 off by {q_err:.2e}"
    return ld_err, q_err


def _inputs(shape, ch, axis, xmode, ext):
    N, H, W = SHAPES[shape]
    x = None if xmode == "none" else seeded_randn((N, ch, H, W), 505)
    t_ext = seeded_randn((N, ch, H, W), 506, 0.3) if ext else None
    perm = None
    xin = torch.zeros(N, ch, H, W) if x is None else x
    if axis:
        perm = torch.from_numpy(np.random.RandomState(7 + axis).permutation({1: ch, 2: H, 3: W}[axis])).long()
        xin = xin.index_select(axis, perm)
    return x, t_ext, perm, xin


# (kind, inverse, ext, ch, perm axis, x, shape, chunk_off, reduction): every coupling_f8_kernel<BF16, INV, EXT> instantiation,
# ch 1..48 (chp8 8..48, BN 16..96: 3 A stages up to BN 80, 2 at BN 96), row / column / no permutation, x given / None,
# external shift, both shapes, the three input slices, in-kernel (ticket) and separate finalize, accumulate on / off.
F8_CASES = [
    ("bf16", False, False, 48, 0, "x", "multi", 0, "ticket"),
    ("bf16", True, False, 24, 2, "x", "multi", 8, "finalize"),
    ("bf16", False, True, 13, 3, "x", "multi", 16, "ticket_noacc"),
    ("bf16", True, True, 48, 0, "none", "multi", 0, "finalize_noacc"),
    ("bf16", True, False, 1, 3, "x", "ragged", 0, "finalize"),
    ("bf16", False, False, 40, 2, "x", "ragged", 16, "ticket"),
    ("fp16", False, False, 5, 3, "x", "ragged", 0, "ticket"),
    ("fp16", True, False, 48, 2, "none", "multi", 16, "ticket"),
    ("fp16", False, True, 1, 2, "x", "ragged", 8, "finalize"),
    ("fp16", True, True, 8, 3, "x", "multi", 0, "ticket_noacc"),
    ("fp16", False, False, 24, 0, "x", "multi", 8, "finalize_noacc"),
    ("fp16", True, True, 24, 0, "x", "ragged", 16, "ticket"),
]


def _run_f8(b8, pc, x8, t8, perm, axis, ch, inverse, N, H, W, chunk_off, kind, red, ticket):
    from cwfa_b200 import _lib, ops, tc
    c8 = tc.ch8(ch)
    tiles = _lib.load().cwfa_coupling_tc_tiles(H, W)
    acc = not red.endswith("noacc")
    y8, ws, sumsq = _nan(N, c8 // 8, H, W, 8), _nan(2 * N * tiles), _nan(N)
    logdet = torch.full((N,), 3.0, device=DEV) if acc else _nan(N)
    use_ticket = red.startswith("ticket")
    _lib.call("cwfa_coupling_f8", b8.data_ptr(), pc.packed.data_ptr(), ops._p(pc.bias), N, H, W, pc.BN, c8, ops._p(x8),
             y8.data_ptr(), ops._p(t8), float(T_SCALE if t8 is not None else 1.0), ops._p(perm), axis, CLAMP, K_ATAN, int(inverse),
             ws.data_ptr(), logdet.data_ptr(), sumsq.data_ptr(), int(acc), ticket.data_ptr() if use_ticket else None, 24, chunk_off,
             int(kind == "bf16"), ops._stream())
    if not use_ticket:
        _lib.call("cwfa_coupling_finalize", ws.data_ptr(), logdet.data_ptr(), sumsq.data_ptr(), N, tiles, int(acc), ops._stream())
    return y8, logdet, sumsq, 3.0 if acc else 0.0


@pytest.mark.parametrize("kind,inverse,ext,ch,axis,xmode,shape,chunk_off,red", F8_CASES)
def test_coupling_f8_vs_fp64(conv_ref, kind, inverse, ext, ch, axis, xmode, shape, chunk_off, red):
    from cwfa_b200 import tc
    N, H, W = SHAPES[shape]
    b, w, bias, a = conv_ref(shape, kind)
    rows = _rows(ch, ext)
    x, t_ext, perm, xin = _inputs(shape, ch, axis, xmode, ext)
    a_c = a[:, rows]
    y_ref, j_ref, sabs = _coupling_reference(a_c, xin.double(), None if t_ext is None else t_ext.double(), T_SCALE, ch, inverse)
    c8 = tc.ch8(ch)
    pc = tc.coupling_weights_f8(w[rows].to(DEV), bias[rows].to(DEV), ch, torch.arange(ch), ext, kind)
    b8 = _c8_slice(b, kind, chunk_off)
    x8 = None if x is None else _to_f8(x, c8).to(DEV)
    t8 = None if t_ext is None else _to_f8(t_ext, c8).to(DEV)
    perm_d = None if perm is None else perm.to(DEV, torch.int32)
    ticket = torch.zeros(1, device=DEV, dtype=torch.int32)
    outs = []
    for rep in range(2):                    # the same ticket serves two consecutive launches
        y8, logdet, sumsq, base = _run_f8(b8, pc, x8, t8, perm_d, axis, ch, inverse, N, H, W, chunk_off, kind, red, ticket)
        torch.cuda.synchronize()
        assert int(ticket[0]) == 0
        outs.append((y8.cpu(), logdet.cpu(), sumsq.cpu()))
    y = _from_f8(outs[0][0])
    assert torch.equal(y[:, ch:], torch.zeros_like(y[:, ch:])), "F8 padding slots must be exactly 0"
    err = _check_elements(y[:, :ch], y_ref, TOL_Y, f"coupling_f8 {kind} inv={inverse} ext={ext} ch={ch}")
    ld_err, q_err = _check_reductions(outs[0][1], outs[0][2], j_ref, sabs, y_ref, base, "coupling_f8")
    assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1]) and torch.equal(outs[0][2], outs[1][2])
    print(f"coupling_f8 {kind} inv={int(inverse)} ext={int(ext)} ch={ch} BN={pc.BN} axis={axis} x={xmode} {shape} {N}x{H}x{W} "
          f"off={chunk_off} {red}: y {err:.2e}  logdet {ld_err:.2e}  sumsq {q_err:.2e}")


# every coupling_tc_kernel<BF16, INV, EXT> instantiation; channel (axis 1) permutations too
TC_CASES = [
    ("bf16", False, False, 48, 1, "x", "multi", 8, "ticket"),
    ("bf16", True, False, 5, 2, "x", "ragged", 0, "finalize"),
    ("bf16", False, True, 24, 3, "x", "multi", 16, "ticket_noacc"),
    ("bf16", True, True, 13, 0, "none", "multi", 0, "finalize_noacc"),
    ("fp16", False, False, 8, 3, "x", "ragged", 16, "ticket"),
    ("fp16", True, False, 48, 1, "x", "multi", 0, "ticket"),
    ("fp16", False, True, 1, 2, "x", "ragged", 8, "finalize"),
    ("fp16", True, True, 40, 1, "x", "multi", 0, "ticket_noacc"),
]


def _run_tc(b8, pc, x, t, perm, axis, ch, inverse, N, H, W, chunk_off, kind, red, ticket):
    from cwfa_b200 import _lib, ops
    tiles = _lib.load().cwfa_coupling_tc_tiles(H, W)
    acc = not red.endswith("noacc")
    y, ws, sumsq = _nan(N, ch, H, W), _nan(2 * N * tiles), _nan(N)
    logdet = torch.full((N,), 3.0, device=DEV) if acc else _nan(N)
    use_ticket = red.startswith("ticket")
    _lib.call("cwfa_coupling_tc", b8.data_ptr(), pc.packed.data_ptr(), ops._p(pc.bias), N, H, W, pc.Cout, pc.Cout_p, ops._p(x),
         y.data_ptr(), ops._p(t), float(T_SCALE if t is not None else 1.0), ops._p(perm), axis, ch, CLAMP, K_ATAN, int(inverse),
         ws.data_ptr(), logdet.data_ptr(), sumsq.data_ptr(), int(acc), ticket.data_ptr() if use_ticket else None, 24, chunk_off,
         int(kind == "bf16"), ops._stream())
    if not use_ticket:
        _lib.call("cwfa_coupling_finalize", ws.data_ptr(), logdet.data_ptr(), sumsq.data_ptr(), N, tiles, int(acc), ops._stream())
    return y, logdet, sumsq, 3.0 if acc else 0.0


@pytest.mark.parametrize("kind,inverse,ext,ch,axis,xmode,shape,chunk_off,red", TC_CASES)
def test_coupling_tc_vs_fp64(conv_ref, kind, inverse, ext, ch, axis, xmode, shape, chunk_off, red):
    from cwfa_b200 import tc
    N, H, W = SHAPES[shape]
    b, w, bias, a = conv_ref(shape, kind)
    rows = _rows(ch, ext)
    x, t_ext, perm, xin = _inputs(shape, ch, axis, xmode, ext)
    y_ref, j_ref, sabs = _coupling_reference(a[:, rows], xin.double(), None if t_ext is None else t_ext.double(), T_SCALE, ch, inverse)
    pc = tc.PackedConv(w[rows].to(DEV), bias[rows].to(DEV), kind, bn=tc.pad16(len(rows)))
    b8 = _c8_slice(b, kind, chunk_off)
    xd = None if x is None else x.to(DEV)
    td = None if t_ext is None else t_ext.to(DEV)
    perm_d = None if perm is None else perm.to(DEV, torch.int32)
    ticket = torch.zeros(1, device=DEV, dtype=torch.int32)
    outs = []
    for rep in range(2):
        y, logdet, sumsq, base = _run_tc(b8, pc, xd, td, perm_d, axis, ch, inverse, N, H, W, chunk_off, kind, red, ticket)
        torch.cuda.synchronize()
        assert int(ticket[0]) == 0
        outs.append((y.cpu(), logdet.cpu(), sumsq.cpu()))
    err = _check_elements(outs[0][0], y_ref, TOL_Y, f"coupling_tc {kind} inv={inverse} ext={ext} ch={ch}")
    ld_err, q_err = _check_reductions(outs[0][1], outs[0][2], j_ref, sabs, y_ref, base, "coupling_tc")
    assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1]) and torch.equal(outs[0][2], outs[1][2])
    print(f"coupling_tc {kind} inv={int(inverse)} ext={int(ext)} ch={ch} Cout_p={pc.Cout_p} axis={axis} x={xmode} {shape} "
          f"{N}x{H}x{W} off={chunk_off} {red}: y {err:.2e}  logdet {ld_err:.2e}  sumsq {q_err:.2e}")


@pytest.mark.parametrize("which", ["f8", "tc"])
def test_coupling_graph_replay_is_bit_reproducible(conv_ref, which):
    """A CUDA graph of one in-kernel-finalized coupling launch, replayed twice: the log-det and sum y^2 come back bit for bit
    equal to each other and to the eager launch, and the ticket is back at zero after each replay."""
    from cwfa_b200 import tc
    kind, ch, shape = "bf16", 24, "multi"
    N, H, W = SHAPES[shape]
    b, w, bias, a = conv_ref(shape, kind)
    rows = _rows(ch, False)
    x, _, perm, _ = _inputs(shape, ch, 2, "x", False)
    b8 = _c8_slice(b, kind, 0)
    ticket = torch.zeros(1, device=DEV, dtype=torch.int32)
    perm_d = perm.to(DEV, torch.int32)
    if which == "f8":
        pc = tc.coupling_weights_f8(w[rows].to(DEV), bias[rows].to(DEV), ch, torch.arange(ch), False, kind)
        xd = _to_f8(x, tc.ch8(ch)).to(DEV)
        run = lambda: _run_f8(b8, pc, xd, None, perm_d, 2, ch, False, N, H, W, 0, kind, "ticket_noacc", ticket)
    else:
        pc = tc.PackedConv(w[rows].to(DEV), bias[rows].to(DEV), kind, bn=tc.pad16(len(rows)))
        xd = x.to(DEV)
        run = lambda: _run_tc(b8, pc, xd, None, perm_d, 2, ch, False, N, H, W, 0, kind, "ticket_noacc", ticket)
    _, ld_eager, q_eager, _ = run()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        with torch.cuda.graph(g, stream=s):
            _, ld, q, _ = run()
    torch.cuda.current_stream().wait_stream(s)
    got = []
    for _ in range(2):
        g.replay()
        torch.cuda.synchronize()
        assert int(ticket[0]) == 0
        got.append((ld.cpu().clone(), q.cpu().clone()))
    assert torch.equal(got[0][0], got[1][0]) and torch.equal(got[0][1], got[1][1])
    assert torch.equal(got[0][0], ld_eager.cpu()) and torch.equal(got[0][1], q_eager.cpu())
    print(f"coupling_{which} graph replay: logdet {got[0][0].tolist()}")


@pytest.mark.parametrize("inverse,ext", [(False, False), (True, True)])
def test_coupling_f8_channel_permutation_matches_tc_gather(conv_ref, inverse, ext):
    """The engine's channel-permutation trick: coupling_f8 with the permutation folded into the packed weights' output columns
    (coupling_weights_f8), read back through slot_to_chan, equals coupling_tc with the same permutation as an axis-1 gather
    on x, to fp32 rounding."""
    from cwfa_b200 import tc
    kind, ch, shape = "bf16", 13, "multi"
    N, H, W = SHAPES[shape]
    b, w, bias, _ = conv_ref(shape, kind)
    rows = _rows(ch, ext)
    x = seeded_randn((N, ch, H, W), 507)
    t_ext = seeded_randn((N, ch, H, W), 508, 0.3) if ext else None
    rs = np.random.RandomState(11)
    perm = torch.from_numpy(rs.permutation(ch)).long()          # the gather of the preceding permutation: xin[c] = x[perm[c]]
    sigma = torch.from_numpy(rs.permutation(ch)).long()         # slot_to_chan: storage slot j holds logical channel sigma[j]
    b8 = _c8_slice(b, kind, 0)
    ticket = torch.zeros(1, device=DEV, dtype=torch.int32)
    pc_tc = tc.PackedConv(w[rows].to(DEV), bias[rows].to(DEV), kind, bn=tc.pad16(len(rows)))
    y_tc, ld_tc, q_tc, _ = _run_tc(b8, pc_tc, x.to(DEV), None if t_ext is None else t_ext.to(DEV),
                                   perm.to(DEV, torch.int32), 1, ch, inverse, N, H, W, 0, kind, "ticket_noacc", ticket)
    # F8 slot j: x of channel perm[sigma[j]], t_ext of channel sigma[j]; columns of the packed conv in slot order
    c8 = tc.ch8(ch)
    pc_f8 = tc.coupling_weights_f8(w[rows].to(DEV), bias[rows].to(DEV), ch, sigma, ext, kind)
    x8 = _to_f8(x[:, perm[sigma]], c8).to(DEV)
    t8 = None if t_ext is None else _to_f8(t_ext[:, sigma], c8).to(DEV)
    y8, ld_f8, q_f8, _ = _run_f8(b8, pc_f8, x8, t8, None, 0, ch, inverse, N, H, W, 0, kind, "ticket_noacc", ticket)
    torch.cuda.synchronize()
    y_f8 = torch.empty(N, ch, H, W)
    y_f8[:, sigma] = _from_f8(y8.cpu())[:, :ch]
    err = rel_l2(y_f8, y_tc)
    print(f"coupling_f8 (permuted columns) vs coupling_tc (axis-1 gather) inv={int(inverse)} ext={int(ext)}: rel_l2 {err:.2e}  "
          f"logdet {ld_f8.tolist()} vs {ld_tc.tolist()}")
    assert err < 2e-6
    assert torch.allclose(ld_f8.cpu(), ld_tc.cpu(), rtol=2e-6, atol=0) and torch.allclose(q_f8.cpu(), q_tc.cpu(), rtol=2e-6, atol=0)
