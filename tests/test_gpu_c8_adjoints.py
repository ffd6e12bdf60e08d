"""The activation adjoints and channel statistics of csrc/c8ops.cu that the C8-native training nodes (autograd._SubnetTC,
autograd._StencilBandedTC) run, called through the C ABI and checked element by element:

- ``cwfa_c8_prelu``: y = v >= 0 ? v : a v;
- ``cwfa_c8_prelu_bwd``: g = pre > 0 ? dy : a dy (torch's PReLU adjoint, the slope at pre = 0), stats = [sum g, sum dy min(pre, 0)];
- ``cwfa_c8_elu_bwd``: g = dy (y > 0 ? 1 : y + 1) from the ELU output y, stats = [sum g, 0];
- ``cwfa_c8_channel_stats``: stats = [sum x, sum x^2].

Half-precision outputs must equal torch's fp32 arithmetic with one rounding bit for bit (signed zeros included).  The inputs
hold +0, -0, values in (-1, 0) and large negatives.  The per-channel sums are of the UNROUNDED fp32 values and are compared
with float64 sums of the same values, within the first-order bound of the kernel's fp32 summation relative to sum |term|;
with quarter-integer operands every partial sum is exact and the sums must match bit for bit.  Outputs, stats and workspace
are NaN-filled before each call (the tc.* wrappers allocate with torch.empty, which can hand back an earlier correct result).

Geometry: the adjoints launch nblk = clamp(ceil(148 * 8 / (Cp / 8)), 32, 256) blocks of 256 threads per 8-channel chunk, each
thread taking two pixels per step, 2 nblk 256 apart; channel statistics use 32 blocks with four loads per step.  Cp = 16, 64
and 1536 give 256, 148 and 32 blocks; P runs from 1 through below one stride, between one and two, to well above two with a
ragged tail, at N = 1 to 3, with the last 3 of the Cp channels being channel padding."""
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
SLOPE = 0.3                      # not a power of two: a v and a dy round
QUARTER = (-0.75, -0.5, -0.25, 0.0, 1.0, 2.0)
PAD = 3                          # channel padding of every case: C = Cp - 3


def _stride(cp):
    """Pixels one step of the activation adjoints covers with its first load (the second is this far behind)."""
    return min(256, max(32, -(-148 * 8 // (cp // 8)))) * 256


def _geoms():
    out = []
    for cp in (16, 64, 1536):
        s = _stride(cp)
        for n, p in ((1, 1), (2, s // 2 + 3), (3, s + s // 3 + 1), (2, 4 * s + s // 2 + 7)):
            out.append((cp, n, p))
    return out


GEOMS = _geoms()
# quarter-integer cases: N * P small enough that sum x^2 (terms <= 4 on a 1/16 grid) stays exact in fp32
QGEOMS = [(16, 2, _stride(16) + _stride(16) // 3 + 1), (64, 1, 4 * _stride(64) + _stride(64) // 2 + 7), (64, 3, 1),
          (1536, 3, 4 * _stride(1536) + _stride(1536) // 2 + 7)]


def _gid(g):
    return f"Cp{g[0]}-N{g[1]}-P{g[2]}"


def _dt(kind):
    return torch.bfloat16 if kind == "bf16" else torch.float16


def _c8(v, cp, kind):
    """(N, C, P) -> C8 [N][Cp/8][P][8] of the given kind, zero channel padding."""
    N, C, P = v.shape
    v = F.pad(v, (0, 0, 0, cp - C)).to(_dt(kind))
    return v.reshape(N, cp // 8, 8, P).permute(0, 1, 3, 2).contiguous()


def _per_channel(c8):
    """C8 [N][Cp/8][P][8] -> (N, Cp, P)."""
    N, G, P, _ = c8.shape
    return c8.permute(0, 1, 3, 2).reshape(N, G * 8, P)


def _operand(geom, kind, seed, elu_out=False):
    """Normal values with every 13th element +0, -0, in (-1, 0] or large negative (-1 for an ELU output), at element positions
    that depend on the seed."""
    cp, N, P = geom
    C = cp - PAD
    g = torch.Generator(DEV).manual_seed(seed)
    v = torch.randn((N, C, P), generator=g, device=DEV) * 2.0
    if elu_out:
        v = F.elu(v)
    u = torch.rand((N, C, P), generator=g, device=DEV)
    k = ((torch.arange(N * C * P, device=DEV) + seed) % 13).reshape(N, C, P)     # shifted by the seed: dy's zeros are not pre's
    v = torch.where(k == 0, torch.zeros_like(v), v)
    v = torch.where(k == 1, torch.full_like(v, -0.0), v)
    v = torch.where(k == 2, -u, v)
    v = torch.where(k == 3, torch.full_like(v, -1.0) if elu_out else -1000.0 * (1.0 + u), v)
    return _c8(v, cp, kind)


def _quarter_operands(geom, kind, seed):
    cp, N, P = geom
    C = cp - PAD
    g = torch.Generator(DEV).manual_seed(seed)
    y = torch.tensor(QUARTER, device=DEV)[torch.randint(0, len(QUARTER), (N, C, P), generator=g, device=DEV)]
    dy = torch.randint(-3, 4, (N, C, P), generator=g, device=DEV).float()
    return _c8(dy, cp, kind), _c8(y, cp, kind)


def _nan_like(t):
    return torch.full_like(t, float("nan"))


def _stats_buffers(cp):
    from cwfa_b200 import _lib
    return (torch.full((2 * cp,), float("nan"), device=DEV),
            torch.full((_lib.load().cwfa_c8_stats_workspace_floats(cp),), float("nan"), device=DEV))


def _assert_bitwise(got, want, what):
    a, b = got.view(torch.int16), want.view(torch.int16)
    if not torch.equal(a, b):
        bad = (a != b).nonzero()
        n, ch, p, j = [int(v) for v in bad[0]]
        raise AssertionError(f"{what}: {bad.shape[0]} elements differ; first at (n={n}, channel={8 * ch + j}, p={p}): got "
                             f"{float(got[n, ch, p, j])!r}, want {float(want[n, ch, p, j])!r}")


def _sum_bound(geom, threads_stride):
    """First-order bound of the kernel's fp32 sums relative to sum |term|: the sequential adds of one thread, the warp and
    block trees (5 + 3 levels) and the final rounding, with some slack."""
    cp, N, P = geom
    return (N * -(-P // threads_stride) + 16) * 2.0 ** -24


def _check_sums(got, terms, bound, what, exact=False):
    """got (Cp,) against float64 per-channel sums of the fp32 C8 terms; channel padding must be exactly zero."""
    t = _per_channel(terms).double()
    want = t.sum(dim=(0, 2))
    scale = t.abs().sum(dim=(0, 2))
    g = got.double()
    assert torch.isfinite(g).all(), f"{what}: {int((~torch.isfinite(g)).sum())} channels never written"
    C = got.numel() - PAD
    assert torch.equal(g[C:], torch.zeros_like(g[C:])), f"{what}: channel padding {g[C:].tolist()}"
    if exact:
        assert torch.equal(g, want), f"{what}: max |diff| {float((g - want).abs().max())}"
        return 0.0
    rel = float(((g - want).abs() / scale.clamp_min(1e-30)).max())
    assert rel <= bound, f"{what}: {rel:.2e} of sum |term| > {bound:.2e}"
    return rel


@pytest.mark.parametrize("kind", ["bf16", "fp16"])
@pytest.mark.parametrize("geom", GEOMS, ids=_gid)
def test_c8_prelu_forward(geom, kind):
    from cwfa_b200 import _lib, ops
    cp, N, P = geom
    x = _operand(geom, kind, 1)
    a = torch.full((1,), SLOPE, device=DEV)
    y = _nan_like(x)
    _lib.call("cwfa_c8_prelu", x.data_ptr(), a.data_ptr(), y.data_ptr(), N, cp, P, int(kind == "bf16"), ops._stream())
    v = x.float()
    _assert_bitwise(y, torch.where(v >= 0, v, v * a).to(_dt(kind)), "prelu")


def _prelu_bwd(dy, pre, a, geom, kind):
    from cwfa_b200 import _lib, ops
    cp, N, P = geom
    g = _nan_like(dy)
    stats, ws = _stats_buffers(cp)
    _lib.call("cwfa_c8_prelu_bwd", dy.data_ptr(), pre.data_ptr(), a.data_ptr(), g.data_ptr(), stats.data_ptr(), ws.data_ptr(),
              N, cp, P, int(kind == "bf16"), ops._stream())
    return g, stats


def _elu_bwd(dy, y, geom, kind):
    from cwfa_b200 import _lib, ops
    cp, N, P = geom
    g = _nan_like(dy)
    stats, ws = _stats_buffers(cp)
    _lib.call("cwfa_c8_elu_bwd", dy.data_ptr(), y.data_ptr(), g.data_ptr(), stats.data_ptr(), ws.data_ptr(), N, cp, P,
              int(kind == "bf16"), ops._stream())
    return g, stats


def _channel_stats(x, geom, kind):
    from cwfa_b200 import _lib, ops
    cp, N, P = geom
    stats, ws = _stats_buffers(cp)
    _lib.call("cwfa_c8_channel_stats", x.data_ptr(), stats.data_ptr(), ws.data_ptr(), N, cp, P, int(kind == "bf16"),
              ops._stream())
    return stats


@pytest.mark.parametrize("kind", ["bf16", "fp16"])
@pytest.mark.parametrize("geom", GEOMS, ids=_gid)
def test_c8_prelu_adjoint(geom, kind):
    cp = geom[0]
    dy, pre = _operand(geom, kind, 2), _operand(geom, kind, 5)
    a = torch.full((1,), SLOPE, device=DEV)
    g, stats = _prelu_bwd(dy, pre, a, geom, kind)
    d, p = dy.float(), pre.float()
    g32 = torch.where(p > 0, d, d * a)
    _assert_bitwise(g, g32.to(_dt(kind)), "prelu adjoint")
    bound = _sum_bound(geom, 2 * _stride(cp))
    e_s = _check_sums(stats[:cp], g32, 2 * bound, "sum g")
    e_q = _check_sums(stats[cp:], d * torch.clamp(p, max=0.0), 2 * bound, "sum dy min(pre, 0)")
    print(f"c8_prelu_bwd {kind} {_gid(geom)}: sums off by {e_s:.2e} / {e_q:.2e} of sum |term| (bound {2 * bound:.2e})")


@pytest.mark.parametrize("kind", ["bf16", "fp16"])
@pytest.mark.parametrize("geom", GEOMS, ids=_gid)
def test_c8_elu_adjoint(geom, kind):
    cp = geom[0]
    dy, y = _operand(geom, kind, 4), _operand(geom, kind, 6, elu_out=True)
    g, stats = _elu_bwd(dy, y, geom, kind)
    d, v = dy.float(), y.float()
    g32 = d * torch.where(v > 0, torch.ones_like(v), v + 1.0)
    _assert_bitwise(g, g32.to(_dt(kind)), "elu adjoint")
    bound = _sum_bound(geom, 2 * _stride(cp))
    e_s = _check_sums(stats[:cp], g32, 2 * bound, "sum g")
    assert torch.equal(stats[cp:], torch.zeros_like(stats[cp:]))
    print(f"c8_elu_bwd {kind} {_gid(geom)}: sum g off by {e_s:.2e} of sum |g| (bound {2 * bound:.2e})")


@pytest.mark.parametrize("kind", ["bf16", "fp16"])
@pytest.mark.parametrize("geom", GEOMS, ids=_gid)
def test_c8_channel_stats(geom, kind):
    cp = geom[0]
    x = _operand(geom, kind, 7)
    stats = _channel_stats(x, geom, kind)
    bound = _sum_bound(geom, 32 * 256)
    v = x.float()
    e_s = _check_sums(stats[:cp], v, bound, "sum x")
    e_q = _check_sums(stats[cp:], v * v, bound, "sum x^2")
    print(f"c8_channel_stats {kind} {_gid(geom)}: sums off by {e_s:.2e} / {e_q:.2e} of sum |term| (bound {bound:.2e})")


@pytest.mark.parametrize("kind", ["bf16", "fp16"])
@pytest.mark.parametrize("geom", QGEOMS, ids=_gid)
def test_c8_sums_exact_on_quarter_integers(geom, kind):
    """dy in -3..3, slope 1/4, pre / y / x in QUARTER: every term lies on a 1/16 grid and every partial sum is bounded by
    sum |term| < 2^20, so all sums are exact in fp32 in any order."""
    cp, N, P = geom
    dy, v = _quarter_operands(geom, kind, 7)
    assert N * P * 4 < 2 ** 20
    a = torch.full((1,), 0.25, device=DEV)
    d, p = dy.float(), v.float()
    g, stats = _prelu_bwd(dy, v, a, geom, kind)
    g32 = torch.where(p > 0, d, d * a)
    _assert_bitwise(g, g32.to(_dt(kind)), "prelu adjoint")
    _check_sums(stats[:cp], g32, 0.0, "prelu sum g", exact=True)
    _check_sums(stats[cp:], d * torch.clamp(p, max=0.0), 0.0, "prelu sum dy min(pre, 0)", exact=True)
    g, stats = _elu_bwd(dy, v, geom, kind)
    g32 = d * torch.where(p > 0, torch.ones_like(p), p + 1.0)
    _assert_bitwise(g, g32.to(_dt(kind)), "elu adjoint")
    _check_sums(stats[:cp], g32, 0.0, "elu sum g", exact=True)
    stats = _channel_stats(v, geom, kind)
    _check_sums(stats[:cp], p, 0.0, "sum x", exact=True)
    _check_sums(stats[cp:], p * p, 0.0, "sum x^2", exact=True)
