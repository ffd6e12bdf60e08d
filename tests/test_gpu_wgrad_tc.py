"""csrc/wgrad_tc.cu (the tensor-core weight gradient of a 1x1 / 3x3 convolution from C8 half-precision x and dy) against a
float64 reference, at the shapes of the training step and at shapes chosen for the kernel's edges.

The kernel launches one CTA per (pixel chunk, input-channel block, M block of 128 output channels); each CTA walks the 8x16
pixel tiles of its chunk with stride gridDim.x through a 4-stage TMA ring and accumulates all of them in one TMEM accumulator,
then a second kernel sums the per-CTA partials in a fixed order.  The small shapes give one tile per CTA, so the cases below
add shapes on which every CTA walks many tiles (up to 512 at the banded stencil's 1536 -> 48 gradient): the ring wraps,
the producer waits on real MMA commits of both barrier parities and the accumulation across tiles runs.
``test_cases_cover_the_kernel_edges`` checks on the CPU, through the library's own workspace size, that the list reaches them.

Two tests per case and kind:
- small-integer operands (x in -2..2, dy in -1..1): every product and every partial sum is an integer below 2^20, so any
  summation order gives the exact value and the result must equal the float64 reference bit for bit.  A lost or repeated
  tile, a wrong halo offset, tap, channel block or M block shows up as an integer difference;
- normal operands rounded to the kind: rel-L2 and a per-element bound relative to sqrt(sum_p (x dy)^2), both growing with
  the tiles per CTA (see TOL_*); at 512x512, two launches must agree bit for bit.
dw and the workspace are NaN-filled before every launch, so an element the kernel never writes cannot pass."""
import pytest
import torch
import torch.nn.functional as F

from conftest import rel_l2

DEV = "cuda:0"
TILE_H, TILE_W, STAGES, NUM_SMS = 8, 16, 4, 148

# (N, Cin, Cout, H, W, K)
TRAINING = [
    (1, 64, 64, 512, 512, 3),       # sub-network trunk 3x3: 74 CTAs along pixels, 27-28 tiles each
    (1, 64, 64, 512, 512, 1),       # sub-network trunk 1x1: 148 CTAs, 13-14 tiles
    (1, 64, 96, 512, 512, 3),       # last sub-network conv
    (1, 48, 1536, 512, 512, 3),     # banded depth stencil dW1: 12 CTAs, 170-171 tiles
    (1, 1536, 48, 512, 512, 3),     # banded depth stencil dW2: 4 CTAs, 512 tiles
]
EDGES = [
    (1, 64, 64, 32, 32, 3), (2, 29, 48, 13, 37, 3), (1, 64, 96, 40, 24, 3), (1, 6, 64, 64, 64, 1), (1, 64, 64, 17, 33, 1),
    (1, 48, 48, 24, 40, 3), (2, 64, 12, 64, 48, 3), (1, 96, 64, 8, 16, 1), (1, 48, 200, 16, 32, 3), (1, 160, 48, 16, 32, 3),
    (1, 16, 1536, 8, 16, 3), (1, 256, 300, 9, 17, 1),
    (2, 200, 136, 45, 70, 3),       # 13 channel blocks of 16, 2 M blocks (the second one 16 channels): 5 CTAs, 12 tiles each
    (3, 100, 200, 45, 70, 1),       # 7 channel blocks of 16, 2 M blocks: 10 CTAs, 9 tiles each, walks cross images
    (2, 1000, 20, 30, 50, 3),       # 21 channel blocks of 48, Cout_p 32: 7 CTAs, 4-5 tiles each
    (2, 24, 40, 1, 1, 3), (1, 29, 7, 1, 37, 3), (1, 13, 30, 19, 1, 1), (3, 16, 16, 5, 9, 3),
]
CASES = TRAINING + EDGES


def _pad16(c):
    return (c + 15) // 16 * 16


def _seed(c):
    return sum(v * 1009 ** i for i, v in enumerate(c)) % (1 << 31)


def _case_id(c):
    return "{}x{}to{}-{}x{}-k{}".format(*c)


def _plan(N, Cin, Cout, H, W, K):
    """The kernel's launch geometry: channel blocking by the rule of wt_plan (csrc/wgrad_tc.cu), the number of pixel chunks
    from the library (workspace = chunks * Cout * Cin * K^2)."""
    from cwfa_b200 import _lib
    cin_p, cout_p = _pad16(Cin), _pad16(Cout)
    nb = min(cin_p, 48 if K == 3 else 64)
    while cin_p % nb:
        nb -= 16
    ws = _lib.load().cwfa_wgrad_tc_workspace_floats(N, H, W, Cin, cin_p, Cout, cout_p, K)
    assert ws % (Cout * Cin * K * K) == 0, ws
    chunks = ws // (Cout * Cin * K * K)
    n_ci_blk, n_m_blk = cin_p // nb, -(-cout_p // 128)
    tiles_per_img = -(-H // TILE_H) * -(-W // TILE_W)
    tiles = N * tiles_per_img
    assert chunks == min(max(1, NUM_SMS // (n_ci_blk * n_m_blk)), tiles), (chunks, n_ci_blk, n_m_blk, tiles)
    cross = any(len({t // tiles_per_img for t in range(b, tiles, chunks)}) > 1 for b in range(chunks))
    return dict(nb=nb, n_ci_blk=n_ci_blk, n_m_blk=n_m_blk, chunks=chunks, tiles=tiles, min_tiles=tiles // chunks,
                cross_image=cross, ws=ws)


def test_cases_cover_the_kernel_edges():
    """Host-side query only, no GPU needed."""
    p = {c: _plan(*c) for c in CASES}
    for K in (1, 3):            # >= 9 tiles on every CTA: each stage is reused twice, after commits of both barrier parities
        assert any(c[5] == K and v["min_tiles"] >= 2 * STAGES + 1 for c, v in p.items()), K
    assert any(c[0] >= 2 and v["cross_image"] for c, v in p.items())
    assert any(v["n_ci_blk"] > 1 and v["nb"] == 32 for v in p.values())
    assert any(v["n_ci_blk"] > 1 and v["nb"] == 16 for v in p.values())
    assert any(v["n_m_blk"] > 1 and _pad16(c[2]) % 128 for c, v in p.items())       # partial last M block: TMA zero-fill
    assert any(_pad16(c[2]) < 128 for c in CASES)                                   # zeroed A rows
    assert any(c[1] % 8 for c in CASES) and any(c[2] % 8 for c in CASES)
    assert any(c[3] % TILE_H and c[4] % TILE_W for c in CASES)
    assert any(c[3] == 1 for c in CASES) and any(c[4] == 1 for c in CASES)
    assert any(c[3] < TILE_H and c[4] < TILE_W for c in CASES)
    # pixel chunks and tiles per CTA of the training shapes (comments of TRAINING)
    assert [(_plan(*c)["chunks"], _plan(*c)["min_tiles"]) for c in TRAINING] == [(74, 27), (148, 13), (74, 27), (12, 170),
                                                                                 (4, 512)]


def _dtype(kind):
    return torch.bfloat16 if kind == "bf16" else torch.float16


def _c8(t, kind):
    """(N, C, H, W) values on the half grid -> the C8 layout [N][Cp/8][H][W][8], zero channel padding (built in torch)."""
    N, C, H, W = t.shape
    cp = _pad16(C)
    t = F.pad(t, (0, 0, 0, 0, 0, cp - C)).to(_dtype(kind))
    return t.reshape(N, cp // 8, 8, H, W).permute(0, 1, 3, 4, 2).contiguous()


def _wgrad_ref(x, dy, K):
    """float64 dW[co, ci, kh, kw] = sum over pixels of dy[co, pix] * x[ci, pix + (kh - p, kw - p)], zero padding."""
    N, Cin, H, W = x.shape
    Cout, p = dy.shape[1], K // 2
    xp = F.pad(x, (p, p, p, p))
    d = dy.transpose(0, 1).reshape(Cout, -1)
    out = torch.empty((Cout, Cin, K, K), dtype=torch.float64, device=x.device)
    for kh in range(K):
        for kw in range(K):
            out[:, :, kh, kw] = d @ xp[:, :, kh:kh + H, kw:kw + W].transpose(0, 1).reshape(Cin, -1).T
    return out


def _launch(x8, dy8, case, kind):
    """cwfa_wgrad_tc into a NaN-filled dW with a NaN-filled workspace."""
    from cwfa_b200 import _lib, ops
    N, Cin, Cout, H, W, K = case
    ws = torch.full((_plan(*case)["ws"],), float("nan"), device=DEV)
    dw = torch.full((Cout, Cin, K, K), float("nan"), device=DEV)
    _lib.call("cwfa_wgrad_tc", x8.data_ptr(), dy8.data_ptr(), dw.data_ptr(), ws.data_ptr(), N, H, W, Cin, _pad16(Cin), Cout,
              _pad16(Cout), K, K, int(kind == "bf16"), ops._stream())
    return dw


def _first_bad(bad, dw, ref):
    co, ci, kh, kw = [int(v) for v in bad.nonzero()[0]]
    return (f"{int(bad.sum())} of {bad.numel()} elements off; first at (co={co}, ci={ci}, kh={kh}, kw={kw}): "
            f"got {float(dw[co, ci, kh, kw]):.9g}, want {float(ref[co, ci, kh, kw]):.9g}")


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["bf16", "fp16"])
@pytest.mark.parametrize("case", CASES, ids=_case_id)
def test_wgrad_tc_small_integers_exact(case, kind):
    N, Cin, Cout, H, W, K = case
    g = torch.Generator(DEV).manual_seed(_seed(case))
    x = torch.randint(-2, 3, (N, Cin, H, W), generator=g, device=DEV).double()
    dy = torch.randint(-1, 2, (N, Cout, H, W), generator=g, device=DEV).double()
    assert 2 * N * H * W < 2 ** 24                       # |every partial sum| <= 2 N H W: exact in fp32 in any order
    dw = _launch(_c8(x, kind), _c8(dy, kind), case, kind)
    ref = _wgrad_ref(x, dy, K)
    bad = dw.double() != ref
    assert not bad.any(), _first_bad(bad, dw, ref)


# Limits of the rounded-normal test.  The error grows linearly with T, the most tiles one CTA accumulates in its TMEM
# accumulator (8 K-steps of 16 pixels per tile): measured on a B200 (1000 W power limit), both kinds, over the cases above,
#   rel-L2 over the whole dW:                          <= 1.95e-7 at T = 1, 1.5e-7 * T at T = 9 ... 512 (7.7e-5 at T = 512)
#   per element |dW - ref| / sqrt(sum_p (x dy)^2):     <= 1.84e-6 at T = 1, 8.0e-7 * T at T = 5 ... 512 (4.1e-4 at T = 512)
# The long-walk errors are biased toward smaller magnitudes (the accumulator's additions do not round to nearest), so they
# add up linearly instead of as a random walk.  Limits: the former 2e-5 rel-L2 of single-tile shapes, and ~4x the measured
# values per tile.  A lost tile of a 512-tile walk moves a typical element by sqrt(128 / 2^18) = 2.2e-2 of its scale.
TOL_REL = (2e-5, 6e-7)           # base + per tile
TOL_ELEM = (8e-6, 3.2e-6)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["bf16", "fp16"])
@pytest.mark.parametrize("case", CASES, ids=_case_id)
def test_wgrad_tc_rounded_random_vs_fp64(case, kind):
    N, Cin, Cout, H, W, K = case
    g = torch.Generator(DEV).manual_seed(_seed(case) + 1)
    x = torch.randn((N, Cin, H, W), generator=g, device=DEV).to(_dtype(kind)).double()
    dy = torch.randn((N, Cout, H, W), generator=g, device=DEV).to(_dtype(kind)).double()
    x8, dy8 = _c8(x, kind), _c8(dy, kind)
    dw = _launch(x8, dy8, case, kind)
    ref = _wgrad_ref(x, dy, K)
    scale = _wgrad_ref(x * x, dy * dy, K).sqrt()
    err = rel_l2(dw, ref)
    elem = (dw.double() - ref).abs() / scale.clamp_min(1e-300)
    plan = _plan(*case)
    T = -(-plan["tiles"] // plan["chunks"])
    tol_rel, tol_elem = TOL_REL[0] + TOL_REL[1] * T, TOL_ELEM[0] + TOL_ELEM[1] * T
    print(f"wgrad_tc {kind} {_case_id(case)} {plan}: rel_l2 {err:.2e} (limit {tol_rel:.1e})  per-element / scale "
          f"{float(elem.max()):.2e} (limit {tol_elem:.1e})")
    assert torch.isfinite(dw).all(), f"{int((~torch.isfinite(dw)).sum())} elements never written"
    bad = elem > tol_elem
    assert not bad.any(), _first_bad(bad, dw, ref)
    assert err < tol_rel, err
    if H * W >= 512 * 512:      # the per-CTA partials are summed in a fixed order: two launches agree bit for bit
        assert torch.equal(_launch(x8, dy8, case, kind), dw)
