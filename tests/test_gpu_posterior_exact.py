"""Exact per-voxel posterior standard deviation in one reconstruction pass: the scale-carrying inverse coupling
(cwfa_coupling_f8_scale), the merge fused with the standard-deviation rule (cwfa_haar1d_inv_std_f8), and
CWFAEngine.reconstruct_posterior_exact / reconstruct_posterior_exact_graphed.

On CAT-only levels the volume is affine in the latents and every voxel depends on exactly one detail element per level, so
std^2 = sigma_T^2 * sum_n (V(z = 1_n) - V(z = 0))^2 with 1_n the all-ones latents of level n: the engine is checked against that
identity run on its own kernels (tight) and on the float64 oracle (the reference error), and against the Monte Carlo estimate of
reconstruct_posterior.  The kernels are checked against float64 on the same half-rounded operands, and y / log-det / x bitwise
against the kernels they extend.  Every output of the kernel tests is NaN-filled before the launch."""
import ctypes
import math

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from conftest import rel_l2
from helpers import build_tiny_model, tiny_inputs
from oracle import cwfa_oracle as O
from oracle.weights import deterministic_fill, seeded_randn

DEV = "cuda:0"
gpu = pytest.mark.gpu
CLAMP, K_ATAN = 2.0, 0.636
T_SCALE = -0.5 ** 0.5
SHAPES = {"ragged": (2, 37, 13), "multi": (3, 230, 230)}
SIGMA_07 = 0.39104826405548904           # sqrt(truncated_normal_var(0.7))


def _round(t, kind):
    return t.to(torch.bfloat16 if kind == "bf16" else torch.float16).float()


def _nan(*shape):
    return torch.full(shape, float("nan"), device=DEV)


def _to_f8(x, c8):
    N, C, H, W = x.shape
    xp = torch.zeros(N, c8, H, W, dtype=x.dtype)
    xp[:, :C] = x
    return xp.view(N, c8 // 8, 8, H, W).permute(0, 1, 3, 4, 2).contiguous()


def _from_f8(y8):
    N, G, H, W, _ = y8.shape
    return y8.permute(0, 1, 4, 2, 3).reshape(N, G * 8, H, W)


def _c8_slice(b, kind, chunk_off):
    """b (N,64,H,W) as the 8-chunk slice at chunk_off of a 192-channel C8 tensor [N][24][H][W][8] (the batched trunks' output)."""
    N, _, H, W = b.shape
    full = _round(1.0e3 * (1.0 + seeded_randn((N, 192, H, W), 1304).abs()), kind)
    full[:, 8 * chunk_off:8 * chunk_off + 64] = b
    dt = torch.bfloat16 if kind == "bf16" else torch.float16
    return full.view(N, 24, 8, H, W).permute(0, 1, 3, 4, 2).contiguous().to(dt).to(DEV)


def test_truncated_normal_var_matches_sampling():
    """CPU: the closed form against the variance of 10^7 draws of the sampler the engine uses (torch.nn.init.trunc_normal_)."""
    from cwfa_b200.pipeline import truncated_normal_var
    assert truncated_normal_var(0.0) == 0.0
    assert abs(math.sqrt(truncated_normal_var(0.7)) - 0.39105) < 5e-6
    g = torch.Generator().manual_seed(1)
    for T in (0.5, 0.7, 2.0):
        z = torch.empty(10_000_000, dtype=torch.float64)
        torch.nn.init.trunc_normal_(z, mean=0.0, std=1.0, a=-T, b=T, generator=g)
        v, ref = float(z.var()), truncated_normal_var(T)
        print(f"truncated_normal_var({T}) = {ref:.6f}, sampled {v:.6f} (rel {abs(v - ref) / ref:.1e})")
        assert abs(v - ref) < 3e-3 * ref                     # the sampling error of 10^7 draws is below 5e-4 relative
    with pytest.raises(ValueError):
        truncated_normal_var(-0.1)


# ------------------------------------------------------------------------------------------------ kernel (1): scale chain
_CONV = {}


def _conv_ref(shape, kind, blk):
    """Condition b (N,64,H,W), 96 rows of 3x3 weights + bias on the half grid for block ``blk`` of a chain, and a = conv(b) in
    float64 (s = rows [0, ch), t = rows [48, 48 + ch))."""
    key = (shape, kind, blk)
    if key not in _CONV:
        N, H, W = SHAPES[shape]
        b = _round(seeded_randn((N, 64, H, W), 1301 + 10 * blk), kind)
        w = _round(seeded_randn((96, 64, 3, 3), 1302 + 10 * blk, 0.04), kind)
        bias = seeded_randn((96,), 1303 + 10 * blk, 0.5)
        _CONV[key] = (b, w, bias, F.conv2d(b.double(), w.double(), bias.double(), padding=1))
    return _CONV[key]


def _perm(n, seed):
    return torch.from_numpy(np.random.RandomState(seed).permutation(n)).long()


# (kind, ch, external shift in the chain's last block, shape, blocks, input chunk offset): blocks = 3 is first (no x, no
# scale) -> middle (row gather) -> last (column gather), in inverse order; blocks = 1 is a level of one block
KERNEL_CASES = [
    ("bf16", 48, False, "multi", 3, 0),
    ("bf16", 1, True, "ragged", 3, 8),
    ("fp16", 48, True, "ragged", 3, 16),
    ("fp16", 20, False, "multi", 3, 8),
    ("bf16", 20, True, "multi", 3, 16),
    ("fp16", 8, False, "ragged", 3, 0),
    ("bf16", 8, True, "ragged", 1, 8),
    ("fp16", 1, False, "multi", 1, 0),
    ("bf16", 48, True, "multi", 1, 16),
]

# Scale error relative to the float64 chain on the same half-rounded operands (atan_fast + ex2.approx per block).  Limit at ~4x
# the worst value measured on a B200 (1000 W power limit) over the cases above: 1.09e-5 (bf16, ch 48 and ch 20, 3 blocks at
# 3x230x230); fp16 at most 4.8e-6.
TOL_SCALE = 4.5e-5


def _launch(name, shape, blk, kind, ch, x8, t8, perm, axis, chunk_off, s_in=None, s_out=None):
    """One inverse launch of cwfa_coupling_f8 / cwfa_coupling_f8_scale for block ``blk``: (y8, logdet, sumsq), NaN-filled before."""
    from cwfa_b200 import _lib, ops, tc
    N, H, W = SHAPES[shape]
    b, w, bias, _ = _conv_ref(shape, kind, blk)
    ext = t8 is not None
    rows = list(range(ch)) + ([] if ext else list(range(48, 48 + ch)))
    pc = tc.coupling_weights_f8(w[rows].to(DEV), bias[rows].to(DEV), ch, torch.arange(ch), ext, kind)
    c8 = tc.ch8(ch)
    tiles = _lib.load().cwfa_coupling_tc_tiles(H, W)
    y8, ws, ld, sq = _nan(N, c8 // 8, H, W, 8), _nan(2 * N * tiles), _nan(N), _nan(N)
    ticket = torch.zeros(1, device=DEV, dtype=torch.int32)
    args = [_c8_slice(b, kind, chunk_off).data_ptr(), pc.packed.data_ptr(), ops._p(pc.bias), N, H, W, pc.BN, c8, ops._p(x8),
            y8.data_ptr(), ops._p(t8), float(T_SCALE if ext else 1.0), ops._p(perm), axis, CLAMP, K_ATAN, 1, ws.data_ptr(),
            ld.data_ptr(), sq.data_ptr(), 0, ticket.data_ptr(), 24, chunk_off, int(kind == "bf16"), ops._stream()]
    if name == "scale":
        _lib.call("cwfa_coupling_f8_scale", *args, ops._p(s_in), s_out.data_ptr())
    else:
        _lib.call("cwfa_coupling_f8", *args)
    torch.cuda.synchronize()
    assert int(ticket[0]) == 0
    return y8, ld, sq


@gpu
@pytest.mark.parametrize("kind,ch,ext,shape,blocks,chunk_off", KERNEL_CASES)
def test_coupling_f8_scale_chain_vs_fp64(kind, ch, ext, shape, blocks, chunk_off):
    from cwfa_b200 import tc
    N, H, W = SHAPES[shape]
    c8 = tc.ch8(ch)
    t_ext = seeded_randn((N, ch, H, W), 1351, 0.3) if ext else None
    gathers = [(None, 0), (_perm(H, 1362), 2), (_perm(W, 1363), 3)][:blocks]
    # float64 reference chain of the scale: gathered like x, then multiplied by exp(-s) of the block
    scale = torch.ones(N, ch, H, W, dtype=torch.float64)
    for blk, (p, axis) in enumerate(gathers):
        a = _conv_ref(shape, kind, blk)[3]
        if p is not None:
            scale = scale.index_select(axis, p)
        scale = scale * torch.exp(-CLAMP * K_ATAN * torch.atan(a[:, :ch]))
    # the GPU chains: coupling_f8_scale and coupling_f8 on the same inputs
    t8 = None if t_ext is None else _to_f8(t_ext, c8).to(DEV)
    xs = xp = s8 = None
    for blk, (p, axis) in enumerate(gathers):
        pd = None if p is None else p.to(DEV, torch.int32)
        tb = t8 if blk == blocks - 1 else None
        s_out = _nan(N, c8 // 8, H, W, 8)
        got = _launch("scale", shape, blk, kind, ch, xs, tb, pd, axis, chunk_off, s8, s_out)
        ref = _launch("plain", shape, blk, kind, ch, xp, tb, pd, axis, chunk_off)
        for g_, r_, what in zip(got, ref, ("y", "log-det", "sum y^2")):
            assert torch.equal(g_, r_), f"block {blk}: {what} differs from cwfa_coupling_f8"
        xs, xp, s8 = got[0], ref[0], s_out
    sf = _from_f8(s8.cpu())
    assert torch.isfinite(sf).all(), "a scale entry was not written"
    err = ((sf[:, :ch].double() - scale) / scale).abs()
    worst = float(err.max())
    print(f"coupling_f8_scale {kind} ch={ch} ext={int(ext)} {shape} {N}x{H}x{W} blocks={blocks} chunk_off={chunk_off}: "
          f"scale rel {worst:.2e} (limit {TOL_SCALE:.0e})")
    assert worst < TOL_SCALE


def test_coupling_f8_scale_rejects_bad_arguments():
    """CPU: argument checks that run before anything touches a device."""
    from cwfa_b200 import _lib
    lib = _lib.load()
    p, q = ctypes.c_void_p(16), ctypes.c_void_p(32)

    def call(inverse=1, s_in=p, s_out=q):
        return lib.cwfa_coupling_f8_scale(p, p, None, 1, 16, 16, 96, 48, p, p, None, 1.0, None, 0, 2.0, 0.636, inverse, p, p, None, 1,
                                          None, 8, 0, 1, None, s_in, s_out)
    assert call(inverse=0) != 0                              # inverse only
    assert b"inverse only" in lib.cwfa_last_error()
    assert call(s_out=None) != 0
    assert call(s_in=q, s_out=q) != 0                        # in place races with the gather
    assert b"alias" in lib.cwfa_last_error()


# ------------------------------------------------------------------------------------------------ kernel (2): std merge
# (B, h channels, H, W, std_lo given, sigma): h not a multiple of 8, P = H * W a multiple of 4 but not of the warp's 128 pixels
MERGE_CASES = [
    (1, 12, 13, 4, False, 0.391),
    (2, 5, 9, 12, True, 0.391),
    (1, 48, 16, 16, True, 1.0),
    (3, 24, 6, 10, False, 1.0),
    (2, 20, 7, 8, True, 0.0),
    (1, 6, 8, 5, False, 0.0),
]
STD_ULPS = 3.0                           # |std - fp64| / (2^-23 std): measured <= 0.94 (B200); the rounding steps bound it near 1.25


@gpu
@pytest.mark.parametrize("B,h,H,W,with_std_lo,sigma", MERGE_CASES)
def test_haar1d_inv_std_f8_vs_fp64(B, h, H, W, with_std_lo, sigma):
    from cwfa_b200 import _lib, ops, tc
    lo = seeded_randn((B, h, H, W), 1401)
    hi = seeded_randn((B, h, H, W), 1402)
    sc = seeded_randn((B, h, H, W), 1403).abs() * 3.0 + 1e-3
    std_lo = seeded_randn((B, h, H, W), 1404).abs() if with_std_lo else None
    c8 = tc.ch8(h)
    lo_d, hi8, sc8 = lo.to(DEV), _to_f8(hi, c8).to(DEV), _to_f8(sc, c8).to(DEV)
    sl_d = None if std_lo is None else std_lo.to(DEV)
    x, sx = _nan(B, 2 * h, H, W), _nan(B, 2 * h, H, W)
    _lib.call("cwfa_haar1d_inv_std_f8", lo_d.data_ptr(), ops._p(sl_d), hi8.data_ptr(), sc8.data_ptr(), sigma, x.data_ptr(), sx.data_ptr(),
              B, 2 * h, H * W, ops._stream())
    torch.cuda.synchronize()
    assert torch.equal(x, tc.haar1d_merge_f8(lo_d, hi8)), "x differs from haar1d_merge_f8"
    sig = float(np.float32(sigma))
    var = 0.5 * ((0.0 if std_lo is None else std_lo.double() ** 2) + (sig * sc.double()) ** 2)
    ref = torch.sqrt(var).repeat_interleave(2, dim=1)
    got = sx.double().cpu()
    if sigma == 0 and std_lo is None:
        assert torch.equal(sx, torch.zeros_like(sx)), "sigma 0 and no std_lo: std must be exactly 0"
        return
    ulp = ref * 2.0 ** -23
    e = float(((got - ref).abs() / ulp).max())
    print(f"haar1d_inv_std_f8 B={B} h={h} {H}x{W} std_lo={int(with_std_lo)} sigma={sigma}: std {e:.2f} ulp (limit {STD_ULPS})")
    assert e <= STD_ULPS
    # the wrapper gives the same
    x2, s2 = tc.haar1d_merge_std_f8(lo_d, sl_d, hi8, sc8, sigma)
    assert torch.equal(x2, x) and torch.equal(s2, sx)


def test_haar1d_inv_std_f8_rejects_bad_arguments():
    """CPU: argument checks that run before anything touches a device."""
    from cwfa_b200 import _lib
    lib = _lib.load()
    p = ctypes.c_void_p(16)

    def call(sigma=0.5, x=p, std_x=p, P=16, C=8):
        return lib.cwfa_haar1d_inv_std_f8(p, None, p, p, sigma, x, std_x, 1, C, P, None)
    assert call(sigma=-0.1) != 0 and b"sigma" in lib.cwfa_last_error()
    assert call(sigma=float("nan")) != 0 and call(sigma=float("inf")) != 0
    assert call(x=None) != 0 and call(std_x=None) != 0
    assert call(P=18) != 0                                   # F8 needs P % 4 == 0
    assert call(C=7) != 0


# ----------------------------------------------------------------------------------------------------------------- engine
def _ones_at(model, n, B):
    return [torch.ones((B,) + tuple(model.conv_inn[k].global_out_shapes[0]), device=DEV) if k == n else
            torch.zeros((B,) + tuple(model.conv_inn[k].global_out_shapes[0]), device=DEV) for k in range(model.n_levels)]


def _linear_std(recon, model, B, sigma):
    """sigma * sqrt(sum_n (V(1_n) - V(0))^2) with V = recon(zs) (float64)."""
    v0 = recon(_ones_at(model, -1, B)).double().cpu()
    acc = torch.zeros_like(v0)
    for n in range(model.n_levels):
        acc += (recon(_ones_at(model, n, B)).double().cpu() - v0) ** 2
    return sigma * acc.sqrt()


def _identity_error(std, mean, ref):
    """max |std - ref| / (1e-4 ref + 1e-6 (1 + |mean|)): the identity on the engine's own kernels holds to fp32 rounding."""
    std, mean = std.double().cpu(), mean.double().cpu()
    return float(((std - ref).abs() / (1e-4 * ref + 1e-6 * (1.0 + mean.abs()))).max())


def _dbl(obj):
    if torch.is_tensor(obj):
        return obj.double() if obj.is_floating_point() else obj
    if isinstance(obj, dict):
        return {k: _dbl(v) for k, v in obj.items()}
    if isinstance(obj, list):
        return [_dbl(v) for v in obj]
    return obj


@pytest.fixture(scope="module")
def tiny(golden_tiny):
    model = build_tiny_model(golden_tiny, DEV)
    views, mean_vols = tiny_inputs(golden_tiny)
    return model, views.to(DEV), [t.to(DEV) for t in mean_vols]


# std against the float64 oracle run of the same identity, rel-L2: limit at ~4x the value measured on a B200 (1000 W power limit),
# 1.03e-2 (bf16) / 1.34e-3 (fp16) -- both inside the engine's stated 2e-2 / 3e-3 on the reconstruction.
TOL_STD_REF = {"bf16": 4e-2, "fp16": 5.5e-3}


@gpu
@pytest.mark.parametrize("kind", ["bf16", "fp16"])
def test_engine_posterior_exact_tiny(tiny, kind):
    from cwfa_b200.engine import CWFAEngine
    model, views, mv = tiny
    eng = CWFAEngine(model, kind)
    mean, std = (t.clone() for t in eng.reconstruct_posterior_exact(views, mv, temperature=0.7))
    assert tuple(mean.shape) == tuple(std.shape) == (1, model.cfg.n_depths, views.shape[2], views.shape[3])
    assert torch.equal(mean, eng.reconstruct(views, mv)), "mean must be bitwise reconstruct()"
    # the linearity identity on the engine's own kernels
    ref = _linear_std(lambda zs: eng.reconstruct(views, mv, zs=zs), model, 1, SIGMA_07)
    e_id = _identity_error(std, mean, ref)
    # the same identity on the float64 oracle: the error against the reference
    om = _dbl(model.export_for_oracle())
    vd, mvd = views.double().cpu(), [m.double().cpu() for m in mv]
    ref64 = _linear_std(lambda zs: O.reconstruct(om, vd, mvd, zs=[z.double().cpu() for z in zs]), model, 1, SIGMA_07)
    e_ref = rel_l2(std, ref64)
    # against the Monte Carlo estimate of reconstruct_posterior, K = 64
    K = 64
    g = torch.Generator().manual_seed(21)
    zs = []
    for n in range(model.n_levels):
        z = torch.empty((K,) + tuple(model.conv_inn[n].global_out_shapes[0]))
        torch.nn.init.trunc_normal_(z, mean=0.0, std=1.0, a=-0.7, b=0.7, generator=g)
        zs.append(z.to(DEV))
    _, s_mc = eng.reconstruct_posterior(views, mv, K, zs=zs)
    ratio = float((s_mc.double() ** 2 / std.double() ** 2).mean())
    print(f"posterior exact tiny {kind}: identity {e_id:.3f} (limit 1), std vs fp64 rel-L2 {e_ref:.2e} (limit {TOL_STD_REF[kind]:.0e}), "
          f"mean s_MC^2 / std^2 (K={K}) {ratio:.4f}; mean |std| {float(std.mean()):.3e}")
    assert e_id < 1.0
    assert e_ref < TOL_STD_REF[kind]
    assert abs(ratio - 1.0) < 0.02
    # temperature 0: the prior is a point mass
    m0, s0 = eng.reconstruct_posterior_exact(views, mv, temperature=0.0)
    assert torch.equal(s0, torch.zeros_like(s0)) and torch.equal(m0, mean)


@gpu
def test_engine_posterior_exact_graphed_sensor_and_batch(tiny):
    from cwfa_b200.data import LensletLayout
    from cwfa_b200.engine import CWFAEngine
    model, views, mv = tiny
    eng = CWFAEngine(model, "bf16")
    eager = {T: [t.clone() for t in eng.reconstruct_posterior_exact(views, mv, temperature=T)] for T in (0.7, 0.3)}
    for T in (0.7, 0.3, 0.7):                                 # a graph per temperature; switching back replays the first
        gm, gs = eng.reconstruct_posterior_exact_graphed(views, mv, temperature=T)
        assert torch.equal(gm, eager[T][0]) and torch.equal(gs, eager[T][1]), T
    assert not torch.equal(eager[0.7][1], eager[0.3][1])
    # raw sensor frame: bitwise the views path
    coords = [[40 + 50 * (i // 6), 35 + 55 * (i % 6)] for i in range(29)]
    layout = LensletLayout(coords, (64, 64), 32768.0, 16384.0, device=DEV)
    gen = torch.Generator().manual_seed(7)
    frame = torch.randint(0, 65536, (1, 1, 300, 340), generator=gen, dtype=torch.int32).to(torch.uint16).to(DEV)
    ref = [t.clone() for t in eng.reconstruct_posterior_exact(layout.views(frame), mv, temperature=0.7)]
    got = eng.reconstruct_posterior_exact(frame, mv, temperature=0.7, sensor=layout)
    assert torch.equal(got[0], ref[0]) and torch.equal(got[1], ref[1])
    gg = eng.reconstruct_posterior_exact_graphed(frame, mv, temperature=0.7, sensor=layout)
    assert torch.equal(gg[0], ref[0]) and torch.equal(gg[1], ref[1])
    # batch 2
    vB = torch.cat([views, seeded_randn(tuple(views.shape), 1501).to(DEV)])
    mvB = [m.repeat(2, 1, 1, 1) for m in mv[:model.n_levels]]
    mean, std = (t.clone() for t in eng.reconstruct_posterior_exact(vB, mvB, temperature=0.7))
    assert tuple(std.shape) == (2, model.cfg.n_depths, views.shape[2], views.shape[3])
    assert torch.equal(mean, eng.reconstruct(vB, mvB))
    e_id = _identity_error(std, mean, _linear_std(lambda zs: eng.reconstruct(vB, mvB, zs=zs), model, 2, SIGMA_07))
    print(f"posterior exact batch 2: identity {e_id:.3f} (limit 1)")
    assert e_id < 1.0
    gm, gs = eng.reconstruct_posterior_exact_graphed(vB, mvB, temperature=0.7)
    assert torch.equal(gm, mean) and torch.equal(gs, std)


def _ragged_model():
    import cwfa_b200
    m = cwfa_b200.CWFAModel(n_depths=24, volume_side_size=72, INN_max_down_steps=3, seed=0)
    for n in range(m.n_levels):
        sd = deterministic_fill(m.conv_inn[n].state_dict(), 400 + n)
        sd.update({k: v for k, v in m.conv_inn[n].state_dict().items() if "perm" in k})
        m.conv_inn[n].load_state_dict(sd)
        m.cond_nets[n].load_state_dict(deterministic_fill(m.cond_nets[n].state_dict(), 500 + n))
    m.cond_nets[-1].load_state_dict(deterministic_fill(m.cond_nets[-1].state_dict(), 600))
    return m.to(DEV)


@gpu
def test_engine_posterior_exact_ragged():
    """24 depths (12- and 6-channel detail halves), 72 x 72: eager and graphed."""
    from cwfa_b200.engine import CWFAEngine
    model = _ragged_model()
    views = seeded_randn((1, 29, 72, 72), 41).to(DEV)
    mv = [seeded_randn((1, 24 // 2 ** (n + 1), 72, 72), 50 + n, 0.1).to(DEV) for n in range(2)] + \
         [seeded_randn((1, 24 // 4, 72, 72), 59, 0.1).to(DEV)]
    eng = CWFAEngine(model, "fp16")
    mean, std = (t.clone() for t in eng.reconstruct_posterior_exact(views, mv, temperature=0.7))
    assert torch.equal(mean, eng.reconstruct(views, mv))
    e_id = _identity_error(std, mean, _linear_std(lambda zs: eng.reconstruct(views, mv, zs=zs), model, 1, SIGMA_07))
    print(f"posterior exact ragged: identity {e_id:.3f} (limit 1)")
    assert e_id < 1.0
    gm, gs = eng.reconstruct_posterior_exact_graphed(views, mv, temperature=0.7)
    assert torch.equal(gm, mean) and torch.equal(gs, std)


def _glow_model(golden_tiny):
    import cwfa_b200
    np.random.seed(0)
    torch.manual_seed(0)
    cfg = golden_tiny["config"]
    m = cwfa_b200.CWFAModel(n_depths=cfg["D"], volume_side_size=cfg["S"], INN_max_down_steps=cfg["MAX"], INN_block_type="GLOW",
                            INN_n_blocks=2)
    for n in range(m.n_levels):
        sd = deterministic_fill(m.conv_inn[n].state_dict(), 900 + n)
        sd.update({k: v for k, v in m.conv_inn[n].state_dict().items() if "perm" in k or k.endswith("w_0")})
        m.conv_inn[n].load_state_dict(sd)
    return m.to(DEV)


@gpu
def test_engine_posterior_exact_rejects(golden_tiny, tiny):
    import cwfa_b200
    from cwfa_b200.engine import CWFAEngine
    model, views, mv = tiny
    cfg = golden_tiny["config"]
    dlr = cwfa_b200.CWFAModel(n_depths=cfg["D"], volume_side_size=cfg["S"], INN_max_down_steps=cfg["MAX"], disable_low_res_input=1,
                              seed=0).to(DEV)
    with pytest.raises(ValueError, match="disable_low_res_input"):
        CWFAEngine(dlr, "bf16").reconstruct_posterior_exact(views, mv)
    glow = CWFAEngine(_glow_model(golden_tiny), "bf16")
    with pytest.raises(ValueError, match="level 0 .*GLOW"):
        glow.reconstruct_posterior_exact(views, mv, temperature=0.7)
    with pytest.raises(ValueError, match="level 0"):
        glow.reconstruct_posterior_exact_graphed(views, mv, temperature=0.7)
    eng = CWFAEngine(model, "bf16")
    eng.use_f8 = False
    with pytest.raises(ValueError, match="use_f8"):
        eng.reconstruct_posterior_exact(views, mv)
    eng.use_f8 = True
    with pytest.raises(ValueError, match="temperature"):
        eng.reconstruct_posterior_exact(views, mv, temperature=-0.1)
    with pytest.raises(ValueError, match="temperature"):
        eng.reconstruct_posterior_exact_graphed(views, mv, temperature=-0.1)


@gpu
def test_engine_posterior_exact_full_config():
    """96 x 512 x 512 (5 steps, bf16), batch 1: the mean bitwise, and the identity over the four flow levels."""
    import cwfa_b200
    from cwfa_b200.engine import CWFAEngine
    model = cwfa_b200.CWFAModel(seed=0).to(DEV)
    g = torch.Generator().manual_seed(1)
    views = torch.randn((1, 29, 512, 512), generator=g).to(DEV)
    mvs = [(0.1 * torch.randn((1, 96 // 2 ** (n + 1), 512, 512), generator=g)).to(DEV) for n in range(4)]
    eng = CWFAEngine(model, "bf16")
    mean, std = (t.clone() for t in eng.reconstruct_posterior_exact(views, mvs, temperature=0.7))
    assert torch.equal(mean, eng.reconstruct(views, mvs))
    e_id = _identity_error(std, mean, _linear_std(lambda zs: eng.reconstruct(views, mvs, zs=zs), model, 1, SIGMA_07))
    print(f"posterior exact full config: identity {e_id:.3f} (limit 1); mean |std| {float(std.mean()):.3e}")
    assert e_id < 1.0
