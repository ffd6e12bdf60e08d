"""Per-voxel NLL maps of the forward pass: the map-writing F8 coupling (cwfa_coupling_f8_map) and
CWFAEngine.forward_nll(nll_map=True) / forward_nll_graphed(nll_map=True).

Every coupling of a level is elementwise (s and t come from the conditions only), so each detail element's NLL is
0.5 z^2 - sum over the level's blocks of s, indexed by the element's coordinate at the level's input.  The kernel is checked
against a float64 chain on the same half-rounded operands, and its y / log-det / sum y^2 bitwise against cwfa_coupling_f8; the
engine against a float64 run of the oracle's pieces that carries an index tensor through every permutation, and exactly by
locality: a perturbation of a small voxel box changes the maps there and nowhere else.  Every output of the kernel tests is
NaN-filled before the launch."""
import ctypes

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
FIRST, LAST = 1, 2

# The map is a difference of terms (0.5 y^2 and the blocks' s) that can be several times larger than it, so its error is taken
# relative to their size: |map - ref| / (1 + 0.5 y^2 + sum |s|), reference values.  Limit at ~4x the worst value measured on a
# B200 (1000 W power limit) over the kernel cases below: 7.1e-5 (bf16, ch 48, 3 blocks at 3x230x230); fp16 at most 1.5e-5.
TOL_MAP = 3e-4


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


def _c8(b, kind):
    N, _, H, W = b.shape
    dt = torch.bfloat16 if kind == "bf16" else torch.float16
    return b.view(N, 8, 8, H, W).permute(0, 1, 3, 4, 2).contiguous().to(dt).to(DEV)


# ------------------------------------------------------------------------------------------------------ kernel
_CONV = {}


def _conv_ref(shape, kind, blk):
    """Condition b (N,64,H,W) and 96 rows of 3x3 weights + bias on the half grid for block ``blk`` of a chain, and a = conv(b)
    in float64 (s = rows [0, ch), t = rows [48, 48 + ch))."""
    key = (shape, kind, blk)
    if key not in _CONV:
        N, H, W = SHAPES[shape]
        b = _round(seeded_randn((N, 64, H, W), 1101 + 10 * blk), kind)
        w = _round(seeded_randn((96, 64, 3, 3), 1102 + 10 * blk, 0.04), kind)
        bias = seeded_randn((96,), 1103 + 10 * blk, 0.5)
        _CONV[key] = (b, w, bias, F.conv2d(b.double(), w.double(), bias.double(), padding=1))
    return _CONV[key]


def _perm(n, seed):
    return torch.from_numpy(np.random.RandomState(seed).permutation(n)).long()


# (kind, ch, external shift in the first block, shape, blocks): blocks = 3 is first -> middle (row gather) -> last (column
# gather); blocks = 1 is a level of one block (FIRST | LAST)
KERNEL_CASES = [
    ("bf16", 48, False, "multi", 3),
    ("bf16", 1, True, "ragged", 3),
    ("fp16", 48, True, "ragged", 3),
    ("fp16", 13, False, "multi", 3),
    ("bf16", 24, True, "multi", 3),
    ("fp16", 1, False, "ragged", 3),
    ("bf16", 40, True, "ragged", 1),
    ("fp16", 8, False, "multi", 1),
]


def _launch(name, shape, blk, kind, ch, x8, t8, perm, axis, m8=None, rsrc=None, csrc=None, mode=0):
    """One launch of cwfa_coupling_f8 / cwfa_coupling_f8_map for block ``blk``: (y8, logdet, sumsq), NaN-filled before."""
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
    args = [_c8(b, kind).data_ptr(), pc.packed.data_ptr(), ops._p(pc.bias), N, H, W, pc.BN, c8, x8.data_ptr(), y8.data_ptr(),
            ops._p(t8), float(T_SCALE if ext else 1.0), ops._p(perm), axis, CLAMP, K_ATAN, 0, ws.data_ptr(), ld.data_ptr(),
            sq.data_ptr(), 0, ticket.data_ptr(), 8, 0, int(kind == "bf16"), ops._stream()]
    if name == "map":
        _lib.call("cwfa_coupling_f8_map", *args, m8.data_ptr(), ops._p(rsrc), ops._p(csrc), mode)
    else:
        _lib.call("cwfa_coupling_f8", *args)
    torch.cuda.synchronize()
    assert int(ticket[0]) == 0
    return y8, ld, sq


@gpu
@pytest.mark.parametrize("kind,ch,ext,shape,blocks", KERNEL_CASES)
def test_coupling_f8_map_chain_vs_fp64(kind, ch, ext, shape, blocks):
    from cwfa_b200 import tc
    N, H, W = SHAPES[shape]
    c8 = tc.ch8(ch)
    x = seeded_randn((N, ch, H, W), 1150)
    t_ext = seeded_randn((N, ch, H, W), 1151, 0.3) if ext else None
    # input coordinates of the first block's positions (as if permutations came before it: a level of one block gets NULL
    # tables, the identity), then one row and one column gather
    R = [_perm(H, 1160) if blocks > 1 else torch.arange(H)]
    C = [_perm(W, 1161) if blocks > 1 else torch.arange(W)]
    gathers = [(None, 0), (_perm(H, 1162), 2), (_perm(W, 1163), 3)][:blocks]
    for p, axis in gathers[1:]:
        R.append(R[-1][p] if axis == 2 else R[-1])
        C.append(C[-1][p] if axis == 3 else C[-1])
    # float64 reference chain
    m_ref = torch.zeros(N, ch, H, W, dtype=torch.float64)
    scale = torch.ones(N, ch, H, W, dtype=torch.float64)
    y = x.double()
    for blk, (p, axis) in enumerate(gathers):
        a = _conv_ref(shape, kind, blk)[3]
        if p is not None:
            y = y.index_select(axis, p)
        s = CLAMP * K_ATAN * torch.atan(a[:, :ch])
        t = T_SCALE * t_ext.double() if (ext and blk == 0) else a[:, 48:48 + ch]
        y = torch.exp(s) * y + t
        m_ref[:, :, R[blk][:, None], C[blk][None, :]] -= s
        scale[:, :, R[blk][:, None], C[blk][None, :]] += s.abs()
    m_ref[:, :, R[-1][:, None], C[-1][None, :]] += 0.5 * y * y
    scale[:, :, R[-1][:, None], C[-1][None, :]] += 0.5 * y * y
    # the GPU chains: coupling_f8_map and coupling_f8 on the same inputs
    m8 = _nan(N, c8 // 8, H, W, 8)
    xm = xp = _to_f8(x, c8).to(DEV)
    t8 = None if t_ext is None else _to_f8(t_ext, c8).to(DEV)
    for blk, (p, axis) in enumerate(gathers):
        mode = (FIRST if blk == 0 else 0) | (LAST if blk == blocks - 1 else 0)
        pd = None if p is None else p.to(DEV, torch.int32)
        tb = t8 if blk == 0 else None
        rs, cs = (None, None) if blocks == 1 else (R[blk].to(DEV, torch.int32), C[blk].to(DEV, torch.int32))
        got = _launch("map", shape, blk, kind, ch, xm, tb, pd, axis, m8, rs, cs, mode)
        ref = _launch("plain", shape, blk, kind, ch, xp, tb, pd, axis)
        for g_, r_, what in zip(got, ref, ("y", "log-det", "sum y^2")):
            assert torch.equal(g_, r_), f"block {blk}: {what} differs from cwfa_coupling_f8"
        xm, xp = got[0], ref[0]
    mf = _from_f8(m8.cpu())
    assert torch.isfinite(mf).all(), "a map entry was not written"
    assert torch.equal(mf[:, ch:], torch.zeros_like(mf[:, ch:])), "padding slots must be exactly 0"
    err = (mf[:, :ch].double() - m_ref).abs() / scale
    worst = float(err.max())
    print(f"coupling_f8_map {kind} ch={ch} ext={int(ext)} {shape} {N}x{H}x{W} blocks={blocks}: map {worst:.2e} (limit {TOL_MAP:.0e})")
    if worst > TOL_MAP:
        n, c, h, w = [int(v) for v in (err > TOL_MAP).nonzero()[0]]
        raise AssertionError(f"{int((err > TOL_MAP).sum())} map entries off, worst {worst:.2e}; first at (n={n}, c={c}, h={h}, w={w}): "
                             f"got {float(mf[n, c, h, w]):.6g}, want {float(m_ref[n, c, h, w]):.6g}")


def test_coupling_f8_map_rejects_bad_arguments():
    """CPU: argument checks that run before anything touches a device."""
    from cwfa_b200 import _lib
    lib = _lib.load()
    p = ctypes.c_void_p(16)

    def call(inverse=0, x=p, nll_map=p, mode=0):
        return lib.cwfa_coupling_f8_map(p, p, None, 1, 16, 16, 96, 48, x, p, None, 1.0, None, 0, 2.0, 0.636, inverse, p, p, p, 1, None,
                                        8, 0, 1, None, nll_map, None, None, mode)
    assert call(inverse=1) != 0                              # forward only
    assert b"forward only" in lib.cwfa_last_error()
    assert call(nll_map=None) != 0
    assert call(mode=4) != 0 and call(mode=-1) != 0
    assert call(x=None) != 0                                 # the forward pass always has x


# ------------------------------------------------------------------------------------------------------ engine
TOL = {"bf16": 2e-2, "fp16": 3e-3}      # the engine's stated rel-L2 tolerances (engine.py)
TOL_MEAN = 1e-5                         # |mean(map) - nll_per_sample| / mean(|map|): summation order only; measured <= 1.2e-7 (B200)


def _dbl(sd):
    return {k: (v.double() if v.is_floating_point() else v) for k, v in sd.items()}


def _map_reference(om, volume, views, mean_vols):
    """float64 forward of every level with the oracle's pieces, an index tensor carried through every permutation: per level
    the map 0.5 z^2 - sum of s, scattered back to the coordinates of the level's detail half."""
    out = []
    x = volume.double()
    for n, lv in enumerate(om["levels"]):
        sd = _dbl(lv["inn"])
        c_lf = O.cond_network(_dbl(lv["cond"]), views.double())
        c_mean = mean_vols[n].double()
        y, _ = O.haar1d(x)
        h = y.shape[1] // 2
        lo, hi = y[:, :h], y[:, h:]
        B, ch, H, W = hi.shape
        idx = torch.arange(ch * H * W).view(1, ch, H, W).expand(B, -1, -1, -1)
        ssum = torch.zeros(B, ch * H * W, dtype=torch.float64)
        for node in lv["spec"]["nodes"]:
            pre = f"module_list.{node['idx']}."
            kind = node["type"]
            if kind == "perm_chan":
                hi, idx = (O.permute_random(t, sd[pre + "perm"], sd[pre + "perm_inv"]) for t in (hi, idx))
            elif kind == "perm_dim":
                hi, idx = (O.permute_dim(t, sd[pre + "perm"], sd[pre + "perm_inv"], node["axis"]) for t in (hi, idx))
            elif kind in ("cat", "cat_first"):
                first = kind == "cat_first"
                a = O.subnet(sd, pre + "subnet.", torch.cat([c_mean, c_lf], 1) if first else c_lf, normal=not first)
                s = O.CLAMP * O.f_clamp(a[:, :ch])
                hi = torch.exp(s) * hi + a[:, ch:]
                ssum.scatter_add_(1, idx.reshape(B, -1), s.reshape(B, -1))
            else:
                raise ValueError(kind)
        q = torch.zeros(B, ch * H * W, dtype=torch.float64).scatter_(1, idx.reshape(B, -1), (0.5 * hi * hi).reshape(B, -1))
        out.append((q - ssum).view(B, ch, H, W))
        x = lo
    return out


def _mean_err(m, nll):
    m = m.double().cpu()
    return float(((m.mean((1, 2, 3)) - nll.double().cpu()).abs() / m.abs().mean((1, 2, 3))).max())


@pytest.fixture(scope="module")
def tiny(golden_tiny):
    model = build_tiny_model(golden_tiny, DEV)
    views, mean_vols = tiny_inputs(golden_tiny)
    B = 2
    vol = seeded_randn((B, golden_tiny["config"]["D"], views.shape[2], views.shape[3]), 1201)
    vB = torch.cat([views, seeded_randn(tuple(views.shape), 1202)])
    mvB = [m.repeat(B, 1, 1, 1) for m in mean_vols[:model.n_levels]]
    return model, vol, vB, mvB


@gpu
@pytest.mark.parametrize("kind", ["bf16", "fp16"])
def test_engine_nll_map_vs_fp64_reference(tiny, kind):
    from cwfa_b200.engine import CWFAEngine
    model, vol, views, mvs = tiny
    ref = _map_reference(model.export_for_oracle(), vol, views, mvs)
    eng = CWFAEngine(model, kind)
    args = (vol.to(DEV), views.to(DEV), [m.to(DEV) for m in mvs])
    plain = [{k: v.clone() for k, v in r.items()} for r in eng.forward_nll(*args)]
    res = eng.forward_nll(*args, nll_map=True)
    for n, (r, p, mref) in enumerate(zip(res, plain, ref)):
        m = r["nll_map"]
        assert tuple(m.shape) == tuple(mref.shape) and m.dtype == torch.float32
        for k in ("z", "logdet", "sumsq", "nll_per_sample"):
            assert torch.equal(r[k], p[k]), f"level {n}: {k} differs from forward_nll(nll_map=False)"
        e, em = rel_l2(m, mref), _mean_err(m, r["nll_per_sample"])
        print(f"nll_map tiny {kind} level {n}: rel-L2 vs fp64 {e:.2e} (limit {TOL[kind]:.0e}), mean vs nll_per_sample {em:.2e}")
        assert e < TOL[kind] and em < TOL_MEAN


@gpu
def test_engine_nll_map_locality_is_exact(tiny):
    """A perturbation inside a small voxel box changes the maps at the detail voxels whose Haar support meets it, and leaves
    every other map entry bitwise unchanged: the map sits at each element's level-input coordinates."""
    from cwfa_b200.engine import CWFAEngine
    model, vol, views, mvs = tiny
    eng = CWFAEngine(model, "bf16")
    d0, d1, h0, h1, w0, w1 = 5, 8, 17, 21, 40, 43
    vol2 = vol.clone()
    vol2[1, d0:d1, h0:h1, w0:w1] += seeded_randn((d1 - d0, h1 - h0, w1 - w0), 1210)
    args = (views.to(DEV), [m.to(DEV) for m in mvs])
    a = [r["nll_map"].clone() for r in eng.forward_nll(vol.to(DEV), *args, nll_map=True)]
    b = [r["nll_map"].clone() for r in eng.forward_nll(vol2.to(DEV), *args, nll_map=True)]
    for n, (ma, mb) in enumerate(zip(a, b)):
        mask = torch.zeros(ma.shape, dtype=torch.bool)
        chans = sorted({d >> (n + 1) for d in range(d0, d1)})
        mask[1, chans, h0:h1, w0:w1] = True
        diff = (ma != mb).cpu()
        print(f"nll_map locality level {n}: {int(diff.sum())} entries changed, {int(mask.sum())} expected (channels {chans})")
        assert not bool(diff[~mask].any()), f"level {n}: map changed outside the perturbed voxels"
        assert bool(diff[mask].all()), f"level {n}: map unchanged at a perturbed voxel"


@gpu
def test_engine_nll_map_graphed_and_sensor(tiny):
    from cwfa_b200.data import LensletLayout
    from cwfa_b200.engine import CWFAEngine
    model, vol, views, mvs = tiny
    eng = CWFAEngine(model, "bf16")
    vd, md = vol.to(DEV), [m.to(DEV) for m in mvs]
    eager = [{k: v.clone() for k, v in r.items()} for r in eng.forward_nll(vd, views.to(DEV), md, nll_map=True)]
    for _ in range(2):
        g = eng.forward_nll_graphed(vd, views.to(DEV), md, nll_map=True)
        for r, e in zip(g, eager):
            for k in ("nll_map", "z", "logdet", "sumsq"):
                assert torch.equal(r[k], e[k]), k
    g0 = eng.forward_nll_graphed(vd, views.to(DEV), md)          # the map-free graph is a graph of its own
    assert "nll_map" not in g0[0]
    # raw sensor frames give the maps of their extracted views
    coords = [[40 + 50 * (i // 6), 35 + 55 * (i % 6)] for i in range(29)]
    layout = LensletLayout(coords, (64, 64), 32768.0, 16384.0, device=DEV)
    gen = torch.Generator().manual_seed(6)
    frame = torch.randint(0, 65536, (2, 1, 300, 340), generator=gen, dtype=torch.int32).to(torch.uint16).to(DEV)
    ref = eng.forward_nll(vd, layout.views(frame), md, nll_map=True)
    ref = [r["nll_map"].clone() for r in ref]
    got = eng.forward_nll(vd, frame, md, sensor=layout, nll_map=True)
    gg = eng.forward_nll_graphed(vd, frame, md, sensor=layout, nll_map=True)
    for r, a, b in zip(ref, got, gg):
        assert torch.equal(a["nll_map"], r) and torch.equal(b["nll_map"], r)


@gpu
def test_engine_nll_map_disable_low_res_input(golden_tiny):
    import cwfa_b200
    from cwfa_b200.engine import CWFAEngine
    cfg = golden_tiny["config"]
    model = cwfa_b200.CWFAModel(n_depths=cfg["D"], volume_side_size=cfg["S"], INN_max_down_steps=cfg["MAX"], disable_low_res_input=1,
                                seed=0).to(DEV)
    vol = seeded_randn((2, cfg["D"], cfg["S"], cfg["S"]), 1220).to(DEV)
    views = seeded_randn((2, 29, cfg["S"], cfg["S"]), 1221).to(DEV)
    eng = CWFAEngine(model, "fp16")
    plain = [{k: v.clone() for k, v in r.items()} for r in eng.forward_nll(vol, views, [None] * model.n_levels)]
    res = eng.forward_nll(vol, views, [None] * model.n_levels, nll_map=True)
    for n, (r, p) in enumerate(zip(res, plain)):
        em = _mean_err(r["nll_map"], r["nll_per_sample"])
        print(f"nll_map disable_low_res_input level {n}: mean vs nll_per_sample {em:.2e}")
        assert em < TOL_MEAN
        assert torch.equal(r["z"], p["z"]) and torch.equal(r["logdet"], p["logdet"])


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
def test_engine_nll_map_rejects_levels_without_f8_plan(golden_tiny):
    import cwfa_b200
    from cwfa_b200.engine import CWFAEngine
    cfg = golden_tiny["config"]
    D, S = cfg["D"], cfg["S"]
    eng = CWFAEngine(_glow_model(golden_tiny), "bf16")
    vol, views = torch.zeros((1, D, S, S), device=DEV), torch.zeros((1, 29, S, S), device=DEV)
    mvs = [torch.zeros((1, D // 2 ** (n + 1), S, S), device=DEV) for n in range(eng.model.n_levels)]
    with pytest.raises(ValueError, match="level 0 .*GLOW"):
        eng.forward_nll(vol, views, mvs, nll_map=True)
    with pytest.raises(ValueError, match="level 0"):
        eng.forward_nll_graphed(vol, views, mvs, nll_map=True)
    S2 = 30                                                      # H * W = 900 is a multiple of 4; 31 * 31 is not
    odd = CWFAEngine(cwfa_b200.CWFAModel(n_depths=D, volume_side_size=S2 + 1, INN_max_down_steps=cfg["MAX"], seed=0).to(DEV), "bf16")
    v2 = torch.zeros((1, D, S2 + 1, S2 + 1), device=DEV)
    with pytest.raises(ValueError, match="multiple of 4"):
        odd.forward_nll(v2, torch.zeros((1, 29, S2 + 1, S2 + 1), device=DEV),
                        [torch.zeros((1, D // 2 ** (n + 1), S2 + 1, S2 + 1), device=DEV) for n in range(odd.model.n_levels)], nll_map=True)


@gpu
def test_engine_nll_map_full_config():
    """96 x 512 x 512, batch 8, bf16, the r2_full probe's weights and forward inputs: the mean invariant per level, and z /
    log-det / sum z^2 bitwise those of the map-free call."""
    import os
    from conftest import GOLDEN
    from helpers import build_full_model, full_inputs
    from cwfa_b200.engine import CWFAEngine
    fx = torch.load(os.path.join(GOLDEN, "r2_full.pt"), weights_only=False)
    model = build_full_model(fx, DEV)
    seeds = fx["config"]["seeds"]
    B = fx["config"]["n_fwd_frames"]
    _, mvs = full_inputs(fx)
    x = torch.cat([seeded_randn((1, 96, 512, 512), seeds["fwd_x"] + b) for b in range(B)]).to(DEV)
    vB = torch.cat([seeded_randn((1, 29, 512, 512), seeds["fwd_views"] + b) for b in range(B)]).to(DEV)
    mvB = [m.to(DEV).repeat(B, 1, 1, 1) for m in mvs]
    eng = CWFAEngine(model, "bf16")
    plain = [{k: v.clone() for k, v in r.items()} for r in eng.forward_nll(x, vB, mvB)]
    res = eng.forward_nll(x, vB, mvB, nll_map=True)
    for n, (r, p) in enumerate(zip(res, plain)):
        for k in ("z", "logdet", "sumsq"):
            assert torch.equal(r[k], p[k]), f"level {n}: {k}"
        em = _mean_err(r["nll_map"], r["nll_per_sample"])
        print(f"nll_map full config level {n}: shape {tuple(r['nll_map'].shape)}, mean vs nll_per_sample {em:.2e}")
        assert tuple(r["nll_map"].shape) == tuple(r["z"].shape) and em < TOL_MEAN
