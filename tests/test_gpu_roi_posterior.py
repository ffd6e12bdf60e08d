"""Exact posterior mean and standard deviation of region readouts (ROIs, e.g. neuron footprints): the RoiSet tables
(cwfa_b200.data.roi_tables), the readout kernel (cwfa_roi_readout_f8) and CWFAEngine.roi_posterior_exact /
roi_posterior_exact_graphed.

On CAT-only levels the volume is affine in the latents, the levels are independent and the Haar merges are orthonormal, so a
readout r = sum_v w_v V_v has Var[r] = sigma_T^2 sum_n || DWT_n(V(z = 1_n) - V(0)) * DWT_n(w) ||^2, with DWT_n the level-n detail
half of the forward depth Haar analysis (oracle.cwfa_oracle.haar1d applied n + 1 times) and 1_n the all-ones latents of level n:
DWT_n(V(1_n) - V(0)) is the level's scale alpha_n, exactly.  The engine is checked against that identity run on its own
reconstructions (tight) and on the float64 oracle (the reference error), so the checks do not depend on the scale tensors."""
import ctypes
import math

import numpy as np
import pytest
import torch

from conftest import rel_l2
from helpers import build_tiny_model, tiny_inputs
from oracle import cwfa_oracle as O
from oracle.weights import seeded_randn
from test_gpu_posterior_exact import SIGMA_07, _dbl, _glow_model, _ones_at, _ragged_model

DEV = "cuda:0"
gpu = pytest.mark.gpu


def _detail(x, n):
    """Level n's detail half of the forward depth Haar analysis of x (B, D, ...): haar1d applied n + 1 times (float64)."""
    x = x.double()
    for _ in range(n):
        x = O.haar1d(x)[0][:, :x.shape[1] // 2]
    return O.haar1d(x)[0][:, x.shape[1] // 2:]


def _f8_flat(x):
    """(C, H, W) -> one batch item of the F8 layout, flattened, channel padding 0 (the tables' offsets index this)."""
    C, H, W = x.shape
    c8 = (C + 7) // 8 * 8
    xp = torch.zeros((c8, H, W), dtype=x.dtype)
    xp[:C] = x
    return xp.view(c8 // 8, 8, H, W).permute(0, 2, 3, 1).reshape(-1)


# ------------------------------------------------------------------------------------------------ synthetic ROIs
def _ellipsoids(D, H, W, R, seed, tiles=None, soft=False):
    """R neuron-like ROIs as (h0, w0, local weights (D, bh, bw) float64): small ellipsoids (lateral radius 1.2-3.5, half-depth
    0.6-2.5 planes) at random centres, borders included, mean readout (weights 1 / |r|).  ``tiles`` = (th, tw): ROI r lies inside
    lateral tile r, so no two ROIs share a pixel column.  ``soft``: Gaussian weights of either sign instead of the mean."""
    rs = np.random.RandomState(seed)
    out = []
    for r in range(R):
        ry, rx = rs.uniform(1.2, 3.5, 2)
        rz = rs.uniform(0.6, 2.5)
        if tiles is not None:
            th, tw = tiles
            t0, t1 = (r // (W // tw)) * th, (r % (W // tw)) * tw
            cy, cx = t0 + rs.uniform(0, th - 1), t1 + rs.uniform(0, tw - 1)
            ry, rx = min(ry, cy - t0, t0 + th - 1 - cy) + 0.5, min(rx, cx - t1, t1 + tw - 1 - cx) + 0.5
        else:
            cy, cx = rs.uniform(-0.5, H - 0.5), rs.uniform(-0.5, W - 0.5)
        cz = rs.uniform(-0.5, D - 0.5)
        h0, h1 = max(0, int(math.floor(cy - ry))), min(H, int(math.ceil(cy + ry)) + 1)
        w0, w1 = max(0, int(math.floor(cx - rx))), min(W, int(math.ceil(cx + rx)) + 1)
        z, y, x = np.meshgrid(np.arange(D), np.arange(h0, h1), np.arange(w0, w1), indexing="ij")
        q = ((z - cz) / rz) ** 2 + ((y - cy) / ry) ** 2 + ((x - cx) / rx) ** 2
        mask = q <= 1.0
        if not mask.any():
            mask[np.unravel_index(np.argmin(q), q.shape)] = True
        if soft:
            wl = np.where(mask, np.exp(-q) * rs.choice([-1.0, 1.0]) * rs.uniform(0.5, 2.0), 0.0)
        else:
            wl = mask / mask.sum()
        out.append((h0, w0, torch.from_numpy(np.ascontiguousarray(wl, dtype=np.float64))))
    return out


def _coo(rois):
    """COO triplets (roi, voxel, weight) of a list of (h0, w0, local weights)."""
    rr, vv, ww = [], [], []
    for r, (h0, w0, wl) in enumerate(rois):
        nz = torch.nonzero(wl)
        rr.append(torch.full((nz.shape[0],), r, dtype=torch.int64))
        vv.append(nz + torch.tensor([0, h0, w0]))
        ww.append(wl[nz[:, 0], nz[:, 1], nz[:, 2]])
    return torch.cat(rr), torch.cat(vv), torch.cat(ww)


def _roiset(rois, shape, L, device=DEV):
    from cwfa_b200 import RoiSet
    r, v, w = _coo(rois)
    return RoiSet(r, v, w, len(rois), shape, L, device=device)


def _column(D, h, w, weight=1.0):
    """An ROI over all D planes of one pixel: its readout is 2^(L/2) times the LRNN voxel, deterministic."""
    return (h, w, torch.full((D, 1, 1), float(weight), dtype=torch.float64))


def _voxel(D, d, h, w, weight=1.0):
    """An ROI of one voxel."""
    wl = torch.zeros((D, 1, 1), dtype=torch.float64)
    wl[d] = weight
    return (h, w, wl)


def _readout(vol, rois):
    """float64 sum_v w_v V_v per (b, roi), and sum_v |w_v V_v| (the scale of its rounding)."""
    vol = vol.double().cpu()
    m, a = torch.zeros(vol.shape[0], len(rois), dtype=torch.float64), torch.zeros(vol.shape[0], len(rois), dtype=torch.float64)
    for r, (h0, w0, wl) in enumerate(rois):
        v = vol[:, :, h0:h0 + wl.shape[1], w0:w0 + wl.shape[2]] * wl
        m[:, r], a[:, r] = v.sum((1, 2, 3)), v.abs().sum((1, 2, 3))
    return m, a


def _identity_std(dvs, rois, sigma):
    """sigma sqrt(sum_n ||DWT_n(dvs[n]) * DWT_n(w)||^2) per (b, roi), float64; dvs[n] = V(1_n) - V(0), (B, D, H, W) on any device."""
    A = [_detail(dv, n) for n, dv in enumerate(dvs)]
    B = A[0].shape[0]
    out = torch.zeros(B, len(rois), dtype=torch.float64)
    for r, (h0, w0, wl) in enumerate(rois):
        acc = torch.zeros(B, dtype=torch.float64, device=A[0].device)
        for n, a in enumerate(A):
            wn = _detail(wl[None].to(a.device), n)
            acc += ((a[:, :, h0:h0 + wl.shape[1], w0:w0 + wl.shape[2]] * wn) ** 2).sum((1, 2, 3))
        out[:, r] = sigma * acc.sqrt().cpu()
    return out


def _identity_error(std, ref, vmax, rois, sigma):
    """max |std - ref| / (1e-4 ref + sigma 1e-6 (1 + max|V|) ||w||_2): the identity on the engine's own reconstructions holds to
    fp32 rounding.  The second term bounds what the fp32 rounding of V(1_n) - V(0) (about 1e-6 (1 + |V|) per voxel) adds to the
    norm, by Cauchy-Schwarz and the orthonormality of the Haar analysis."""
    wn = torch.tensor([float(wl.norm()) for _, _, wl in rois], dtype=torch.float64)
    return float(((std.double().cpu() - ref).abs() / (1e-4 * ref + sigma * 1e-6 * (1.0 + vmax) * wn)).max())


# ------------------------------------------------------------------------------------------------ tables (CPU)
def _check_tables(rs, rois, D, H, W, L):
    """The tables against the dense float64 reference: per ROI, the weight volume and its recursive oracle Haar details, read at
    the tables' offsets; every nonzero detail coefficient is present, entries sorted by offset, no padding channel indexed."""
    t = {k: getattr(rs, k).cpu() for k in ("mean_ptr", "mean_idx", "mean_w", "coef_ptr", "coef_idx", "coef_val")}
    worst = 0.0
    for r, (h0, w0, wl) in enumerate(rois):
        dense = torch.zeros((1, D, H, W), dtype=torch.float64)
        dense[0, :, h0:h0 + wl.shape[1], w0:w0 + wl.shape[2]] += wl
        a, b = int(t["mean_ptr"][r]), int(t["mean_ptr"][r + 1])
        idx = t["mean_idx"][a:b].long()
        ref = dense.reshape(-1)
        assert torch.equal(idx, torch.nonzero(ref).reshape(-1)), f"roi {r}: mean offsets"
        assert torch.allclose(t["mean_w"][a:b].double(), ref[idx], rtol=1e-7, atol=0)
        x = dense
        for n in range(L):
            out = O.haar1d(x)[0]
            h = x.shape[1] // 2
            ref = _f8_flat(out[0, h:])
            x = out[:, :h]
            a, b = int(t["coef_ptr"][n, r]), int(t["coef_ptr"][n, r + 1])
            idx, val = t["coef_idx"][a:b].long(), t["coef_val"][a:b].double()
            want = torch.nonzero(ref.abs() > 1e-12 * ref.abs().max().clamp_min(1e-300)).reshape(-1)
            assert torch.equal(idx, want), f"roi {r} level {n}: the offsets are not the nonzero detail coefficients"
            assert bool((idx % 8 < h - (idx // (8 * H * W)) * 8).all()), f"roi {r} level {n}: a padding channel is indexed"
            if b > a:
                worst = max(worst, float(((val - ref[idx]).abs() / ref[idx].abs()).max()))
    assert worst < 2e-7, worst                               # fp32 storage of the float64 sums
    return t


@pytest.mark.parametrize("D,H,W,L", [(16, 9, 7, 2), (24, 10, 13, 3)])
def test_roi_tables_vs_dense_haar(D, H, W, L):
    """D = 16 with 2 levels and D = 24 with 3 (12- and 6-channel ragged halves): mean ellipsoids touching the borders, soft
    overlapping ROIs of either sign, an ROI of one voxel and a voxel listed twice."""
    from cwfa_b200.data import RoiSet
    rois = _ellipsoids(D, H, W, 12, 7) + _ellipsoids(D, H, W, 6, 8, soft=True)
    rois += [_voxel(D, 0, 0, 0), _voxel(D, D - 1, H - 1, W - 1, -0.5)]
    rois.append((0, 0, torch.rand((D, H, W), dtype=torch.float64, generator=torch.Generator().manual_seed(3)) - 0.5))
    r, v, w = _coo(rois)
    for axis, val in ((1, 0), (1, H - 1), (2, 0), (2, W - 1), (0, 0), (0, D - 1)):
        assert bool((v[:, axis] == val).any()), "the ROIs must touch every border"
    rs = RoiSet(r, v, w, len(rois), (D, H, W), L, device="cpu")
    _check_tables(rs, rois, D, H, W, L)
    # a voxel listed twice adds up
    r2, v2, w2 = torch.cat([r, r[:1]]), torch.cat([v, v[:1]]), torch.cat([w, w[:1]])
    rois2 = list(rois)
    h0, w0, wl = rois2[0]
    wl = wl.clone()
    wl[v[0, 0], v[0, 1] - h0, v[0, 2] - w0] *= 2
    rois2[0] = (h0, w0, wl)
    _check_tables(RoiSet(r2, v2, w2, len(rois), (D, H, W), L, device="cpu"), rois2, D, H, W, L)


def test_roi_from_labels():
    from cwfa_b200.data import RoiSet
    D, H, W, L = 24, 11, 9, 3
    rois = _ellipsoids(D, H, W, 9, 11)
    labels = torch.zeros((D, H, W), dtype=torch.int32)
    for r, (h0, w0, wl) in enumerate(rois):                   # later ROIs overwrite earlier ones where they overlap
        labels[:, h0:h0 + wl.shape[1], w0:w0 + wl.shape[2]][wl > 0] = r + 1
    want = []
    for r in range(len(rois)):
        m = (labels == r + 1).double()
        want.append((0, 0, m / m.sum()))
    rs = RoiSet.from_labels(labels.numpy(), L, device="cpu")
    assert rs.n_rois == len(rois) and rs.volume_shape == (D, H, W) and rs.n_levels == L
    _check_tables(rs, want, D, H, W, L)
    # a label value no voxel carries is an empty ROI
    labels[labels == 3] = 0
    rs = RoiSet.from_labels(labels, L, device="cpu")
    assert rs.n_rois == len(rois) and int(rs.mean_ptr[3] - rs.mean_ptr[2]) == 0
    assert bool((rs.coef_ptr[:, 3] == rs.coef_ptr[:, 2]).all())


def test_roi_all_planes_has_no_coefficients():
    """A readout over all D planes of a pixel is 2^(L/2) times the deterministic LRNN voxel: no detail coefficient survives, with
    weight 1 and as a label (weight 1 / D)."""
    from cwfa_b200.data import RoiSet
    D, H, W, L = 24, 5, 6, 3
    rs = _roiset([_column(D, 2, 3), _column(D, 0, 5, 0.1)], (D, H, W), L, device="cpu")
    assert rs.n_coef_entries == 0 and bool((rs.coef_ptr == 0).all())
    assert rs.n_mean_entries == 2 * D
    labels = torch.zeros((D, H, W), dtype=torch.int64)
    labels[:, 1, 1] = 1
    labels[:, 4, 0] = 2
    labels[:, 4, 1] = 2
    rs = RoiSet.from_labels(labels, L, device="cpu")
    assert rs.n_coef_entries == 0, "equal weights on both halves of every Haar block must cancel to exactly 0"
    # two planes {2i, 2i+1} with equal weights: nothing at level 0, one coefficient per level above
    rs = _roiset([(1, 1, torch.tensor([0.0, 0.0, 1.0, 1.0] + [0.0] * (D - 4), dtype=torch.float64).view(D, 1, 1))], (D, H, W), L,
                 device="cpu")
    assert [int(rs.coef_ptr[n, 1] - rs.coef_ptr[n, 0]) for n in range(L)] == [0, 1, 1]


def test_roi_validation():
    from cwfa_b200.data import RoiSet
    D, H, W = 16, 4, 4
    r, v, w = torch.tensor([0, 1]), torch.tensor([[0, 0, 0], [15, 3, 3]]), torch.tensor([1.0, 2.0])
    RoiSet(r, v, w, 2, (D, H, W), 2, device="cpu")
    for bad in ([-1, 0, 0], [16, 0, 0], [0, 4, 0], [0, 0, 4], [0, -1, 0]):
        with pytest.raises(ValueError, match="out of range"):
            RoiSet(r, torch.tensor([[0, 0, 0], bad]), w, 2, (D, H, W), 2, device="cpu")
    for bad in (float("nan"), float("inf"), -float("inf")):
        with pytest.raises(ValueError, match="finite"):
            RoiSet(r, v, torch.tensor([1.0, bad]), 2, (D, H, W), 2, device="cpu")
    with pytest.raises(ValueError, match="roi indices"):
        RoiSet(torch.tensor([0, 2]), v, w, 2, (D, H, W), 2, device="cpu")
    with pytest.raises(ValueError, match="roi indices"):
        RoiSet(torch.tensor([-1, 0]), v, w, 2, (D, H, W), 2, device="cpu")
    with pytest.raises(ValueError, match="n_rois"):
        RoiSet(r, v, w, 0, (D, H, W), 2, device="cpu")
    with pytest.raises(ValueError, match="divisible"):
        RoiSet(r, v, w, 2, (D, H, W), 5, device="cpu")
    with pytest.raises(ValueError, match="divisible"):
        RoiSet(r, torch.tensor([[0, 0, 0], [11, 3, 3]]), w, 2, (12, H, W), 3, device="cpu")
    with pytest.raises(ValueError, match="n_levels"):
        RoiSet(r, v, w, 2, (D, H, W), 0, device="cpu")
    with pytest.raises(ValueError, match="entries"):
        RoiSet(r, v, w[:1], 2, (D, H, W), 2, device="cpu")
    with pytest.raises(ValueError, match="integer"):
        RoiSet(r, v.double(), w, 2, (D, H, W), 2, device="cpu")
    with pytest.raises(ValueError, match="no positive label"):
        RoiSet.from_labels(torch.zeros((D, H, W), dtype=torch.int32), 2, device="cpu")
    with pytest.raises(ValueError, match="integer"):
        RoiSet.from_labels(torch.ones((D, H, W)), 2, device="cpu")
    with pytest.raises(ValueError, match="divisible"):
        RoiSet.from_labels(torch.ones((12, H, W), dtype=torch.int32), 3, device="cpu")


def test_roi_readout_f8_rejects_bad_arguments():
    """CPU: argument checks that run before anything touches a device (every call has at least one bad argument)."""
    from cwfa_b200 import _lib
    lib = _lib.load()
    p = ctypes.c_void_p(16)
    sc = (ctypes.c_void_p * 3)(16, 32, 48)
    st = (ctypes.c_int64 * 3)(64, 32, 16)

    def call(vol=p, scales=sc, strides=st, L=3, mean_ptr=p, coef_val=p, B=1, R=4, sigma=0.5, mean=p, std=p):
        return lib.cwfa_roi_readout_f8(vol, 100, scales, strides, L, mean_ptr, p, p, p, p, coef_val, B, R, sigma, mean, std, None)
    assert call(L=0) != 0 and b"L must be" in lib.cwfa_last_error()
    assert call(L=9) != 0 and b"L must be" in lib.cwfa_last_error()
    for s in (-0.1, float("nan"), float("inf")):
        assert call(sigma=s) != 0 and b"sigma" in lib.cwfa_last_error()
    assert call(R=0) != 0 and b"R >= 1" in lib.cwfa_last_error()
    assert call(B=0) != 0
    for kw in ("vol", "scales", "strides", "mean_ptr", "coef_val", "mean", "std"):
        assert call(**{kw: None}) != 0 and b"NULL" in lib.cwfa_last_error(), kw
    assert call(scales=(ctypes.c_void_p * 3)(16, None, 48)) != 0 and b"level 1" in lib.cwfa_last_error()
    assert call(strides=(ctypes.c_int64 * 3)(64, 32, 0)) != 0 and b"level 2" in lib.cwfa_last_error()


# ------------------------------------------------------------------------------------------------ kernel (GPU)
@gpu
def test_roi_readout_f8_vs_fp64():
    """Random volumes and scales (batch 2, ragged 10 x 13 lateral, 24 depths, 3 levels with 12 / 6 / 3-channel halves whose F8
    padding channels hold NaN), ROIs of 1 to 3120 entries including one with no coefficient, against float64 on the same inputs;
    NaN-filled outputs; two launches bitwise equal."""
    from cwfa_b200 import _lib, ops, tc
    B, D, H, W, L = 2, 24, 10, 13, 3
    sigma = 0.391
    rois = [_voxel(D, 5, 3, 4), _column(D, 9, 12)]
    rois += _ellipsoids(D, H, W, 20, 21) + _ellipsoids(D, H, W, 10, 22, soft=True)
    rois.append((0, 0, torch.rand((D, H, W), dtype=torch.float64, generator=torch.Generator().manual_seed(5)) + 0.1))
    rs = _roiset(rois, (D, H, W), L)
    sizes = [int(rs.mean_ptr[r + 1] - rs.mean_ptr[r]) + int((rs.coef_ptr[:, r + 1] - rs.coef_ptr[:, r]).sum()) for r in range(len(rois))]
    assert sizes[0] == 1 + L and int((rs.coef_ptr[:, 2] - rs.coef_ptr[:, 1]).sum()) == 0 and max(sizes) > 3000
    vol = seeded_randn((B, D, H, W), 2101)
    scales = [seeded_randn((B, D >> (n + 1), H, W), 2102 + n).abs() * 2.0 + 1e-2 for n in range(L)]
    s8 = []
    for s in scales:
        f8 = torch.stack([_f8_flat(s[b]) for b in range(B)]).view(B, -1, H, W, 8)
        c = s.shape[1]
        if c % 8:
            f8[:, -1, :, :, c % 8:] = float("nan")
        s8.append(f8.contiguous().to(DEV))
    vol_d = vol.to(DEV)
    # float64 reference from the dense weights (independent of the tables)
    m_ref, m_abs = _readout(vol, rois)
    s_ref = torch.zeros(B, len(rois), dtype=torch.float64)
    for r, (h0, w0, wl) in enumerate(rois):
        acc = torch.zeros(B, dtype=torch.float64)
        for n, s in enumerate(scales):
            acc += ((s[:, :, h0:h0 + wl.shape[1], w0:w0 + wl.shape[2]].double() * _detail(wl[None], n)) ** 2).sum((1, 2, 3))
        s_ref[:, r] = float(np.float32(sigma)) * acc.sqrt()
    outs = []
    for _ in range(2):
        mean, std = torch.full((B, len(rois)), float("nan"), device=DEV), torch.full((B, len(rois)), float("nan"), device=DEV)
        ptrs = (ctypes.c_void_p * L)(*[t.data_ptr() for t in s8])
        strides = (ctypes.c_int64 * L)(*[t[0].numel() for t in s8])
        _lib.call("cwfa_roi_readout_f8", vol_d.data_ptr(), D * H * W, ptrs, strides, L, rs.mean_ptr.data_ptr(), rs.mean_idx.data_ptr(),
                  rs.mean_w.data_ptr(), rs.coef_ptr.data_ptr(), rs.coef_idx.data_ptr(), rs.coef_val.data_ptr(), B, len(rois), sigma,
                  mean.data_ptr(), std.data_ptr(), ops._stream())
        torch.cuda.synchronize()
        outs.append((mean, std))
    mean, std = outs[0]
    assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1]), "two launches differ"
    assert bool(torch.isfinite(mean).all() and torch.isfinite(std).all()), "an output was not written, or padding was read"
    assert bool((std[:, 1] == 0).all()), "an ROI without coefficients must have std exactly 0"
    em = float(((mean.double().cpu() - m_ref).abs() / m_abs.clamp_min(1e-300)).max())
    es = float(((std.double().cpu() - s_ref).abs() / s_ref.clamp_min(1e-300)).max())
    print(f"roi_readout_f8: {len(rois)} ROIs of {min(sizes)}..{max(sizes)} entries, mean rel {em:.2e}, std rel {es:.2e} (limit 1e-5)")
    assert em < 1e-5 and es < 1e-5
    m2, s2 = tc.roi_readout_f8(vol_d, s8, rs, sigma)
    assert torch.equal(m2, mean) and torch.equal(s2, std)


# ------------------------------------------------------------------------------------------------ engine (GPU)
@pytest.fixture(scope="module")
def tiny(golden_tiny):
    model = build_tiny_model(golden_tiny, DEV)
    views, mean_vols = tiny_inputs(golden_tiny)
    return model, views.to(DEV), [t.to(DEV) for t in mean_vols]


def _tiny_rois(D, S):
    """64 mean ellipsoids, one per 8 x 8 lateral tile (no two share a pixel column, so their readouts are independent), then
    soft overlapping ROIs of either sign and a few all-plane columns."""
    return _ellipsoids(D, S, S, 64, 31, tiles=(8, 8)) + _ellipsoids(D, S, S, 12, 32, soft=True) + \
        [_column(D, 0, 0), _column(D, S - 1, 17), _column(D, 30, S - 1, -2.0)]


def _dvs(recon, model, B):
    """V(1_n) - V(0) per level, float64 (device of the reconstruction)."""
    v0 = recon(_ones_at(model, -1, B)).double()
    return [recon(_ones_at(model, n, B)).double() - v0 for n in range(model.n_levels)], v0


# ROI std against the float64 oracle run of the same identity, rel-L2 over the ROIs: limit at ~4x the value measured on a B200
# (1000 W power limit), 5.39e-3 (bf16) / 6.79e-4 (fp16) -- half the per-voxel std's error (test_gpu_posterior_exact.TOL_STD_REF):
# a readout averages the voxels' independent rounding.
TOL_ROI_STD_REF = {"bf16": 2.2e-2, "fp16": 2.8e-3}


@gpu
@pytest.mark.parametrize("kind", ["bf16", "fp16"])
def test_engine_roi_posterior_exact_tiny(tiny, kind):
    from cwfa_b200.engine import CWFAEngine
    model, views, mv = tiny
    D, S, L = model.cfg.n_depths, views.shape[2], model.n_levels
    eng = CWFAEngine(model, kind)
    rois = _tiny_rois(D, S)
    rs = _roiset(rois, (D, S, S), L)
    vol, rm, rsd = (t.clone() for t in eng.roi_posterior_exact(views, mv, rs, temperature=0.7))
    assert tuple(rm.shape) == tuple(rsd.shape) == (1, len(rois))
    assert torch.equal(vol, eng.reconstruct(views, mv)), "volume must be bitwise reconstruct()"
    m_ref, m_abs = _readout(vol, rois)
    e_mean = float(((rm.double().cpu() - m_ref).abs() / m_abs).max())
    # the identity on the engine's own reconstructions
    dvs, v0 = _dvs(lambda zs: eng.reconstruct(views, mv, zs=zs), model, 1)
    ref = _identity_std(dvs, rois, SIGMA_07)
    e_id = _identity_error(rsd, ref, float(v0.abs().max()), rois, SIGMA_07)
    # the same identity on the float64 oracle: the error against the reference
    om = _dbl(model.export_for_oracle())
    vd, mvd = views.double().cpu(), [m.double().cpu() for m in mv]
    dvs64, _ = _dvs(lambda zs: O.reconstruct(om, vd, mvd, zs=[z.double().cpu() for z in zs]), model, 1)
    e_ref = rel_l2(rsd, _identity_std(dvs64, rois, SIGMA_07))
    print(f"roi posterior tiny {kind}: mean rel {e_mean:.2e} (limit 1e-5), identity {e_id:.3f} (limit 1), std vs fp64 rel-L2 "
          f"{e_ref:.2e} (limit {TOL_ROI_STD_REF[kind]:.0e}); mean roi std {float(rsd.mean()):.3e}")
    assert e_mean < 1e-5
    assert e_id < 1.0
    assert e_ref < TOL_ROI_STD_REF[kind]
    # all-plane columns: deterministic readouts
    assert bool((rsd[0, -3:] == 0).all())
    # single-voxel ROIs are the per-voxel exact std
    _, pstd = eng.reconstruct_posterior_exact(views, mv, temperature=0.7)
    g = torch.Generator().manual_seed(41)
    vox = torch.stack([torch.randint(0, n, (40,), generator=g) for n in (D, S, S)], 1)
    single = [_voxel(D, d, h, w) for d, h, w in vox.tolist()]
    _, _, s1 = eng.roi_posterior_exact(views, mv, _roiset(single, (D, S, S), L), temperature=0.7)
    want = pstd[0, vox[:, 0], vox[:, 1], vox[:, 2]].double().cpu()
    e_single = float(((s1[0].double().cpu() - want).abs() / want).max())
    # pairs {2i, 2i+1} of one pixel with weights (1, 1) and (1, -1): Cov(x[2i], x[2i+1]) = (Var lo_i - Var hi_i) / 2 with
    # Var hi_i = sigma^2 alpha_0[i]^2, alpha_0 = DWT_0(V(1_0) - V(0)); the naive sqrt(std_2i^2 + std_2i+1^2) ignores it
    pairs = [(int(h), int(w), 2 * (int(d) // 2)) for d, h, w in vox.tolist()]
    def pair(sign):
        return [(h, w, torch.tensor([1.0 if k == d0 else (sign if k == d0 + 1 else 0.0) for k in range(D)],
                                    dtype=torch.float64).view(D, 1, 1)) for h, w, d0 in pairs]
    _, _, s_sum = (t.clone() for t in eng.roi_posterior_exact(views, mv, _roiset(pair(1.0), (D, S, S), L), temperature=0.7))
    _, _, s_dif = eng.roi_posterior_exact(views, mv, _roiset(pair(-1.0), (D, S, S), L), temperature=0.7)
    a0 = _detail(dvs[0], 0).cpu()
    p = pstd[0].double().cpu()
    e_sym, e_pair, n_apart = 0.0, 0.0, 0
    for k, (h, w, d0) in enumerate(pairs):
        naive2 = float(p[d0, h, w] ** 2 + p[d0 + 1, h, w] ** 2)
        var_hi = SIGMA_07 ** 2 * float(a0[0, d0 // 2, h, w]) ** 2
        cov = (naive2 - 2 * var_hi) / 2                        # naive^2 = Var lo + Var hi
        # Var(x + x') + Var(x - x') = 2 (Var lo + Var hi) = 2 naive^2, whatever the covariance
        e_sym = max(e_sym, abs(float(s_sum[0, k]) ** 2 + float(s_dif[0, k]) ** 2 - 2 * naive2) / naive2)
        for got, want2 in ((float(s_sum[0, k]) ** 2, naive2 + 2 * cov), (float(s_dif[0, k]) ** 2, naive2 - 2 * cov)):
            e_pair = max(e_pair, abs(got - want2) / naive2)
        if abs(cov) > 1e-2 * naive2:
            n_apart += 1
            assert (float(s_sum[0, k]) ** 2 - naive2) * cov > 0 and (float(s_dif[0, k]) ** 2 - naive2) * cov < 0
    # Monte Carlo: K = 256 latent draws through reconstruct(zs=...), readouts in float64
    K = 256
    gen = torch.Generator().manual_seed(43)
    zs = []
    for n in range(L):
        z = torch.empty((K,) + tuple(model.conv_inn[n].global_out_shapes[0]))
        torch.nn.init.trunc_normal_(z, mean=0.0, std=1.0, a=-0.7, b=0.7, generator=gen)
        zs.append(z.to(DEV))
    tiles = rois[:64]
    reads = []
    for c in range(0, K, 64):
        vB = views.expand(64, -1, -1, -1).contiguous()
        mvB = [m.expand(64, -1, -1, -1).contiguous() for m in mv]
        reads.append(_readout(eng.reconstruct(vB, mvB, zs=[z[c:c + 64] for z in zs]), tiles)[0])
    reads = torch.cat(reads)
    # a footprint that is the same on every plane of aligned 2^L-plane blocks has no detail coefficient: its readout is an LRNN
    # quantity, deterministic (std exactly 0, s_MC at fp32 rounding); the others enter the ratio
    sd64 = rsd[0, :64].double().cpu()
    live = sd64 > 0
    n_live = int(live.sum())
    ratio = float((reads.var(0)[live] / sd64[live] ** 2).mean())
    # the tile ROIs share no pixel column, hence no latent: independent, each s^2 / std^2 with sd <= sqrt(2 / (K - 1))
    bound = 4.0 * math.sqrt(2.0 / (K - 1)) / math.sqrt(n_live)
    # temperature 0
    v0_, m0, s0 = eng.roi_posterior_exact(views, mv, rs, temperature=0.0)
    print(f"  single voxels vs per-voxel std rel {e_single:.2e} (limit 1e-5); pairs: sum rule {e_sym:.2e} (limit 1e-5), vs "
          f"predicted Cov {e_pair:.2e} (limit 1e-3), {n_apart}/{len(pairs)} with |Cov| > 1e-2 naive^2; mean s_MC^2 / std^2 (K={K}, {n_live} ROIs) {ratio:.4f} (bound 1 +- {bound:.3f})")
    assert e_single < 1e-5
    assert e_sym < 1e-5 and e_pair < 1e-3 and n_apart >= len(pairs) // 2
    assert n_live >= 50 and abs(ratio - 1.0) < bound
    assert torch.equal(s0, torch.zeros_like(s0)) and torch.equal(v0_, vol) and torch.equal(m0, rm)


@gpu
def test_engine_roi_posterior_exact_graphed_sensor_and_batch(tiny):
    from cwfa_b200.data import LensletLayout
    from cwfa_b200.engine import CWFAEngine
    model, views, mv = tiny
    D, S, L = model.cfg.n_depths, views.shape[2], model.n_levels
    eng = CWFAEngine(model, "bf16")
    rois = _tiny_rois(D, S)
    rs = _roiset(rois, (D, S, S), L)
    eager = {T: [t.clone() for t in eng.roi_posterior_exact(views, mv, rs, temperature=T)] for T in (0.7, 0.3)}
    for T in (0.7, 0.3, 0.7):                                 # a graph per temperature; switching back replays the first
        got = eng.roi_posterior_exact_graphed(views, mv, rs, temperature=T)
        assert all(torch.equal(a, b) for a, b in zip(got, eager[T])), T
    assert not torch.equal(eager[0.7][2], eager[0.3][2])
    # another RoiSet gets a graph of its own
    rs2 = _roiset(rois[:5], (D, S, S), L)
    got = eng.roi_posterior_exact_graphed(views, mv, rs2, temperature=0.7)
    assert torch.equal(got[2], eager[0.7][2][:, :5]) and torch.equal(got[1], eager[0.7][1][:, :5])
    # raw sensor frame: bitwise the views path
    coords = [[40 + 50 * (i // 6), 35 + 55 * (i % 6)] for i in range(29)]
    layout = LensletLayout(coords, (64, 64), 32768.0, 16384.0, device=DEV)
    frame = torch.randint(0, 65536, (1, 1, 300, 340), generator=torch.Generator().manual_seed(7), dtype=torch.int32).to(torch.uint16).to(DEV)
    ref = [t.clone() for t in eng.roi_posterior_exact(layout.views(frame), mv, rs, temperature=0.7)]
    got = eng.roi_posterior_exact(frame, mv, rs, temperature=0.7, sensor=layout)
    assert all(torch.equal(a, b) for a, b in zip(got, ref))
    got = eng.roi_posterior_exact_graphed(frame, mv, rs, temperature=0.7, sensor=layout)
    assert all(torch.equal(a, b) for a, b in zip(got, ref))
    # batch 2
    vB = torch.cat([views, seeded_randn(tuple(views.shape), 1501).to(DEV)])
    mvB = [m.repeat(2, 1, 1, 1) for m in mv[:model.n_levels]]
    vol, rm, rsd = (t.clone() for t in eng.roi_posterior_exact(vB, mvB, rs, temperature=0.7))
    assert tuple(rsd.shape) == (2, len(rois))
    assert torch.equal(vol, eng.reconstruct(vB, mvB))
    m_ref, m_abs = _readout(vol, rois)
    assert float(((rm.double().cpu() - m_ref).abs() / m_abs).max()) < 1e-5
    dvs, v0 = _dvs(lambda zs: eng.reconstruct(vB, mvB, zs=zs), model, 2)
    e_id = _identity_error(rsd, _identity_std(dvs, rois, SIGMA_07), float(v0.abs().max()), rois, SIGMA_07)
    print(f"roi posterior batch 2: identity {e_id:.3f} (limit 1)")
    assert e_id < 1.0
    got = eng.roi_posterior_exact_graphed(vB, mvB, rs, temperature=0.7)
    assert torch.equal(got[0], vol) and torch.equal(got[1], rm) and torch.equal(got[2], rsd)


@gpu
def test_engine_roi_posterior_exact_ragged():
    """24 depths (12- and 6-channel detail halves), 72 x 72, fp16: eager and graphed."""
    from cwfa_b200.engine import CWFAEngine
    model = _ragged_model()
    views = seeded_randn((1, 29, 72, 72), 41).to(DEV)
    mv = [seeded_randn((1, 24 // 2 ** (n + 1), 72, 72), 50 + n, 0.1).to(DEV) for n in range(2)] + \
         [seeded_randn((1, 24 // 4, 72, 72), 59, 0.1).to(DEV)]
    eng = CWFAEngine(model, "fp16")
    rois = _ellipsoids(24, 72, 72, 40, 61) + _ellipsoids(24, 72, 72, 8, 62, soft=True) + [_column(24, 71, 0)]
    rs = _roiset(rois, (24, 72, 72), model.n_levels)
    vol, rm, rsd = (t.clone() for t in eng.roi_posterior_exact(views, mv, rs, temperature=0.7))
    assert torch.equal(vol, eng.reconstruct(views, mv))
    m_ref, m_abs = _readout(vol, rois)
    e_mean = float(((rm.double().cpu() - m_ref).abs() / m_abs).max())
    dvs, v0 = _dvs(lambda zs: eng.reconstruct(views, mv, zs=zs), model, 1)
    e_id = _identity_error(rsd, _identity_std(dvs, rois, SIGMA_07), float(v0.abs().max()), rois, SIGMA_07)
    print(f"roi posterior ragged: mean rel {e_mean:.2e}, identity {e_id:.3f} (limit 1)")
    assert e_mean < 1e-5 and e_id < 1.0 and float(rsd[0, -1]) == 0.0
    got = eng.roi_posterior_exact_graphed(views, mv, rs, temperature=0.7)
    assert torch.equal(got[0], vol) and torch.equal(got[1], rm) and torch.equal(got[2], rsd)


@gpu
def test_engine_roi_posterior_exact_rejects(golden_tiny, tiny):
    import cwfa_b200
    from cwfa_b200.engine import CWFAEngine
    model, views, mv = tiny
    cfg = golden_tiny["config"]
    D, S, L = model.cfg.n_depths, views.shape[2], model.n_levels
    rs = _roiset(_ellipsoids(D, S, S, 4, 71), (D, S, S), L)
    dlr = cwfa_b200.CWFAModel(n_depths=cfg["D"], volume_side_size=cfg["S"], INN_max_down_steps=cfg["MAX"], disable_low_res_input=1,
                              seed=0).to(DEV)
    with pytest.raises(ValueError, match="disable_low_res_input"):
        CWFAEngine(dlr, "bf16").roi_posterior_exact(views, mv, rs)
    glow = CWFAEngine(_glow_model(golden_tiny), "bf16")
    with pytest.raises(ValueError, match="level 0 .*GLOW"):
        glow.roi_posterior_exact(views, mv, rs, temperature=0.7)
    with pytest.raises(ValueError, match="level 0"):
        glow.roi_posterior_exact_graphed(views, mv, rs, temperature=0.7)
    eng = CWFAEngine(model, "bf16")
    eng.use_f8 = False
    with pytest.raises(ValueError, match="use_f8"):
        eng.roi_posterior_exact(views, mv, rs)
    eng.use_f8 = True
    for fn in (eng.roi_posterior_exact, eng.roi_posterior_exact_graphed):
        with pytest.raises(ValueError, match="temperature"):
            fn(views, mv, rs, temperature=-0.1)
        with pytest.raises(ValueError, match=rf"for \({2 * D}, {S}, {S}\) volumes"):
            fn(views, mv, _roiset(_ellipsoids(2 * D, S, S, 2, 72), (2 * D, S, S), L), temperature=0.7)
        with pytest.raises(ValueError, match=f"with {L + 1} levels"):
            fn(views, mv, _roiset(_ellipsoids(D, S, S, 2, 73), (D, S, S), L + 1), temperature=0.7)
        with pytest.raises(ValueError, match="RoiSet is on cpu"):
            fn(views, mv, _roiset(_ellipsoids(D, S, S, 2, 74), (D, S, S), L, device="cpu"), temperature=0.7)
        with pytest.raises(TypeError, match="RoiSet"):
            fn(views, mv, None, temperature=0.7)


@gpu
def test_engine_roi_posterior_exact_full_config():
    """96 x 512 x 512 (5 steps, bf16), batch 1: the volume bitwise, the readout mean, and the identity on 1000 synthetic ROIs."""
    import cwfa_b200
    from cwfa_b200.engine import CWFAEngine
    model = cwfa_b200.CWFAModel(seed=0).to(DEV)
    g = torch.Generator().manual_seed(1)
    views = torch.randn((1, 29, 512, 512), generator=g).to(DEV)
    mvs = [(0.1 * torch.randn((1, 96 // 2 ** (n + 1), 512, 512), generator=g)).to(DEV) for n in range(4)]
    eng = CWFAEngine(model, "bf16")
    rois = _ellipsoids(96, 512, 512, 1000, 81)
    rs = _roiset(rois, (96, 512, 512), model.n_levels)
    vol, rm, rsd = (t.clone() for t in eng.roi_posterior_exact(views, mvs, rs, temperature=0.7))
    assert torch.equal(vol, eng.reconstruct(views, mvs))
    m_ref, m_abs = _readout(vol, rois)
    e_mean = float(((rm.double().cpu() - m_ref).abs() / m_abs).max())
    dvs, v0 = _dvs(lambda zs: eng.reconstruct(views, mvs, zs=zs), model, 1)
    e_id = _identity_error(rsd, _identity_std(dvs, rois, SIGMA_07), float(v0.abs().max()), rois, SIGMA_07)
    print(f"roi posterior full config: mean rel {e_mean:.2e}, identity {e_id:.3f} (limit 1); mean roi std {float(rsd.mean()):.3e}")
    assert e_mean < 1e-5 and e_id < 1.0
