"""Posterior statistics over K latent samples of one frame: the K-sample coupling kernel (cwfa_coupling_f8_samples), the last
merge fused with the per-voxel mean / standard deviation (cwfa_haar1d_inv_stats), and CWFAEngine.reconstruct_posterior /
reconstruct_posterior_graphed.

The K-sample coupling must give every sample bitwise what the single-sample kernel gives on that sample's rows (the engine's
tight tolerances below rest on it); the statistics kernel is checked against the existing merge kernels run on the K rows and
float64 statistics in torch, including an offset case (mean ~ 1e3, spread ~ 1e-2) that the naive fp32 sum-of-squares formula
fails.  Every output buffer of the kernel tests is NaN-filled before the launch."""
import ctypes

import numpy as np
import pytest
import torch

from conftest import rel_l2
from helpers import build_tiny_model, tiny_inputs
from oracle.weights import deterministic_fill, seeded_randn

DEV = "cuda:0"
gpu = pytest.mark.gpu
CLAMP, K_ATAN = 2.0, 0.636
T_SCALE = -0.5 ** 0.5
SHAPES = {"ragged": (37, 13), "multi": (230, 230)}      # (H, W): 3 x 1 partial tiles / 225 tiles per condition image


def _nan(*shape):
    return torch.full(shape, float("nan"), device=DEV)


def _round(t, kind):
    return t.to(torch.bfloat16 if kind == "bf16" else torch.float16).float()


def _c8_slice(b, kind, chunk_off):
    """b (N,64,H,W) as the 8-chunk slice at chunk_off of a 192-channel C8 tensor [N][24][H][W][8] (the batched trunks' output)."""
    N, _, H, W = b.shape
    full = _round(1.0e3 * (1.0 + seeded_randn((N, 192, H, W), 704).abs()), kind)
    full[:, 8 * chunk_off:8 * chunk_off + 64] = b
    dt = torch.bfloat16 if kind == "bf16" else torch.float16
    return full.view(N, 24, 8, H, W).permute(0, 1, 3, 4, 2).contiguous().to(dt).to(DEV)


def _to_f8(x, c8):
    N, C, H, W = x.shape
    xp = torch.zeros(N, c8, H, W, dtype=x.dtype)
    xp[:, :C] = x
    return xp.view(N, c8 // 8, 8, H, W).permute(0, 1, 3, 4, 2).contiguous()


# ------------------------------------------------------------------------------------------------ kernel (1): K-sample coupling
# (kind, ch, samples S, condition images N, external shift, perm axis, shape, input chunk offset, reduction)
COUPLING_CASES = [
    ("bf16", 48, 2, 1, True, 0, "multi", 0, "ticket"),
    ("bf16", 24, 3, 2, False, 2, "ragged", 8, "finalize"),
    ("fp16", 12, 8, 2, True, 3, "ragged", 16, "ticket"),
    ("fp16", 6, 3, 1, False, 3, "multi", 0, "finalize"),
    ("bf16", 6, 8, 2, False, 0, "ragged", 0, "ticket"),
    ("fp16", 48, 2, 2, False, 2, "multi", 8, "ticket"),
    ("bf16", 12, 2, 1, True, 2, "multi", 16, "finalize"),
    ("fp16", 24, 8, 1, True, 0, "ragged", 0, "ticket"),
    ("bf16", 48, 3, 2, True, 3, "multi", 8, "ticket"),
]


def _coupling_setup(kind, ch, S, N, ext, axis, shape, chunk_off):
    from cwfa_b200 import tc
    H, W = SHAPES[shape]
    c8 = tc.ch8(ch)
    b = _round(seeded_randn((N, 64, H, W), 701), kind)
    rows = list(range(ch)) + ([] if ext else list(range(48, 48 + ch)))
    w = _round(seeded_randn((96, 64, 3, 3), 702, 0.04), kind)[rows]
    bias = seeded_randn((96,), 703, 0.5)[rows]
    pc = tc.coupling_weights_f8(w.to(DEV), bias.to(DEV), ch, torch.arange(ch), ext, kind)
    b8 = _c8_slice(b, kind, chunk_off)
    x8 = _to_f8(seeded_randn((N * S, ch, H, W), 705), c8).to(DEV)
    t8 = _to_f8(seeded_randn((N, ch, H, W), 706, 0.3), c8).to(DEV) if ext else None
    perm = None
    if axis:
        perm = torch.from_numpy(np.random.RandomState(17 + axis).permutation({2: H, 3: W}[axis])).to(DEV, torch.int32)
    return pc, b8, x8, t8, perm


def _launch(name, pc, b8, x8, t8, perm, axis, ch, N, S, H, W, chunk_off, kind, red, ticket, y8=None, ws=None, logdet=None):
    """One launch of cwfa_coupling_f8_samples (name = "samples") or cwfa_coupling_f8 (N rows of x8) into NaN-filled buffers."""
    from cwfa_b200 import _lib, ops, tc
    c8 = tc.ch8(ch)
    tiles = _lib.load().cwfa_coupling_tc_tiles(H, W)
    rows = N * S if name == "samples" else N
    y8 = _nan(rows, c8 // 8, H, W, 8) if y8 is None else y8
    ws = _nan(2 * N * tiles) if ws is None else ws
    logdet = torch.full((N,), 3.0, device=DEV) if logdet is None else logdet
    use_ticket = red == "ticket"
    common = (pc.BN, c8, x8.data_ptr(), y8.data_ptr(), ops._p(t8), float(T_SCALE if t8 is not None else 1.0), ops._p(perm), axis,
              CLAMP, K_ATAN, 1, ws.data_ptr(), logdet.data_ptr(), None, 1, ticket.data_ptr() if use_ticket else None, 24, chunk_off,
              int(kind == "bf16"), ops._stream())
    if name == "samples":
        _lib.call("cwfa_coupling_f8_samples", b8.data_ptr(), pc.packed.data_ptr(), ops._p(pc.bias), N, S, H, W, *common)
    else:
        _lib.call("cwfa_coupling_f8", b8.data_ptr(), pc.packed.data_ptr(), ops._p(pc.bias), N, H, W, *common)
    if not use_ticket:
        _lib.call("cwfa_coupling_finalize", ws.data_ptr(), logdet.data_ptr(), None, N, tiles, 1, ops._stream())
    return y8, logdet


@gpu
@pytest.mark.parametrize("kind,ch,S,N,ext,axis,shape,chunk_off,red", COUPLING_CASES)
def test_coupling_f8_samples_bitwise_equals_single_sample(kind, ch, S, N, ext, axis, shape, chunk_off, red):
    """Sample k of condition image n (row n * S + k) is bitwise the single-sample kernel on x[n * S + k] with image n's
    conditions; the per-image log-det is bitwise the single-sample log-det; padding slots stay 0."""
    H, W = SHAPES[shape]
    pc, b8, x8, t8, perm = _coupling_setup(kind, ch, S, N, ext, axis, shape, chunk_off)
    ticket = torch.zeros(1, device=DEV, dtype=torch.int32)
    y8, ld = _launch("samples", pc, b8, x8, t8, perm, axis, ch, N, S, H, W, chunk_off, kind, red, ticket)
    xs = x8.view(N, S, *x8.shape[1:])
    refs, lds = [], []
    for k in range(S):
        yk, ldk = _launch("single", pc, b8, xs[:, k].contiguous(), t8, perm, axis, ch, N, S, H, W, chunk_off, kind, red, ticket)
        refs.append(yk)
        lds.append(ldk)
    torch.cuda.synchronize()
    assert int(ticket[0]) == 0
    y = y8.view(N, S, *y8.shape[1:]).cpu()
    assert torch.isfinite(y).all(), "a tile or sample was not written"
    for k in range(S):
        assert torch.equal(y[:, k], refs[k].cpu()), f"sample {k} differs from the single-sample kernel"
        assert torch.equal(ld.cpu(), lds[k].cpu()), (ld.tolist(), lds[k].tolist())
    yf = y.reshape(N * S, -1, H, W, 8).permute(0, 1, 4, 2, 3).reshape(N * S, -1, H, W)
    assert torch.equal(yf[:, ch:], torch.zeros_like(yf[:, ch:])), "F8 padding slots must be exactly 0"


@gpu
def test_coupling_f8_samples_graph_replay():
    """A CUDA graph of one ticket-finalized K-sample launch, replayed twice: output and log-det bitwise equal to the eager
    launch, ticket back at zero."""
    kind, ch, S, N, ext, axis, shape = "bf16", 24, 3, 2, True, 2, "multi"
    H, W = SHAPES[shape]
    pc, b8, x8, t8, perm = _coupling_setup(kind, ch, S, N, ext, axis, shape, 0)
    ticket = torch.zeros(1, device=DEV, dtype=torch.int32)
    ref_y, ref_ld = _launch("samples", pc, b8, x8, t8, perm, axis, ch, N, S, H, W, 0, kind, "ticket", ticket)
    torch.cuda.synchronize()
    y8, ld = _nan(*ref_y.shape), torch.full((N,), 3.0, device=DEV)
    g = torch.cuda.CUDAGraph()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        with torch.cuda.graph(g, stream=s):
            _launch("samples", pc, b8, x8, t8, perm, axis, ch, N, S, H, W, 0, kind, "ticket", ticket, y8=y8, logdet=ld)
    torch.cuda.current_stream().wait_stream(s)
    for _ in range(2):
        y8.fill_(float("nan"))
        ld.fill_(3.0)
        g.replay()
        torch.cuda.synchronize()
        assert int(ticket[0]) == 0
        assert torch.equal(y8, ref_y) and torch.equal(ld, ref_ld)


def test_new_entry_points_reject_bad_arguments():
    """CPU: argument checks that run before anything touches a device."""
    from cwfa_b200 import _lib
    lib = _lib.load()
    p = ctypes.c_void_p(16)

    def samples(S, inverse=1, x=p, sumsq=None, H=16, W=16, chp8=48):
        return lib.cwfa_coupling_f8_samples(p, p, None, 1, S, H, W, 96, chp8, x, p, None, 1.0, None, 0, 2.0, 0.636, inverse, p, p,
                                            sumsq, 1, None, 8, 0, 1, None)
    assert samples(0) != 0
    assert samples(2, inverse=0) != 0                     # the K-sample variant is inverse-only
    assert samples(2, x=None) != 0
    assert samples(2, sumsq=p) != 0
    assert samples(1 << 12, H=512, W=512) != 0            # samples * chp8 * H * W beyond the 32-bit in-sample offsets
    assert b"2^31" in lib.cwfa_last_error()

    def stats(K, C=8, P=16, f8=1, ptr=p):
        return lib.cwfa_haar1d_inv_stats(ptr, 0, ptr, f8, ptr, ptr, K, C, P, None)
    assert stats(1) != 0                                  # at least two samples
    assert stats(2, C=7) != 0
    assert stats(2, P=18) != 0                            # F8 needs P % 4 == 0
    assert stats(2, ptr=ctypes.c_void_p(20)) != 0         # F8 needs 16-byte alignment


# ------------------------------------------------------------------------------------ kernel (2): merge with sample statistics
def _stats_reference(lo, hi, K):
    """The existing merge kernels on K rows (lo expanded when shared), then float64 mean / unbiased std."""
    from cwfa_b200 import ops, tc
    lo_k = lo.expand(K, -1, -1, -1).contiguous() if lo.shape[0] == 1 else lo
    v = tc.haar1d_merge_f8(lo_k, hi) if hi.dim() == 5 else ops.haar1d_merge(lo_k, hi)
    vd = v.double()
    return v, vd.mean(0, keepdim=True), vd.std(0, keepdim=True)


# Limits: mean within 1e-6 (1 + |mean|); std within 2e-7 |mean| + 1e-5 std + 1e-7 (a few fp32 ulps of the mean: Welford's
# deviations carry the rounding of the running mean).  Measured worst values are printed per case.
def _stats_errors(mean, std, m_ref, s_ref):
    mean, std = mean.double().cpu(), std.double().cpu()
    m_ref, s_ref = m_ref.cpu(), s_ref.cpu()
    e_m = ((mean - m_ref).abs() / (1.0 + m_ref.abs())).max().item()
    e_s = ((std - s_ref).abs() / (2e-7 * m_ref.abs() + 1e-5 * s_ref + 1e-7)).max().item()
    return e_m, e_s


# (detail-half layout, lo shared, K, h channels, H, W, case)
STATS_CASES = [
    ("f8", False, 2, 12, 24, 20, "plain"),
    ("f8", True, 3, 48, 16, 16, "plain"),
    ("f8", False, 8, 6, 8, 36, "plain"),
    ("f8", True, 16, 24, 12, 12, "offset"),
    ("nchw", False, 3, 12, 13, 7, "plain"),
    ("nchw", True, 16, 6, 9, 11, "offset"),
    ("nchw", False, 8, 24, 16, 16, "offset"),
    ("nchw", True, 2, 4, 10, 10, "plain"),
    ("f8", True, 8, 12, 16, 16, "identical"),
    ("nchw", False, 3, 6, 7, 5, "identical"),
]


@gpu
@pytest.mark.parametrize("layout,shared,K,h,H,W,case", STATS_CASES)
def test_haar1d_inv_stats(layout, shared, K, h, H, W, case):
    from cwfa_b200 import tc
    lo = seeded_randn((1 if shared else K, h, H, W), 801)
    hi = seeded_randn((K, h, H, W), 802)
    if case == "offset":                      # every voxel ~ 1e3, spread over the samples ~ 1e-2
        lo = 1.0e3 + 1.0e-2 * lo
        hi = 1.0e-2 * hi
    elif case == "identical":
        lo = lo[:1].expand(lo.shape[0], -1, -1, -1).contiguous()
        hi = hi[:1].expand(K, -1, -1, -1).contiguous()
    lo_d = lo.to(DEV)
    hi_d = _to_f8(hi, tc.ch8(h)).to(DEV) if layout == "f8" else hi.to(DEV)
    v, m_ref, s_ref = _stats_reference(lo_d, hi_d, K)
    mean, std = _nan(1, 2 * h, H, W), _nan(1, 2 * h, H, W)
    from cwfa_b200 import _lib, ops
    _lib.call("cwfa_haar1d_inv_stats", lo_d.data_ptr(), int(shared), hi_d.data_ptr(), int(layout == "f8"), mean.data_ptr(),
              std.data_ptr(), K, 2 * h, H * W, ops._stream())
    torch.cuda.synchronize()
    assert torch.isfinite(mean).all() and torch.isfinite(std).all()
    if case == "identical":
        assert torch.equal(std, torch.zeros_like(std)), "identical samples must give std exactly 0"
        assert torch.equal(mean, v[:1]), "identical samples: the mean is the merged value"
        return
    e_m, e_s = _stats_errors(mean, std, m_ref, s_ref)
    print(f"haar1d_inv_stats {layout} shared={shared} K={K} h={h} {H}x{W} {case}: mean {e_m:.2e} (limit 1e-6), std {e_s:.2f} "
          f"(limit 1 = 2e-7 |mean| + 1e-5 std + 1e-7)")
    assert e_m < 1e-6 and e_s < 1.0, (e_m, e_s)
    # the wrapper gives the same
    m2, s2 = tc.haar1d_merge_stats(lo_d, hi_d)
    assert torch.equal(m2, mean) and torch.equal(s2, std)
    if case == "offset":
        # the cancelling one-pass formula sum x^2 - (sum x)^2 / K, in fp32 on the same merged values, fails these limits
        vf = v.float()
        s1 = torch.zeros_like(vf[:1])
        s2_ = torch.zeros_like(vf[:1])
        for k in range(K):
            s1 = s1 + vf[k:k + 1]
            s2_ = s2_ + vf[k:k + 1] * vf[k:k + 1]
        naive = ((s2_ - s1 * s1 / K) / (K - 1)).clamp_min(0).sqrt()
        _, e_naive = _stats_errors(s1 / K, naive, m_ref, s_ref)
        print(f"  naive fp32 sum-of-squares formula on the same values: std error {e_naive:.1f} x the limit")
        assert e_naive > 10.0


# ----------------------------------------------------------------------------------------------------------------- engine
def _zs(model, K, seed, T=0.7):
    g = torch.Generator().manual_seed(seed)
    out = []
    for n in range(model.n_levels):
        z = torch.empty((K,) + tuple(model.conv_inn[n].global_out_shapes[0]))
        torch.nn.init.trunc_normal_(z, mean=0.0, std=1.0, a=-T, b=T, generator=g)
        out.append(z.to(DEV))
    return out


def _sample_stats(vols):
    v = torch.cat([x.double() for x in vols], 0)
    return v.mean(0, keepdim=True), v.std(0, keepdim=True)


def _engine_errors(mean, std, m_ref, s_ref):
    """(max |mean - ref| / (1 + |ref|), max |std - ref| / (1e-6 (1 + |mean|) + 1e-4 std)): tight limits for the engine against
    its own single-sample reconstructions, which run the same kernels."""
    mean, std, m_ref, s_ref = (t.double().cpu() for t in (mean, std, m_ref, s_ref))
    e_m = ((mean - m_ref).abs() / (1.0 + m_ref.abs())).max().item()
    e_s = ((std - s_ref).abs() / (1e-6 * (1.0 + m_ref.abs()) + 1e-4 * s_ref)).max().item()
    return e_m, e_s


@pytest.fixture(scope="module")
def tiny(golden_tiny):
    model = build_tiny_model(golden_tiny, DEV)
    views, mean_vols = tiny_inputs(golden_tiny)
    return model, views.to(DEV), [t.to(DEV) for t in mean_vols]


TOL = {"bf16": 2e-2, "fp16": 3e-3}      # the engine's stated rel-L2 tolerances (engine.py)
# std against the fp32 module path, rel-L2, at about 4x the values measured on a B200 (1000 W power limit): 1.06e-2 (bf16),
# 1.36e-3 (fp16); the mean measured 1.27e-2 / 1.53e-3 against the engine tolerances above.
TOL_STD_MODULE = {"bf16": 4.5e-2, "fp16": 6e-3}


@gpu
@pytest.mark.parametrize("kind", ["bf16", "fp16"])
def test_engine_posterior_tiny(tiny, kind):
    from cwfa_b200.engine import CWFAEngine
    model, views, mv = tiny
    K = 4
    zs = _zs(model, K, 11)
    eng = CWFAEngine(model, kind)
    mean, std = eng.reconstruct_posterior(views, mv, K, zs=zs)
    assert tuple(mean.shape) == tuple(std.shape) == (1, model.cfg.n_depths, views.shape[2], views.shape[3])
    # against K single-sample reconstructions of the engine (same kernels: sample k bitwise)
    singles = [eng.reconstruct(views, mv, zs=[z[k:k + 1] for z in zs]) for k in range(K)]
    m_ref, s_ref = _sample_stats(singles)
    e_m, e_s = _engine_errors(mean, std, m_ref, s_ref)
    # against the fp32 module path, sample by sample
    mods = [model.reconstruct(views, mv, zs=[z[k:k + 1] for z in zs]) for k in range(K)]
    mm, sm = _sample_stats(mods)
    r_m, r_s = rel_l2(mean, mm), rel_l2(std, sm)
    # the mean-only multi-sample path
    r_multi = rel_l2(mean, eng.reconstruct(views, mv, zs=zs, n_samples=K))
    print(f"posterior tiny {kind} K={K}: vs engine singles mean {e_m:.2e} (limit 4e-6) std {e_s:.3f} (limit 1); vs fp32 module "
          f"mean {r_m:.2e} std {r_s:.2e}; vs reconstruct(n_samples) mean {r_multi:.2e}; mean |std| {float(std.mean()):.3e}")
    assert e_m < 4e-6 and e_s < 1.0, (e_m, e_s)
    assert r_m < TOL[kind] and r_s < TOL_STD_MODULE[kind], (r_m, r_s)
    assert r_multi < TOL[kind]
    # graphed == eager, bitwise, for given zs
    gm, gs = eng.reconstruct_posterior_graphed(views, mv, K, zs=zs)
    assert torch.equal(gm, mean) and torch.equal(gs, std)


@gpu
def test_engine_posterior_graphed_sampling(tiny):
    from cwfa_b200.engine import CWFAEngine
    model, views, mv = tiny
    eng = CWFAEngine(model, "bf16")
    m1, s1 = (t.clone() for t in eng.reconstruct_posterior_graphed(views, mv, 3, temperature=0.7))
    m2, s2 = (t.clone() for t in eng.reconstruct_posterior_graphed(views, mv, 3, temperature=0.7))
    assert not torch.equal(m1, m2) and not torch.equal(s1, s2), "fresh latent samples per replay"
    for s in (s1, s2):
        assert torch.isfinite(s).all() and bool((s >= 0).all()) and float(s.mean()) > 0
    m0, s0 = eng.reconstruct_posterior_graphed(views, mv, 3, temperature=0.0)
    assert torch.equal(s0, torch.zeros_like(s0)), "temperature 0: every sample is the z = 0 reconstruction"
    r = rel_l2(m0, eng.reconstruct(views, mv))
    print(f"posterior temperature 0 vs reconstruct(): rel-L2 {r:.2e}")
    assert r < 1e-6
    m0e, s0e = eng.reconstruct_posterior(views, mv, 3, temperature=0.0)
    assert torch.equal(m0e, m0) and torch.equal(s0e, s0)


@gpu
def test_engine_posterior_from_sensor_frame(tiny):
    from cwfa_b200.data import LensletLayout
    from cwfa_b200.engine import CWFAEngine
    model, _, mv = tiny
    coords = [[40 + 50 * (i // 6), 35 + 55 * (i % 6)] for i in range(29)]
    layout = LensletLayout(coords, (64, 64), 32768.0, 16384.0, device=DEV)
    g = torch.Generator().manual_seed(5)
    frame = torch.randint(0, 65536, (1, 1, 300, 340), generator=g, dtype=torch.int32).to(torch.uint16).to(DEV)
    zs = _zs(model, 3, 12)
    eng = CWFAEngine(model, "fp16")
    ref = eng.reconstruct_posterior(layout.views(frame), mv, 3, zs=zs)
    got = eng.reconstruct_posterior(frame, mv, 3, zs=zs, sensor=layout)
    assert torch.equal(got[0], ref[0]) and torch.equal(got[1], ref[1])
    gg = eng.reconstruct_posterior_graphed(frame, mv, 3, zs=zs, sensor=layout)
    assert torch.equal(gg[0], ref[0]) and torch.equal(gg[1], ref[1])


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
        m.cond_nets[n].load_state_dict(deterministic_fill(m.cond_nets[n].state_dict(), 200 + n))
    m.cond_nets[-1].load_state_dict(deterministic_fill(m.cond_nets[-1].state_dict(), 300))
    return m.to(DEV)


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


# Limits against the engine's own single-sample reconstructions when the levels run the K-row NCHW path: that path applies
# the coefficients to the K rows through the affine kernel (GLOW: the block's own forward on K rows) instead of the fused
# coupling, so sample k agrees with its single-sample reconstruction to fp32 rounding, not bitwise.
TOL_NCHW_MEAN, TOL_NCHW_STD = 1e-5, 1e-3


@gpu
@pytest.mark.parametrize("which", ["glow", "ragged_nchw", "ragged_f8"])
def test_engine_posterior_other_level_types(golden_tiny, which):
    from cwfa_b200.engine import CWFAEngine
    if which == "glow":
        model = _glow_model(golden_tiny)
        views, mean_vols = tiny_inputs(golden_tiny)
        views, mv = views.to(DEV), [t.to(DEV) for t in mean_vols[:model.n_levels]] + [None]
    else:
        model = _ragged_model()
        views = seeded_randn((1, 29, 72, 72), 41).to(DEV)
        mv = [seeded_randn((1, 24 // 2 ** (n + 1), 72, 72), 50 + n, 0.1).to(DEV) for n in range(2)] + \
             [seeded_randn((1, 24 // 4, 72, 72), 59, 0.1).to(DEV)]
    eng = CWFAEngine(model, "fp16")
    if which == "ragged_nchw":
        eng.use_f8 = False                       # every level on the NCHW coupling path
    K = 3
    zs = _zs(model, K, 13)
    mean, std = eng.reconstruct_posterior(views, mv, K, zs=zs)
    singles = [eng.reconstruct(views, mv, zs=[z[k:k + 1] for z in zs]) for k in range(K)]
    m_ref, s_ref = _sample_stats(singles)
    mean_d, std_d = mean.double().cpu(), std.double().cpu()
    e_m = ((mean_d - m_ref.cpu()).abs() / (1.0 + m_ref.cpu().abs())).max().item()
    e_s = rel_l2(std_d, s_ref)
    print(f"posterior {which} K={K}: vs engine singles mean {e_m:.2e} std rel-L2 {e_s:.2e}")
    if which == "ragged_f8":
        assert e_m < 4e-6 and _engine_errors(mean, std, m_ref, s_ref)[1] < 1.0
    else:
        assert e_m < TOL_NCHW_MEAN and e_s < TOL_NCHW_STD, (e_m, e_s)
    gm, gs = eng.reconstruct_posterior_graphed(views, mv, K, zs=zs)
    assert torch.equal(gm, mean) and torch.equal(gs, std)


@gpu
def test_engine_posterior_rejects(golden_tiny, tiny):
    import cwfa_b200
    from cwfa_b200.engine import CWFAEngine
    model, views, mv = tiny
    eng = CWFAEngine(model, "bf16")
    with pytest.raises(ValueError, match="n_samples"):
        eng.reconstruct_posterior(views, mv, 1)
    with pytest.raises(ValueError, match="batch"):
        eng.reconstruct_posterior(views.expand(2, -1, -1, -1).contiguous(), mv, 2)
    zs = _zs(model, 3, 14)
    with pytest.raises(ValueError, match="rows"):
        eng.reconstruct_posterior(views, mv, 2, zs=zs)
    with pytest.raises(ValueError, match="rows"):
        eng.reconstruct_posterior_graphed(views, mv, 2, zs=zs)
    cfg = golden_tiny["config"]
    dlr = cwfa_b200.CWFAModel(n_depths=cfg["D"], volume_side_size=cfg["S"], INN_max_down_steps=cfg["MAX"], disable_low_res_input=1,
                              seed=0).to(DEV)
    with pytest.raises(ValueError, match="disable_low_res_input"):
        CWFAEngine(dlr, "bf16").reconstruct_posterior(views, mv, 2)


@gpu
def test_engine_posterior_full_config():
    """96 x 512 x 512 (5 steps, bf16), K = 3: against three single-sample reconstructions, eager and graphed."""
    import cwfa_b200
    from cwfa_b200.engine import CWFAEngine
    model = cwfa_b200.CWFAModel(seed=0).to(DEV)
    g = torch.Generator().manual_seed(1)
    views = torch.randn((1, 29, 512, 512), generator=g).to(DEV)
    mvs = [(0.1 * torch.randn((1, 96 // 2 ** (n + 1), 512, 512), generator=g)).to(DEV) for n in range(4)]
    K = 3
    zs = _zs(model, K, 15)
    eng = CWFAEngine(model, "bf16")
    mean, std = eng.reconstruct_posterior(views, mvs, K, zs=zs)
    singles = [eng.reconstruct(views, mvs, zs=[z[k:k + 1] for z in zs]) for k in range(K)]
    m_ref, s_ref = _sample_stats(singles)
    e_m, e_s = _engine_errors(mean, std, m_ref, s_ref)
    print(f"posterior full config K={K}: vs engine singles mean {e_m:.2e} std {e_s:.3f}; mean |std| {float(std.mean()):.3e}")
    assert e_m < 4e-6 and e_s < 1.0
    gm, gs = eng.reconstruct_posterior_graphed(views, mvs, K, zs=zs)
    assert torch.equal(gm, mean) and torch.equal(gs, std)
