"""Raw sensor frames as an input of the throughput path: ``LensletLayout`` and the one-pass sensor -> C8 lenslet-view kernel
(csrc/sensor.cu), bitwise against the two-pass route ``to_c8(extract_views(frame.float()))``; ``extract_views`` on uint16
frames; the engine, its CUDA graphs and the streaming reconstructor fed with frames instead of views, bitwise against the
same calls fed with the frames' views.  Kernel outputs are NaN-filled before every launch so that an unwritten byte fails."""
import os

import pytest
import torch

from conftest import GOLDEN
from helpers import build_tiny_model, tiny_inputs
from oracle.weights import seeded_randn

DEV = "cuda:0"
gpu = pytest.mark.gpu
DTYPES = {"uint16": torch.uint16, "float16": torch.float16, "float32": torch.float32}


def _frame(shape, dtype, seed):
    """A seeded frame built on the host: uint16 frames as int32 first (values 0..65535, both ends present), float frames from a
    normal sample.  Returns (frame in ``dtype``, the same values in fp32) on the device."""
    g = torch.Generator().manual_seed(seed)
    if dtype == torch.uint16:
        src = torch.randint(0, 65536, shape, generator=g, dtype=torch.int32)
        src.view(-1)[:2] = torch.tensor([0, 65535], dtype=torch.int32)
        src.view(-1)[-1] = 65535
    else:
        src = torch.randn(shape, generator=g) * 3.0
    host = src.to(dtype)
    return host.to(DEV), host.float().to(DEV)


def _norm(dtype):
    return (3000.5, 517.3) if dtype == torch.uint16 else (0.25, 1.75)


def _bits(t: torch.Tensor) -> torch.Tensor:
    """Bit pattern of a 16/32-bit tensor (signed zeros and NaN payloads compare as bits)."""
    return t.view(torch.int16 if t.element_size() == 2 else torch.int32)


def _c8_nan_filled(layout, frame, kind):
    """The kernel through the C ABI into a NaN-filled C8 buffer (an unwritten chunk stays NaN)."""
    from cwfa_b200 import _lib, tc
    from cwfa_b200.data import _IMAGE_DTYPES
    from cwfa_b200.ops import _stream
    img = layout._frame(frame)
    B, Hi, Wi = img.shape
    out = tc.C8.empty(B, layout.n_lenslets, *layout.subimage_shape, img.device, kind)
    out.data.fill_(float("nan"))
    _lib.call("cwfa_extract_views_c8", img.data_ptr(), _IMAGE_DTYPES[img.dtype], layout.coords.data_ptr(), out.data.data_ptr(), B,
              Hi, Wi, layout.n_lenslets, out.Cp, *layout.subimage_shape, layout.mean, layout.std, int(layout.normalise), out.is_bf16,
              _stream())
    return out


def _grid_coords(L, Hi, Wi, side):
    """L lenslet centres on a grid that reaches past every border of the frame (clipped windows on all four sides); from
    L = 16 on, the last window lies wholly outside the frame (a view of the normalised zero only)."""
    rows, cols = 6, (L + 5) // 6
    c = [[-side // 4 + (Hi + side // 2) * (i % rows) // (rows - 1), -side // 3 + (Wi + side // 2) * (i // rows) // max(cols - 1, 1)]
         for i in range(L)]
    if L >= 16:
        c[-1] = [Hi + side, -side]
    return c


def _clipped_coords(side, Hi=700, Wi=1002):
    """The windows of test_gpu_data.py::test_extract_views_wide_views_clipped_windows."""
    h = side // 2
    return [[10, 17], [Hi - 5, Wi - 9], [h, h], [Hi - h, Wi - h], [h + 1, Wi - 3], [Hi - 2, h + 3], [350, 501], [351, 502], [352, 503]]


def _case(name, golden_modules):
    """(frame shape (B, 1, Hi, Wi), coordinates, view side)."""
    if name == "golden":
        return (2, 1, 90, 100), golden_modules["extract_views/coords"].tolist(), 64
    if name.startswith("clip"):
        side = int(name[4:])
        return ((3 if side % 8 else 1), 1, 700, 1002), _clipped_coords(side), side
    if name.startswith("L"):
        L = int(name[1:])
        return ((3 if L % 2 else 1), 1, 300, 340), _grid_coords(L, 300, 340, 64), 64
    assert name == "full"
    return (1, 1, 2160, 2160), [[300 + 370 * (i // 6), 280 + 330 * (i % 6)] for i in range(29)], 512


CASES = ["golden", "clip128", "clip60", "clip37", "L1", "L8", "L16", "L29", "full"]


@gpu
@pytest.mark.parametrize("dtype", list(DTYPES))
@pytest.mark.parametrize("case", CASES)
def test_views_c8_bitwise_equals_extract_views_to_c8(golden_modules, case, dtype):
    """Both kinds, with and without normalisation: the one-pass kernel (NaN-filled output, and through ``views_c8``) is bitwise
    ``to_c8(extract_views(frame.float()))``, padding slots included; ``views`` equals ``extract_views``."""
    from cwfa_b200 import tc
    from cwfa_b200.data import LensletLayout, extract_views
    dt = DTYPES[dtype]
    shape, coords, side = _case(case, golden_modules)
    frame, frame32 = _frame(shape, dt, seed=sum(map(ord, case + dtype)))
    for norm in (False, True):
        mean, std = _norm(dt) if norm else (None, None)
        layout = LensletLayout(coords, (side, side), mean, std, device=DEV)
        ref32 = extract_views(frame32, coords, [side, side], mean, std)
        assert torch.equal(_bits(layout.views(frame)), _bits(ref32))
        assert torch.equal(_bits(layout.views(frame[:, 0])), _bits(ref32))          # (B, Hi, Wi) frames
        for kind in ("bf16", "fp16"):
            ref = tc.to_c8(ref32, kind)
            got = _c8_nan_filled(layout, frame, kind)
            assert (got.C, got.Cp, tuple(got.data.shape)) == (ref.C, ref.Cp, tuple(ref.data.shape))
            assert torch.equal(_bits(got.data), _bits(ref.data)), (case, dtype, norm, kind)
            api = layout.views_c8(frame, kind)
            assert api.kind == kind and torch.equal(_bits(api.data), _bits(ref.data))
            if got.Cp > got.C:                                                       # padding slots are +0, not the normalised zero
                pad = tc.from_c8(tc.C8(got.data, got.Cp, kind))[:, got.C:]
                assert torch.equal(_bits(pad), torch.zeros_like(_bits(pad)))


@gpu
@pytest.mark.parametrize("case", CASES)
def test_extract_views_uint16_equals_float(golden_modules, case):
    """``extract_views`` reads uint16 frames as they are (no fp32 copy of the frame): bitwise equal to the fp32 frame's views."""
    from cwfa_b200 import _lib
    from cwfa_b200.data import extract_views
    from cwfa_b200.ops import _stream
    shape, coords, side = _case(case, golden_modules)
    frame, frame32 = _frame(shape, torch.uint16, seed=7 + len(case))
    c = torch.tensor(coords, dtype=torch.int32, device=DEV)
    for mean, std in ((None, None), _norm(torch.uint16)):
        out = torch.full((shape[0], len(coords), side, side), float("nan"), device=DEV)
        norm = mean is not None
        _lib.call("cwfa_extract_views", frame.data_ptr(), 2, c.data_ptr(), out.data_ptr(), shape[0], shape[2], shape[3], len(coords),
                  side, side, mean or 0.0, std or 1.0, int(norm), _stream())
        ref = extract_views(frame32, coords, [side, side], mean, std)
        assert torch.equal(_bits(out), _bits(ref))
        assert torch.equal(_bits(extract_views(frame, coords, [side, side], mean, std)), _bits(ref))


# ---- the engine fed with frames ---------------------------------------------------------------------------------------------
TINY_COORDS = [[40 + 50 * (i // 6), 35 + 55 * (i % 6)] for i in range(29)]     # 64 x 64 views of a 300 x 340 frame, right edge clipped


def _tiny_layout():
    from cwfa_b200.data import LensletLayout
    return LensletLayout(TINY_COORDS, (64, 64), 32768.0, 16384.0, device=DEV)


def _frames(n, B=1, seed=0, dtype=torch.uint16, pinned=False):
    out = []
    for i in range(n):
        f = _frame((B, 1, 300, 340), dtype, seed + i)[0]
        out.append(f.cpu().pin_memory() if pinned else f)
    return out


@pytest.fixture(scope="module")
def tiny_model(golden_tiny):
    return build_tiny_model(golden_tiny, DEV)


@gpu
@pytest.mark.parametrize("kind", ["bf16", "fp16"])
def test_engine_reconstruct_from_frames(golden_tiny, tiny_model, kind):
    """reconstruct / reconstruct_graphed / reconstruct_host with ``sensor=``: bitwise the same calls on the frames' views; two
    different frames replayed through one graph."""
    from cwfa_b200.engine import CWFAEngine
    _, mean_vols = tiny_inputs(golden_tiny)
    mv = [t.to(DEV) for t in mean_vols]
    layout = _tiny_layout()
    eng = CWFAEngine(tiny_model, kind)
    f1, f2 = _frames(2, seed=11)
    ref1, ref2 = eng.reconstruct(layout.views(f1), mv), eng.reconstruct(layout.views(f2), mv)
    assert torch.isfinite(ref1).all() and not torch.equal(ref1, ref2)
    assert torch.equal(eng.reconstruct(f1, mv, sensor=layout), ref1)
    assert torch.equal(eng.reconstruct(f1[:, 0], mv, sensor=layout), ref1)
    g1 = eng.reconstruct_graphed(f1, mv, sensor=layout).clone()
    g2 = eng.reconstruct_graphed(f2, mv, sensor=layout).clone()
    assert torch.equal(g1, ref1) and torch.equal(g2, ref2)
    # the views graph of the same shapes is a separate graph, fed with views
    assert torch.equal(eng.reconstruct_graphed(layout.views(f2), mv), ref2)
    assert sum(k[-1] == (id(layout), torch.uint16) for k in eng._graphs) == 1
    assert torch.equal(eng.reconstruct_host(f1.cpu().pin_memory(), mv, sensor=layout), ref1.cpu())
    assert eng._frame_dev.dtype == torch.uint16
    # all outputs of the multi-level call too
    outs, jacs = eng.reconstruct(f2, mv, return_all=True, sensor=layout)
    routs, rjacs = eng.reconstruct(layout.views(f2), mv, return_all=True)
    assert all(torch.equal(outs[n], routs[n]) for n in routs) and all(torch.equal(jacs[n], rjacs[n]) for n in rjacs)


@gpu
@pytest.mark.parametrize("kind", ["bf16", "fp16"])
def test_engine_forward_nll_from_frames(golden_tiny, tiny_model, kind):
    from cwfa_b200.engine import CWFAEngine
    cfg = golden_tiny["config"]
    B, D, S = 2, cfg["D"], cfg["S"]
    _, mean_vols = tiny_inputs(golden_tiny)
    mvB = [m.repeat(B, 1, 1, 1).to(DEV) for m in mean_vols[:tiny_model.n_levels]]
    layout = _tiny_layout()
    eng = CWFAEngine(tiny_model, kind)
    x1, x2 = seeded_randn((B, D, S, S), 2).to(DEV), seeded_randn((B, D, S, S), 3).to(DEV)
    f1, f2 = _frames(2, B=B, seed=21)
    keys = ("z", "lo", "logdet", "sumsq", "nll_per_sample", "nll_ref")

    def same(a, b):
        return all(torch.equal(ra[k], rb[k]) for ra, rb in zip(a, b) for k in keys)

    ref1 = eng.forward_nll(x1, layout.views(f1), mvB)
    ref2 = eng.forward_nll(x2, layout.views(f2), mvB)
    assert same(eng.forward_nll(x1, f1, mvB, sensor=layout), ref1)
    g1 = [{k: v.clone() for k, v in r.items()} for r in eng.forward_nll_graphed(x1, f1, mvB, sensor=layout)]
    g2 = eng.forward_nll_graphed(x2, f2, mvB, sensor=layout)
    assert same(g1, ref1) and same(g2, ref2)


@gpu
def test_engine_from_frames_disable_low_res_input(golden_tiny):
    """disable_low_res_input=1: only the LRNN reads the conditions."""
    from cwfa_b200.engine import CWFAEngine
    from test_oracle_golden_r2 import build_dlr_model
    small = torch.load(os.path.join(GOLDEN, "r2_small.pt"), weights_only=False)
    m = build_dlr_model(golden_tiny, small, DEV)
    _, mean_vols = tiny_inputs(golden_tiny)
    mv = [t.to(DEV) for t in mean_vols[:m.n_levels]] + [None]
    layout = _tiny_layout()
    f1, f2 = _frames(2, seed=31)
    for kind in ("bf16", "fp16"):
        eng = CWFAEngine(m, kind)
        ref1, ref2 = eng.reconstruct(layout.views(f1), mv), eng.reconstruct(layout.views(f2), mv)
        assert torch.equal(eng.reconstruct(f1, mv, sensor=layout), ref1)
        assert torch.equal(eng.reconstruct_graphed(f1, mv, sensor=layout).clone(), ref1)
        assert torch.equal(eng.reconstruct_graphed(f2, mv, sensor=layout), ref2)


@gpu
def test_engine_from_frames_multi_sample(golden_tiny, tiny_model):
    """n_samples=2 with given latent samples, eager and graphed."""
    from cwfa_b200.engine import CWFAEngine
    _, mean_vols = tiny_inputs(golden_tiny)
    mv = [t.to(DEV) for t in mean_vols]
    zs = [seeded_randn((2,) + tuple(tiny_model.conv_inn[n].global_out_shapes[0]), 140 + n, 0.6).to(DEV) for n in range(tiny_model.n_levels)]
    layout = _tiny_layout()
    (f1,) = _frames(1, seed=41)
    eng = CWFAEngine(tiny_model, "fp16")
    ref = eng.reconstruct(layout.views(f1), mv, zs=zs, n_samples=2)
    assert torch.equal(eng.reconstruct(f1, mv, zs=zs, n_samples=2, sensor=layout), ref)
    assert torch.equal(eng.reconstruct_graphed(f1, mv, zs=zs, n_samples=2, sensor=layout), ref)


@gpu
@pytest.mark.parametrize("out_dtype", [torch.float32, torch.float16])
def test_streaming_from_pinned_uint16_frames(golden_tiny, tiny_model, out_dtype):
    """6 different pinned uint16 frames at depth 2 (a stale static buffer would repeat a frame): each output is bitwise the
    one-by-one ``reconstruct_graphed`` of that frame's views; device-resident frames as well."""
    from cwfa_b200.engine import CWFAEngine, StreamingReconstructor
    _, mean_vols = tiny_inputs(golden_tiny)
    mv = [t.to(DEV) for t in mean_vols]
    layout = _tiny_layout()
    eng = CWFAEngine(tiny_model, "bf16")
    frames = _frames(6, seed=51, pinned=True)
    D, S = golden_tiny["config"]["D"], golden_tiny["config"]["S"]
    refs = [eng.reconstruct_graphed(layout.views(f.to(DEV)), mv).to(out_dtype).cpu() for f in frames]
    assert all(not torch.equal(refs[i], refs[i + 1]) for i in range(5))
    st = StreamingReconstructor(eng, tuple(frames[0].shape), mv, depth=2, out_dtype=out_dtype, sensor=layout)
    outs = [torch.full((1, D, S, S), float("nan"), dtype=out_dtype).pin_memory() for _ in frames]
    st.run(frames, outs)
    for i, (o, r) in enumerate(zip(outs, refs)):
        assert torch.equal(o, r), f"frame {i}"
    if out_dtype == torch.float32:
        dev_frames = [f.to(DEV) for f in frames]
        douts = [torch.full((1, D, S, S), float("nan"), device=DEV) for _ in frames]
        StreamingReconstructor(eng, tuple(frames[0].shape), mv, depth=2, sensor=layout).run(dev_frames, douts)
        assert all(torch.equal(o.cpu(), r) for o, r in zip(douts, refs))


@gpu
def test_full_config_from_2160_frame():
    """96 x 512 x 512 (5 steps), a 2160 x 2160 uint16 frame, 29 x 512 x 512 views, bf16: the sensor path is bitwise the views
    path, eager and graphed."""
    import cwfa_b200
    from cwfa_b200.data import LensletLayout
    from cwfa_b200.engine import CWFAEngine
    model = cwfa_b200.CWFAModel(seed=0).to(DEV)
    assert (model.cfg.n_depths, model.cfg.volume_side_size) == (96, 512)
    g = torch.Generator().manual_seed(1)
    mvs = [(0.1 * torch.randn((1, 96 // 2 ** (n + 1), 512, 512), generator=g)).to(DEV) for n in range(4)]
    coords = [[300 + 370 * (i // 6), 280 + 330 * (i % 6)] for i in range(29)]
    layout = LensletLayout(coords, (512, 512), 32768.0, 16384.0, device=DEV)
    frame = _frame((1, 1, 2160, 2160), torch.uint16, 61)[0]
    eng = CWFAEngine(model, "bf16")
    ref = eng.reconstruct(layout.views(frame), mvs)
    assert torch.isfinite(ref).all()
    assert torch.equal(eng.reconstruct(frame, mvs, sensor=layout), ref)
    assert torch.equal(eng.reconstruct_graphed(frame, mvs, sensor=layout), ref)


@gpu
def test_layout_rejects_bad_frames():
    from cwfa_b200 import _lib
    layout = _tiny_layout()
    with pytest.raises(TypeError, match="uint16, float16 or float32"):
        layout.views_c8(torch.zeros((1, 1, 300, 340), dtype=torch.int32, device=DEV))
    with pytest.raises(ValueError, match=r"\(B, 1, Hi, Wi\)"):
        layout.views(torch.zeros((300, 340), device=DEV))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        layout.views(torch.zeros((1, 1, 300, 340)))
    f = torch.zeros((1, 1, 300, 340), device=DEV)
    out = torch.empty(32 * 64 * 64 + 8, dtype=torch.bfloat16, device=DEV)
    with pytest.raises(_lib.CwfaError, match="16-byte aligned"):
        _lib.call("cwfa_extract_views_c8", f.data_ptr(), 0, layout.coords.data_ptr(), out.data_ptr() + 2, 1, 300, 340, 29, 32, 64, 64,
                  0.0, 1.0, 0, 1, None)
    with pytest.raises(_lib.CwfaError, match="bad arguments"):          # Cp < L
        _lib.call("cwfa_extract_views_c8", f.data_ptr(), 0, layout.coords.data_ptr(), out.data_ptr(), 1, 300, 340, 29, 24, 64, 64,
                  0.0, 1.0, 0, 1, None)


# ---- CPU: argument checks of LensletLayout (before any device work) -----------------------------------------------------------
@pytest.mark.parametrize("coords, shape, mean, std, err", [
    ([[1, 2, 3]], (8, 8), None, None, "must be \\(L, 2\\)"),
    ([], (8, 8), None, None, "must be \\(L, 2\\)"),
    ([[1, 2]], (0, 8), None, None, "positive view sides"),
    ([[1, 2]], (8,), None, None, "positive view sides"),
    ([[1, 2]], (8, 8), 0.5, 0.0, "non-zero"),
    ([[1, 2]], (8, 8), 0.5, None, "both mean and std"),
    ([[1.5, 2]], (8, 8), None, None, "integer"),
])
def test_layout_validates_arguments(coords, shape, mean, std, err):
    from cwfa_b200.data import LensletLayout
    with pytest.raises(ValueError, match=err):
        LensletLayout(coords, shape, mean, std)


def test_layout_needs_cuda_device():
    from cwfa_b200.data import LensletLayout
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        LensletLayout([[1, 2]], (8, 8), device="cpu")
