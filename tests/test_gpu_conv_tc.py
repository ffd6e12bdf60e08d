"""GPU: the tcgen05 implicit-GEMM convolution vs torch CPU convolution on operands rounded to the same
half-precision grid (so the only difference is fp32 accumulation order)."""
import pytest
import torch
import torch.nn.functional as F

from conftest import max_abs, rel_l2
from oracle.weights import seeded_randn
from test_gpu_coupling import _coupling_reference

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _round(t, kind):
    return t.to(torch.bfloat16 if kind == "bf16" else torch.float16).float()


CASES = [
    # cin, cout, k, H, W, mb, bn
    (64, 64, 3, 32, 32, 1, 64),
    (64, 64, 3, 32, 32, 2, 64),
    (64, 64, 1, 16, 24, 2, 64),
    (16, 16, 3, 16, 16, 1, 16),
    (6, 64, 1, 20, 13, 1, 64),
    (48, 96, 3, 40, 24, 2, 96),
    (29, 48, 3, 33, 17, 2, 48),
    (64, 12, 3, 16, 16, 2, 16),
    (128, 64, 3, 32, 16, 2, 64),
    (256, 256, 3, 32, 32, 2, 256),
    (64, 64, 7, 32, 32, 2, 64),
    (256, 512, 3, 16, 16, 1, 256),
]


@pytest.mark.parametrize("cin,cout,k,H,W,mb,bn", CASES)
@pytest.mark.parametrize("kind", ["bf16", "fp16"])
def test_conv_tc_vs_cpu(cin, cout, k, H, W, mb, bn, kind):
    from cwfa_b200 import ops, tc
    x = _round(seeded_randn((2, cin, H, W), 1), kind)
    w = _round(seeded_randn((cout, cin, k, k), 2, (1.0 / (cin * k * k)) ** 0.5), kind)
    b = seeded_randn((cout,), 3)
    ref = F.conv2d(x.double(), w.double(), b.double(), padding=k // 2).float()
    xc = tc.to_c8(x.to(DEV), kind)
    assert torch.equal(tc.from_c8(xc).cpu(), x), "C8 round trip must be exact on representable values"
    pc = tc.PackedConv(w.to(DEV), b.to(DEV), kind, bn=bn)
    y = tc.conv_tc(xc, pc, out_nchw=True, mb=mb)
    torch.cuda.synchronize()
    err = rel_l2(y, ref)
    print(f"conv_tc {cin}->{cout} k{k} {H}x{W} mb{mb} bn{bn} {kind}: rel_l2={err:.2e} max_abs={max_abs(y, ref):.2e}")
    assert err < 2e-5
    # C8 output with fused ELU + residual (pre-activation add), rounded to half on store
    r = _round(seeded_randn((2, cout, H, W), 4), kind)
    y2 = tc.from_c8(tc.conv_tc(xc, pc, act=ops.ACT_ELU, res=tc.to_c8(r.to(DEV), kind), res_mode=1, mb=mb))
    ref2 = F.elu(ref + r)
    tol = 6e-3 if kind == "bf16" else 8e-4
    assert rel_l2(y2, ref2) < tol


@pytest.mark.parametrize("kind", ["bf16", "fp16"])
@pytest.mark.parametrize("N,H,W", [(1, 16, 16), (2, 48, 32), (1, 40, 24), (1, 128, 128), (3, 64, 80)])
def test_fused_resblock_vs_unfused_and_cpu(kind, N, H, W):
    """Fused persistent trunk block == the two-kernel sequence (same roundings) and ~= fp64 CPU."""
    from cwfa_b200 import ops, tc
    x = _round(seeded_randn((N, 64, H, W), 11), kind)
    w3 = _round(seeded_randn((64, 64, 3, 3), 12, (1.0 / 576) ** 0.5), kind)
    w1 = _round(seeded_randn((64, 64, 1, 1), 13, (1.0 / 64) ** 0.5), kind)
    b3, b1 = seeded_randn((64,), 14, 0.1), seeded_randn((64,), 15, 0.1)
    xc = tc.to_c8(x.to(DEV), kind)
    p3, p1 = tc.PackedConv(w3.to(DEV), b3.to(DEV), kind, bn=64), tc.PackedConv(w1.to(DEV), b1.to(DEV), kind, bn=64)
    y = tc.from_c8(tc.resblock_tc(xc, p3, p1))
    t = tc.conv_tc(xc, p3, act=ops.ACT_ELU)
    y_ref2 = tc.from_c8(tc.conv_tc(t, p1, act=ops.ACT_ELU, res=xc, res_mode=1))
    torch.cuda.synchronize()
    tmid = _round(F.elu(F.conv2d(x.double(), w3.double(), b3.double(), padding=1)).float(), kind)
    ref = F.elu(F.conv2d(tmid.double(), w1.double(), b1.double()) + x.double()).float()
    tol = 6e-3 if kind == "bf16" else 8e-4
    print(f"resblock {kind} {N}x{H}x{W}: vs unfused {rel_l2(y, y_ref2):.2e}  vs cpu {rel_l2(y, ref):.2e}")
    assert rel_l2(y, y_ref2) < tol
    assert rel_l2(y, ref) < tol


FAST_CASES = [
    # cin, cout, k, N, H, W, mb, bn  -- lean epilogue (C8 out, no residual); ragged edges, >1 item per CTA, every tile plan
    (16, 320, 1, 2, 128, 128, 2, 64),     # 640 items on a 296-CTA persistent grid, double-buffered TMEM
    (6, 192, 3, 1, 37, 53, 1, 192),       # ragged H and W, one M-block, two CTAs per SM
    (12, 384, 3, 1, 40, 72, 2, 128),      # 256 TMEM columns, single buffer
    (24, 768, 3, 2, 24, 40, 1, 256),
    (48, 96, 3, 3, 33, 17, 2, 48),
    (64, 48, 3, 1, 50, 30, 2, 48),
    (256, 256, 3, 3, 128, 128, 2, 256),   # WIDE variant, 192 items on 148 CTAs
    (64, 64, 7, 1, 45, 45, 2, 64),        # one A stage (shared-memory plan for two CTAs per SM)
]


@pytest.mark.parametrize("cin,cout,k,N,H,W,mb,bn", FAST_CASES)
@pytest.mark.parametrize("act", ["none", "prelu"])
def test_conv_tc_lean_epilogue_and_persistent_walk(cin, cout, k, N, H, W, mb, bn, act):
    """C8-output convolutions without residual take the compile-time lean epilogue; the grid is persistent, so these
    shapes also exercise CTAs walking several (n-block, sample, tile) items, ragged tile edges and each tile plan."""
    from cwfa_b200 import ops, tc
    kind = "bf16"
    x = _round(seeded_randn((N, cin, H, W), 21), kind)
    w = _round(seeded_randn((cout, cin, k, k), 22, (1.0 / (cin * k * k)) ** 0.5), kind)
    b = seeded_randn((cout,), 23)
    ref = F.conv2d(x, w, b, padding=k // 2)
    slope = torch.full((1,), -0.3 if cin == 6 else 0.2)
    if act == "prelu":
        ref = torch.where(ref >= 0, ref, slope * ref)
    xc = tc.to_c8(x.to(DEV), kind)
    pc = tc.PackedConv(w.to(DEV), b.to(DEV), kind, bn=bn)
    y8 = tc.conv_tc(xc, pc, act=ops.ACT_PRELU if act == "prelu" else ops.ACT_NONE,
                    slope=slope.to(DEV) if act == "prelu" else None, mb=mb)
    y = tc.from_c8(y8)
    torch.cuda.synchronize()
    assert y.shape == ref.shape
    err = rel_l2(y, ref)
    print(f"lean conv {cin}->{cout} k{k} {N}x{H}x{W} mb{mb} bn{bn} {act}: rel_l2={err:.2e}")
    assert err < 6e-3
    # padded output channels of the C8 tensor must be exactly zero (the next conv reads them as K padding)
    if y8.Cp != cout:
        raw = y8.data.float().view(N, y8.Cp // 8, H, W, 8).permute(0, 1, 4, 2, 3).reshape(N, y8.Cp, H, W)
        assert float(raw[:, cout:].abs().max()) == 0.0
    # same result from the default tile plan (heuristic BN / MB)
    y_def = tc.from_c8(tc.conv_tc(xc, tc.PackedConv(w.to(DEV), b.to(DEV), kind), act=ops.ACT_PRELU if act == "prelu" else ops.ACT_NONE,
                                  slope=slope.to(DEV) if act == "prelu" else None))
    assert rel_l2(y_def, ref) < 6e-3


@pytest.mark.parametrize("N,H,W,cin,cout", [(1, 9, 13, 64, 32), (2, 16, 24, 128, 64), (1, 64, 64, 512, 256)])
def test_conv_transpose_tc_with_skip(N, H, W, cin, cout):
    """ConvTranspose2d(k=2, s=2) + skip add (unet.py:166,190): scatter epilogue with the one-group-ahead residual prefetch."""
    from cwfa_b200 import tc
    kind = "bf16"
    x = _round(seeded_randn((N, cin, H, W), 31), kind)
    w = _round(seeded_randn((cin, cout, 2, 2), 32, (1.0 / cin) ** 0.5), kind)
    b = seeded_randn((cout,), 33)
    skip = _round(seeded_randn((N, cout, 2 * H, 2 * W), 34), kind)
    ref = F.conv_transpose2d(x, w, b, stride=2) + skip
    pc = tc.PackedConv(w.to(DEV), b.to(DEV), kind, transposed=True)
    y = tc.from_c8(tc.conv_transpose_tc(tc.to_c8(x.to(DEV), kind), pc, tc.to_c8(skip.to(DEV), kind)))
    y0 = tc.from_c8(tc.conv_transpose_tc(tc.to_c8(x.to(DEV), kind), pc))
    torch.cuda.synchronize()
    assert rel_l2(y, ref) < 6e-3
    assert rel_l2(y0, ref - skip) < 6e-3


@pytest.mark.parametrize("cin,cout,N,H,W,bn", [(96, 12, 2, 20, 24, None), (256, 6, 1, 33, 17, None), (512, 48, 1, 32, 48, 144)])
def test_conv3x3_as_1x1_plus_col2im(cin, cout, N, H, W, bn):
    """3x3 conv with huge Cin / tiny Cout evaluated as one 1x1 tensor-core conv to 9 tap partials + col2im
    (second depth-stencil conv of the conditioning net): equals the direct 3x3 conv; channel padding stays zero."""
    from cwfa_b200 import tc
    kind = "bf16"
    x = _round(seeded_randn((N, cin, H, W), 41), kind)
    w = _round(seeded_randn((cout, cin, 3, 3), 42, (1.0 / (cin * 9)) ** 0.5), kind)
    b = seeded_randn((cout,), 43)
    ref = F.conv2d(x, w, b, padding=1)
    wg = tc.col2im3x3_weights(w.to(DEV))
    pc = tc.PackedConv(wg, None, kind, bn=bn)
    g = tc.conv_tc(tc.to_c8(x.to(DEV), kind), pc)
    y8 = tc.col2im3x3_c8(g, b.to(DEV), cout)
    y = tc.from_c8(y8)
    torch.cuda.synchronize()
    assert y.shape == ref.shape
    assert rel_l2(y, ref) < 8e-3
    if y8.Cp != cout:
        raw = y8.data.float().view(N, y8.Cp // 8, H, W, 8).permute(0, 1, 4, 2, 3).reshape(N, y8.Cp, H, W)
        assert float(raw[:, cout:].abs().max()) == 0.0


def test_conv_tc_skips_zero_weight_blocks():
    """Block-banded weights (each 64-channel output block reads only two 64-channel input blocks): the packer marks the
    all-zero K-blocks and the kernel skips them -- same result as the dense evaluation, incl. an all-zero output block."""
    from cwfa_b200 import tc
    kind = "bf16"
    cin, cout, H, W = 256, 256, 24, 40
    w = _round(seeded_randn((cout, cin, 3, 3), 51, (1.0 / (128 * 9)) ** 0.5), kind)
    mask = torch.zeros(cout, cin)
    for g in range(3):
        mask[64 * g:64 * g + 64, 64 * g:64 * g + 128] = 1.0       # output block 3 stays entirely zero
    w = w * mask[:, :, None, None]
    x = _round(seeded_randn((2, cin, H, W), 52), kind)
    b = seeded_randn((cout,), 53)
    ref = F.conv2d(x, w, b, padding=1)
    y = tc.from_c8(tc.conv_tc(tc.to_c8(x.to(DEV), kind), tc.PackedConv(w.to(DEV), b.to(DEV), kind, bn=64), mb=2))
    torch.cuda.synchronize()
    assert rel_l2(y, ref) < 6e-3
    assert rel_l2(y[:, 192:], ref[:, 192:]) < 6e-3              # bias only


@pytest.mark.parametrize("ch,axis,inverse,ext,zero_x", [
    (48, 1, True, False, False), (48, 3, True, False, False), (24, 2, False, False, False), (12, 1, False, True, False),
    (6, 0, True, True, True), (6, 3, False, False, False), (48, 0, True, False, True), (24, 1, True, True, False)])
@pytest.mark.parametrize("persistent", [True, False, "ticket"])
def test_fused_coupling_conv_vs_reference(ch, axis, inverse, ext, zero_x, persistent):
    """Last sub-network conv (64 -> 2 ch, 3x3) + affine coupling + log-det / sum y^2 + preceding permutation (gather on x)
    in ONE kernel (persistent coupling_tc and the general conv_tc<COUPLING>) vs conv2d + coupling_layers.py:490-500 in torch."""
    from cwfa_b200 import tc
    kind, N, H, W = "bf16", 2, 40, 56
    cout = ch if ext else 2 * ch
    b = _round(seeded_randn((N, 64, H, W), 61), kind)
    w = _round(seeded_randn((cout, 64, 3, 3), 62, 0.04), kind)
    bias = seeded_randn((cout,), 63, 0.1)
    a = F.conv2d(b, w, bias, padding=1)
    x = None if zero_x else seeded_randn((N, ch, H, W), 64)
    t_ext = seeded_randn((N, ch, H, W), 65, 0.3) if ext else None
    perm = None
    xin = torch.zeros(N, ch, H, W) if x is None else x
    if axis and x is not None:
        n_ax = {1: ch, 2: H, 3: W}[axis]
        perm = torch.from_numpy(__import__("numpy").random.RandomState(7).permutation(n_ax)).long()
        xin = xin.index_select(axis, perm)                 # the permutation preceding the coupling (fixed_transforms.py:37-41)
    y_ref, j_ref, _ = _coupling_reference(a, xin, t_ext, -0.5 ** 0.5 if ext else 1.0, ch, inverse)
    pc = tc.PackedConv(w.to(DEV), bias.to(DEV), kind, bn=tc.pad16(cout))
    # "ticket": the persistent kernel reduces its own partial sums (last-CTA finalize); the int32 must come back as zero
    ticket = torch.zeros(1, device=DEV, dtype=torch.int32) if persistent == "ticket" else None
    persistent = bool(persistent)
    logdet = torch.full((N,), 3.0, device=DEV)
    sumsq = torch.zeros(N, device=DEV)
    y = tc.conv_tc_coupling(tc.to_c8(b.to(DEV), kind), pc, None if x is None else x.to(DEV), ch=ch, inverse=inverse,
                            t_ext=None if t_ext is None else t_ext.to(DEV), t_scale=-0.5 ** 0.5 if ext else 1.0,
                            perm=None if perm is None else perm.to(DEV).to(torch.int32), perm_axis=axis if perm is not None else 0,
                            logdet=logdet, sumsq=sumsq, accumulate=True, persistent=persistent, ticket=ticket)
    torch.cuda.synchronize()
    assert ticket is None or int(ticket[0]) == 0
    assert rel_l2(y, y_ref) < 2e-5 * 50                     # fp32 accumulation-order + fast atan/exp differences only
    assert torch.allclose(logdet.cpu() - 3.0, j_ref, rtol=2e-4, atol=2e-2)
    assert torch.allclose(sumsq.cpu(), (y_ref.double() ** 2).sum(dim=(1, 2, 3)).float(), rtol=2e-3)
    # bit-reproducible reductions
    logdet2 = torch.full((N,), 3.0, device=DEV)
    tc.conv_tc_coupling(tc.to_c8(b.to(DEV), kind), pc, None if x is None else x.to(DEV), ch=ch, inverse=inverse,
                        t_ext=None if t_ext is None else t_ext.to(DEV), t_scale=-0.5 ** 0.5 if ext else 1.0,
                        perm=None if perm is None else perm.to(DEV).to(torch.int32), perm_axis=axis if perm is not None else 0,
                        logdet=logdet2, persistent=persistent, ticket=ticket)
    assert torch.equal(logdet, logdet2)


@pytest.mark.parametrize("N,C,H,W,kind", [(1, 64, 32, 32, "bf16"), (2, 6, 17, 23, "bf16"), (1, 64, 24, 40, "fp16")])
def test_layernorm_c8(N, C, H, W, kind):
    """LayerNorm([C,H,W]) with element-wise affine (ConvNeXt, networks.py:486-503) on the C8 layout vs F.layer_norm."""
    from cwfa_b200 import tc
    x = _round(seeded_randn((N, C, H, W), 81) * 1.7 + 0.3, kind)
    g = _round(seeded_randn((C, H, W), 82, 0.3) + 1.0, kind)
    b = _round(seeded_randn((C, H, W), 83, 0.2), kind)
    ref = F.layer_norm(x, [C, H, W], g, b, 1e-6)
    y8 = tc.layernorm_c8(tc.to_c8(x.to(DEV), kind), tc.to_c8(g[None].to(DEV), kind), tc.to_c8(b[None].to(DEV), kind), 1e-6)
    y = tc.from_c8(y8)
    torch.cuda.synchronize()
    assert rel_l2(y, ref) < (5e-3 if kind == "bf16" else 7e-4)
    if y8.Cp != C:
        raw = y8.data.float().view(N, y8.Cp // 8, H, W, 8).permute(0, 1, 4, 2, 3).reshape(N, y8.Cp, H, W)
        assert float(raw[:, C:].abs().max()) == 0.0


@pytest.mark.parametrize("kind,N,H,W,nsets", [("bf16", 1, 48, 80, 5), ("fp16", 2, 33, 19, 3), ("bf16", 1, 16, 16, 2), ("bf16", 3, 64, 64, 5)])
def test_batched_trunk_block_equals_per_subnetwork_launches(kind, N, H, W, nsets):
    """One launch over the block row of several independent sub-networks (cwfa_resblock_tc_batched: contiguous tile ranges, one
    weight switch per CTA) must equal the per-sub-network launches BIT FOR BIT (same MMAs, same epilogues), ragged shapes and
    set boundaries that fall inside a CTA's range included."""
    from cwfa_b200 import tc
    x = _round(seeded_randn((N, 64 * nsets, H, W), 91), kind)
    x8 = tc.to_c8(x.to(DEV), kind)
    sets = []
    for k in range(nsets):
        w3 = _round(seeded_randn((64, 64, 3, 3), 100 + k, 0.05), kind)
        w1 = _round(seeded_randn((64, 64, 1, 1), 200 + k, 0.12), kind)
        sets.append((tc.PackedConv(w3.to(DEV), seeded_randn((64,), 300 + k, 0.1).to(DEV), kind, bn=64),
                     tc.PackedConv(w1.to(DEV), seeded_randn((64,), 400 + k, 0.1).to(DEV), kind, bn=64)))
    y = tc.from_c8(tc.resblock_tc_batched(x8, sets))
    for k, (p3, p1) in enumerate(sets):
        yk = tc.from_c8(tc.resblock_tc(x8, p3, p1, 8 * k))
        assert torch.equal(y[:, 64 * k:64 * (k + 1)], yk), k
    torch.cuda.synchronize()
