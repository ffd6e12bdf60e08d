"""Per-kernel roofline table at the full-config shapes (CUDA events around a CUDA-graph replay of the calls, best of 5, tensors rotated through > L2).
Writes profiles/r02_kernel_rooflines.md.  HBM peak / tensor peak from MEASURED_PEAKS.json."""
import json, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from cwfa_b200 import ops, tc
from cwfa_b200.data import extract_views

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pk = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))) if os.path.exists(os.path.join(ROOT, "MEASURED_PEAKS.json")) else {}
HBM, TF = pk.get("hbm_gbs", 6650.0), pk.get("bf16_tflops", 1590.0)
DEV = "cuda:0"
P = 512 * 512
rows = []


def timeit(fn, nbuf):
    """Replays the nbuf calls from a CUDA graph so host launch overhead does not pollute short kernels."""
    for i in range(nbuf):
        fn(i)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        keep = [fn(i) for i in range(nbuf)]
    g.replay()
    torch.cuda.synchronize()
    best = 1e9
    for _ in range(5):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        g.replay()
        e1.record()
        torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1) / nbuf)
    del keep, g
    return best * 1e-3


def hbm(name, bytes_, fn, nbuf):
    t = timeit(fn, nbuf)
    rows.append((name, "HBM", f"{bytes_/1e6:.1f} MB", f"{t*1e6:.1f}", f"{bytes_/t/1e9:.0f} GB/s", f"{bytes_/t/1e9/HBM:.2f}"))


def tensor(name, flop, fn, nbuf):
    t = timeit(fn, nbuf)
    rows.append((name, "tensor", f"{flop/1e9:.1f} GFLOP", f"{t*1e6:.1f}", f"{flop/t/1e12:.0f} TFLOP/s", f"{flop/t/1e12/TF:.2f}"))


nb = 4
# K1 Haar (level 0: C = 96)
xs = [torch.randn(1, 96, 512, 512, device=DEV) for _ in range(nb)]
los = [torch.randn(1, 48, 512, 512, device=DEV) for _ in range(nb)]
hbm("haar1d_fwd C=96 (level 0)", 2 * 96 * P * 4, lambda i: ops.haar1d_split(xs[i]), nb)
hbm("haar1d_inv C=96 (level 0, Split^-1 fused)", 2 * 96 * P * 4, lambda i: ops.haar1d_merge(los[i], los[(i + 1) % nb]), nb)
perm_c = torch.randperm(48)
perm_s = torch.randperm(512)
hbm("permute channels ch=48", 8 * 48 * P, lambda i: ops.permute(los[i], perm_c, 1), nb)
hbm("permute rows ch=48", 8 * 48 * P, lambda i: ops.permute(los[i], perm_s, 2), nb)
hbm("permute columns ch=48", 8 * 48 * P, lambda i: ops.permute(los[i], perm_s, 3), nb)
hbm("affine (standalone K3) ch=48", 16 * 48 * P, lambda i: ops.affine(los[i], xs[i][:, :48], xs[i][:, 48:], inverse=True), nb)
hbm("haar2d_down C=96", 2 * 96 * P * 4, lambda i: ops.haar2d_down(xs[i], True, 0.5), nb)
c8s = [tc.to_c8(torch.randn(1, 256, 512, 512, device=DEV)) for _ in range(nb)]
g = torch.ones(256, device=DEV); b = torch.zeros(256, device=DEV)
hbm("c8 BatchNorm stats+apply+maxpool 256ch", int(256 * P * 2 * (1 + 2 + 0.25)), lambda i: tc.batchnorm_c8(c8s[i], g, b, None, None, batch_stats=True, pool=True), nb)
hbm("nchw_to_c8 96ch", 96 * P * 6, lambda i: tc.to_c8(xs[i]), nb)
imgs = [torch.rand(1, 1, 2160, 2160, device=DEV) for _ in range(nb)]
coords = torch.tensor([[300 + 370 * (i // 6), 280 + 330 * (i % 6)] for i in range(29)], dtype=torch.int32, device=DEV)
hbm("extract_views 2160^2 -> 29x512x512 (+normalise)", 29 * P * 8, lambda i: extract_views(imgs[i], coords, [512, 512], 0.1, 1.3), nb)
del xs, los, c8s, imgs
# tensor kernels
def conv_case(cin, cout, k, H, W, bn=None, name=None):
    per = H * W * (tc.pad16(cin) + tc.pad16(cout)) * 2
    n = max(2, min(32, (300 << 20) // per + 1))
    xin = [tc.to_c8(torch.randn(1, cin, H, W, device=DEV)) for _ in range(n)]
    pc = tc.PackedConv(torch.randn(cout, cin, k, k, device=DEV) * 0.05, torch.zeros(cout, device=DEV), bn=bn)
    tensor(name or f"conv_tc {cin}->{cout} {k}x{k} @{H}x{W}", 2.0 * H * W * cin * cout * k * k, lambda i: tc.conv_tc(xin[i], pc, act=ops.ACT_PRELU, slope=torch.tensor([0.2], device=DEV)) if False else tc.conv_tc(xin[i], pc, act=ops.ACT_ELU), n)
conv_case(256, 256, 3, 512, 512)
conv_case(512, 512, 3, 256, 256)
conv_case(1024, 1024, 3, 128, 128)
conv_case(64, 64, 7, 512, 512)
def small_conv_case(cin, cout, k):
    """Small-channel convs of the conditioning nets / mean-volume branch: streaming passes, rated against HBM (operand + output bytes)."""
    per = P * (tc.pad16(cin) + tc.pad16(cout)) * 2
    n_ = max(2, min(32, (300 << 20) // per + 1))
    xin_ = [tc.to_c8(torch.randn(1, cin, 512, 512, device=DEV)) for _ in range(n_)]
    pc_ = tc.PackedConv(torch.randn(cout, cin, k, k, device=DEV) * 0.05, torch.zeros(cout, device=DEV))
    sl_ = torch.tensor([0.2], device=DEV)
    hbm(f"conv_tc {cin}->{cout} {k}x{k} @512x512 (resident weights; C8 bytes in + out)", per, lambda i: tc.conv_tc(xin_[i], pc_, act=ops.ACT_PRELU, slope=sl_), n_)
small_conv_case(29, 48, 3)
small_conv_case(48, 48, 3)
small_conv_case(6, 6, 3)
small_conv_case(6, 6, 7)
n = 8
xin = [tc.to_c8(torch.randn(1, 64, 512, 512, device=DEV)) for _ in range(n)]
p3 = tc.PackedConv(torch.randn(64, 64, 3, 3, device=DEV) * 0.04, torch.zeros(64, device=DEV), bn=64)
p1 = tc.PackedConv(torch.randn(64, 64, 1, 1, device=DEV) * 0.1, torch.zeros(64, device=DEV), bn=64)
tensor("resblock_tc (3x3+ELU+1x1+res+ELU, 64 ch) @512x512", 2.0 * P * 64 * 64 * 10, lambda i: tc.resblock_tc(xin[i], p3, p1), n)
pco = tc.PackedConv(torch.randn(96, 64, 3, 3, device=DEV) * 0.04, torch.zeros(96, device=DEV), bn=96)
xs48 = [torch.randn(1, 48, 512, 512, device=DEV) for _ in range(n)]
ld = torch.zeros(1, device=DEV)
pi = torch.randperm(48).to(torch.int32).to(DEV)
tensor("coupling_tc: last conv + coupling, NCHW state (64->96, ch=48, channel perm; module-API path)", 2.0 * P * 64 * 96 * 9, lambda i: tc.conv_tc_coupling(xin[i], pco, xs48[i], ch=48, inverse=True, perm=pi, perm_axis=1, logdet=ld), n)
tk = torch.zeros(8, device=DEV, dtype=torch.int32)
for ch_ in (48, 24, 12, 6):
    pcf = tc.coupling_weights_f8(torch.randn(2 * ch_, 64, 3, 3, device=DEV) * 0.04, torch.zeros(2 * ch_, device=DEV), ch_, torch.randperm(ch_), False, "bf16")
    xf = [tc.to_f8(torch.randn(1, ch_, 512, 512, device=DEV)) for _ in range(n)]
    rp = torch.randperm(512, device=DEV).to(torch.int32)
    tensor(f"coupling_f8: last conv + coupling, F8 state (64->{2 * tc.ch8(ch_)}, ch={ch_}, row perm; engine path)", 2.0 * P * 64 * 2 * ch_ * 9,
           lambda i: tc.coupling_f8(xin[i], pcf, xf[i], ch=ch_, inverse=True, perm=rp, perm_axis=2, logdet=ld, ticket=tk[:1]), n)
    del xf
x5 = [tc.to_c8(torch.randn(1, 320, 512, 512, device=DEV)) for _ in range(4)]
sets5 = [(tc.PackedConv(torch.randn(64, 64, 3, 3, device=DEV) * 0.04, torch.zeros(64, device=DEV), bn=64),
          tc.PackedConv(torch.randn(64, 64, 1, 1, device=DEV) * 0.1, torch.zeros(64, device=DEV), bn=64)) for _ in range(5)]
tensor("resblock_tc_batched: the block row of 5 sub-network trunks in one launch (5 x 64 ch) @512x512", 5 * 2.0 * P * 64 * 64 * 10, lambda i: tc.resblock_tc_batched(x5[i], sets5), 4)
del x5
lf48 = [tc.to_c8(torch.randn(1, 48, 512, 512, device=DEV)) for _ in range(4)]
ent5 = [tc.PackedEntry(torch.randn(64, 48, 1, 1, device=DEV) * 0.14, torch.randn(64, device=DEV) * 0.1, torch.randn(64, 64, 3, 3, device=DEV) * 0.04, torch.zeros(64, device=DEV), sets5[k][1], "bf16") for k in range(5)]
# algorithmic flops of the pair it replaces (1x1 conv 48 -> 64 + the block); the launch executes fewer: W3' has 48 input channels
tensor("resblock_tc_entry_batched: 1x1 input conv folded into the first block, 5 trunks (48 -> 5 x 64) @512x512",
       5 * 2.0 * P * (48 * 64 + 64 * 64 * 10), lambda i: tc.resblock_tc_entry_batched(lf48[i], ent5), 4)
del lf48
hx = [torch.randn(1, 96, 512, 512, device=DEV) for _ in range(4)]
hbm("haar1d split, detail half in F8 (C=96)", 2 * 96 * P * 4, lambda i: tc.haar1d_split_f8(hx[i]), 4)
lo4 = [torch.randn(1, 48, 512, 512, device=DEV) for _ in range(4)]
hi4 = [tc.to_f8(torch.randn(1, 48, 512, 512, device=DEV)) for _ in range(4)]
hbm("haar1d merge, detail half in F8 (C=96)", 2 * 96 * P * 4, lambda i: tc.haar1d_merge_f8(lo4[i], hi4[i]), 4)
del hx, lo4, hi4

# conditioning-net depth stencil (48 depths): banded 3x3 conv s1 (hidden tensor write), s2 as 1x1 conv to tap partials, col2im
del xin, xs48
D, Cm = 48, 32
w1 = torch.randn(Cm, 3, 3, 3, device=DEV) * 0.2
w2 = torch.randn(Cm, 3, 3, 3, device=DEV) * 0.05
W1 = torch.zeros(D, Cm, D, 3, 3, device=DEV)
W2 = torch.zeros(D, D, Cm, 3, 3, device=DEV)
for kd in range(3):
    for d in range(D):
        dp = d + kd - 1
        if 0 <= dp < D:
            W1[d, :, dp] = w1[:, :, :, kd]
            W2[d, dp] = w2[:, :, :, kd]
s1 = tc.PackedConv(W1.reshape(D * Cm, D, 3, 3), torch.zeros(D * Cm, device=DEV))
s2g = tc.PackedConv(tc.col2im3x3_weights(W2.reshape(D, D * Cm, 3, 3)), None, bn=144)
slope = torch.full((1,), 0.25, device=DEV)
xd = [tc.to_c8(torch.randn(1, D, 512, 512, device=DEV)) for _ in range(4)]
hd = [tc.conv_tc(x, s1, act=ops.ACT_PRELU, slope=slope) for x in xd]
gd = [tc.conv_tc(h, s2g, mb=1) for h in hd[:2]]
bias2 = torch.zeros(48, device=DEV)
hbm("depth stencil s1: banded 3x3 conv 48 -> 1536 ch + PReLU (tcgen05, zero K-steps skipped)", (D + D * Cm) * P * 2, lambda i: tc.conv_tc(xd[i], s1, act=ops.ACT_PRELU, slope=slope), 4)
hbm("depth stencil s2: 1x1 conv 1536 -> 432 tap partials (tcgen05, zero K-blocks skipped)", (D * Cm + 432) * P * 2, lambda i: tc.conv_tc(hd[i], s2g, mb=1), 4)
hbm("depth stencil s2: col2im of the 9 tap partials -> 48 ch", (432 + 48) * P * 2, lambda i: tc.col2im3x3_c8(gd[i % 2], bias2, 48), 4)
# the fused voxel-row kernel that replaces the three rows above in the engine (csrc/stencil_tc.cu)
del hd, gd, s1, s2g, W1, W2
sw = tc.StencilWeights(w1.unsqueeze(1), torch.zeros(Cm, device=DEV), w2.unsqueeze(0), torch.zeros(1, device=DEV), "bf16")
tensor("stencil3d_tc: fused Conv3d(1,32,3) + PReLU + Conv3d(32,1,3), 48 depths (true 3-D flops; MMA-ISSUE-bound, not math-bound: 1.15 M M128 MMAs of N <= 32 at >= 44 cycles each = a ~180 us floor, 0.44 of it)",
       2.0 * 27 * 32 * 2 * D * P, lambda i: tc.stencil3d_tc(xd[i], sw, slope, D), 4)
for Dl in (24, 12, 6):
    xl = [tc.to_c8(torch.randn(1, Dl, 512, 512, device=DEV)) for _ in range(4)]
    tensor(f"stencil3d_tc: {Dl} depths", 2.0 * 27 * 32 * 2 * Dl * P, lambda i: tc.stencil3d_tc(xl[i], sw, slope, Dl), 4)
    del xl

md = ["# Per-kernel roofline (round 2, one B200; CUDA events around a CUDA-graph replay, best of 5, tensors rotated through > L2)", "",
      f"Peaks: HBM {HBM} GB/s, bf16 {TF} TFLOP/s burst (MEASURED_PEAKS.json; kernels timed in isolation).", "",
      "| kernel | bound | algorithmic work | us | achieved | frac of measured peak |", "|---|---|---|---|---|---|"]
md += ["| " + " | ".join(r) + " |" for r in rows]
md += ["", "Notes: the trunk block and the coupling convs issue N <= 96 MMAs.  An SS-mode (both operands from shared memory) M = 128, K = 16",
       "MMA costs ~59 cycles on this chip INDEPENDENT of N <= 64 (measured: `profiles/r02_resblock_experiments.md` -- N sweep 64/32/16,",
       "operand alignment, accumulator-chain experiments all flat), so these kernels have a ceiling of 32/59 = 0.54 of the tensor peak;",
       "batching the five sub-networks of a level into one launch removes most of the per-launch prologue / tail (24 us per block instead",
       "of 28-31).  The banded depth-stencil rows are HBM rows: their tensor work is small once the zero blocks of the banded weights are",
       "skipped, the traffic is the 1536-channel hidden tensor.  The engine now runs the stencil as ONE fused voxel-row kernel",
       "(`stencil3d_tc`: 406 us instead of 571 us at 48 depths); its tensor-roofline fraction is small by construction -- the true 3-D",
       "work is 3456 flop per voxel with K = 9 / 32 and N = 32 / 9, so it is bound by the 44-cycle minimum of an M = 128 MMA and by its",
       "epilogues, not by tensor math or HBM (`profiles/r02_stencil3d_notes.md`).  A clean SS-mode instruction stream measures 48 cycles",
       "per N = 64 MMA (`experiments/ts_mma_probe.cu`); the 55-59 cycles inside the trunk block include its epilogue traffic on the",
       "shared-memory port."]
open(os.path.join(ROOT, "profiles", "r02_kernel_rooflines.md"), "w").write("\n".join(md) + "\n")
print("\n".join(md))
