"""GPU: the training step of a flow level (SURVEY.md 8f-3, BASELINE.json configs[3]).

(a) every adjoint kernel of csrc/backward.cu through cwfa_b200.autograd against torch CPU autograd of the same op,
    on ragged shapes; (b) the whole flow-level loss + gradients against the CPU oracle's autograd AND against the gradients
    of the unmodified reference (tests/golden/train.pt); (c) the Lion kernel against the oracle's restatement; (d) a few
    optimiser steps (loss goes down, run-to-run bit-reproducible).  Tolerances are rel-L2 in fp32 and stated per test.
"""
import math
import os

import pytest
import torch
import torch.nn.functional as F

from conftest import GOLDEN, max_abs, rel_l2
from helpers import build_tiny_model
from oracle import cwfa_oracle as O
from oracle.weights import seeded_randn
from test_training_oracle import check_against_golden, train_inputs

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
TOL = 2e-4        # rel-L2 of fp32 gradients (different summation order than torch's CPU kernels)


@pytest.fixture(scope="module")
def golden_train():
    return torch.load(os.path.join(GOLDEN, "train.pt"), weights_only=False)


@pytest.fixture(autouse=True)
def _restore_shared_prelu():
    """networks._SHARED_PRELU is ONE module-level instance (as in the reference, networks.py:209): put it back after tests
    that load other weights into it or train it."""
    from cwfa_b200 import networks
    w = networks._SHARED_PRELU.weight
    keep = w.detach().cpu().clone()
    yield
    with torch.no_grad():
        w.data = keep.to(w.device)
    w.grad = None
    if hasattr(w, "_cwfa_flat"):
        del w._cwfa_flat


def leaf(t, dev=None):
    t = t.clone().to(dev) if dev else t.clone()
    return t.requires_grad_(True)


# ---------------------------------------------------------------------------------------------
# (a) single ops
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("N,Cin,Cout,H,W,K,act,use_res", [
    (1, 64, 64, 32, 32, 3, "elu", False), (2, 29, 48, 13, 37, 3, "none", False), (1, 64, 96, 40, 24, 3, "none", False),
    (2, 5, 7, 9, 11, 1, "none", False), (1, 64, 64, 17, 33, 1, "elu", True), (1, 6, 64, 64, 64, 1, "none", False),
    (3, 3, 2, 8, 32, 3, "prelu", True), (1, 33, 65, 8, 8, 3, "elu", True)])
def test_conv2d_adjoints(N, Cin, Cout, H, W, K, act, use_res):
    from cwfa_b200 import ops
    x, w, b = seeded_randn((N, Cin, H, W), 1), seeded_randn((Cout, Cin, K, K), 2, 0.2), seeded_randn((Cout,), 3)
    r = seeded_randn((N, Cout, H, W), 4) if use_res else None
    a = torch.tensor([0.25])
    gy = seeded_randn((N, Cout, H, W), 5)
    # CPU autograd reference
    xc, wc, bc, ac = leaf(x), leaf(w), leaf(b), leaf(a)
    rc = leaf(r) if use_res else None
    v = F.conv2d(xc, wc, bc, padding=K // 2)
    if use_res:
        v = v + rc
    yc = {"none": lambda t: t, "elu": F.elu, "prelu": lambda t: F.prelu(t, ac)}[act](v)
    yc.backward(gy)
    # ours
    xg, wg, bg, ag_ = leaf(x, DEV), leaf(w, DEV), leaf(b, DEV), leaf(a, DEV)
    rg = leaf(r, DEV) if use_res else None
    code = {"none": ops.ACT_NONE, "elu": ops.ACT_ELU, "prelu": ops.ACT_PRELU}[act]
    yg = ops.conv2d(xg, wg, bg, act=code, slope=ag_ if act == "prelu" else None, res=rg, res_mode=1 if use_res else 0)
    assert yg.requires_grad and rel_l2(yg, yc) < 1e-5
    yg.backward(gy.to(DEV))
    assert rel_l2(xg.grad, xc.grad) < TOL and rel_l2(wg.grad, wc.grad) < TOL and rel_l2(bg.grad, bc.grad) < TOL
    if use_res:
        assert rel_l2(rg.grad, rc.grad) < TOL
    if act == "prelu":
        assert rel_l2(ag_.grad, ac.grad) < TOL


@pytest.mark.parametrize("inverse", [False, True])
@pytest.mark.parametrize("mode", ["packed", "split_tscale", "x_none"])
def test_affine_adjoint(inverse, mode):
    from cwfa_b200 import ops
    if mode == "x_none" and not inverse:
        pytest.skip("x = None (z = 0) exists in the inverse direction only")
    B, ch, H, W = 2, 6, 9, 20
    x = seeded_randn((B, ch, H, W), 1)
    a = seeded_randn((B, 2 * ch, H, W), 2)
    lowc = seeded_randn((B, 2 * ch, H, W), 3)          # cat(meanvol, LF): the shift is read from its first half
    gy, gj = seeded_randn((B, ch, H, W), 4), seeded_randn((B,), 5)
    ts = -1.0 / math.sqrt(2.0)

    def ref(xt, at, lt):
        if mode == "split_tscale":
            s_raw, t = at[:, :ch], lt[:, :ch] * ts
        else:
            s_raw, t = at[:, :ch], at[:, ch:]
        s = 2.0 * 0.636 * torch.atan(s_raw)
        xx = xt if xt is not None else torch.zeros(B, ch, H, W)
        y = (xx - t) * torch.exp(-s) if inverse else torch.exp(s) * xx + t
        j = s.sum((1, 2, 3)) * (-1.0 if inverse else 1.0)
        return y, j

    xc, ac, lc = (None if mode == "x_none" else leaf(x)), leaf(a), leaf(lowc)
    yc, jc = ref(xc, ac, lc)
    ((yc * gy).sum() + (jc * gj).sum()).backward()

    xg, agd, lg = (None if mode == "x_none" else leaf(x, DEV)), leaf(a, DEV), leaf(lowc, DEV)
    if mode == "split_tscale":
        s_in = agd[:, :ch].contiguous()
        yg, jg = ops.affine(xg, s_in, lg[:, :ch], inverse=inverse, t_scale=ts)
    else:
        yg, jg = ops.affine(xg, agd[:, :ch], agd[:, ch:], inverse=inverse)
    assert rel_l2(yg, yc) < 1e-5 and rel_l2(jg, jc) < 1e-5
    ((yg * gy.to(DEV)).sum() + (jg * gj.to(DEV)).sum()).backward()
    if mode == "split_tscale":
        assert rel_l2(agd.grad[:, :ch], ac.grad[:, :ch]) < TOL and rel_l2(lg.grad, lc.grad) < TOL
    else:
        assert rel_l2(agd.grad, ac.grad) < TOL
    if xg is not None:
        assert rel_l2(xg.grad, xc.grad) < TOL


def test_permute_haar_reductions_adjoints():
    from cwfa_b200 import ops, autograd as ag
    B, C, H, W = 2, 6, 8, 12
    x = seeded_randn((B, C, H, W), 1)
    for axis, n in ((1, C), (2, H), (3, W)):
        perm = torch.randperm(n, generator=torch.Generator().manual_seed(axis))
        gy = seeded_randn((B, C, H, W), 2)
        xc = leaf(x); xc.index_select(axis, perm).backward(gy)
        xg = leaf(x, DEV); ops.permute(xg, perm.to(DEV), axis).backward(gy.to(DEV))
        assert max_abs(xg.grad, xc.grad) == 0.0
    # Haar: all four entry points against the oracle's differentiable restatement
    gy = seeded_randn((B, C, H, W), 3)
    for rev in (False, True):
        xc = leaf(x); O.haar1d(xc, rev=rev)[0].backward(gy)
        xg = leaf(x, DEV); (ops.haar1d_inverse(xg) if rev else ops.haar1d_forward(xg)).backward(gy.to(DEV))
        assert max_abs(xg.grad, xc.grad) < 1e-6
    xg = leaf(x, DEV)
    lo, hi = ops.haar1d_split(xg)
    (lo * gy[:, :3].to(DEV)).sum().backward()                     # only ONE of the two outputs is used
    xc = leaf(x); (O.haar1d(xc)[0][:, :3] * gy[:, :3]).sum().backward()
    assert max_abs(xg.grad, xc.grad) < 1e-6
    lo_g, hi_g = leaf(x[:, :3], DEV), leaf(x[:, 3:], DEV)
    ops.haar1d_merge(lo_g, hi_g).backward(gy.to(DEV))
    lo_c, hi_c = leaf(x[:, :3]), leaf(x[:, 3:])
    O.haar1d(torch.cat((lo_c, hi_c), 1), rev=True)[0].backward(gy)
    assert max_abs(lo_g.grad, lo_c.grad) < 1e-6 and max_abs(hi_g.grad, hi_c.grad) < 1e-6
    # sum of squares and MSE
    gs = seeded_randn((B,), 4)
    xc = leaf(x); (xc.square().sum((1, 2, 3)) * gs).sum().backward()
    xg = leaf(x, DEV); (ops.sum_squares(xg) * gs.to(DEV)).sum().backward()
    assert rel_l2(xg.grad, xc.grad) < 1e-6
    y = seeded_randn((B, C, H, W), 5)
    xc = leaf(x); lc = F.mse_loss(y, xc); (3.0 * lc).backward()
    xg = leaf(x, DEV); lg = ag.mse_loss(y.to(DEV), xg); (3.0 * lg).backward()
    assert abs(float(lg) - float(lc)) < 1e-5 * float(lc) and rel_l2(xg.grad, xc.grad) < 1e-5


@pytest.mark.parametrize("B,D,H,W,Cm", [(1, 8, 12, 16, 32), (2, 3, 5, 7, 4), (1, 1, 4, 4, 2)])
def test_depth_stencil_adjoint(B, D, H, W, Cm):
    from cwfa_b200 import ops
    x = seeded_randn((B, D, H, W), 1)
    w1, b1 = seeded_randn((Cm, 1, 3, 3, 3), 2, 0.3), seeded_randn((Cm,), 3)
    w2, b2 = seeded_randn((1, Cm, 3, 3, 3), 4, 0.3), seeded_randn((1,), 5)
    a = torch.tensor([0.25])
    gy = seeded_randn((B, D, H, W), 6)
    cl = [leaf(t) for t in (x, w1, b1, a, w2, b2)]
    v = cl[0].permute(0, 2, 3, 1).unsqueeze(1)                    # networks.py:236-241
    v = F.conv3d(F.prelu(F.conv3d(v, cl[1], cl[2], padding=1), cl[3]), cl[4], cl[5], padding=1)
    yc = v[:, 0].permute(0, 3, 1, 2)
    yc.backward(gy)
    gl = [leaf(t, DEV) for t in (x, w1, b1, a, w2, b2)]
    yg = ops.depth_stencil3d(*gl)
    assert rel_l2(yg, yc) < 1e-5
    with torch.no_grad():                                         # the unfused training forward == the fused inference kernel
        assert rel_l2(ops.depth_stencil3d(*[t.detach() for t in gl]), yc) < 1e-5
    yg.backward(gy.to(DEV))
    for g, c, name in zip(gl, cl, ("x", "w1", "b1", "slope", "w2", "b2")):
        assert rel_l2(g.grad, c.grad) < TOL, name


def test_lion_kernel_vs_oracle():
    from cwfa_b200.training import Lion
    torch.manual_seed(0)
    ps = [torch.nn.Parameter(seeded_randn(s, 10 + i).to(DEV)) for i, s in enumerate([(7, 3, 3, 3), (5,), (1,), (64, 64)])]
    opt = Lion([{"params": ps[:2], "lr": 1e-2, "weight_decay": 1e-2}, {"params": ps[2:]}], lr=3e-3, betas=(0.9, 0.99))
    ref_p = [p.detach().cpu().clone() for p in ps]
    ref_m = [torch.zeros_like(p) for p in ref_p]
    hyp = [(1e-2, 1e-2), (1e-2, 1e-2), (3e-3, 0.0), (3e-3, 0.0)]
    for it in range(3):
        opt.zero_grad()
        gs = [seeded_randn(tuple(p.shape), 100 * it + i) for i, p in enumerate(ps)]
        gs[3][0, :8] = 0.0                                        # sign(0) = 0 on the first step
        for p, g in zip(ps, gs):
            p.grad.copy_(g.to(DEV))
        opt.mark_all_used()                                   # gradients written by hand into the flat views
        opt.step()
        for i in range(4):
            ref_p[i], ref_m[i] = O.lion_step(ref_p[i], gs[i], ref_m[i], hyp[i][0], 0.9, 0.99, hyp[i][1])
    for p, r in zip(ps, ref_p):
        assert max_abs(p, r) < 1e-6


# ---------------------------------------------------------------------------------------------
# (b) whole flow level: loss and all gradients vs the oracle and vs the reference's own autograd
# ---------------------------------------------------------------------------------------------
def _our_level_grads(model, n, inputs, w):
    from cwfa_b200.training import flow_level_loss
    for p in model.parameters():
        p.grad = None
    gt, views, mean_vol, vol_in = (t.to(DEV) for t in inputs)
    loss, parts = flow_level_loss(model, n, gt, views, mean_vol, vol_in, cond_weight=w)
    loss.backward()
    gi = {k: p.grad for k, p in model.conv_inn[n].named_parameters() if p.requires_grad and p.grad is not None}
    gc = {k: p.grad for k, p in model.cond_nets[n].named_parameters() if p.grad is not None}
    return loss, parts, gi, gc


@pytest.mark.parametrize("n", [0, 1])
def test_flow_level_gradients_vs_oracle_and_reference(golden_tiny, golden_train, n):
    lv = build_tiny_model(golden_tiny).export_for_oracle()["levels"][n]    # CPU copies first: the PReLU instance is shared
    model = build_tiny_model(golden_tiny, DEV)
    w = golden_train["config"]["cond_weight"]
    inputs = train_inputs(golden_train, n)
    loss, parts, gi, gc = _our_level_grads(model, n, inputs, w)
    g = golden_train[f"level{n}"]
    assert abs(float(loss) - float(g["loss"])) < 1e-4 * abs(float(g["loss"]))
    assert abs(float(parts["mse"]) - float(g["mse"])) < 1e-4 * abs(float(g["mse"]))
    assert abs(float(parts["nll"]) - float(g["nll"])) < 1e-4 * abs(float(g["nll"]))
    # vs the reference's own gradients (norm / probe / small tensors in full)
    check_against_golden({k: v.cpu() for k, v in gi.items()}, g["inn"], 5e-4)
    check_against_golden({k: v.cpu() for k, v in gc.items()}, g["cond"], 5e-4)
    # vs the pinned oracle: every gradient tensor in full
    r = O.level_train_grads(lv["inn"], lv["cond"], lv["spec"], *inputs, w)
    worst = ("", 0.0)
    for k, v in gi.items():
        e = rel_l2(v, r["inn"][k]); worst = max(worst, (k, e), key=lambda t: t[1])
    for k, v in gc.items():
        e = rel_l2(v, r["cond"][k]); worst = max(worst, (k, e), key=lambda t: t[1])
    print(f"level {n}: loss {float(loss):.6f} (ref {float(g['loss']):.6f}); worst gradient rel-L2 {worst[1]:.2e} at {worst[0]}")
    assert worst[1] < 5e-4, worst
    # parameters the reference never touches get no gradient here either
    for k in g["no_grad_keys"]:
        p = dict(model.conv_inn[n].named_parameters()).get(k)
        assert p is None or p.grad is None or float(p.grad.abs().max()) == 0.0, k


def test_flow_level_gradients_mid_size_vs_oracle():
    """Level 0 of a D=96 model on 96x80 frames (ragged tiles, ch = 48 as in the full config), batch 1."""
    import cwfa_b200
    from oracle.weights import deterministic_fill
    import numpy as np
    np.random.seed(3); torch.manual_seed(3)
    m = cwfa_b200.CWFAModel(n_depths=96, volume_side_size=80, INN_max_down_steps=2)
    m.conv_inn[0].load_state_dict({**deterministic_fill(m.conv_inn[0].state_dict(), 7),
                                   **{k: v for k, v in m.conv_inn[0].state_dict().items() if "perm" in k}})
    m.cond_nets[0].load_state_dict(deterministic_fill(m.cond_nets[0].state_dict(), 8))
    lv = m.export_for_oracle()["levels"][0]
    m = m.to(DEV)
    S = 80
    inputs = (seeded_randn((1, 96, S, S), 1), seeded_randn((1, 29, S, S), 2), seeded_randn((1, 48, S, S), 3, 0.1),
              seeded_randn((1, 48, S, S), 4))
    loss, parts, gi, gc = _our_level_grads(m, 0, inputs, 0.40984)
    r = O.level_train_grads(lv["inn"], lv["cond"], lv["spec"], *inputs, 0.40984)
    assert abs(float(loss) - float(r["loss"])) < 1e-4 * abs(float(r["loss"]))
    errs = {k: rel_l2(v, r["inn"][k]) for k, v in gi.items()}
    errs.update({"cond." + k: rel_l2(v, r["cond"][k]) for k, v in gc.items()})
    k = max(errs, key=errs.get)
    print(f"mid-size level 0: loss {float(loss):.5f}, worst gradient rel-L2 {errs[k]:.2e} at {k}")
    assert errs[k] < 1e-3, (k, errs[k])


@pytest.mark.parametrize("kind,tol_all,tol_each", [("bf16", 3e-2, 1.5e-1), ("fp16", 4e-3, 2e-2)])
def test_flow_level_gradients_tensor_core_path(golden_tiny, golden_train, kind, tol_all, tol_each):
    """Training precision 'bf16' / 'fp16': every convolution of the step (forward and data gradient) runs on the tcgen05
    kernel with half-precision operands and fp32 accumulation; weight gradients, couplings, log-dets stay fp32.
    Tolerance vs the fp32 oracle: rel-L2 over ALL gradients <= tol_all, every tensor <= tol_each (stated; printed)."""
    from cwfa_b200 import _lib, autograd as ag
    n = 1
    lv = build_tiny_model(golden_tiny).export_for_oracle()["levels"][n]
    model = build_tiny_model(golden_tiny, DEV)
    w = golden_train["config"]["cond_weight"]
    inputs = train_inputs(golden_train, n)
    prev = ag.set_training_precision(kind)
    before = dict(_lib.launch_hist)
    try:
        loss, parts, gi, gc = _our_level_grads(model, n, inputs, w)
    finally:
        ag.set_training_precision(prev)
    assert _lib.launch_hist.get("cwfa_conv_tc", 0) - before.get("cwfa_conv_tc", 0) >= 80       # fwd + dgrad convs on tensor cores
    r = O.level_train_grads(lv["inn"], lv["cond"], lv["spec"], *inputs, w)
    num = den = 0.0
    worst = ("", 0.0)
    for ours, ref in ((gi, r["inn"]), (gc, r["cond"])):
        for k, v in ours.items():
            d = (v.double().cpu() - ref[k].double()).norm().item()
            b = ref[k].double().norm().item()
            num, den = num + d * d, den + b * b
            if b > 0 and d / b > worst[1]:
                worst = (k, d / b)
    total = (num / den) ** 0.5
    print(f"{kind}: loss {float(loss):.5f} (fp32 oracle {float(r['loss']):.5f}); gradients rel-L2 all {total:.2e}, worst {worst[1]:.2e} at {worst[0]}")
    assert abs(float(loss) - float(r["loss"])) < 2e-2 * abs(float(r["loss"]))
    assert total < tol_all and worst[1] < tol_each, (total, worst)


# ---------------------------------------------------------------------------------------------
# (d) optimiser steps
# ---------------------------------------------------------------------------------------------
def test_training_steps_reduce_loss_and_are_reproducible(golden_tiny, golden_train):
    from cwfa_b200.training import FlowLevelTrainer
    inputs = [t.to(DEV) for t in train_inputs(golden_train, 1)]
    runs = []
    for _ in range(2):
        model = build_tiny_model(golden_tiny, DEV)
        tr = FlowLevelTrainer(model, 1, lr=2e-4, lr_cond=2e-4)
        unused0 = model.conv_inn[1].module_list[2].subnet.block_grad_up.weight.detach().clone()
        losses = [float(tr.step(*inputs)["loss"]) for _ in range(5)]
        # parameters that never receive a gradient (kept for checkpoint compatibility) are skipped, as lion_pytorch does (no decay)
        assert torch.equal(unused0, model.conv_inn[1].module_list[2].subnet.block_grad_up.weight.detach())
        runs.append((losses, torch.cat([p.detach().reshape(-1) for p in model.conv_inn[1].parameters() if p.requires_grad]).clone()))
        assert tr.collectives == 0
    print("losses", runs[0][0])
    assert runs[0][0][-1] < runs[0][0][0]
    assert runs[0][0] == runs[1][0] and torch.equal(runs[0][1], runs[1][1])      # deterministic reductions everywhere


def test_coarse_to_fine_schedule_and_ood_rule(golden_tiny):
    """The reference's fine-tune schedule over the flow levels (coarsest first, per-frame cache handed down) on two tiny
    frames, then the OOD rule on forward-NLL scores."""
    from cwfa_b200.training import fine_tune_flow_levels, ood_decision
    model = build_tiny_model(golden_tiny, DEV)
    cfg = golden_tiny["config"]
    D, S, L = cfg["D"], cfg["S"], cfg["MAX"]
    frames = []
    for i in range(2):
        mv = [seeded_randn((1, D // 2 ** (n + 1), S, S), 70 + 10 * i + n, 0.1).to(DEV) for n in range(L - 1)]
        frames.append(dict(views=seeded_randn((1, 29, S, S), 60 + i).to(DEV), gt=seeded_randn((1, D, S, S), 50 + i).to(DEV), mean_vols=mv))
    before = model.reconstruct(frames[0]["views"], frames[0]["mean_vols"]).clone()
    hist, cache = fine_tune_flow_levels(model, frames, levels=[2, 1, 0], epochs_per_step=2, lr=1e-4, lr_cond=1e-4, lr_first_step=1e-4)
    assert sorted(hist) == [0, 1, 2] and all(len(v) == 4 for v in hist.values())          # LRNN step first, then the flow levels
    assert hist[2][-2] < hist[2][0]
    assert all(math.isfinite(x) for v in hist.values() for x in v)
    assert hist[1][-2] < hist[1][0] and hist[0][-2] < hist[0][0]              # same frame, one epoch later
    assert cache[0].shape == (1, D, S, S)
    after = model.reconstruct(frames[0]["views"], frames[0]["mean_vols"])
    # the cache is the fine-tuned reconstruction; not bit-equal to a fresh one because the conditioning nets of ALL levels share
    # ONE PReLU instance (networks.py:209), which kept training while level 0 was optimised
    assert rel_l2(cache[0], after) < 2e-2 and max_abs(after, before) > 1e-4
    res = model.forward_nll(torch.cat([f["gt"] for f in frames]), torch.cat([f["views"] for f in frames]),
                            [torch.cat([f["mean_vols"][n] for f in frames]) for n in range(L - 1)])
    nll = [r["nll_per_sample"] for r in res]
    flags = ood_decision(nll, 0, -1.33)
    assert flags.shape == (2,) and flags.dtype == torch.bool
    assert torch.equal(flags.cpu(), (-nll[0] < -1.33).cpu())


def test_full_size_training_step_properties():
    """BASELINE.json configs[3] at FULL size (level 0: 96 -> 48+48 channels, 512x512, batch 1), size-independent properties:
    (1) directional derivative: (loss(theta + eps d) - loss(theta - eps d)) / (2 eps) = <grad, d> with d = grad / |grad|, the
        two losses evaluated under no_grad, i.e. through the FUSED inference kernels (tolerance 3 %);
    (2) the tensor-core (bf16) step -- conv_tc forward / data gradient, wgrad_tc incl. the 1536-channel banded stencil shapes --
        against the fp32 step on the same weights: all-gradient rel-L2 <= 3e-2, cosine >= 0.999."""
    import cwfa_b200
    from cwfa_b200 import autograd as ag
    from cwfa_b200.training import flow_level_loss
    model = cwfa_b200.CWFAModel(n_depths=96, volume_side_size=512, INN_max_down_steps=2, seed=0).to(DEV)
    S = 512
    gt, views = seeded_randn((1, 96, S, S), 1).to(DEV), seeded_randn((1, 29, S, S), 2).to(DEV)
    mv, vin = seeded_randn((1, 48, S, S), 3, 0.1).to(DEV), seeded_randn((1, 48, S, S), 4).to(DEV)
    params = [p for p in list(model.conv_inn[0].parameters()) + list(model.cond_nets[0].parameters()) if p.requires_grad]

    def grads(kind):
        for p in params:
            p.grad = None
        prev = ag.set_training_precision(kind)
        try:
            loss, _ = flow_level_loss(model, 0, gt, views, mv, vin)
            loss.backward()
        finally:
            ag.set_training_precision(prev)
        return float(loss), [None if p.grad is None else p.grad.detach().clone() for p in params]

    loss0, g32 = grads("fp32")
    used = [i for i, g in enumerate(g32) if g is not None]
    gnorm = math.sqrt(sum(float(g32[i].double().pow(2).sum()) for i in used))
    assert gnorm > 0 and math.isfinite(loss0)
    ratios = []
    for target in (2e-3, 5e-4):                               # intended loss change across the symmetric difference
        eps = 0.5 * target / gnorm
        vals = []
        with torch.no_grad():
            for sign in (+1.0, -1.0):
                for i in used:
                    params[i].add_(g32[i], alpha=sign * eps / gnorm)
                vals.append(float(flow_level_loss(model, 0, gt, views, mv, vin)[0]))
                for i in used:
                    params[i].sub_(g32[i], alpha=sign * eps / gnorm)
        ratios.append((vals[0] - vals[1]) / (2 * eps) / gnorm)
    print(f"full-size level 0: loss {loss0:.6f}, |grad| {gnorm:.4e}, finite difference / <grad, d> = {ratios}")
    assert min(abs(r - 1.0) for r in ratios) < 3e-2, ratios
    loss16, g16 = grads("bf16")
    num = sum(float((g16[i].double() - g32[i].double()).pow(2).sum()) for i in used)
    dot = sum(float((g16[i].double() * g32[i].double()).sum()) for i in used)
    n16 = math.sqrt(sum(float(g16[i].double().pow(2).sum()) for i in used))
    print(f"bf16 vs fp32 at full size: loss {loss16:.6f} vs {loss0:.6f}; gradient rel-L2 {math.sqrt(num) / gnorm:.2e}, cosine {dot / (gnorm * n16):.5f}")
    assert abs(loss16 - loss0) < 2e-2 * abs(loss0)
    assert math.sqrt(num) / gnorm < 3e-2 and dot / (gnorm * n16) > 0.999


# ---------------------------------------------------------------------------------------------
# LRNN step: U-Net adjoints (BatchNorm, max-pool, transposed conv as 1x1 conv + pixel shuffle)
# ---------------------------------------------------------------------------------------------
def test_unet_ops_adjoints():
    from cwfa_b200 import ops
    N, C, H, W = 2, 5, 12, 20
    x, gy = seeded_randn((N, C, H, W), 1), seeded_randn((N, C, H, W), 2)
    gam, bet = seeded_randn((C,), 3) * 0.3 + 1.0, seeded_randn((C,), 4)
    rm, rv = seeded_randn((C,), 5) * 0.1, seeded_randn((C,), 6).abs() + 0.5
    for batch_stats in (True, False):
        xc, gc, bc = leaf(x), leaf(gam), leaf(bet)
        F.batch_norm(xc, None if batch_stats else rm, None if batch_stats else rv, gc, bc, training=batch_stats, eps=1e-5).backward(gy)
        xg, gg, bg = leaf(x, DEV), leaf(gam, DEV), leaf(bet, DEV)
        y = ops.batchnorm(xg, gg, bg, rm.to(DEV), rv.to(DEV), batch_stats=batch_stats, eps=1e-5)
        y.backward(gy.to(DEV))
        assert rel_l2(xg.grad, xc.grad) < TOL and rel_l2(gg.grad, gc.grad) < TOL and rel_l2(bg.grad, bc.grad) < TOL
    # max-pool incl. ties (torch routes the gradient to the first maximum in scan order)
    xt = x.clone(); xt[:, :, ::4, ::4] = xt[:, :, 1::4, 1::4]; xt[0, 0, :2, :2] = 7.0
    g2 = seeded_randn((N, C, H // 2, W // 2), 7)
    xc = leaf(xt); F.max_pool2d(xc, 2).backward(g2)
    xg = leaf(xt, DEV); ops.maxpool2(xg).backward(g2.to(DEV))
    assert max_abs(xg.grad, xc.grad) == 0.0
    # transposed conv + skip
    Cin, Cout = 6, 4
    xi, w, b = seeded_randn((N, Cin, H, W), 8), seeded_randn((Cin, Cout, 2, 2), 9, 0.3), seeded_randn((Cout,), 10)
    sk, g3 = seeded_randn((N, Cout, 2 * H, 2 * W), 11), seeded_randn((N, Cout, 2 * H, 2 * W), 12)
    cl = [leaf(t) for t in (xi, w, b, sk)]
    yc = F.conv_transpose2d(cl[0], cl[1], cl[2], stride=2) + cl[3]
    yc.backward(g3)
    gl = [leaf(t, DEV) for t in (xi, w, b, sk)]
    yg = ops.conv_transpose2x2(*gl)
    assert rel_l2(yg, yc) < 1e-5
    yg.backward(g3.to(DEV))
    for a_, c_ in zip(gl, cl):
        assert rel_l2(a_.grad, c_.grad) < TOL


def test_grad_scaler_matches_torch_semantics_and_skips_overflowed_steps(golden_tiny, golden_train):
    """``GradScaler(init_scale=4)`` as the reference drives it (CWFA.py:613,1005-1015): (a) scale trajectory equals
    torch.amp.GradScaler's for the same good / overflowed step pattern; (b) a power-of-two loss scale is exact in fp32, so a
    scaled fp32 run is bit-identical to an unscaled one; (c) an overflowed gradient skips the step and halves the scale."""
    from cwfa_b200.training import FlowLevelTrainer, GradScaler
    # (a) trajectory vs torch
    ref = torch.amp.GradScaler("cuda", init_scale=4.0, growth_interval=3)
    ours = GradScaler(init_scale=4.0, growth_interval=3)
    w = torch.nn.Parameter(torch.ones(4, device=DEV))
    opt = torch.optim.SGD([w], lr=0.0)
    for bad in (False, False, True, False, False, False, True, True, False):
        ref.scale(torch.ones((), device=DEV))                      # torch initialises its scale tensor lazily in scale()
        w.grad = torch.full((4,), float("inf") if bad else 1.0, device=DEV)
        ref.step(opt)
        ref.update()
        ours._found_inf = bad
        ours.update()
        assert ours.get_scale() == ref.get_scale(), (ours.get_scale(), ref.get_scale())
    # (b) exactness of a power-of-two scale in fp32
    inputs = [t.to(DEV) for t in train_inputs(golden_train, 1)]
    runs = []
    for scaler in (None, GradScaler(init_scale=4.0)):
        model = build_tiny_model(golden_tiny, DEV)
        tr = FlowLevelTrainer(model, 1, lr=2e-4, lr_cond=2e-4, grad_scaler=scaler)
        for _ in range(3):
            tr.step(*inputs)
        runs.append(torch.cat([p.detach().reshape(-1) for p in model.conv_inn[1].parameters() if p.requires_grad]).clone())
        tr.release()
    assert torch.equal(runs[0], runs[1])
    # (c) overflow -> skipped step, scale halves, later steps resume
    model = build_tiny_model(golden_tiny, DEV)
    tr = FlowLevelTrainer(model, 1, lr=2e-4, lr_cond=2e-4, precision="fp16")
    assert tr.scaler is not None and tr.scaler.get_scale() == 4.0          # on by default for the reference's fp16 arithmetic
    before = torch.cat([p.detach().reshape(-1) for p in model.conv_inn[1].parameters() if p.requires_grad]).clone()
    tr.scaler.update(new_scale=2.0 ** 120)                                  # forces an overflow of the scaled loss / gradients
    tr.step(*inputs)
    after = torch.cat([p.detach().reshape(-1) for p in model.conv_inn[1].parameters() if p.requires_grad])
    assert torch.equal(before, after) and tr.scaler.get_scale() == 2.0 ** 119 and tr.scaler.skipped_steps == 1
    tr.scaler.update(new_scale=4.0)
    parts = tr.step(*inputs)
    after2 = torch.cat([p.detach().reshape(-1) for p in model.conv_inn[1].parameters() if p.requires_grad])
    assert not torch.equal(before, after2) and parts["loss_scale"] == 4.0 and torch.isfinite(after2).all()
    tr.release()


def test_zero_grad_set_to_none_between_steps(golden_tiny, golden_train):
    """``model.zero_grad()`` (set_to_none=True is torch's default) drops the ``.grad`` views of the flat buffer; the next
    backward then allocates fresh gradient tensors.  The optimiser must pick those up (and re-home them) instead of crashing or
    stepping on zeros: the run must equal one that never called ``model.zero_grad()``, bit for bit."""
    from cwfa_b200.training import FlowLevelTrainer
    inputs = [t.to(DEV) for t in train_inputs(golden_train, 1)]
    runs = []
    for foreign_zero in (False, True):
        model = build_tiny_model(golden_tiny, DEV)
        tr = FlowLevelTrainer(model, 1, lr=2e-4, lr_cond=2e-4)
        losses = []
        for _ in range(3):
            if foreign_zero:
                model.zero_grad()                                   # sets every p.grad to None
                assert model.conv_inn[1].module_list[2].subnet.block2[0].weight.grad is None
            losses.append(float(tr.step(*inputs)["loss"]))
        runs.append((losses, torch.cat([p.detach().reshape(-1) for p in model.conv_inn[1].parameters() if p.requires_grad]).clone()))
        tr.release()
    assert runs[0][0] == runs[1][0] and torch.equal(runs[0][1], runs[1][1])


def _grad_errors(ours, ref):
    """(total rel-L2 over all tensors, {key: rel-L2}, |g|-weighted fraction of entries whose SIGN agrees -- the only thing the
    Lion update consumes at the first step: sign(b1 m + (1 - b1) g) with m = 0)."""
    num = den = agree = weight = 0.0
    per = {}
    for k, r in ref.items():
        v, r = ours[k].double().cpu(), r.double()
        d, b_ = (v - r).norm().item(), r.norm().item()
        num, den = num + d * d, den + b_ * b_
        per[k] = d / b_ if b_ > 0 else 0.0
        w = r.abs()
        agree += float((w * (torch.sign(v) == torch.sign(r))).sum())
        weight += float(w.sum())
    return (num / den) ** 0.5, per, agree / weight


@pytest.mark.parametrize("kind", ["fp32", "fp16", "bf16"])
def test_lrnn_step_gradients_vs_oracle_and_reference(golden_tiny, golden_train, kind):
    """Reference for the comparison: the oracle evaluated in float64.  The U-Net gradient is ill-conditioned (max-pool arg-max
    and PReLU kinks flip on tiny perturbations of the activations; BatchNorm over 512 samples at the deepest level): the
    oracle's OWN fp32 run differs from its fp64 run by 1.4e-3 rel-L2 over all gradients (worst tensor 8.4e-3), which sets the
    fp32 tolerances (5e-3 / 5e-2).  For the half-precision modes the yardstick is computed, not assumed: the float64 oracle is
    re-run with every convolution operand (input, weight, output cotangent) rounded to fp16 / bf16 (tests/helpers.py:
    half_operand_emulation) -- the error the ARITHMETIC TYPE causes on this network (fp16 4.6e-2 total, bf16 1.31e-1 on the
    deterministic-fill fixture, a worst case; measured on the B200: kernels 4.8e-2 / 1.32e-1, i.e. the kernels add nothing
    beyond the operand rounding).  The tensor-core kernels must stay within 2x of that in total, within 4x per non-scalar
    tensor (floor: the emulation's total), and agree with float64 on the gradient SIGNS -- all Lion consumes -- as often as
    the emulation does (minus 2 %; measured 0.9993 / 0.9947 for both)."""
    from cwfa_b200 import autograd as ag
    from cwfa_b200.training import lrnn_loss
    cfg, g = golden_train["config"], golden_train["lrnn"]
    D, S, B, MAX = cfg["D"], cfg["S"], cfg["B"], cfg["MAX"]
    views = seeded_randn((B, 29, S, S), g["seeds"]["views"])
    gt = seeded_randn((B, D // 2 ** (MAX - 1), S, S), g["seeds"]["gt"])
    om = build_tiny_model(golden_tiny).export_for_oracle()
    model = build_tiny_model(golden_tiny, DEV)
    for p in model.parameters():
        p.grad = None
    prev = ag.set_training_precision(kind)
    try:
        loss, _ = lrnn_loss(model, gt.to(DEV), views.to(DEV))
        loss.backward()
    finally:
        ag.set_training_precision(prev)
    ours = {k: p.grad for k, p in model.cond_nets[-1].named_parameters() if p.grad is not None}
    sd64 = {k: (v.double() if v.dtype.is_floating_point else v) for k, v in om["lrnn"].items()}
    r = O.lrnn_train_grads(sd64, views.double(), gt.double())
    assert set(ours) == set(r["grads"]) == set(g["grads"])
    total, per, signs = _grad_errors(ours, r["grads"])
    worst = max(per.items(), key=lambda kv: kv[1])
    probe_keys = ["net.deconv.1.last.0.weight", "net.deconv.1.up_path.1.conv_block.block.3.weight", "net.deconv.1.up_path.1.up.weight",
                  "net.deconv.1.down_path.2.block.0.weight", "net.deconv.1.down_path.0.block.0.weight", "net.deconv.0.weight"]
    print({k.replace("net.deconv.", ""): f"{per[k]:.1e}" for k in probe_keys})
    print(f"LRNN step {kind}: loss {float(loss):.6f} (reference {float(g['loss']):.6f}); gradients vs float64 oracle: rel-L2 all {total:.2e}, "
          f"worst {worst[1]:.2e} at {worst[0]}, |g|-weighted sign agreement {signs:.4f}")
    assert per["net.deconv.1.last.0.weight"] < (1e-4 if kind == "fp32" else 3e-2)
    assert abs(float(loss) - float(g["loss"])) < (1e-4 if kind == "fp32" else 2e-2) * abs(float(g["loss"]))
    if kind == "fp32":
        assert total < 5e-3 and worst[1] < 5e-2 and signs > 0.999, (total, worst, signs)
        check_against_golden({k: v.cpu() for k, v in ours.items()}, g["grads"], 5e-2)
        return
    from helpers import half_operand_emulation
    with half_operand_emulation(kind):
        emu = O.lrnn_train_grads(sd64, views.double(), gt.double())
    e_total, e_per, e_signs = _grad_errors(emu["grads"], r["grads"])
    print(f"  float64 oracle with {kind}-rounded conv operands: rel-L2 all {e_total:.2e}, worst {max(e_per.values()):.2e}, sign agreement {e_signs:.4f}")
    assert total < 2.0 * e_total, (total, e_total)
    # (scalar tensors -- the PReLU slopes -- are sums over whole feature maps with heavy cancellation: emulation and kernels both
    #  show O(1) relative scatter on them; they are covered by the total and the sign agreement)
    bad = {k: (v, e_per[k]) for k, v in per.items() if ours[k].numel() > 1 and v > 4.0 * max(e_per[k], e_total)}
    assert not bad, bad
    assert signs > e_signs - 0.02, (signs, e_signs)


def test_lrnn_trainer_reduces_loss(golden_tiny, golden_train):
    from cwfa_b200.training import LRNNTrainer
    cfg, g = golden_train["config"], golden_train["lrnn"]
    D, S, B, MAX = cfg["D"], cfg["S"], cfg["B"], cfg["MAX"]
    views = seeded_randn((B, 29, S, S), g["seeds"]["views"]).to(DEV)
    gt = seeded_randn((B, D // 2 ** (MAX - 1), S, S), g["seeds"]["gt"]).to(DEV)
    model = build_tiny_model(golden_tiny, DEV)
    tr = LRNNTrainer(model, lr=1e-4)
    losses = [float(tr.step(gt, views)["loss"]) for _ in range(4)]
    print("LRNN losses", losses)
    assert losses[-1] < losses[0]


# ---------------------------------------------------------------------------------------------
# LRNN mean-volume branch: ConvNeXt (7x7 conv, LayerNorm([C,H,W]), GELU + skip) and the attention gate
# ---------------------------------------------------------------------------------------------
def test_mean_volume_branch_ops_adjoints():
    from cwfa_b200 import ops, autograd as ag
    # 7x7 convolution (fp32 weight gradient kernel, 16x16 channel blocks), ragged channels / tiles
    for (N, Cin, Cout, H, W) in ((1, 20, 18, 13, 37), (2, 6, 64, 16, 32)):
        x, w, b = seeded_randn((N, Cin, H, W), 1), seeded_randn((Cout, Cin, 7, 7), 2, 0.05), seeded_randn((Cout,), 3)
        gy = seeded_randn((N, Cout, H, W), 4)
        cl = [leaf(t) for t in (x, w, b)]
        F.conv2d(cl[0], cl[1], cl[2], padding=3).backward(gy)
        gl = [leaf(t, DEV) for t in (x, w, b)]
        ops.conv2d(*gl).backward(gy.to(DEV))
        for a_, c_ in zip(gl, cl):
            assert rel_l2(a_.grad, c_.grad) < TOL
    # gelu(conv1x1) + skip
    N, C, H, W = 2, 7, 9, 20
    x, w, b, r = seeded_randn((N, C, H, W), 5), seeded_randn((C, C, 1, 1), 6, 0.5), seeded_randn((C,), 7), seeded_randn((N, C, H, W), 8)
    gy = seeded_randn((N, C, H, W), 9)
    cl = [leaf(t) for t in (x, w, b, r)]
    yc = F.gelu(F.conv2d(cl[0], cl[1], cl[2])) + cl[3]
    yc.backward(gy)
    gl = [leaf(t, DEV) for t in (x, w, b, r)]
    yg = ops.conv2d(gl[0], gl[1], gl[2], act=ops.ACT_GELU, res=gl[3], res_mode=2)
    assert rel_l2(yg, yc) < 1e-5
    yg.backward(gy.to(DEV))
    for a_, c_ in zip(gl, cl):
        assert rel_l2(a_.grad, c_.grad) < TOL
    # LayerNorm([C,H,W]) with element-wise affine
    gam, bet = seeded_randn((C, H, W), 10) * 0.3 + 1.0, seeded_randn((C, H, W), 11)
    cl = [leaf(t) for t in (x * 1.5 + 0.3, gam, bet)]
    F.layer_norm(cl[0], (C, H, W), cl[1], cl[2], 1e-5).backward(gy)
    gl = [leaf(t, DEV) for t in (x * 1.5 + 0.3, gam, bet)]
    ops.layernorm_chw(gl[0], gl[1], gl[2], 1e-5).backward(gy.to(DEV))
    for a_, c_ in zip(gl, cl):
        assert rel_l2(a_.grad, c_.grad) < TOL
    # Conv1d over the flattened H*W axis with ReLU / sigmoid, then the gate
    L = H * W
    f = seeded_randn((N, C, L), 12)
    w3, b3, w1, b1 = seeded_randn((C, C, 3), 13, 0.4), seeded_randn((C,), 14), seeded_randn((C, C, 1), 15, 0.4), seeded_randn((C,), 16)
    xx, mm = seeded_randn((N, C, L), 17), seeded_randn((N, C, L), 18)
    gz = seeded_randn((N, C, L), 19)
    cl = [leaf(t) for t in (w3, b3, w1, b1, xx, mm)]
    gc = torch.sigmoid(F.conv1d(F.relu(F.conv1d(f, cl[0], cl[1], padding=1)), cl[2], cl[3]))
    (cl[4] + cl[5] * 2 * (gc - 0.5)).backward(gz)
    gl = [leaf(t, DEV) for t in (w3, b3, w1, b1, xx, mm)]
    gg = ops.conv1d_flat(ops.conv1d_flat(f.to(DEV), gl[0], gl[1], ops.ACT_RELU), gl[2], gl[3], ops.ACT_SIGMOID)
    assert rel_l2(gg, gc) < 1e-5
    ag.gate_add(gl[4], gl[5], gg).backward(gz.to(DEV))
    for a_, c_ in zip(gl, cl):
        assert rel_l2(a_.grad, c_.grad) < TOL


def test_lrnn_step_with_mean_volume_vs_oracle_and_reference(golden_tiny, golden_train):
    """fp32 LRNN step incl. the mean-volume branch: every one of the 79 parameters gets its gradient; reference = the float64
    oracle (conditioning of the U-Net part: see the test above) and the reference's own autograd (golden)."""
    from cwfa_b200.training import lrnn_loss
    cfg, g = golden_train["config"], golden_train["lrnn_mv"]
    D, S, B, MAX = cfg["D"], cfg["S"], cfg["B"], cfg["MAX"]
    nd = D // 2 ** (MAX - 1)
    views, gt = seeded_randn((B, 29, S, S), g["seeds"]["views"]), seeded_randn((B, nd, S, S), g["seeds"]["gt"])
    mv = seeded_randn((B, nd, S, S), g["seeds"]["mean_vol"], 0.1)
    om = build_tiny_model(golden_tiny).export_for_oracle()
    model = build_tiny_model(golden_tiny, DEV)
    for p in model.parameters():
        p.grad = None
    loss, _ = lrnn_loss(model, gt.to(DEV), views.to(DEV), mv.to(DEV))
    loss.backward()
    ours = {k: p.grad for k, p in model.cond_nets[-1].named_parameters() if p.grad is not None}
    sd64 = {k: (v.double() if v.dtype.is_floating_point else v) for k, v in om["lrnn"].items()}
    r = O.lrnn_train_grads(sd64, views.double(), gt.double(), mv.double())
    assert set(ours) == set(r["grads"]) == set(g["grads"])
    branch = {k: rel_l2(v, r["grads"][k]) for k, v in ours.items() if "conv3d" in k or "attention" in k}
    kb = max(branch, key=branch.get)
    unet = {k: rel_l2(v, r["grads"][k]) for k, v in ours.items() if k not in branch}
    ku = max(unet, key=unet.get)
    print(f"LRNN + mean volume: loss {float(loss):.6f} (reference {float(g['loss']):.6f}); mean-volume branch worst {branch[kb]:.2e} at {kb}; U-Net worst {unet[ku]:.2e} at {ku}")
    assert abs(float(loss) - float(g["loss"])) < 1e-4 * abs(float(g["loss"]))
    assert branch[kb] < 2e-3 and unet[ku] < 5e-2
    check_against_golden({k: v.cpu() for k, v in ours.items()}, g["grads"], 5e-2)


@pytest.mark.parametrize("kind", ["bf16", "fp16"])
@pytest.mark.parametrize("N,C,H,W", [(1, 64, 32, 32), (2, 6, 9, 14), (1, 3, 5, 7), (1, 96, 16, 20), (1, 17, 8, 8)])
@pytest.mark.parametrize("elu", [True, False])
def test_dy_prep_fused_cotangent_pass(kind, N, C, H, W, elu):
    """``tc.dy_prep`` (ELU adjoint + C8 conversion + bias gradient in one pass) against the three separate steps, incl. channel
    counts whose last 8-channel chunk is partly or wholly padding and odd pixel counts (scalar path)."""
    from cwfa_b200 import tc
    g = torch.Generator().manual_seed(C * 10 + W)
    dy = torch.randn(N, C, H, W, generator=g).to(DEV)
    y = (torch.randn(N, C, H, W, generator=g) * 0.7).to(DEV) if elu else None
    ref = dy * torch.where(y > 0, torch.ones_like(y), y + 1.0) if elu else dy
    g8, g32, db = tc.dy_prep(dy, y, kind, want_f32=True, want_bias=True)
    assert torch.equal(g32, ref)
    assert torch.equal(g8.data, tc.to_c8(ref, kind).data)                 # same rounding, zero channel padding
    want = ref.double().sum(dim=(0, 2, 3))
    assert float((db.double() - want).abs().max()) <= 1e-5 * max(1.0, float(want.abs().max()))
    g8b, none32, noneb = tc.dy_prep(dy, y, kind)
    assert none32 is None and noneb is None and torch.equal(g8b.data, g8.data)


@pytest.mark.parametrize("kind,tol", [("bf16", 4e-2), ("fp16", 6e-3)])
@pytest.mark.parametrize("first", [False, True])
@pytest.mark.parametrize("N,H,W", [(2, 20, 28), (2, 160, 272)])
def test_subnet_c8_native_node_matches_per_conv_nodes_and_fp32(kind, tol, first, N, H, W):
    """``autograd._SubnetTC`` (activations and cotangents in C8 through the whole sub-network) against the chain of one node per
    convolution at the same precision and against the fp32 path: output, input gradient and all 16 parameter gradients.
    At 2x160x272 the 64-channel weight gradients walk several tiles per CTA (9-10 at 3x3, 4-5 at 1x1)."""
    from cwfa_b200 import autograd as ag, networks
    torch.manual_seed(7)
    net = (networks.wavelet_flow_subnetwork2D_first if first else networks.wavelet_flow_subnetwork2D)(24, 24).to(DEV)
    gen = torch.Generator().manual_seed(11)
    with torch.no_grad():
        for p in net.parameters():
            p.copy_((torch.randn(p.shape, generator=gen) * (0.5 / max(1.0, float(p[0].numel()) ** 0.5) if p.dim() > 1 else 0.1)).to(DEV))
    x0 = torch.randn(N, 24, H, W, generator=gen).to(DEV)
    r = torch.randn(N, 12 if first else 24, H, W, generator=gen).to(DEV)

    def run(prec, node):
        prev, old = ag.set_training_precision(prec), ag._SUBNET_NODE
        ag._SUBNET_NODE = node
        try:
            net.zero_grad(set_to_none=True)
            x = x0.clone().requires_grad_(True)
            y = net.forward_split(x)[0] if first else net(x)
            (y * r).sum().backward()
            names = [n for n, p in net.named_parameters() if p.grad is not None]
            return y.detach(), x.grad.clone(), {n: dict(net.named_parameters())[n].grad.clone() for n in names}
        finally:
            ag.set_training_precision(prev)
            ag._SUBNET_NODE = old

    y32, dx32, g32 = run("fp32", False)
    yn, dxn, gn = run(kind, True)
    yc, dxc, gc = run(kind, False)
    assert set(gn) == set(gc) == set(g32) and len(gn) == 16
    assert rel_l2(yn, y32) < tol and rel_l2(dxn, dx32) < tol
    worst = 0.0
    for n in gn:
        e_node, e_chain = rel_l2(gn[n], g32[n]), rel_l2(gc[n], g32[n])
        worst = max(worst, e_node)
        assert e_node < max(tol, 2.0 * e_chain), (n, e_node, e_chain)
    print(f"subnet node {kind} first={first} {N}x{H}x{W}: out {rel_l2(yn, y32):.2e}, dx {rel_l2(dxn, dx32):.2e}, worst parameter gradient {worst:.2e} "
          f"(per-conv chain: dx {rel_l2(dxc, dx32):.2e})")


@pytest.mark.parametrize("kind,tol", [("bf16", 3e-2), ("fp16", 4e-3)])
@pytest.mark.parametrize("D,H,W", [(12, 18, 22), (48, 64, 96)])
def test_stencil_c8_native_node_matches_generic_chain_and_fp32(kind, tol, D, H, W):
    """``autograd._StencilBandedTC`` (hidden tensor only in C8) against the generic conv -> PReLU -> conv chain and the fp32 stencil.
    At D = 48, 64x96 the banded weight gradients walk several tiles per CTA (12 for dW2, 4 for dW1)."""
    from cwfa_b200 import autograd as ag
    gen = torch.Generator().manual_seed(3)
    mk = lambda *s, sc=1.0: (torch.randn(*s, generator=gen) * sc).to(DEV)
    Cm = 32
    x0, r = mk(1, D, H, W), mk(1, D, H, W)
    P = [mk(Cm, 1, 3, 3, 3, sc=0.3), mk(Cm, sc=0.2), torch.tensor([0.25], device=DEV), mk(1, Cm, 3, 3, 3, sc=0.1), mk(1, sc=0.2)]

    def run(prec, node):
        prev, old = ag.set_training_precision(prec), ag._STENCIL_NODE
        ag._STENCIL_NODE = node
        try:
            x = x0.clone().requires_grad_(True)
            ps = [p.clone().requires_grad_(True) for p in P]
            y = ag.depth_stencil3d(x, ps[0], ps[1], ps[2], ps[3], ps[4])
            (y * r).sum().backward()
            return [y.detach(), x.grad] + [p.grad for p in ps]
        finally:
            ag.set_training_precision(prev)
            ag._STENCIL_NODE = old

    ref, node, chain = run("fp32", False), run(kind, True), run(kind, False)
    names = ["out", "dx", "dw1", "db1", "dslope", "dw2", "db2"]
    for nm, a, b, c in zip(names, node, chain, ref):
        e_node, e_chain = rel_l2(a, c), rel_l2(b, c)
        print(f"stencil node {kind} D={D} {H}x{W} {nm}: {e_node:.2e} (generic chain {e_chain:.2e})")
        assert e_node < max(tol, 2.0 * e_chain), nm


@pytest.mark.parametrize("which", ["level", "lrnn"])
def test_graph_captured_step_equals_eager_steps(golden_tiny, golden_train, which):
    """``graph=True``: the captured whole-step graph (forward + backward + Lion) leaves exactly the parameters, optimiser state and
    BatchNorm buffers that the same number of eager steps leaves -- including the FIRST call (warm-up steps are undone)."""
    import copy
    import cwfa_b200
    from cwfa_b200.training import FlowLevelTrainer, LRNNTrainer
    cfg = golden_tiny["config"]
    D, S, MAX = cfg["D"], cfg["S"], cfg["MAX"]
    gen = torch.Generator().manual_seed(21)
    mk = lambda *s, sc=1.0: (torch.randn(*s, generator=gen) * sc).to(DEV)
    views = mk(2, 29, S, S)
    if which == "level":
        args = (mk(2, D, S, S), views, mk(2, D // 2, S, S, sc=0.1), mk(2, D // 2, S, S))
    else:
        args = (mk(2, D // 2 ** (MAX - 1), S, S), views)
    results = []
    from cwfa_b200 import networks
    slope0 = networks._SHARED_PRELU.weight.data.clone()    # the reference's ONE PReLU shared by every ResidualBlock / LRNN (a default
    for graph in (False, True):                             # argument, networks.py:209): training it in run 1 must not leak into run 2
        with torch.no_grad():
            networks._SHARED_PRELU.weight.data.copy_(slope0.to(networks._SHARED_PRELU.weight.device))
        model = cwfa_b200.CWFAModel(n_depths=D, volume_side_size=S, INN_max_down_steps=MAX, seed=0).to(DEV)
        tr = (FlowLevelTrainer(model, 0, lr=1e-3, lr_cond=1e-3, precision="bf16", graph=graph) if which == "level"
              else LRNNTrainer(model, lr=1e-3, precision="bf16", graph=graph))
        losses = [float(tr.step(*args)["loss"]) for _ in range(3)]
        sd = copy.deepcopy({k: v.clone() for k, v in model.state_dict().items()})
        moms = [g["exp_avg"].clone() for o in tr._optimizers() for g in o.param_groups]
        results.append((losses, sd, moms))
        tr.release()
    (l0, sd0, m0), (l1, sd1, m1) = results
    assert l0 == l1
    assert all(torch.equal(sd0[k], sd1[k]) for k in sd0)
    assert all(torch.equal(a, b) for a, b in zip(m0, m1))
    with torch.no_grad():
        networks._SHARED_PRELU.weight.data.copy_(slope0.to(networks._SHARED_PRELU.weight.device))
