"""Throughput engine for the CWFA hot path: the same arithmetic as ``CWFAModel.reconstruct`` /
``forward_nll`` (pipeline.py) but with every wide convolution on the tcgen05 tensor-core kernel
(C8 half-precision activations, fp32 accumulation), weights packed once, no per-call parameter
handling, and optional whole-frame CUDA-graph replay.

Numerics: operands are rounded to ``kind`` ('bf16' default, 'fp16'); the coupling coefficients
(the last conv of every sub-network), the affine couplings, log-dets, the Haar transforms, the
depth stencil of the conditioning net and the 6-channel mean-volume branch stay in fp32.
Stated tolerance vs the fp32 reference: rel-L2 <= 2e-2 (bf16) / 3e-3 (fp16) on the reconstruction
(tests/test_gpu_engine.py reports the measured values per level).

Reference path: CWFA.py:865-924 (inverse), :156-196 / :966-978 (forward NLL).
"""
from __future__ import annotations

import math
from typing import Dict, List, Optional, Sequence

import torch

from . import modules as Fm
from . import networks, ops, tc
from .data import LensletLayout, RoiSet
from .pipeline import CWFAModel, lrnn_mean_volume


from .packed import _CondNet, _LRNN, _Subnet, _UNet  # noqa: F401  (executors shared with the module-API fast path)


class CWFAEngine:
    """``engine = CWFAEngine(model); vol = engine.reconstruct(views, mean_vols)``.

    The model's parameters are packed at construction; call ``refresh()`` after changing them.

    Every graph the reference's ``conditional_wavelet_flow`` can build runs here: ``ConditionalAffineTransform`` blocks (the
    default, networks.py:289-297) use the fused trunk / coupling kernels; any other invertible block (GLOW / RNVP / GIN / AI1 /
    ...) is executed through its own ``forward`` with the tensor-core inference switch on (``cwfa_b200.packed``: its sub-networks
    run on tcgen05 and, where the clamp allows, with the coupling fused into the last convolution).
    ``disable_low_res_input=1`` (networks.py:331-338, CWFA.py:899-901) makes the levels sequential: the condition of level n is
    the volume reconstructed by level n+1."""

    def __init__(self, model: CWFAModel, kind: str = "bf16"):
        if kind not in ("bf16", "fp16"):
            raise ValueError(kind)
        if not next(model.parameters()).is_cuda:
            raise RuntimeError("CWFAEngine needs the model on a CUDA device (no CPU fallback)")
        self.model, self.kind = model, kind
        self.parallel_branches = True      # LRNN and per-level coefficient nets as parallel CUDA-graph branches
        self.refresh()

    def refresh(self):
        m, kind = self.model, self.kind
        self.dlr = bool(m.cfg.disable_low_res_input)
        self.levels = []
        for n in range(m.n_levels):
            inn = m.conv_inn[n]
            nodes = []
            for mod in inn.module_list:
                if isinstance(mod, Fm.ConditionalAffineTransform) and mod._clamp_kw is not None and not mod._clamp_kw["tanh_clamp"]:
                    nodes.append(("cat", mod, _Subnet(mod.subnet, kind)))
                elif isinstance(mod, Fm.PermuteRandom):
                    nodes.append(("perm", mod, 1))
                elif isinstance(mod, Fm.PermuteDim):
                    nodes.append(("perm", mod, mod.axis))
                elif isinstance(mod, (Fm.HaarTransform1D, Fm.Split)):
                    continue
                elif isinstance(mod, Fm.InvertibleModule):
                    nodes.append(("module", mod, None))          # generic block: its own forward, tensor-core inference switch on
                else:
                    raise NotImplementedError(f"CWFAEngine: {type(mod).__name__} is not an invertible module of this package")
            subs = [x[2] for x in nodes if x[0] == "cat"]
            batched = None
            if len(subs) > 1 and all(sn.inp.Cout_p == 64 and sn.inp.Cin_p == subs[0].inp.Cin_p and sn.inp.Cin == subs[0].inp.Cin for sn in subs):
                # one 1x1 conv for the input layers of all sub-networks of the level (they all read the LF condition)
                ws = [(mod.subnet.block12 if mod.subnet.normal else mod.subnet.block1) for k_, mod, _ in nodes if k_ == "cat"]
                batched = tc.PackedConv(torch.cat([w.weight.detach() for w in ws], 0), torch.cat([w.bias.detach() for w in ws], 0),
                                        kind, bn=64)
            self.levels.append(dict(nodes=nodes, cond=None if self.dlr else _CondNet(m.cond_nets[n], kind), batched_in=batched,
                                    entry=self._plan_entry(nodes, kind), f8=self._plan_f8(nodes, kind)))
        self.lrnn = _LRNN(m.cond_nets[-1], kind)
        self._graphs: Dict = {}

    @staticmethod
    def _plan_entry(nodes, kind):
        """The first trunk block of every fused sub-network folded onto its 1x1 input conv (``tc.PackedEntry``), or None when a
        sub-network's input conv is not 1x1 Cin_p <= 64 -> 64, and for fp16.  fp16 keeps the separate input conv: its rounding
        of W3' instead of Win and W3 moved the level-0 log-det of the full-size forward pass from 1.94e-3 to 2.24e-3 against the
        fp32 reference (B200), past the fp16 engine's stated 2e-3."""
        subs = [(mod.subnet, sn) for k, mod, sn in nodes if k == "cat"]
        if kind != "bf16" or not subs or any(sn.inp.KH != 1 or sn.inp.Cout != 64 or sn.inp.Cin_p > 64
                                             or sn.inp.Cin_p != subs[0][1].inp.Cin_p for _, sn in subs):
            return None
        out = []
        for sub, sn in subs:
            first = sub.block12 if sub.normal else sub.block1
            out.append(tc.PackedEntry(first.weight, first.bias, sub.block2[0].weight, sub.block2[0].bias, sn.res[0][1], kind))
        return out

    use_f8 = True          # lean coupling path on the F8 layout (csrc/coupling_f8.cu) for levels made of CAT blocks + permutations

    @staticmethod
    def _plan_f8(nodes, kind):
        """F8 plan of a level whose flow is CAT blocks + permutations (the default graph, networks.py:305-366): the detail half
        stays in the channel order it ENTERED the flow; a channel permutation (fixed_transforms.py:37-41) only updates the map
        ``m`` (logical channel -> storage slot: m <- m[perm]) and every coupling's last conv is packed with its output channels
        in storage order.  Returns None when the level has other block types (they run on the NCHW path)."""
        if not nodes or any(k == "module" for k, _, _ in nodes):
            return None
        cats = [mod for k, mod, _ in nodes if k == "cat"]
        if not cats or any(sub.inp.Cout_p != 64 or sub.out.KH != 3 for k, _, sub in nodes if k == "cat") or cats[0].channels > 48:
            return None
        ch = cats[0].channels
        dev = next(cats[0].parameters()).device
        m = torch.arange(ch)
        packed = []
        # NLL maps (forward): (R_b, C_b) per CAT block in forward order = the level-input row / column of the element block b
        # writes at (h, w).  A row / column permutation is gathered by the next coupling (y[h] = x[perm[h]]): R <- R[perm].
        rc, src, pending = [None, None], [], None
        for k, mod, extra in nodes:
            if k == "perm" and extra == 1:
                m = m[mod.perm.detach().cpu().long()]
            elif k == "perm":
                pending = (mod.perm.detach().cpu().long(), extra)
            elif k == "cat":
                minv = torch.empty_like(m)
                minv[m] = torch.arange(ch)
                last = mod.subnet.block72[1] if mod.subnet.normal else mod.subnet.block7[1]
                packed.append(tc.coupling_weights_f8(last.weight, last.bias, ch, minv, not mod.subnet.normal, kind))
                if pending is not None:
                    a = pending[1] - 2
                    rc[a] = pending[0] if rc[a] is None else rc[a][pending[0]]
                    pending = None
                src.append(tuple(None if t is None else t.to(dev, torch.int32).contiguous() for t in rc))
        minv = torch.empty_like(m)
        minv[m] = torch.arange(ch)
        return dict(ch=ch, out=packed, z_from_storage=m.to(dev, torch.int32).contiguous(), storage_from_z=minv.to(dev, torch.int32).contiguous(),
                    map_src=src)

    def _f8_unsupported(self, n: int, H: int, W: int) -> Optional[str]:
        """Why level n does not run on the F8 coupling kernels (which give the per-voxel NLL maps and the exact posterior std),
        or None."""
        lv = self.levels[n]
        if lv["f8"] is not None and self.use_f8 and (H * W) % 4 == 0:
            return None
        if not self.use_f8:
            return "the F8 coupling path is switched off (use_f8 = False)"
        if lv["f8"] is not None:
            return f"H * W = {H} * {W} is not a multiple of 4"
        tanh = lambda mod: isinstance(mod, Fm.ConditionalAffineTransform) and bool(mod._clamp_kw and mod._clamp_kw["tanh_clamp"])
        others = sorted({type(mod).__name__ + (" with a tanh clamp" if tanh(mod) else "") for k, mod, _ in lv["nodes"] if k == "module"})
        if others:
            return "its flow has blocks other than (non-tanh-clamped) ConditionalAffineTransform: " + ", ".join(others)
        cats = [(mod, sub) for k, mod, sub in lv["nodes"] if k == "cat"]
        if not cats:
            return "its flow has no coupling block"
        if cats[0][0].channels > 48:
            return f"its detail half has {cats[0][0].channels} channels (at most 48)"
        return "its coupling sub-networks are not 64 hidden channels with a 3x3 last conv"

    # -------------------------------------------------------------------------------------
    batch_trunks = True    # the block rows of a level's sub-network trunks as ONE launch each (cwfa_resblock_tc_batched)
    # the first trunk block reads the LF condition directly (tc.PackedEntry): no 1x1 input-conv launch, its output never in HBM;
    # CWFA_COMPOSED_ENTRY=0 keeps the input conv + block pair (A/B measurements)
    composed_entry = __import__("os").environ.get("CWFA_COMPOSED_ENTRY", "1") == "1"

    def _trunks(self, n: int, lf8: tc.C8, allow_batched: bool = True):
        """The trunks of all fused sub-networks of level n from the level's LF condition (C8).  They depend on the conditions
        only (CAT blocks, coupling_layers.py:475-500), so forward and inverse share them and levels are independent.
        Items: (kind, module, executor, trunk output C8, chunk offset of this sub-network's 64-channel slice in it).
        With a batched input conv the three block rows of the (<= 5) trunks run as three launches over all sub-networks."""
        lv = self.levels[n]
        subs = [extra for kind, _, extra in lv["nodes"] if kind == "cat"]
        out, k = [], 0
        if lv["entry"] is not None and self.composed_entry:
            b_all = None
            if allow_batched and self.batch_trunks and 2 <= len(subs) <= 5:
                b_all = tc.resblock_tc_entry_batched(lf8, lv["entry"])
                for r in (1, 2):
                    b_all = tc.resblock_tc_batched(b_all, [sn.res[r] for sn in subs])
            for kind, mod, extra in lv["nodes"]:
                if kind != "cat":
                    out.append((kind, mod, extra, None, 0))
                    continue
                if b_all is not None:
                    out.append(("cat", mod, extra, b_all, 8 * k))
                else:
                    b = tc.resblock_tc_entry_batched(lf8, [lv["entry"][k]])
                    for p3, p1 in extra.res[1:]:
                        b = tc.resblock_tc(b, p3, p1)
                    out.append(("cat", mod, extra, b, 0))
                k += 1
            return out
        b_all = tc.conv_tc(lf8, lv["batched_in"]) if lv["batched_in"] is not None else None
        if b_all is not None and allow_batched and self.batch_trunks and 2 <= len(subs) <= 5:
            for r in range(3):
                b_all = tc.resblock_tc_batched(b_all, [sn.res[r] for sn in subs])
            for kind, mod, extra in lv["nodes"]:
                if kind == "cat":
                    out.append(("cat", mod, extra, b_all, 8 * k))
                    k += 1
                else:
                    out.append((kind, mod, extra, None, 0))
            return out
        for kind, mod, extra in lv["nodes"]:
            if kind == "cat":
                out.append(("cat", mod, extra, extra.trunk(lf8, b_all, 8 * k) if b_all is not None else extra.trunk(lf8), 0))
                k += 1
            else:
                out.append((kind, mod, extra, None, 0))
        return out

    def _views_c8(self, views: torch.Tensor, sensor: Optional[LensletLayout]) -> tc.C8:
        """The conditions in the C8 layout: from fp32 views, or in one pass from a raw sensor frame."""
        return tc.to_c8(views, self.kind) if sensor is None else sensor.views_c8(views, self.kind)

    def _lf(self, n: int, v8: Optional[tc.C8], low_res: Optional[torch.Tensor]) -> tc.C8:
        """LF condition of level n: conditioning net of the views, or (disable_low_res_input) the volume of the level below."""
        if self.dlr:
            return tc.to_c8(low_res, self.kind)
        return self.levels[n]["cond"](v8)

    @staticmethod
    def _jac_and_tickets(n_samples: int, device, n_tickets: int = 8):
        """One zero-filled allocation (one memset) per level: the (B,) log-det accumulator plus the int32 tickets of the
        level's coupling kernels (in-kernel last-CTA finalize, cwfa_coupling_tc)."""
        buf = torch.zeros(n_samples + n_tickets, device=device, dtype=torch.float32)
        return buf[:n_samples], buf[n_samples:].view(torch.int32)

    def _couple(self, item, x, mean_vol, pending, inverse, logdet, sumsq=None, ticket=None):
        """Final conv of one sub-network with the coupling fused in its epilogue.  When ``x`` carries more samples than the
        conditions (multi-sample reconstruction, CWFA.py:903-914) the coefficients are computed ONCE and broadcast over the
        samples by the affine kernel."""
        _, mod, sub, b8, off = item
        first = not sub.normal
        t_scale = (-1.0 / math.sqrt(2)) if first else 1.0
        if x is not None and x.shape[0] != b8.N:
            K = x.shape[0]
            if pending is not None:
                x = ops.permute(x, pending[0], pending[1])
            a = tc.conv_tc(b8, sub.out, out_nchw=True)                       # (1, 2ch | ch, H, W)
            ch = mod.channels
            a_s = a[:, :ch].expand(K, -1, -1, -1)
            a_t = (mean_vol if first else a[:, ch:]).expand(K, -1, -1, -1)
            y, j, q = ops.affine(x, a_s, a_t, inverse=inverse, clamp=mod.clamp, t_scale=t_scale, want_sumsq=True)
            logdet += j
            if sumsq is not None:
                sumsq.copy_(q)
            return y
        perm, axis = (None, 0) if pending is None else (ops.perm_i32(pending[0], b8.data.device), pending[1])
        return tc.conv_tc_coupling(b8, sub.out, x, ch=mod.channels, inverse=inverse, clamp=mod.clamp,
                                   t_ext=mean_vol if first else None, t_scale=t_scale,
                                   perm=perm, perm_axis=axis, logdet=logdet, sumsq=sumsq, ticket=ticket, chunk_off=off)

    def _run_module(self, mod, hi, lf_nchw, rev, logdet):
        """A generic invertible block through its own forward (module-API fast path: sub-networks on tcgen05)."""
        from . import packed
        with packed.inference_precision(self.kind):
            (hi,), j = mod((hi,), c=[lf_nchw], rev=rev) if mod.dims_c else mod((hi,), rev=rev)
        if torch.is_tensor(j):
            logdet += j
        elif j != 0:
            logdet += float(j)
        return hi

    def _level_detail_inverse(self, n, lf8, mean_vol, z=None, rows: int = 1):
        """Detail half ``hi`` of level n in the inverse direction and its log-det.  Independent of the other levels unless
        ``disable_low_res_input``.  ``z`` None = zeros (INN_z_temperature = 0, CWFA.py:906-907: z is never materialised);
        otherwise the latent sample(s) of this level (``sample_z_truncated``, CWFA.py:47-64), ``rows`` of them."""
        items = self._trunks(n, lf8, allow_batched=(z is None or z.shape[0] == lf8.N))
        plan = self.levels[n]["f8"] if (self.use_f8 and (lf8.H * lf8.W) % 4 == 0) else None
        if plan is not None and (z is None or z.shape[0] == lf8.N):
            return self._level_detail_inverse_f8(n, items, plan, lf8, mean_vol, z)
        hi, pending = z, None
        jac, tickets = self._jac_and_tickets(rows if z is None else z.shape[0], lf8.data.device)
        lf_nchw, k = None, 0
        for item in reversed(items):
            if item[0] == "cat":
                hi = self._couple(item, hi, mean_vol, pending, True, jac, ticket=tickets[k:k + 1])
                pending, k = None, (k + 1) % tickets.numel()
            elif item[0] == "perm":
                if hi is not None:
                    pending = (item[1].perm_inv, item[2])       # gathered by the next coupling's epilogue
            else:
                if hi is None:
                    hi = torch.zeros((rows,) + tuple(item[1].dims_in[0]), device=lf8.data.device, dtype=torch.float32)
                if pending is not None:
                    hi, pending = ops.permute(hi, pending[0], pending[1]), None
                if lf_nchw is None:
                    lf_nchw = tc.from_c8(lf8)
                    if lf_nchw.shape[0] != hi.shape[0]:
                        lf_nchw = lf_nchw.expand(hi.shape[0], -1, -1, -1).contiguous()
                hi = self._run_module(item[1], hi, lf_nchw, True, jac)
        if pending is not None:
            hi = ops.permute(hi, pending[0], pending[1])
        return hi, jac

    def _couple_f8(self, item, pc, x8, mv8, pending, inverse, logdet, sumsq, ticket, nll_map=None, map_src=(None, None), map_mode=0,
                   with_scale=False, scale8=None):
        _, mod, sub, b8, off = item
        first = not sub.normal
        perm, axis = (None, 0) if pending is None else (ops.perm_i32(pending[0], b8.data.device), pending[1])
        if with_scale:
            return tc.coupling_f8_scale(b8, pc, x8, scale8, ch=mod.channels, clamp=mod.clamp, t_ext8=mv8 if first else None,
                                        t_scale=(-1.0 / math.sqrt(2)) if first else 1.0, perm=perm, perm_axis=axis, logdet=logdet,
                                        ticket=ticket, chunk_off=off)
        if nll_map is not None:
            return tc.coupling_f8_map(b8, pc, x8, nll_map, ch=mod.channels, map_mode=map_mode, row_src=map_src[0], col_src=map_src[1],
                                      clamp=mod.clamp, t_ext8=mv8 if first else None, t_scale=(-1.0 / math.sqrt(2)) if first else 1.0,
                                      perm=perm, perm_axis=axis, logdet=logdet, sumsq=sumsq, ticket=ticket, chunk_off=off)
        return tc.coupling_f8(b8, pc, x8, ch=mod.channels, inverse=inverse, clamp=mod.clamp, t_ext8=mv8 if first else None,
                              t_scale=(-1.0 / math.sqrt(2)) if first else 1.0, perm=perm, perm_axis=axis, logdet=logdet, sumsq=sumsq,
                              ticket=ticket, chunk_off=off)

    @staticmethod
    def _permute_f8(x8, ch, perm, axis):
        """Row / column permutation of an F8 tensor that no coupling follows (never the case in CWFA's graphs): via NCHW."""
        return tc.to_f8(ops.permute(tc.from_f8(x8, ch), perm, axis))

    def _level_detail_inverse_f8(self, n, items, plan, lf8, mean_vol, z, with_scale=False):
        """Inverse of a CAT-only level on the F8 layout: returns (("f8", hi8), logdet).  ``with_scale``: the couplings also
        carry each element's scale d hi / d z (``coupling_f8_scale``), returned as (("f8", hi8, scale8), logdet)."""
        ch = plan["ch"]
        hi = None if z is None else tc.to_f8(z, plan["storage_from_z"])
        mv8 = None if mean_vol is None else tc.to_f8(mean_vol)
        jac, tickets = self._jac_and_tickets(lf8.N, lf8.data.device)
        pending, k = None, 0
        pcs = plan["out"]
        ci = len(pcs)
        sc = None                                               # scale of the chain so far; None = 1 (nothing gathered yet)
        for item in reversed(items):
            if item[0] == "cat":
                ci -= 1
                if with_scale:
                    hi, sc = self._couple_f8(item, pcs[ci], hi, mv8, pending, True, jac, None, tickets[k:k + 1], with_scale=True,
                                             scale8=sc)
                else:
                    hi = self._couple_f8(item, pcs[ci], hi, mv8, pending, True, jac, None, tickets[k:k + 1])
                pending, k = None, (k + 1) % tickets.numel()
            elif item[2] != 1 and hi is not None:               # row / column permutation: gathered by the next coupling
                pending = (item[1].perm_inv, item[2])
        if pending is not None:
            hi = self._permute_f8(hi, ch, pending[0], pending[1])
            if with_scale:
                sc = self._permute_f8(sc, ch, pending[0], pending[1])
        return (("f8", hi, sc) if with_scale else ("f8", hi)), jac

    @torch.no_grad()
    def reconstruct(self, views: torch.Tensor, mean_vols: Sequence[Optional[torch.Tensor]], return_all: bool = False,
                    _side_streams=None, zs: Optional[Sequence[Optional[torch.Tensor]]] = None, n_samples: int = 1,
                    temperature: Optional[float] = None, sensor: Optional[LensletLayout] = None):
        """Inverse reconstruction (CWFA.py:865-924); z = 0 unless ``zs[n]`` gives level n's latent sample(s) or
        ``temperature`` (default ``cfg.INN_z_temperature`` = 0) is non-zero (then z ~ ``sample_z_truncated``).
        ``n_samples`` > 1 (batch 1): the reference's multi-sample path (CWFA.py:903-914) -- the coefficients of a level are
        computed once, applied to ``n_samples`` latent samples, and the samples are averaged (the Haar merge is linear, so the
        mean is taken on the detail half before the merge).

        The LRNN and the coupling coefficients of every level depend only on the views / mean volumes, not on
        each other, so under CUDA-graph capture they are issued on side streams (``_side_streams``) and become
        parallel branches of the graph; only the four Haar merges are sequential.

        ``sensor``: ``views`` is then a raw sensor frame (``LensletLayout``: uint16 / fp16 / fp32, (B, 1, Hi, Wi) or (B, Hi, Wi)),
        cropped and normalised straight into the tensor-core input layout; the result is bitwise that of
        ``reconstruct(sensor.views(frame), ...)``."""
        from .pipeline import sample_z_truncated
        L1 = self.model.n_levels
        T = self.model.cfg.INN_z_temperature if temperature is None else temperature
        B = views.shape[0]
        if n_samples > 1 and B != 1:
            raise ValueError("n_samples > 1 needs batch size 1 (CWFA.py:904)")
        v8 = self._views_c8(views, sensor)
        mv_last = lrnn_mean_volume(mean_vols, L1)            # CWFA.py:882: mean_vols_cache[L-2] unless given explicitly

        def z_of(n):
            if zs is not None and zs[n] is not None:
                return zs[n]
            if T != 0:
                return sample_z_truncated((B * n_samples,) + tuple(self.model.conv_inn[n].global_out_shapes[0]), device=views.device,
                                          temperature=T)
            return None

        def merge(vol, hi):
            """Split^-1 + IDWT of a level; the detail half arrives in NCHW or (CAT-only levels) in the F8 layout."""
            if isinstance(hi, tuple):
                return tc.haar1d_merge_f8(vol, hi[1])
            if n_samples > 1 and hi.shape[0] > 1:
                hi = ops.batch_mean(hi)
            return ops.haar1d_merge(vol, hi)

        if self.dlr:                                         # sequential pyramid: the condition is the volume of the level below
            vol = self.lrnn(v8, mv_last)
            outs, jacs = {L1: vol}, {}
            for n in range(L1 - 1, -1, -1):
                hi, jac = self._level_detail_inverse(n, self._lf(n, None, vol), None, z_of(n), B)
                vol = merge(vol, hi)
                outs[n], jacs[n] = vol, jac
            return (outs, jacs) if return_all else vol
        jobs = [lambda: self.lrnn(v8, mv_last)] + [(lambda n=n: self._level_detail_inverse(n, self._lf(n, v8, None), mean_vols[n], z_of(n), B))
                                                    for n in range(L1 - 1, -1, -1)]
        results = self._run_jobs(jobs, _side_streams)
        vol = results[0]
        outs, jacs = {L1: vol}, {}
        for k, n in enumerate(range(L1 - 1, -1, -1)):
            hi, jac = results[1 + k]
            vol = merge(vol, hi)                     # Split^-1 + IDWT: the only sequential part of the pyramid
            outs[n], jacs[n] = vol, jac
        return (outs, jacs) if return_all else vol

    @staticmethod
    def _run_jobs(jobs, side_streams):
        """Runs independent jobs in order, or each on its own side stream (forked from and joined back into the current
        stream: parallel branches under CUDA-graph capture).  Returns their results in order."""
        if not side_streams:
            return [job() for job in jobs]
        main = torch.cuda.current_stream()
        fork = torch.cuda.Event()
        fork.record(main)
        results, joins = [], []
        for st, job in zip(side_streams, jobs):
            st.wait_event(fork)
            with torch.cuda.stream(st):
                results.append(job())
                ev = torch.cuda.Event()
                ev.record(st)
            joins.append(ev)
        for ev in joins:
            main.wait_event(ev)
        return results

    # ---- posterior statistics: per-voxel mean and standard deviation over K latent samples ------------------------------
    def _level_detail_samples(self, n, lf8, mean_vol, z):
        """Detail halves of level n for the K latent samples ``z`` (K rows) of one frame: ("f8", K-row F8 tensor) on the F8 plan
        (batched trunks, one K-sample coupling per block: s and t computed once), else the K-row NCHW path of
        ``_level_detail_inverse``.  Sample k is what ``_level_detail_inverse`` gives for ``z[k:k+1]`` (bitwise on the F8 plan)."""
        K = z.shape[0]
        plan = self.levels[n]["f8"] if (self.use_f8 and (lf8.H * lf8.W) % 4 == 0) else None
        if plan is None:
            return self._level_detail_inverse(n, lf8, mean_vol, z, K)[0]
        items = self._trunks(n, lf8)
        hi = tc.to_f8(z, plan["storage_from_z"])
        mv8 = None if mean_vol is None else tc.to_f8(mean_vol)
        jac, tickets = self._jac_and_tickets(lf8.N, lf8.data.device)          # log-det: computed by the kernels, not returned
        pending, k = None, 0
        pcs = plan["out"]
        ci = len(pcs)
        for item in reversed(items):
            if item[0] == "cat":
                ci -= 1
                _, mod, sub, b8, off = item
                first = not sub.normal
                perm, axis = (None, 0) if pending is None else (ops.perm_i32(pending[0], b8.data.device), pending[1])
                hi = tc.coupling_f8_samples(b8, pcs[ci], hi, K, ch=mod.channels, clamp=mod.clamp, t_ext8=mv8 if first else None,
                                            t_scale=(-1.0 / math.sqrt(2)) if first else 1.0, perm=perm, perm_axis=axis,
                                            logdet=jac, ticket=tickets[k:k + 1], chunk_off=off)
                pending, k = None, (k + 1) % tickets.numel()
            elif item[2] != 1:                                  # row / column permutation: gathered by the next coupling
                pending = (item[1].perm_inv, item[2])
        if pending is not None:
            hi = self._permute_f8(hi, plan["ch"], pending[0], pending[1])
        return ("f8", hi)

    def _independent_levels_check(self):
        if self.dlr:
            raise ValueError("posterior statistics need independent levels: with disable_low_res_input each level is conditioned "
                             "on the volume reconstructed below it, so the samples are not a chain of independent levels")

    def _posterior_check(self, views, n_samples, zs):
        self._independent_levels_check()
        if int(n_samples) < 2:
            raise ValueError("posterior statistics need n_samples >= 2")
        if views.shape[0] != 1:
            raise ValueError("posterior statistics take one frame (batch size 1, CWFA.py:904)")
        if zs is not None:
            for n, z in enumerate(zs):
                if z is not None and z.shape[0] != int(n_samples):
                    raise ValueError(f"zs[{n}] has {z.shape[0]} rows, expected n_samples = {int(n_samples)}")

    @torch.no_grad()
    def reconstruct_posterior(self, views: torch.Tensor, mean_vols: Sequence[Optional[torch.Tensor]], n_samples: int,
                              temperature: Optional[float] = None, zs: Optional[Sequence[Optional[torch.Tensor]]] = None,
                              sensor: Optional[LensletLayout] = None, _side_streams=None):
        """Per-voxel posterior mean and unbiased standard deviation over ``n_samples`` = K >= 2 latent samples of one frame:
        ``(mean, std)``, each (1, D, H, W) fp32.  Sample k's volume V_k is ``reconstruct(views, mean_vols, zs=[z_n[k:k+1]])``
        with ``z_n`` = ``zs[n]`` (K rows) or, for levels without one, K draws of ``sample_z_truncated(temperature)``
        (default ``cfg.INN_z_temperature``; temperature 0: z = 0, so std = 0).  mean = sum_k V_k / K,
        std = sqrt(sum_k (V_k - mean)^2 / (K - 1)).

        The LRNN, the conditioning nets and the sub-network trunks run once for all samples; every coupling of the F8 levels
        computes its s and t once and applies them to the K samples; the last merge computes the statistics in registers, so
        the K full-resolution volumes are never written.  Not for ``disable_low_res_input`` models (their levels are not
        independent).  ``sensor``: ``views`` is a raw sensor frame (see ``reconstruct``)."""
        from .pipeline import sample_z_truncated
        self._posterior_check(views, n_samples, zs)
        K = int(n_samples)
        L1 = self.model.n_levels
        T = self.model.cfg.INN_z_temperature if temperature is None else temperature
        v8 = self._views_c8(views, sensor)
        mv_last = lrnn_mean_volume(mean_vols, L1)

        def z_of(n):
            if zs is not None and zs[n] is not None:
                return zs[n]
            shape = (K,) + tuple(self.model.conv_inn[n].global_out_shapes[0])
            if T != 0:
                return sample_z_truncated(shape, device=views.device, temperature=T)
            return torch.zeros(shape, device=views.device, dtype=torch.float32)

        jobs = [lambda: self.lrnn(v8, mv_last)] + [(lambda n=n: self._level_detail_samples(n, self._lf(n, v8, None), mean_vols[n], z_of(n)))
                                                    for n in range(L1 - 1, -1, -1)]
        results = self._run_jobs(jobs, _side_streams)
        vol = results[0]
        for k, n in enumerate(range(L1 - 1, -1, -1)):
            hi = results[1 + k]
            hi = hi[1] if isinstance(hi, tuple) else hi
            if n == 0:
                return tc.haar1d_merge_stats(vol, hi)            # one LRNN row is shared when level 0 is the only flow level
            if vol.shape[0] != K:
                vol = vol.expand(K, -1, -1, -1).contiguous()
            vol = tc.haar1d_merge_f8(vol, hi) if hi.dim() == 5 else ops.haar1d_merge(vol, hi)

    def reconstruct_posterior_graphed(self, views: torch.Tensor, mean_vols: Sequence[Optional[torch.Tensor]], n_samples: int,
                                      temperature: Optional[float] = None, zs: Optional[Sequence[Optional[torch.Tensor]]] = None,
                                      sensor: Optional[LensletLayout] = None):
        """``reconstruct_posterior`` as one CUDA-graph replay.  The latent samples are graph inputs (K rows per level), filled
        before each replay from ``zs`` or fresh ``sample_z_truncated`` draws as in ``reconstruct_graphed``; the LRNN and the
        levels are parallel branches.  The returned (mean, std) are the graph's static outputs, overwritten by the next call."""
        self._posterior_check(views, n_samples, zs)
        K = int(n_samples)
        T = self.model.cfg.INN_z_temperature if temperature is None else temperature
        key = ("posterior", tuple(views.shape), tuple(None if m is None else tuple(m.shape) for m in mean_vols), views.device.index, K,
               None if sensor is None else (id(sensor), views.dtype))
        g = self._graphs.get(key)
        if g is None:
            sv = views.clone()
            sm = [None if m is None else m.clone() for m in mean_vols]
            sz = [torch.zeros((K,) + tuple(self.model.conv_inn[n].global_out_shapes[0]), device=views.device, dtype=torch.float32)
                  for n in range(self.model.n_levels)]
            s = torch.cuda.Stream()
            s.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(s):
                for _ in range(2):
                    self.reconstruct_posterior(sv, sm, K, zs=sz, sensor=sensor)
            torch.cuda.current_stream().wait_stream(s)
            graph = torch.cuda.CUDAGraph()
            side = [torch.cuda.Stream() for _ in range(self.model.n_levels + 1)] if self.parallel_branches else None
            with torch.cuda.graph(graph):
                out = self.reconstruct_posterior(sv, sm, K, zs=sz, sensor=sensor, _side_streams=side)
            g = self._graphs[key] = (graph, sv, sm, out, sz, sensor)    # the graph reads the layout's coordinates: keep it alive
        graph, sv, sm, out, sz = g[:5]
        sv.copy_(views, non_blocking=True)
        for d, s_ in zip(sm, mean_vols):
            if d is not None:
                d.copy_(s_, non_blocking=True)
        self._fill_z(sz, zs, T)
        graph.replay()
        return out

    # ---- exact posterior standard deviation: the volume is affine in the latents on CAT-only levels -------------------------
    def _posterior_exact_sigma(self, temperature: Optional[float]) -> float:
        """Checks that the exact moments exist for this model and returns sigma_T, the std of one latent at ``temperature``."""
        from .pipeline import truncated_normal_var
        self._independent_levels_check()
        T = self.model.cfg.INN_z_temperature if temperature is None else temperature
        var = truncated_normal_var(T)                             # ValueError for T < 0
        for n in range(self.model.n_levels):
            _, H, W = self.model.conv_inn[n].global_out_shapes[0]
            why = self._f8_unsupported(n, H, W)
            if why is not None:
                raise ValueError(f"reconstruct_posterior_exact: level {n} has no exact posterior std: {why} (the exact moments "
                                 "need every level affine in its latent: CAT blocks on the F8 coupling path)")
        return math.sqrt(var)

    @torch.no_grad()
    def reconstruct_posterior_exact(self, views: torch.Tensor, mean_vols: Sequence[Optional[torch.Tensor]],
                                    temperature: Optional[float] = None, sensor: Optional[LensletLayout] = None, _side_streams=None):
        """Exact per-voxel posterior mean and standard deviation of the reconstruction under the latent prior, in one inverse
        pass and for any batch size: ``(mean, std)``, each (B, D, H, W) fp32.

        Every coupling of a level is a CAT block whose s and t come from the conditions only, so level n's detail half is affine in
        its latent, hi_n = beta_n + alpha_n * z_n (alpha_n = exp(-sum of the blocks' s), carried along the chain by
        ``coupling_f8_scale``); the levels are independent, the LRNN volume is deterministic and the Haar merge is linear.  Hence
        mean = V(z = 0), bitwise ``reconstruct(views, mean_vols, temperature=0)``, and at every merge Var x[2i] = Var x[2i+1] =
        (Var lo_i + Var hi_i) / 2 with Var hi_n = sigma_T^2 alpha_n^2, sigma_T^2 = ``truncated_normal_var(temperature)`` (default
        ``cfg.INN_z_temperature``; 0 gives std = 0).  Only the mean and std are exact: a sum of scaled truncated normals is not
        Gaussian.  ``reconstruct_posterior`` estimates the same two moments from K samples.

        Raises ValueError for ``disable_low_res_input`` models (each level is conditioned on the volume below it, so the volume
        is not affine in z), for levels without the F8 coupling plan (GLOW / RNVP / GIN / AI1 or tanh-clamped blocks, which are
        not affine in z; more than 48 detail channels; H * W not a multiple of 4; ``use_f8 = False``) and for a negative
        temperature.  ``sensor``: ``views`` is a raw sensor frame (see ``reconstruct``)."""
        sigma = self._posterior_exact_sigma(temperature)
        vol, levels = self._scale_pass(views, mean_vols, sensor, _side_streams)
        std = None                                                # the LRNN volume is deterministic: std 0 (NULL)
        for hi8, sc8 in levels:
            vol, std = tc.haar1d_merge_std_f8(vol, std, hi8, sc8, sigma)
        return vol, std

    def _scale_pass(self, views, mean_vols, sensor, side_streams):
        """The LRNN volume and, from the top level down (n = L-1 .. 0), every level's z = 0 detail half and scale d hi / d z as
        ``(hi8, scale8)`` F8 tensors: the LRNN and the levels as independent jobs (parallel branches under graph capture)."""
        L1 = self.model.n_levels
        v8 = self._views_c8(views, sensor)
        mv_last = lrnn_mean_volume(mean_vols, L1)

        def level(n):
            lf8 = self._lf(n, v8, None)
            (_, hi8, sc8), _ = self._level_detail_inverse_f8(n, self._trunks(n, lf8), self.levels[n]["f8"], lf8, mean_vols[n], None,
                                                             with_scale=True)
            return hi8, sc8

        jobs = [lambda: self.lrnn(v8, mv_last)] + [(lambda n=n: level(n)) for n in range(L1 - 1, -1, -1)]
        results = self._run_jobs(jobs, side_streams)
        return results[0], results[1:]

    def reconstruct_posterior_exact_graphed(self, views: torch.Tensor, mean_vols: Sequence[Optional[torch.Tensor]],
                                            temperature: Optional[float] = None, sensor: Optional[LensletLayout] = None):
        """``reconstruct_posterior_exact`` as one CUDA-graph replay, the LRNN and the levels as parallel branches.  sigma_T is a
        kernel argument, so every temperature has a graph of its own.  The returned (mean, std) are the graph's static outputs,
        overwritten by the next call with the same shapes and temperature."""
        sigma = self._posterior_exact_sigma(temperature)
        key = ("posterior_exact", tuple(views.shape), tuple(None if m is None else tuple(m.shape) for m in mean_vols), views.device.index,
               sigma, None if sensor is None else (id(sensor), views.dtype))
        g = self._graphs.get(key)
        if g is None:
            sv = views.clone()
            sm = [None if m is None else m.clone() for m in mean_vols]
            s = torch.cuda.Stream()
            s.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(s):
                for _ in range(2):
                    self.reconstruct_posterior_exact(sv, sm, temperature, sensor=sensor)
            torch.cuda.current_stream().wait_stream(s)
            graph = torch.cuda.CUDAGraph()
            side = [torch.cuda.Stream() for _ in range(self.model.n_levels + 1)] if self.parallel_branches else None
            with torch.cuda.graph(graph):
                out = self.reconstruct_posterior_exact(sv, sm, temperature, sensor=sensor, _side_streams=side)
            g = self._graphs[key] = (graph, sv, sm, out, sensor)    # the graph reads the layout's coordinates: keep it alive
        graph, sv, sm, out = g[:4]
        sv.copy_(views, non_blocking=True)
        for d, s_ in zip(sm, mean_vols):
            if d is not None:
                d.copy_(s_, non_blocking=True)
        graph.replay()
        return out

    # ---- exact posterior mean and standard deviation of region readouts (neuron traces) ----------------------------------
    def _roi_check(self, rois: RoiSet, device: torch.device):
        if not isinstance(rois, RoiSet):
            raise TypeError(f"rois must be a cwfa_b200.RoiSet, got {type(rois).__name__}")
        ch0, H, W = self.model.conv_inn[0].global_out_shapes[0]
        shape = (2 * int(ch0), int(H), int(W))
        if tuple(rois.volume_shape) != shape or rois.n_levels != self.model.n_levels:
            raise ValueError(f"the RoiSet is for {tuple(rois.volume_shape)} volumes with {rois.n_levels} levels; this model "
                             f"reconstructs {shape} volumes with {self.model.n_levels} levels")
        if rois.device != device:
            raise ValueError(f"the RoiSet is on {rois.device}, the views on {device}")

    @torch.no_grad()
    def roi_posterior_exact(self, views: torch.Tensor, mean_vols: Sequence[Optional[torch.Tensor]], rois: RoiSet,
                            temperature: Optional[float] = None, sensor: Optional[LensletLayout] = None, _side_streams=None):
        """The reconstruction and the exact posterior mean and standard deviation of every readout of ``rois`` (a neuron's
        trace value: a weighted sum over its footprint), in one inverse pass, for any batch size: ``(volume, roi_mean,
        roi_std)``, volume (B, D, H, W) bitwise ``reconstruct(views, mean_vols, temperature=0)``, roi_mean and roi_std (B, R) fp32.

        On CAT-only levels level n's detail half is affine in its latent, hi_n[e] = beta_n[e] + alpha_n[e] z_n[pi_n(e)] (alpha_n
        carried by ``coupling_f8_scale``), the levels are independent and the Haar merges are orthonormal, so for r = sum_v w_v V_v,
        exactly, E[r] = sum_v w_v V(z = 0)_v and Var[r] = sigma_T^2 sum_n sum_e (alpha_n[e] w~_n[e])^2, w~_n being level n's
        Haar detail coefficients of the weight volume (``RoiSet``).  This accounts for every covariance between the ROI's voxels:
        the per-voxel std of ``reconstruct_posterior_exact`` cannot be combined into a readout's std.  sigma_T^2 =
        ``truncated_normal_var(temperature)`` (default ``cfg.INN_z_temperature``).  Only the mean and std are exact.

        Raises ValueError as ``reconstruct_posterior_exact`` does, and for a RoiSet whose volume shape or level count is not the
        model's, or which is on another device.  ``sensor``: ``views`` is a raw sensor frame (see ``reconstruct``)."""
        sigma = self._posterior_exact_sigma(temperature)
        self._roi_check(rois, views.device)
        vol, levels = self._scale_pass(views, mean_vols, sensor, _side_streams)
        for hi8, _ in levels:
            vol = tc.haar1d_merge_f8(vol, hi8)
        roi_mean, roi_std = tc.roi_readout_f8(vol, [sc8 for _, sc8 in reversed(levels)], rois, sigma)
        return vol, roi_mean, roi_std

    def roi_posterior_exact_graphed(self, views: torch.Tensor, mean_vols: Sequence[Optional[torch.Tensor]], rois: RoiSet,
                                    temperature: Optional[float] = None, sensor: Optional[LensletLayout] = None):
        """``roi_posterior_exact`` as one CUDA-graph replay, the LRNN and the levels as parallel branches.  A graph per shapes,
        temperature and RoiSet (the graph reads its tables and keeps it alive).  The returned (volume, roi_mean, roi_std) are the
        graph's static outputs, overwritten by the next call with the same key."""
        sigma = self._posterior_exact_sigma(temperature)
        self._roi_check(rois, views.device)
        key = ("roi_posterior_exact", tuple(views.shape), tuple(None if m is None else tuple(m.shape) for m in mean_vols),
               views.device.index, sigma, id(rois), None if sensor is None else (id(sensor), views.dtype))
        g = self._graphs.get(key)
        if g is None:
            sv = views.clone()
            sm = [None if m is None else m.clone() for m in mean_vols]
            s = torch.cuda.Stream()
            s.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(s):
                for _ in range(2):
                    self.roi_posterior_exact(sv, sm, rois, temperature, sensor=sensor)
            torch.cuda.current_stream().wait_stream(s)
            graph = torch.cuda.CUDAGraph()
            side = [torch.cuda.Stream() for _ in range(self.model.n_levels + 1)] if self.parallel_branches else None
            with torch.cuda.graph(graph):
                out = self.roi_posterior_exact(sv, sm, rois, temperature, sensor=sensor, _side_streams=side)
            g = self._graphs[key] = (graph, sv, sm, out, rois, sensor)   # the graph reads the tables and the layout: keep them alive
        graph, sv, sm, out = g[:4]
        sv.copy_(views, non_blocking=True)
        for d, s_ in zip(sm, mean_vols):
            if d is not None:
                d.copy_(s_, non_blocking=True)
        graph.replay()
        return out

    def _level_forward_f8(self, n, plan, hi8, lf8, mean_vol, nll_map=False):
        ch = plan["ch"]
        jac, tickets = self._jac_and_tickets(hi8.shape[0], hi8.device)
        sumsq = torch.empty_like(jac)
        mv8 = None if mean_vol is None else tc.to_f8(mean_vol)
        map8 = torch.empty_like(hi8) if nll_map else None        # the first coupling writes every entry: no memset
        last = len(plan["out"]) - 1
        pending, k, ci = None, 0, 0
        for item in self._trunks(n, lf8):
            if item[0] == "cat":
                if map8 is None:
                    hi8 = self._couple_f8(item, plan["out"][ci], hi8, mv8, pending, False, jac, sumsq, tickets[k:k + 1])   # sumsq: last coupling wins
                else:
                    mode = (tc.NLL_MAP_FIRST if ci == 0 else 0) | (tc.NLL_MAP_LAST if ci == last else 0)
                    hi8 = self._couple_f8(item, plan["out"][ci], hi8, mv8, pending, False, jac, sumsq, tickets[k:k + 1],
                                          nll_map=map8, map_src=plan["map_src"][ci], map_mode=mode)
                pending, k, ci = None, (k + 1) % tickets.numel(), ci + 1
            elif item[2] != 1:
                pending = (item[1].perm, item[2])
        if pending is not None:
            hi8 = self._permute_f8(hi8, ch, pending[0], pending[1])     # moves z only: the map is in level-input coordinates
        z = tc.from_f8(hi8, ch, plan["z_from_storage"])
        if map8 is None:
            return z, jac, sumsq
        return z, jac, sumsq, tc.from_f8(map8, ch)

    def _level_forward(self, n, hi, lf8, mean_vol, nll_map=False):
        """Detail half of level n through the flow in the forward direction: (z, logdet[B], sumsq[B]), plus the (B, ch, H, W) NLL
        map with ``nll_map`` (F8 levels only).  ``hi``: NCHW tensor, or ("f8", tensor) from ``haar1d_split_f8`` for CAT-only levels."""
        if isinstance(hi, tuple):
            return self._level_forward_f8(n, self.levels[n]["f8"], hi[1], lf8, mean_vol, nll_map)
        jac, tickets = self._jac_and_tickets(hi.shape[0], hi.device)
        sumsq = None
        pending, k, lf_nchw = None, 0, None
        last_was_cat = False
        for item in self._trunks(n, lf8):
            if item[0] == "cat":
                sumsq = torch.empty_like(jac) if sumsq is None else sumsq
                hi = self._couple(item, hi, mean_vol, pending, False, jac, sumsq, ticket=tickets[k:k + 1])   # sumsq: last coupling wins
                pending, k, last_was_cat = None, (k + 1) % tickets.numel(), True
            elif item[0] == "perm":
                pending = (item[1].perm, item[2])
            else:
                if pending is not None:
                    hi, pending = ops.permute(hi, pending[0], pending[1]), None
                if lf_nchw is None:
                    lf_nchw = tc.from_c8(lf8)
                hi = self._run_module(item[1], hi, lf_nchw, False, jac)
                last_was_cat = False
        if pending is not None:          # trailing permutation: does not change ||z||^2
            hi = ops.permute(hi, pending[0], pending[1])
        if not last_was_cat or sumsq is None:
            sumsq = ops.sum_squares(hi)
        return hi, jac, sumsq

    @torch.no_grad()
    def forward_nll(self, volume: torch.Tensor, views: torch.Tensor, mean_vols: Sequence[torch.Tensor],
                    low_res_conditions: Optional[Sequence[torch.Tensor]] = None, _side_streams=None,
                    sensor: Optional[LensletLayout] = None, nll_map: bool = False):
        """Forward pyramid + per-level NLL (CWFA.py:966-978); same outputs as CWFAModel.forward_nll.  ``sensor``: ``views`` is
        a raw sensor frame (see ``reconstruct``).

        ``nll_map``: every level's dict also holds ``"nll_map"``, (B, ch, H, W) fp32: the NLL of each detail voxel,
        0.5 z^2 - sum over the level's couplings of s, in the coordinates of the level's detail half (``haar1d_split(x)[1]``)
        -- the couplings are elementwise, so this is exact, and ``nll_map.mean((1, 2, 3))`` is ``nll_per_sample``.  Channel c
        of level n covers depths [c 2^(n+1), (c+1) 2^(n+1)) of the volume; ``.sum(1)`` is a lateral map.  Levels without the
        F8 coupling plan (GLOW / RNVP / GIN / AI1 or tanh-clamped blocks, more than 48 detail channels, H * W not a multiple
        of 4) raise ValueError.  z, the log-dets and the NLLs are bitwise those of ``nll_map=False``.

        The conditioning nets and trunks of the four levels depend on the views only, so under CUDA-graph capture
        (``forward_nll_graphed``) they run as parallel branches next to the Haar pyramid of the volume."""
        L1 = self.model.n_levels
        if nll_map:
            self._nll_map_check(volume)
        v8 = None if self.dlr else self._views_c8(views, sensor)
        # Haar pyramid of the volume first (cheap, sequential): lo_n / hi_n of every level
        los, his = [], []
        x = volume
        for n in range(L1):
            if self.use_f8 and self.levels[n]["f8"] is not None and (x.shape[2] * x.shape[3]) % 4 == 0:
                lo, hi8 = tc.haar1d_split_f8(x)
                hi = ("f8", hi8)
            else:
                lo, hi = ops.haar1d_split(x)
            los.append(lo)
            his.append(hi)
            x = lo

        def job(n):
            if self.dlr:
                given = low_res_conditions[n] if low_res_conditions is not None and n < len(low_res_conditions) else None
                lf8 = tc.to_c8(given if given is not None else los[n], self.kind)
                return self._level_forward(n, his[n], lf8, None, nll_map)
            return self._level_forward(n, his[n], self._lf(n, v8, None), mean_vols[n], nll_map)

        if _side_streams:
            main = torch.cuda.current_stream()
            fork = torch.cuda.Event()
            fork.record(main)
            results, joins = [], []
            for st, n in zip(_side_streams, range(L1)):
                st.wait_event(fork)
                with torch.cuda.stream(st):
                    results.append(job(n))
                    ev = torch.cuda.Event()
                    ev.record(st)
                joins.append(ev)
            for ev in joins:
                main.wait_event(ev)
        else:
            results = [job(n) for n in range(L1)]
        res = []
        for n, r in enumerate(results):
            z, jac, sumsq = r[:3]
            lo = los[n]
            per = (0.5 * sumsq - jac) / z[0].numel()
            ref = (0.5 * sumsq.sum() - jac) / lo.numel()
            res.append(dict(z=z, lo=lo, logdet=jac, sumsq=sumsq, nll_per_sample=per, nll_ref=ref))
            if nll_map:
                res[-1]["nll_map"] = r[3]
        return res

    def _nll_map_check(self, volume: torch.Tensor):
        for n in range(self.model.n_levels):
            why = self._f8_unsupported(n, volume.shape[2], volume.shape[3])
            if why is not None:
                raise ValueError(f"forward_nll(nll_map=True): level {n} has no per-voxel NLL map: {why}")

    # ---- CUDA-graph replay of the forward pyramid (BASELINE.json configs[2]) ---------------------------------------------
    def forward_nll_graphed(self, volume: torch.Tensor, views: torch.Tensor, mean_vols: Sequence[torch.Tensor],
                            sensor: Optional[LensletLayout] = None, nll_map: bool = False):
        """``forward_nll`` as one CUDA-graph replay (static shapes; inputs are copied into static buffers, the returned tensors
        are the graph's static outputs, overwritten by the next call): the four levels' conditioning nets / trunks / couplings
        are parallel branches of the graph.  ``sensor``: ``views`` is a raw sensor frame; the static input is the frame in its
        own dtype and the lenslet extraction is part of the graph.  ``nll_map``: as in ``forward_nll``, a graph of its own whose
        maps are static outputs too."""
        if nll_map:
            self._nll_map_check(volume)
        key = ("nll", tuple(volume.shape), tuple(views.shape), tuple(tuple(m.shape) for m in mean_vols), volume.device.index,
               None if sensor is None else (id(sensor), views.dtype))
        if nll_map:
            key = key + ("nll_map",)
        g = self._graphs.get(key)
        if g is None:
            sx, sv, sm = volume.clone(), views.clone(), [m.clone() for m in mean_vols]
            s = torch.cuda.Stream()
            s.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(s):
                for _ in range(2):
                    self.forward_nll(sx, sv, sm, sensor=sensor, nll_map=nll_map)
            torch.cuda.current_stream().wait_stream(s)
            graph = torch.cuda.CUDAGraph()
            side = [torch.cuda.Stream() for _ in range(self.model.n_levels)] if self.parallel_branches else None
            with torch.cuda.graph(graph):
                out = self.forward_nll(sx, sv, sm, _side_streams=side, sensor=sensor, nll_map=nll_map)
            g = self._graphs[key] = (graph, sx, sv, sm, out, sensor)     # the graph reads the layout's coordinates: keep it alive
        graph, sx, sv, sm, out = g[:5]
        sx.copy_(volume, non_blocking=True)
        sv.copy_(views, non_blocking=True)
        for d, s_ in zip(sm, mean_vols):
            d.copy_(s_, non_blocking=True)
        graph.replay()
        return out

    # ---- CUDA-graph replay of the whole frame -------------------------------------------
    def _graph_slot(self, views: torch.Tensor, mean_vols, slot: int = 0, z_rows: int = 0, sensor: Optional[LensletLayout] = None):
        """(graph, static_views, static_mean_vols, static_out, static_zs) for this shape; ``slot`` selects an independent
        instance (own static buffers) so that several frames can be in flight.  ``z_rows`` > 0: the graph takes the latent
        samples of every level as inputs (``z_rows`` rows each; temperature > 0 / multi-sample reconstruction) -- they are
        sampled outside the graph into the static buffers.  ``sensor``: the static input is a raw frame in its own dtype and
        the lenslet extraction is captured in the graph."""
        key = (tuple(views.shape), tuple(None if m is None else tuple(m.shape) for m in mean_vols), views.device.index, slot, z_rows,
               None if sensor is None else (id(sensor), views.dtype))
        g = self._graphs.get(key)
        if g is None:
            sv = views.clone()
            sm = [None if m is None else m.clone() for m in mean_vols]
            sz = None
            if z_rows:
                sz = [torch.zeros((z_rows,) + tuple(self.model.conv_inn[n].global_out_shapes[0]), device=views.device, dtype=torch.float32)
                      for n in range(self.model.n_levels)]
            ns = max(1, z_rows // views.shape[0])
            s = torch.cuda.Stream()
            s.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(s):
                for _ in range(2):
                    self.reconstruct(sv, sm, zs=sz, n_samples=ns, sensor=sensor)
            torch.cuda.current_stream().wait_stream(s)
            graph = torch.cuda.CUDAGraph()
            side = [torch.cuda.Stream() for _ in range(self.model.n_levels + 1)] if (self.parallel_branches and not self.dlr) else None
            with torch.cuda.graph(graph):
                out = self.reconstruct(sv, sm, _side_streams=side, zs=sz, n_samples=ns, sensor=sensor)
            g = self._graphs[key] = (graph, sv, sm, out, sz, sensor)      # the graph reads the layout's coordinates: keep it alive
        return g

    def _fill_z(self, sz, zs, temperature):
        """Latent samples of one frame into a graph slot's static z buffers (current stream): given ``zs`` or fresh draws."""
        for n, d in enumerate(sz):
            if zs is not None and zs[n] is not None:
                d.copy_(zs[n], non_blocking=True)
            elif temperature:
                torch.nn.init.trunc_normal_(d, mean=0.0, std=1.0, a=-temperature, b=temperature)     # sample_z_truncated, CWFA.py:47-64
            else:
                d.zero_()

    def reconstruct_graphed(self, views: torch.Tensor, mean_vols: Sequence[Optional[torch.Tensor]],
                            zs: Optional[Sequence[Optional[torch.Tensor]]] = None, n_samples: int = 1,
                            temperature: Optional[float] = None, sensor: Optional[LensletLayout] = None) -> torch.Tensor:
        """Same as ``reconstruct`` but replays a captured CUDA graph (static shapes; inputs are copied into
        static buffers, the returned tensor is the graph's static output buffer).  With ``zs`` / a non-zero temperature /
        ``n_samples`` > 1 the latent samples are graph INPUTS filled before the replay.  ``sensor``: ``views`` is a raw sensor
        frame, copied as it is into the graph's frame buffer; the lenslet extraction runs inside the graph."""
        T = self.model.cfg.INN_z_temperature if temperature is None else temperature
        z_rows = views.shape[0] * n_samples if (zs is not None or T != 0 or n_samples > 1) else 0
        graph, sv, sm, out, sz = self._graph_slot(views, mean_vols, z_rows=z_rows, sensor=sensor)[:5]
        sv.copy_(views, non_blocking=True)
        for d, s_ in zip(sm, mean_vols):
            if d is not None:
                d.copy_(s_, non_blocking=True)
        if sz is not None:
            self._fill_z(sz, zs, T)
        graph.replay()
        return out

    # ---- reference-facing call with HOST buffers ------------------------------------------
    def reconstruct_host(self, views_host: torch.Tensor, mean_vols: Sequence[Optional[torch.Tensor]],
                         out_host: Optional[torch.Tensor] = None, sensor: Optional[LensletLayout] = None) -> torch.Tensor:
        """views on the HOST (pinned for full speed) -> H2D copy -> graph replay -> D2H copy of the
        reconstructed volume into ``out_host``.  The mean-volume conditions are dataset constants and
        stay resident on the device.  Returns ``out_host`` (synchronised).  ``sensor``: ``views_host`` is a raw sensor frame,
        copied in its own dtype (a uint16 frame is a third of the bytes of the fp32 views it becomes)."""
        dev = mean_vols[0].device
        attr = "_views_dev" if sensor is None else "_frame_dev"
        dtype = torch.float32 if sensor is None else views_host.dtype
        vd = getattr(self, attr, None)
        if vd is None or vd.shape != views_host.shape or vd.dtype != dtype:
            vd = torch.empty(views_host.shape, device=dev, dtype=dtype)
            setattr(self, attr, vd)
        vd.copy_(views_host, non_blocking=True)
        out = self.reconstruct_graphed(vd, mean_vols, sensor=sensor)
        if out_host is None:
            out_host = torch.empty(out.shape, dtype=torch.float32, pin_memory=True)
        out_host.copy_(out, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        return out_host


class StreamingReconstructor:
    """Streaming reconstruction of a sequence of frames (BASELINE.json configs[4]): ``depth`` independent graph
    instances, each on its own stream, so that (a) the H2D copy of frame i+1 and the D2H copy of frame i-1 overlap
    the replay of frame i, and (b) consecutive frames overlap on the GPU itself (the tail / dependency bubbles of
    one frame's graph are filled by the next frame's kernels).  Frames are independent, results are bit-identical
    to one-by-one reconstruction.  Inputs / outputs may live on the host (pinned) or on the device.
    The mean-volume pyramid is a dataset constant and stays on the device."""

    def __init__(self, engine: CWFAEngine, views_shape, mean_vols: Sequence[Optional[torch.Tensor]], depth: int = 2,
                 out_dtype: torch.dtype = torch.float32, sensor: Optional[LensletLayout] = None,
                 frame_dtype: torch.dtype = torch.uint16):
        """``out_dtype=torch.float16``: host-resident outputs are narrowed on the device (one cast kernel) so the device->host
        transfer carries half the bytes (the reference's own GPU output is fp16 under autocast, CWFA.py:845); the host buffers
        passed to ``run`` must then be fp16.

        ``sensor``: the inputs passed to ``run`` are raw sensor frames of shape ``views_shape`` ((B, 1, Hi, Wi) or (B, Hi, Wi))
        and dtype ``frame_dtype`` (uint16, float16 or float32); they are copied to the device as they are and cropped into
        views inside each frame's graph.  A uint16 2160 x 2160 frame is 9.3 MB against 30.4 MB of fp32 views."""
        if out_dtype not in (torch.float32, torch.float16):
            raise ValueError("out_dtype must be torch.float32 or torch.float16")
        if sensor is not None and frame_dtype not in (torch.uint16, torch.float16, torch.float32):
            raise ValueError("frame_dtype must be torch.uint16, torch.float16 or torch.float32")
        self.eng, self.depth, self.out_dtype = engine, depth, out_dtype
        dev = mean_vols[0].device
        probe = torch.empty(views_shape, device=dev, dtype=torch.float32 if sensor is None else frame_dtype)
        (probe.view(torch.int16) if probe.dtype == torch.uint16 else probe).zero_()      # (few torch ops take uint16)
        self.slots = [engine._graph_slot(probe, mean_vols, slot=k, sensor=sensor)[:4] for k in range(depth)]
        for (graph, sv, sm, out) in self.slots:
            for d, s_ in zip(sm, mean_vols):
                if d is not None:
                    d.copy_(s_)
        self.s_in = [torch.cuda.Stream(dev) for _ in range(depth)]
        self.s_run = [torch.cuda.Stream(dev) for _ in range(depth)]
        self.s_out = [torch.cuda.Stream(dev) for _ in range(depth)]
        self.ev_in = [torch.cuda.Event() for _ in range(depth)]
        self.ev_run = [torch.cuda.Event() for _ in range(depth)]
        self.ev_out = [torch.cuda.Event() for _ in range(depth)]
        torch.cuda.synchronize(dev)

    def _staging(self, like_in: torch.Tensor, like_out: torch.Tensor):
        """Device staging buffers for host-resident frames: the H2D copy of frame i+1 and the D2H copy of frame i-1 use
        them, so a graph slot's static input/output tensors are tied up only for a device-to-device copy."""
        if getattr(self, "_stage", None) is None:
            n = self.depth + 1
            dev = like_out.device
            self._stage = ([torch.empty_like(like_in, device=dev) for _ in range(n)],
                           [torch.empty(like_out.shape, device=dev, dtype=self.out_dtype) for _ in range(n)],
                           [torch.cuda.Event() for _ in range(n)], [torch.cuda.Event() for _ in range(n)],
                           [torch.cuda.Event() for _ in range(n)], [torch.cuda.Event() for _ in range(n)])
        return self._stage

    def run(self, views: Sequence[torch.Tensor], outs: Sequence[torch.Tensor], latency_events: Optional[list] = None) -> None:
        """Reconstructs ``views[i]`` into ``outs[i]``; returns when every output has been written.
        ``latency_events``: a list that receives one (start, end) pair of timing events per frame -- start when the frame's
        input copy is issued to the device queue position it can run at, end when its output has been written."""
        n = len(views)
        lat = latency_events
        cur = torch.cuda.current_stream()
        for st in self.s_in + self.s_run + self.s_out:
            st.wait_stream(cur)
        host_io = n > 0 and (not views[0].is_cuda or not outs[0].is_cuda)
        if host_io:
            _, sv0, _, out0 = self.slots[0]
            st_in, st_out, ev_h2d, ev_in_free, ev_staged, ev_out_free = self._staging(sv0, out0)
            ns = len(st_in)
            s_in, s_out = self.s_in[0], self.s_out[0]
            for i in range(n):
                k, j = i % self.depth, i % ns
                graph, sv, sm, out = self.slots[k]
                with torch.cuda.stream(s_in):
                    if i >= ns:
                        s_in.wait_event(ev_in_free[j])           # the slot that used this staging buffer has copied it in
                    if lat is not None:
                        e0 = torch.cuda.Event(enable_timing=True)
                        e0.record(s_in)
                    st_in[j].copy_(views[i], non_blocking=True)
                    ev_h2d[j].record(s_in)
                with torch.cuda.stream(self.s_run[k]):           # stream order serialises the replays of one slot
                    self.s_run[k].wait_event(ev_h2d[j])
                    sv.copy_(st_in[j], non_blocking=True)
                    ev_in_free[j].record(self.s_run[k])
                    graph.replay()
                    if i >= ns:
                        self.s_run[k].wait_event(ev_out_free[j]) # the D2H copy that used this staging buffer has finished
                    if self.out_dtype == torch.float16:
                        ops.cast_f16(out, st_out[j])
                    else:
                        st_out[j].copy_(out, non_blocking=True)
                    ev_staged[j].record(self.s_run[k])
                with torch.cuda.stream(s_out):
                    s_out.wait_event(ev_staged[j])
                    outs[i].copy_(st_out[j], non_blocking=True)
                    ev_out_free[j].record(s_out)
                    if lat is not None:
                        e1 = torch.cuda.Event(enable_timing=True)
                        e1.record(s_out)
                        lat.append((e0, e1))
        else:
            for i in range(n):
                k = i % self.depth
                graph, sv, sm, out = self.slots[k]
                with torch.cuda.stream(self.s_in[k]):
                    if i >= self.depth:
                        self.s_in[k].wait_event(self.ev_run[k])      # previous replay of this slot has consumed its input
                    if lat is not None:
                        e0 = torch.cuda.Event(enable_timing=True)
                        e0.record(self.s_in[k])
                    sv.copy_(views[i], non_blocking=True)
                    self.ev_in[k].record(self.s_in[k])
                with torch.cuda.stream(self.s_run[k]):
                    self.s_run[k].wait_event(self.ev_in[k])
                    if i >= self.depth:
                        self.s_run[k].wait_event(self.ev_out[k])     # previous output of this slot has been copied out
                    graph.replay()
                    self.ev_run[k].record(self.s_run[k])
                with torch.cuda.stream(self.s_out[k]):
                    self.s_out[k].wait_event(self.ev_run[k])
                    outs[i].copy_(out, non_blocking=True)
                    self.ev_out[k].record(self.s_out[k])
                    if lat is not None:
                        e1 = torch.cuda.Event(enable_timing=True)
                        e1.record(self.s_out[k])
                        lat.append((e0, e1))
        for st in self.s_out + self.s_run:
            cur.wait_stream(st)
        cur.synchronize()
