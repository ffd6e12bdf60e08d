"""Model assembly and the drivers of the hot path: inverse reconstruction and forward NLL.

Mirrors the parts of the reference's ``run_CWFA`` that touch the flow:
model assembly CWFA.py:478-529, inverse loop CWFA.py:865-924, forward pyramid / NLL
CWFA.py:156-196 and :966-978.  Training loop, metrics, TIFF/TensorBoard output are out of
scope (SURVEY.md section 8).
"""
from __future__ import annotations

import math
from dataclasses import dataclass, asdict
from typing import List, Optional, Sequence

import numpy as np
import torch
import torch.nn as nn

from . import networks, ops


@dataclass
class CWFAConfig:
    """Shape-relevant flags of the reference's argparse namespace (main.py:65-110 defaults)."""
    n_depths: int = 96
    volume_side_size: int = 512
    INN_max_down_steps: int = 5
    INN_n_blocks: int = 4
    INN_internal_chans: int = 64
    INN_cond_chans: int = 32
    INN_block_type: str = "CAT"
    INN_use_perm: int = 1
    INN_use_bias: int = 1
    INN_z_temperature: float = 0.0
    disable_low_res_input: int = 0
    n_views: int = 29


def lrnn_mean_volume(mean_vols: Sequence[Optional[torch.Tensor]], n_levels: int) -> Optional[torch.Tensor]:
    """The mean volume the LRNN receives.  The reference calls ``cond_nets[L-1](views, mean_vols_cache[n_net-1])`` (CWFA.py:882),
    i.e. the mean-volume condition of the LAST flow level (index L-2), so a list with one entry per flow level -- the
    reference's ``mean_vols_cache`` -- gives exactly that.  An explicit extra entry ``mean_vols[L-1]`` overrides it
    (``None`` = run the LRNN without its mean-volume branch, ``Encoder(im)``, networks.py:581-582)."""
    if len(mean_vols) > n_levels:
        return mean_vols[n_levels]
    return mean_vols[n_levels - 1] if n_levels >= 1 else None


class CWFAModel(nn.Module):
    """``conv_inn[n]`` (flow level n, n < L-1), ``cond_nets[n]`` (conditioning nets, last one is the
    LRNN ``Encoder``) exactly as ``run_CWFA`` assembles them (CWFA.py:478-529)."""

    def __init__(self, cfg: Optional[CWFAConfig] = None, seed: Optional[int] = None, **overrides):
        super().__init__()
        cfg = cfg or CWFAConfig()
        for k, v in overrides.items():
            if not hasattr(cfg, k):
                raise TypeError(f"unknown config field {k!r}")
            setattr(cfg, k, v)
        self.cfg = cfg
        if seed is not None:
            torch.manual_seed(seed)
            np.random.seed(seed)
        D, S, L = cfg.n_depths, cfg.volume_side_size, cfg.INN_max_down_steps
        if D % (2 ** (L - 1)) != 0:
            raise ValueError(f"n_depths={D} is not divisible by 2^{L-1}")
        self.conv_inn = nn.ModuleList()
        self.cond_nets = nn.ModuleList()
        for ix in range(L - 1):
            ch = D // 2 ** (ix + 1)
            ctor = lambda ch=ch, ix=ix: networks.cond_network(cfg.n_views, ch, ix + 1, L, [], cfg.INN_cond_chans)
            cn, graphs = networks.conditional_wavelet_flow(
                input_volume_shape=[D, S, S], condition_shape=[1, cfg.n_views, S, S],
                st_subnet=networks.wavelet_flow_subnetwork2D, conditional_network=ctor,
                n_internal_ch=cfg.INN_internal_chans, n_down_steps=ix + 1,
                use_permutations=cfg.INN_use_perm == 1, block_type=cfg.INN_block_type,
                n_blocks=cfg.INN_n_blocks, disable_low_res_input=bool(cfg.disable_low_res_input))
            self.conv_inn.append(graphs[ix])
            self.cond_nets.append(cn)
        self.cond_nets.append(networks.Encoder(cfg.n_views, D // 2 ** (L - 1), L, cfg.INN_internal_chans,
                                               cfg.INN_use_bias, size=S))
        # reference: everything .eval(), then the LRNN back to .train() (CWFA.py:528-532)
        self.eval()
        self.cond_nets[-1].train()

    @property
    def n_levels(self) -> int:
        return len(self.conv_inn)

    # ---- inverse reconstruction (CWFA.py:865-924) -------------------------------------------
    def level_conditions(self, n: int, views: torch.Tensor, mean_vols: Sequence[Optional[torch.Tensor]], low_res: torch.Tensor):
        """The condition list of flow level n as the reference's driver assembles it (CWFA.py:891-901):
        ``[cond_net(views), mean_vols_cache[n]]``, or -- with ``disable_low_res_input=1`` -- the single condition
        ``[low_res]`` (the volume of the level below: the previous up-sampled reconstruction in the inverse loop)."""
        if self.cfg.disable_low_res_input:
            return [low_res]
        return [self.cond_nets[n](views)[-1], mean_vols[n]]

    @torch.no_grad()
    def reconstruct(self, views: torch.Tensor, mean_vols: Sequence[Optional[torch.Tensor]],
                    zs: Optional[Sequence[torch.Tensor]] = None, return_all: bool = False,
                    n_samples: int = 1, temperature: Optional[float] = None):
        """views (B,29,S,S) normalised lenslet views; mean_vols[n] the mean-volume delta condition of
        level n (n < L-1) -- the reference's ``mean_vols_cache``; the LRNN receives ``mean_vols[L-2]`` as in CWFA.py:882
        unless an extra entry ``mean_vols[L-1]`` (a tensor, or None for no mean-volume branch) is supplied
        (``lrnn_mean_volume``).  z = 0 unless ``zs`` is given or ``temperature`` (default ``cfg.INN_z_temperature`` = 0,
        CWFA.py:906-907) is non-zero, in which case z ~ ``sample_z_truncated``.

        ``n_samples`` > 1 at batch 1 is the reference's multi-sample path (``INN_n_samples``, CWFA.py:903-914): every level
        runs on ``n_samples`` copies of (low-res volume, conditions) with independent z and the level output is the mean over
        the samples.  ``zs[n]`` then has ``n_samples`` rows."""
        L1 = self.n_levels
        T = self.cfg.INN_z_temperature if temperature is None else temperature
        if n_samples > 1 and views.shape[0] != 1:
            raise ValueError("n_samples > 1 needs batch size 1 (CWFA.py:904: n_samples = INN_n_samples if batch_size == 1 else 1)")
        mv_last = lrnn_mean_volume(mean_vols, L1)
        vol = self.cond_nets[L1](views, mv_last)[-1]
        outs, jacs = {L1: vol}, {}
        for n in range(L1 - 1, -1, -1):
            inn = self.conv_inn[n]
            conds = self.level_conditions(n, views, mean_vols, vol)
            rows = vol.shape[0] * n_samples
            if zs is not None and zs[n] is not None:
                z = zs[n]
            else:
                z = sample_z_truncated((rows,) + tuple(inn.global_out_shapes[0]), device=vol.device, temperature=T)
            if n_samples > 1:
                vol = vol.repeat(n_samples, 1, 1, 1)
                conds = [c.repeat(n_samples, 1, 1, 1) for c in conds]
            vol, jac = inn([z, vol], c=conds, rev=True)
            if n_samples > 1:
                vol = ops.batch_mean(vol)                               # upsampled_vol.mean(0).unsqueeze(0), CWFA.py:913-914
            outs[n], jacs[n] = vol, jac
        return (outs, jacs) if return_all else vol

    # ---- forward pyramid + NLL (CWFA.py:156-196, :966-978) -------------------------------------
    @torch.no_grad()
    def forward_nll(self, volume: torch.Tensor, views: torch.Tensor, mean_vols: Sequence[torch.Tensor],
                    low_res_conditions: Optional[Sequence[torch.Tensor]] = None):
        """Per level: z, lo, logdet[B], sumsq[B], nll_per_sample[B] = (0.5*sumsq - logdet)/(ch*P) and the
        reference's batch-coupled ``nll_ref`` = (0.5*||Z||^2_batch - logdet)/lo.numel() (CWFA.py:183-189).
        With ``disable_low_res_input=1`` the single condition of level n is ``low_res_conditions[n]`` (what the training step
        passes: the reconstruction of the level below, CWFA.py:900-901,966); by default the volume's own low-resolution half."""
        res = []
        x = volume
        for n in range(self.n_levels):
            if self.cfg.disable_low_res_input:
                given = low_res_conditions[n] if low_res_conditions is not None and n < len(low_res_conditions) else None
                conds = [given if given is not None else ops.haar1d_split(x)[0]]
            else:
                conds = self.level_conditions(n, views, mean_vols, None)
            (z, lo), jac = self.conv_inn[n](x, c=conds)
            sumsq = ops.sum_squares(z)
            per = (0.5 * sumsq - jac) / z[0].numel()
            ref = (0.5 * sumsq.sum() - jac) / lo.numel()
            res.append(dict(z=z, lo=lo, logdet=jac, sumsq=sumsq, nll_per_sample=per, nll_ref=ref))
            x = lo
        return res

    # ---- the reference's GT-pyramid pass (CWFA.py:134-196) ----------------------------------------
    @torch.no_grad()
    def evaluate_INN_forward(self, gt_volume: torch.Tensor, extra_cond_in=None, fix_empty_depths: bool = True):
        """``evaluate_INN_forward`` of the reference: the forward pyramid with ZERO LF conditions (and zero or given
        mean-volume conditions), used to build the low-resolution ground-truth cache.  Returns
        ``(losses, gt_cache, prior_errors, log_jacobians)`` with the reference's batch-coupled formulas
        (CWFA.py:183-192).  ``check_empty_depths`` (CWFA.py:84-96) adds N(0, 1e-3) noise to all-constant depth
        columns; disable it for deterministic runs."""
        if fix_empty_depths:
            gt_volume = check_empty_depths(gt_volume)
        losses, prior_errors, log_jacobians = [], [], []
        gt_cache = [None] * self.cfg.INN_max_down_steps
        gt_cache[0] = gt_volume
        for n in range(self.n_levels):
            inn = self.conv_inn[n]
            B = gt_volume.shape[0]
            cond_in = [torch.zeros((B,) + tuple(inn.dims_c[0]), device=gt_volume.device)]
            if len(inn.dims_c) > 1:
                cond_in.append(torch.zeros((B,) + tuple(inn.dims_c[1]), device=gt_volume.device) if extra_cond_in is None
                               else extra_cond_in[n].clone())
            Z, log_jac_det = inn(gt_volume, c=cond_in)
            err = ops.sum_squares(Z[0]).sum()                       # torch.norm(Z)**2 over the whole batch
            loss = (0.5 * err - log_jac_det) / Z[-1].numel()
            losses.append(loss.mean())
            prior_errors.append(0.5 * err / Z[-1].numel())
            log_jacobians.append(log_jac_det.mean() / Z[-1].numel())
            gt_volume = Z[1]
            gt_cache[n + 1] = gt_volume
        return losses, gt_cache, prior_errors, log_jacobians

    # ---- test / bench helper ---------------------------------------------------------------
    def export_for_oracle(self) -> dict:
        """CPU copies of all state_dicts plus the per-level node specs, in the structure
        oracle/cwfa_oracle.py consumes.  (The oracle itself is never imported by this package.)"""
        cpu = lambda sd: {k: v.detach().cpu().clone() for k, v in sd.items()}
        levels = [dict(inn=cpu(self.conv_inn[n].state_dict()), cond=cpu(self.cond_nets[n].state_dict()),
                       spec=networks.level_spec(self.conv_inn[n])) for n in range(self.n_levels)]
        return dict(levels=levels, lrnn=cpu(self.cond_nets[-1].state_dict()), config=asdict(self.cfg))


def check_empty_depths(gt_volume: torch.Tensor) -> torch.Tensor:
    """CWFA.py:84-96: pixels whose depth column is constant get N(0, 1e-3) noise on all depths (host-level data hygiene)."""
    empty = gt_volume.std(dim=1, keepdim=True) == 0
    if bool(empty.any()):
        gt_volume = gt_volume + empty * torch.normal(0.0, 0.001, gt_volume.shape, device=gt_volume.device)
    return gt_volume


def sample_z_truncated(shape, device="cpu", temperature: float = 1.0) -> torch.Tensor:
    """CWFA.py:47-64: zeros at temperature 0, otherwise a normal truncated to [-T, T] with std T.  (The reference's
    non-zero branch raises NameError because ``_no_grad_trunc_normal_`` is never imported, SURVEY.md section 0 item 5.)"""
    z = torch.zeros(tuple(shape), device=device)
    if temperature != 0:
        torch.nn.init.trunc_normal_(z, mean=0.0, std=1.0, a=-temperature, b=temperature)
    return z


def truncated_normal_var(temperature: float) -> float:
    """Variance of one ``sample_z_truncated`` draw: a unit normal truncated to [-T, T], 1 - 2 T phi(T) / (2 Phi(T) - 1), in double
    precision; 0 at T = 0 (z = 0).  sigma_T = 0.39105 at T = 0.7."""
    T = float(temperature)
    if not (T >= 0.0 and math.isfinite(T)):
        raise ValueError(f"temperature must be finite and >= 0, got {temperature}")
    if T < 1e-3:
        return T * T / 3.0 * (1.0 - 2.0 * T * T / 15.0)      # series: the closed form cancels to nothing as T -> 0
    return 1.0 - 2.0 * T * math.exp(-0.5 * T * T) / math.sqrt(2.0 * math.pi) / math.erf(T / math.sqrt(2.0))
