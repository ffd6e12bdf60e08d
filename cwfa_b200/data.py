"""The data formats either side of the hot path (SURVEY.md section 8f): lenslet-view extraction before it,
reference checkpoints and output de-normalisation after it.

Mirrors: ``XLFMDatasetFull.extract_views`` (XLFMDataset.py:212-242), ``serialize_INN_step`` / ``load_INN_steps``
(networks.py:708-756), checkpoint discovery of ``run_CWFA`` (CWFA.py:424-469, 488-522), de-normalisation (CWFA.py:1041).
"""
from __future__ import annotations

import argparse
import glob
import os
import re
from typing import Dict, Optional, Sequence, Tuple

import torch

from . import _lib, tc
from .ops import _stream


_IMAGE_DTYPES = {torch.float32: 0, torch.float16: 1, torch.uint16: 2}     # image_dtype codes of cwfa_extract_views(_c8)


def extract_views(image: torch.Tensor, lenslet_coords, subimage_shape: Sequence[int], mean: Optional[float] = None,
                  std: Optional[float] = None, debug: bool = False) -> torch.Tensor:
    """``(B,1,Hi,Wi)`` sensor image -> ``(B, n_lenslets, S0, S1)`` stacked views (XLFMDataset.py:212-242) in ONE gather
    kernel; with ``mean``/``std`` also ``(x - mean) / std`` (CWFA.py:797).  Output is fp32.  fp32, fp16 and uint16 (raw
    sensor) images are read as they are; any other dtype is converted to fp32 first.  For a stream of frames with fixed
    coordinates see ``LensletLayout``, which uploads them once."""
    if not image.is_cuda:
        raise RuntimeError("cwfa_b200.extract_views needs a CUDA tensor (no CPU fallback)")
    if image.dim() != 4 or image.shape[1] < 1:
        raise ValueError("image must be (B, C>=1, H, W); channel 0 is used, as in the reference")
    img = image[:, 0].contiguous()
    if img.dtype not in _IMAGE_DTYPES:
        img = img.float()
    coords = torch.as_tensor(lenslet_coords, dtype=torch.int32).reshape(-1, 2).to(image.device).contiguous()
    norm = mean is not None and std is not None
    return _views_f32(img, coords, subimage_shape, float(mean) if norm else 0.0, float(std) if norm else 1.0, norm)


def _views_f32(img: torch.Tensor, coords: torch.Tensor, subimage_shape, mean: float, std: float, norm: bool) -> torch.Tensor:
    B, Hi, Wi = img.shape
    L = coords.shape[0]
    S0, S1 = int(subimage_shape[0]), int(subimage_shape[1])
    out = torch.empty((B, L, S0, S1), device=img.device, dtype=torch.float32)
    _lib.call("cwfa_extract_views", img.data_ptr(), _IMAGE_DTYPES[img.dtype], coords.data_ptr(), out.data_ptr(), B, Hi, Wi, L,
              S0, S1, mean, std, int(norm), _stream())
    return out


class LensletLayout:
    """The lenslet geometry of a dataset, held once on the device, so that raw sensor frames become views inside a captured
    CUDA graph or a stream: ``layout = LensletLayout(coords, (512, 512), mean, std)``, then per frame
    ``layout.views(frame)`` (fp32 NCHW, identical to ``extract_views``) or ``layout.views_c8(frame, kind)`` (the tensor-core
    engine's input, bitwise equal to ``tc.to_c8(layout.views(frame), kind)`` in one pass without the fp32 views).

    Frames are ``(B, 1, Hi, Wi)`` (channel 0 is used, as in ``extract_views``) or ``(B, Hi, Wi)`` in uint16, float16 or float32,
    on the layout's device.  Neither method touches the host: no host allocation, no host-to-device copy."""

    def __init__(self, lenslet_coords, subimage_shape: Sequence[int], mean: Optional[float] = None, std: Optional[float] = None,
                 device="cuda"):
        coords = torch.as_tensor(lenslet_coords).detach()
        if coords.dim() != 2 or coords.shape[1] != 2 or coords.shape[0] < 1:
            raise ValueError(f"lenslet_coords must be (L, 2) (row, col) centres with L >= 1, got shape {tuple(coords.shape)}")
        if coords.is_floating_point() and not torch.equal(coords, coords.round()):
            raise ValueError("lenslet_coords must be integer pixel positions")
        if int(coords.min()) < -2 ** 31 or int(coords.max()) >= 2 ** 31:
            raise ValueError("lenslet_coords do not fit int32")
        if len(subimage_shape) != 2 or int(subimage_shape[0]) <= 0 or int(subimage_shape[1]) <= 0:
            raise ValueError(f"subimage_shape must be two positive view sides, got {tuple(subimage_shape)}")
        if (mean is None) != (std is None):
            raise ValueError("give both mean and std (normalised views) or neither")
        if std is not None and float(std) == 0.0:
            raise ValueError("std must be non-zero")
        device = torch.device(device)
        if device.type != "cuda":
            raise RuntimeError("cwfa_b200.LensletLayout needs a CUDA device (no CPU fallback)")
        if device.index is None:
            device = torch.device("cuda", torch.cuda.current_device())
        self.device = device
        self.coords = coords.to(torch.int32).to(device).contiguous()
        self.n_lenslets = int(coords.shape[0])
        self.subimage_shape = (int(subimage_shape[0]), int(subimage_shape[1]))
        self.normalise = mean is not None
        self.mean = float(mean) if self.normalise else 0.0
        self.std = float(std) if self.normalise else 1.0

    def _frame(self, image: torch.Tensor) -> torch.Tensor:
        """The frame as a contiguous (B, Hi, Wi) tensor of a supported dtype on the layout's device (a view when it already is)."""
        if not image.is_cuda:
            raise RuntimeError("cwfa_b200.LensletLayout needs the frame on a CUDA device (no CPU fallback)")
        if image.device != self.device:
            raise ValueError(f"frame on {image.device}, lenslet layout on {self.device}")
        if image.dtype not in _IMAGE_DTYPES:
            raise TypeError(f"frames must be uint16, float16 or float32, got {image.dtype}")
        if image.dim() == 4 and image.shape[1] >= 1:
            image = image[:, 0]
        elif image.dim() != 3:
            raise ValueError(f"frame must be (B, 1, Hi, Wi) or (B, Hi, Wi), got shape {tuple(image.shape)}")
        if not image.is_contiguous():
            image = torch.empty(image.shape, device=image.device, dtype=image.dtype).copy_(image)
        return image

    def views(self, image: torch.Tensor) -> torch.Tensor:
        """``(B, L, S0, S1)`` fp32 views of the frame, identical to ``extract_views(image, coords, shape, mean, std)``."""
        return _views_f32(self._frame(image), self.coords, self.subimage_shape, self.mean, self.std, self.normalise)

    def views_c8(self, image: torch.Tensor, kind: str = "bf16") -> tc.C8:
        """The views as a ``tc.C8`` tensor (``Cp = pad16(L)``; lenslet slots L..Cp-1 are 0) in one pass over the frame."""
        img = self._frame(image)
        B, Hi, Wi = img.shape
        S0, S1 = self.subimage_shape
        out = tc.C8.empty(B, self.n_lenslets, S0, S1, img.device, kind)
        _lib.call("cwfa_extract_views_c8", img.data_ptr(), _IMAGE_DTYPES[img.dtype], self.coords.data_ptr(), out.data.data_ptr(),
                  B, Hi, Wi, self.n_lenslets, out.Cp, S0, S1, self.mean, self.std, int(self.normalise), out.is_bf16, _stream())
        return out


_ROI_MAX_LEVELS = 8                      # the readout kernel's per-level pointer table (cwfa_roi_readout_f8)


def _roi_csr(roi: torch.Tensor, off: torch.Tensor, plus: torch.Tensor, minus: torch.Tensor, size: int, n_rois: int, scale: float):
    """CSR over ROIs of ``(offset, scale * (sum of plus - sum of minus))`` per distinct (roi, offset), entries of an ROI sorted
    by offset, exact zeros dropped.  The two sums are accumulated apart in float64 (index_add_ on the CPU, in entry order), so
    equal weights on both halves of a Haar block cancel to exactly 0 instead of to a rounding residue."""
    key = roi * size + off
    uniq, inv = torch.unique(key, sorted=True, return_inverse=True)
    p = torch.zeros(uniq.numel(), dtype=torch.float64).index_add_(0, inv, plus)
    m = torch.zeros(uniq.numel(), dtype=torch.float64).index_add_(0, inv, minus)
    val = (p - m) * scale
    keep = val != 0
    uniq, val = uniq[keep], val[keep]
    ptr = torch.zeros(n_rois + 1, dtype=torch.int64)
    ptr[1:] = torch.cumsum(torch.bincount(uniq // size, minlength=n_rois), 0)
    return ptr, (uniq % size).to(torch.int32), val.to(torch.float32)


def roi_tables(roi, voxel, weight, n_rois: int, volume_shape: Sequence[int], n_levels: int) -> Dict[str, torch.Tensor]:
    """The readout tables of ``RoiSet`` from COO triplets, in pure torch on the CPU (float64 sums, fp32 storage).

    ROI r reads ``r = sum_v w_v V[d_v, h_v, w_v]`` over its triplets ``(roi = r, voxel = (d, h, w), weight = w)``; repeated
    voxels add up.  Returns

      * ``mean_ptr`` (R + 1,) int64, ``mean_idx`` int32, ``mean_w`` fp32: a CSR over ROIs of (offset ``(d H + h) W + w`` into one
        (D, H, W) volume, summed weight);
      * ``coef_ptr`` (L, R + 1) int64, ``coef_idx`` int32, ``coef_val`` fp32: per level n a CSR over ROIs, with offsets into the
        shared ``coef_idx`` / ``coef_val`` (level n's entries follow level n - 1's), of (offset into level n's F8 scale tensor of one
        batch item, ``((i >> 3) H W + h W + w) 8 + (i & 7)``, coefficient ``w~_n[i, h, w]``).  ``w~_n`` is level n's detail half
        of the forward depth Haar analysis of the weight volume (``oracle.cwfa_oracle.haar1d``, applied n + 1 times):
        ``w~_n[i, h, w] = 2^(-(n+1)/2) (sum of w[d, h, w] over the first half of depths [i 2^(n+1), (i+1) 2^(n+1)) - sum over
        the second half)``.

    Within an ROI the entries are sorted by offset; entries that are exactly 0 are dropped.  Raises ValueError for voxels out of
    range, non-finite weights, ``roi`` outside [0, n_rois), ``n_rois < 1``, ``n_levels`` outside 1..8, and D not divisible by
    2^n_levels."""
    n_rois, n_levels = int(n_rois), int(n_levels)
    if n_rois < 1:
        raise ValueError(f"n_rois must be >= 1, got {n_rois}")
    if not 1 <= n_levels <= _ROI_MAX_LEVELS:
        raise ValueError(f"n_levels must be in 1..{_ROI_MAX_LEVELS}, got {n_levels}")
    if len(volume_shape) != 3 or any(int(s) < 1 for s in volume_shape):
        raise ValueError(f"volume_shape must be three positive sizes (D, H, W), got {tuple(volume_shape)}")
    D, H, W = (int(s) for s in volume_shape)
    if D % (1 << n_levels):
        raise ValueError(f"D = {D} is not divisible by 2^n_levels = {1 << n_levels}")
    if D * H * W >= 2 ** 31 or ((D // 2 + 7) // 8) * 8 * H * W >= 2 ** 31:
        raise ValueError(f"volume {D}x{H}x{W} is too large for the tables' int32 offsets")
    roi, voxel, weight = (torch.as_tensor(t).detach().cpu() for t in (roi, voxel, weight))
    if roi.is_floating_point() or roi.is_complex() or roi.dtype == torch.bool or roi.dim() != 1:
        raise ValueError(f"roi must be a 1-D integer array, got {roi.dtype} of shape {tuple(roi.shape)}")
    if voxel.is_floating_point() or voxel.is_complex() or voxel.dtype == torch.bool or voxel.dim() != 2 or voxel.shape[1] != 3:
        raise ValueError(f"voxel must be an (N, 3) integer array of (d, h, w), got {voxel.dtype} of shape {tuple(voxel.shape)}")
    if not (weight.is_floating_point() or weight.dtype in (torch.int32, torch.int64)) or weight.dim() != 1:
        raise ValueError(f"weight must be a 1-D float array, got {weight.dtype} of shape {tuple(weight.shape)}")
    if not roi.shape[0] == voxel.shape[0] == weight.shape[0]:
        raise ValueError(f"roi, voxel and weight have {roi.shape[0]}, {voxel.shape[0]} and {weight.shape[0]} entries")
    roi, voxel, wt = roi.long(), voxel.long(), weight.double()
    if roi.numel() and (int(roi.min()) < 0 or int(roi.max()) >= n_rois):
        raise ValueError(f"roi indices must lie in [0, {n_rois})")
    d, h, w = voxel.unbind(1)
    for name, a, n in (("d", d, D), ("h", h, H), ("w", w, W)):
        if a.numel() and (int(a.min()) < 0 or int(a.max()) >= n):
            raise ValueError(f"voxel {name} index out of range [0, {n})")
    if not bool(torch.isfinite(wt).all()):
        raise ValueError("weights must be finite")
    zero = torch.zeros_like(wt)
    mean_ptr, mean_idx, mean_w = _roi_csr(roi, (d * H + h) * W + w, wt, zero, D * H * W, n_rois, 1.0)
    ptrs, idxs, vals, base = [], [], [], 0
    for n in range(n_levels):
        i = d >> (n + 1)
        first = ((d >> n) & 1) == 0                             # first half of the 2^(n+1)-plane block of element i
        size = ((D // 2 ** (n + 1) + 7) // 8) * 8 * H * W       # one batch item of level n's F8 tensor
        off = ((i >> 3) * (H * W) + h * W + w) * 8 + (i & 7)
        ptr, idx, val = _roi_csr(roi, off, torch.where(first, wt, zero), torch.where(first, zero, wt), size, n_rois,
                                 2.0 ** (-(n + 1) / 2))
        ptrs.append(ptr + base)
        idxs.append(idx)
        vals.append(val)
        base += idx.numel()
    return dict(mean_ptr=mean_ptr, mean_idx=mean_idx, mean_w=mean_w, coef_ptr=torch.stack(ptrs),
                coef_idx=torch.cat(idxs), coef_val=torch.cat(vals))


class RoiSet:
    """Region readouts of a reconstructed volume, e.g. neuron footprints, held on the device once per recording:
    ``rois = RoiSet.from_labels(labels, n_levels)``, then per frame ``engine.roi_posterior_exact_graphed(views, mean_vols, rois)``
    gives each ROI's posterior mean and exact standard deviation.

    ``RoiSet(roi, voxel, weight, n_rois, volume_shape=(D, H, W), n_levels=L)``: COO triplets; ROI r reads
    ``sum_v w_v V[d_v, h_v, w_v]`` (soft footprints and overlapping ROIs are fine; repeated voxels add up).  ``n_levels`` is the
    model's number of flow levels.  The tables (``roi_tables``: the weights, and per level the Haar detail coefficients of the
    weight volume at the offsets of the engine's F8 scale tensors) are built on the CPU in float64, so they are the same on
    every run, then copied to ``device``.  An ROI without voxels reads 0 with std 0."""

    def __init__(self, roi, voxel, weight, n_rois: int, volume_shape: Sequence[int], n_levels: int, device="cuda"):
        t = roi_tables(roi, voxel, weight, n_rois, volume_shape, n_levels)
        self.n_rois, self.n_levels = int(n_rois), int(n_levels)
        self.volume_shape: Tuple[int, int, int] = tuple(int(s) for s in volume_shape)
        device = torch.device(device)
        if device.type == "cuda" and device.index is None:
            device = torch.device("cuda", torch.cuda.current_device())
        self.device = device
        self.n_mean_entries, self.n_coef_entries = int(t["mean_idx"].numel()), int(t["coef_idx"].numel())
        for k, v in t.items():
            if v.numel() == 0:                  # the kernel takes non-NULL pointers; no ptr range ever reaches this element
                v = torch.zeros(1, dtype=v.dtype)
            setattr(self, k, v.to(device).contiguous())

    @classmethod
    def from_labels(cls, labels, n_levels: int, device="cuda") -> "RoiSet":
        """ROIs from a (D, H, W) integer label volume: 0 is background, ROI r is label r + 1 and reads the mean over its voxels
        (weight 1 / |r|).  ``n_rois`` is the largest label; a label value that no voxel carries is an empty ROI."""
        lab = torch.as_tensor(labels).detach().cpu()
        if lab.is_floating_point() or lab.is_complex() or lab.dtype == torch.bool or lab.dim() != 3:
            raise ValueError(f"labels must be a (D, H, W) integer volume, got {lab.dtype} of shape {tuple(lab.shape)}")
        lab = lab.long()
        if lab.numel() == 0 or int(lab.max()) < 1:
            raise ValueError("labels has no positive label (0 is background)")
        if int(lab.min()) < 0:
            raise ValueError("labels must be >= 0 (0 is background)")
        vox = torch.nonzero(lab)
        roi = lab[vox[:, 0], vox[:, 1], vox[:, 2]] - 1
        n_rois = int(lab.max())
        count = torch.bincount(roi, minlength=n_rois).double()
        return cls(roi, vox, 1.0 / count[roi], n_rois, tuple(lab.shape), n_levels, device)

    @property
    def n_entries(self) -> int:
        """Table entries the readout kernel walks per batch item: the mean's and every level's coefficients."""
        return self.n_mean_entries + self.n_coef_entries


def denormalize(volume: torch.Tensor, mean_vols, std_vols) -> torch.Tensor:
    """``(vol * 2**len(vol)) * std + mean`` exactly as CWFA.py:1041 writes it (``len`` of a (B,...) tensor = B)."""
    return (volume * 2 ** len(volume)) * std_vols + mean_vols


# ---- checkpoints (networks.py:708-756) -------------------------------------------------------
def serialize_INN_step(INN, cond, optimizer, std_train_stats, args, epoch, path, posfix=""):
    step = args.INN_down_steps if hasattr(args, "INN_down_steps") else args["INN_down_steps"]
    path = path + "/model_step_" + str(step) + "__ep_" + str(epoch) + posfix
    torch.save({"epoch": epoch, "args": args,
                "INN_state_dict": INN.state_dict() if INN else None,
                "condition_state_dict": cond.state_dict() if cond else None,
                "optimizer_state_dict": optimizer.state_dict() if optimizer else None,
                "training_statistics": std_train_stats}, path)
    return path


def load_INN_steps(path, prefix="model_step_*__ep_*", epoch=-1) -> Dict[int, list]:
    """{step: [epoch, file]} keeping the highest epoch per step (or exactly ``epoch``).  networks.py:732-756."""
    found: Dict[int, list] = {}
    for m in glob.glob(path + "/" + prefix):
        step, it = map(int, re.findall(r"\d+", m.split("/")[-1])[:2])
        if epoch == -1:
            if step in found and it < found[step][0]:
                continue
            found[step] = [it, m]
        elif it == epoch:
            found[step] = [it, m]
    return found


def load_checkpoints(model, path: str, epoch: int = -1, strict: bool = True, permute_dim_axes: Optional[Dict[int, Dict[int, int]]] = None):
    """Loads reference-format step checkpoints into a ``CWFAModel`` (step k -> conv_inn[k-1] / cond_nets[k-1], as in
    CWFA.py:488-522) and returns the stored ``training_statistics`` (or None).  ``PermuteDim`` axes are not part of the
    reference's ``state_dict`` (INN_utils.py:58-61); a file written by ``save_checkpoints`` carries them as
    ``permute_dim_axes``; for files written by the reference pass ``permute_dim_axes={step: {module_idx: axis}}``.

    SECURITY: the reference format pickles an argparse.Namespace, so the files are read with ``weights_only=False`` like the
    reference does (CWFA.py:483) -- unpickling executes code: load checkpoints from TRUSTED sources only."""
    steps = load_INN_steps(path, epoch=epoch)
    stats = None
    for step, (_, fname) in sorted(steps.items()):
        data = torch.load(fname, map_location="cpu", weights_only=False)
        ix = step - 1
        if ix < model.n_levels and data.get("INN_state_dict") is not None:
            model.conv_inn[ix].load_state_dict(data["INN_state_dict"], strict=strict)
            axes = dict(data.get("permute_dim_axes") or {})
            axes.update((permute_dim_axes or {}).get(step, {}))
            for idx, axis in axes.items():
                model.conv_inn[ix].module_list[int(idx)].dims_to_permute = [1, int(axis)]
        if data.get("condition_state_dict") is not None and ix < len(model.cond_nets):
            model.cond_nets[ix].load_state_dict(data["condition_state_dict"], strict=strict)
        if stats is None:
            stats = data.get("training_statistics")
    return stats


def _args_namespace(model, args, step: int) -> argparse.Namespace:
    """The ``args`` entry of a reference checkpoint is the run's argparse.Namespace; the reference loader reads it by
    ATTRIBUTE (``args_model.INN_down_steps = ix+1``, ``.INN_internal_chans``, ``.INN_use_perm``, ``.INN_block_type``,
    ``.INN_n_blocks``, ``.INN_use_bias``, ``.INN_max_down_steps``, ``'force_last_step_NF' in args_model``; CWFA.py:486-508).
    Accepts a Namespace, a dict or None; the model's shape flags (``CWFAConfig``) fill whatever the caller did not give."""
    from dataclasses import asdict, is_dataclass
    base = vars(args) if isinstance(args, argparse.Namespace) else dict(args or {})
    cfg = asdict(model.cfg) if is_dataclass(getattr(model, "cfg", None)) else {}
    ns = argparse.Namespace(**{**cfg, **base})
    ns.INN_down_steps = step
    return ns


def save_checkpoints(model, path: str, epoch: int = 0, training_statistics=None, args=None):
    """One reference-format file per step (model_step_{k}__ep_{E}) that the reference's own loader accepts: ``args`` is an
    argparse.Namespace (see ``_args_namespace``).  Adds the PermuteDim axes as an extra key (``permute_dim_axes``), which the
    reference ignores and ``load_checkpoints`` uses (the axis is not part of the reference's state_dict, INN_utils.py:58-61)."""
    from .modules import PermuteDim
    os.makedirs(path, exist_ok=True)
    for ix in range(len(model.cond_nets)):
        inn = model.conv_inn[ix] if ix < model.n_levels else None
        a = _args_namespace(model, args, ix + 1)
        fname = serialize_INN_step(inn, model.cond_nets[ix], None, training_statistics, a, epoch, path)
        if inn is not None:
            data = torch.load(fname, weights_only=False)
            data["permute_dim_axes"] = {i: m.axis for i, m in enumerate(inn.module_list) if isinstance(m, PermuteDim)}
            torch.save(data, fname)
