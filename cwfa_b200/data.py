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
