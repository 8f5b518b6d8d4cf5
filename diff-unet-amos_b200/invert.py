"""Output side of the validation pre-pass: labels on the grid of the array handed to ``val_transform``.

MONAI's answer is ``Invertd(keys="pred", transform=val_transforms, orig_keys="image")`` (undo Spacingd, then
CropForegroundd's crop as a zero BorderPad) followed by ``AsDiscreted``.  Here that is one CUDA kernel,
``dunet_invert_labels``: it reads the finalised fp32 volume of the window driver and writes uint8 labels on the original
grid, so no fp32 volume of the original grid is ever formed.  Orientationd and the NIfTI affine stay file-side.
"""
from __future__ import annotations

import ctypes
from typing import Optional, Sequence

import torch

from . import _lib
from .inference import sliding_window_inference
from .preprocess import ValTransformMeta, val_transform

INTERP_MODES = {"nearest": 0, "bilinear": 1}  # kernel modes; nearest is Invertd's default (nearest_interp=True)


def _ptr(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def invert_labels(blended: torch.Tensor, vol: Sequence[int], meta: ValTransformMeta, mode: str = "nearest", binary: bool = True,
                  argmax: bool = False):
    """Labels on the original grid from the finalised blended volume of the window driver.

    blended: fp32 [C, *vol], what ``StitchBuffers.finalize()`` leaves in ``StitchBuffers.out`` (divided by the coverage; any
    blend mode or ensemble count); ``vol`` is the driver's volume shape (``StitchBuffers.vol``), which holds the resampled
    volume ``meta.res_shape`` at ``meta.offset_in(vol)``.  ``mode``: "nearest" (Invertd's nearest_interp=True) or "bilinear"
    (trilinear, nearest_interp=False).  Returns (binary uint8 [C, *orig_shape] or None, argmax uint8 [*orig_shape] or None):
    sigmoid > 0.5 per class and the first-maximum class, 0 outside the foreground box."""
    if not blended.is_cuda:
        raise RuntimeError("invert_labels runs on the GPU only (no CPU fallback)")
    if mode not in INTERP_MODES:
        raise ValueError(f"mode must be one of {tuple(INTERP_MODES)}, got {mode!r}")
    if not (binary or argmax):
        raise ValueError("nothing to compute: binary and argmax are both False")
    vol = tuple(int(v) for v in vol)
    if blended.dtype != torch.float32 or blended.dim() != 4 or tuple(blended.shape[1:]) != vol or not blended.is_contiguous():
        raise ValueError(f"blended must be contiguous fp32 [C, *vol] with vol = {vol}, got {blended.dtype} {tuple(blended.shape)}")
    C = blended.shape[0]
    out = meta.orig_shape
    b = torch.empty((C,) + out, dtype=torch.uint8, device=blended.device) if binary else None
    a = torch.empty(out, dtype=torch.uint8, device=blended.device) if argmax else None
    ratio = (ctypes.c_double * 3)(*[si / so for si, so in zip(meta.spacing_in, meta.pixdim)])
    with torch.cuda.device(blended.device):
        _lib.check(_lib.load().dunet_invert_labels(_ptr(blended), C, _lib.i32x3(vol), _lib.i32x3(meta.offset_in(vol)),
                                                   _lib.i32x3(meta.res_shape), ratio, _lib.i32x3(meta.box_start),
                                                   _lib.i32x3(meta.box_shape), _lib.i32x3(out), INTERP_MODES[mode], _ptr(b),
                                                   _ptr(a), _stream()))
    return b, a


@torch.no_grad()
def predict_original(model, image: torch.Tensor, spacing_in: Sequence[float], pixdim: Sequence[float] = (1.5, 1.5, 2.0),
                     sw_batch_size: int = 4, overlap: float = 0.25, interp: str = "nearest", argmax: bool = False,
                     seed: Optional[int] = None, noise_fn=None, ensemble: int = 1, mode: str = "constant"):
    """Segment one raw-intensity volume and return the labels on its own grid.

    image: [in_channels, D, H, W] raw intensities (HU for CT) on the GPU, spacing_in its voxel spacing per array axis.
    Runs ``val_transform`` (intensity window, foreground crop, resample to ``pixdim``), the fused sliding-window DDIM
    driver (``seed`` / ``noise_fn`` / ``ensemble`` / ``mode`` as in ``sliding_window_inference``; window indices start at 0),
    the division by the coverage and ``invert_labels``.  Returns uint8 binary [C, D, H, W], or (binary, argmax [D, H, W])
    with ``argmax=True``."""
    if image.dim() != 4:
        raise ValueError(f"image must be [in_channels, D, H, W], got {tuple(image.shape)}")
    img, _, meta = val_transform(image, None, spacing_in, pixdim, return_meta=True)
    (buf,) = sliding_window_inference(img[None], model.patch, sw_batch_size, model, overlap, mode=mode, finalize=False,
                                      noise_fn=noise_fn, seed=seed, ensemble=ensemble, pred_type="ddim_sample")
    blended, _, _ = buf.finalize()
    b, a = invert_labels(blended, buf.vol, meta, interp, binary=True, argmax=argmax)
    return (b, a) if argmax else b
