"""Input side of the path as a GPU pre-pass (SURVEY 8f-3): the array transforms of the reference's validation pipeline
(utils.py:165-181) that run between file loading and the window driver,

    ScaleIntensityRanged(a_min=-175, a_max=250, b_min=0, b_max=1, clip=True)          utils.py:167-170
    CropForegroundd(keys=["image", "label"], source_key="image")                      utils.py:171
    Spacingd(pixdim=(1.5, 1.5, 2.0), mode=("bilinear", "nearest"))                    utils.py:173-177

as CUDA kernels through the C ABI.  LoadImaged (NIfTI decoding) and Orientationd (an axis permutation / flip decided by
the file's affine) stay on the CPU side: they are file-format logic, not array arithmetic (out of scope, DESIGN.md).
Tensors are [C, D, H, W] fp32 on the GPU; there is no CPU fallback.
"""
from __future__ import annotations

import ctypes
from dataclasses import dataclass
from typing import Optional, Sequence, Tuple

import torch

from . import _lib
from .inference import scale_intensity_range


def _ptr(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _chw(t: torch.Tensor, name: str) -> torch.Tensor:
    if not t.is_cuda:
        raise RuntimeError(f"{name} must be a CUDA tensor: the B200 path has no CPU fallback")
    if t.dim() != 4:
        raise ValueError(f"{name} must be [C, D, H, W], got {tuple(t.shape)}")
    return t.float().contiguous()


def foreground_bbox(image: torch.Tensor) -> Tuple[Tuple[int, int, int], Tuple[int, int, int]]:
    """(start, end) of the bounding box of ``image > 0`` over all channels (MONAI generate_spatial_bounding_box with
    select_fn=is_positive, margin=0); end is exclusive.  An all-background image gives the empty box ((0,0,0),(0,0,0))
    like MONAI's fallback."""
    image = _chw(image, "image")
    box = torch.empty(6, dtype=torch.int32, device=image.device)
    with torch.cuda.device(image.device):
        _lib.check(_lib.load().dunet_foreground_bbox(_ptr(image), image.shape[0], _lib.i32x3(image.shape[1:]), _ptr(box), _stream()))
    b = box.cpu().tolist()
    if b[3] <= b[0]:
        return (0, 0, 0), (0, 0, 0)
    return tuple(b[:3]), tuple(b[3:])


def crop_box(t: torch.Tensor, start: Sequence[int], end: Sequence[int]) -> torch.Tensor:
    t = _chw(t, "tensor")
    size = tuple(int(e) - int(s) for s, e in zip(start, end))
    out = torch.empty((t.shape[0],) + size, dtype=torch.float32, device=t.device)
    with torch.cuda.device(t.device):
        _lib.check(_lib.load().dunet_crop_box(_ptr(t), t.shape[0], _lib.i32x3(t.shape[1:]), _ptr(out), _lib.i32x3(size), _lib.i32x3(start),
                                              _stream()))
    return out


def crop_foreground(image: torch.Tensor, label: Optional[torch.Tensor] = None):
    """CropForegroundd(keys=["image", "label"], source_key="image"): both tensors cropped to the image's foreground box."""
    start, end = foreground_bbox(image)
    if end == (0, 0, 0):  # nothing positive: MONAI keeps a degenerate box; keep the tensors unchanged instead of emptying them
        return (image, label, (start, end)) if label is not None else (image, (start, end))
    img = crop_box(image, start, end)
    if label is None:
        return img, (start, end)
    return img, crop_box(label, start, end), (start, end)


def resampled_shape(shape: Sequence[int], spacing_in: Sequence[float], pixdim: Sequence[float]) -> Tuple[int, ...]:
    """MONAI compute_shape_offset (scale_extent=False) for axis-aligned affines: round((n - 1) * s_in / s_out) + 1."""
    return tuple(int(round((n - 1) * float(si) / float(so))) + 1 for n, si, so in zip(shape, spacing_in, pixdim))


def spacing_resample(t: torch.Tensor, spacing_in: Sequence[float], pixdim: Sequence[float] = (1.5, 1.5, 2.0),
                     mode: str = "bilinear") -> torch.Tensor:
    """Spacingd for an axis-aligned affine: output voxel i samples the input at index i * pixdim / spacing_in."""
    t = _chw(t, "tensor")
    if mode not in ("bilinear", "nearest"):
        raise NotImplementedError(f"mode {mode!r}: the reference uses ('bilinear', 'nearest')")
    out_shape = resampled_shape(t.shape[1:], spacing_in, pixdim)
    ratio = (ctypes.c_double * 3)(*[float(so) / float(si) for si, so in zip(spacing_in, pixdim)])
    out = torch.empty((t.shape[0],) + out_shape, dtype=torch.float32, device=t.device)
    with torch.cuda.device(t.device):
        _lib.check(_lib.load().dunet_resample_spacing(_ptr(t), t.shape[0], _lib.i32x3(t.shape[1:]), _ptr(out), _lib.i32x3(out_shape), ratio,
                                                      0 if mode == "bilinear" else 1, _stream()))
    return out


@dataclass(frozen=True)
class ValTransformMeta:
    """Geometry of one ``val_transform`` call, what its inverse (``invert_labels``) needs: the shape of the array handed
    to ``val_transform`` (the "original" grid), the foreground box [box_start, box_end) on it, the two spacings and the
    resampled shape of the box."""
    orig_shape: Tuple[int, int, int]
    box_start: Tuple[int, int, int]
    box_end: Tuple[int, int, int]
    spacing_in: Tuple[float, float, float]
    pixdim: Tuple[float, float, float]
    res_shape: Tuple[int, int, int]

    @property
    def box_shape(self) -> Tuple[int, ...]:
        return tuple(e - s for s, e in zip(self.box_start, self.box_end))

    def offset_in(self, vol: Sequence[int]) -> Tuple[int, ...]:
        """Corner of the resampled volume inside the window driver's volume ``vol``: the driver pads a volume smaller than
        the roi symmetrically, with the floor on the low side (``crop_to``)."""
        if len(vol) != 3 or any(int(v) < r for v, r in zip(vol, self.res_shape)):
            raise ValueError(f"driver volume {tuple(vol)} does not contain the resampled volume {self.res_shape}")
        return tuple((int(v) - r) // 2 for v, r in zip(vol, self.res_shape))


def val_meta(shape: Sequence[int], box, spacing_in: Sequence[float], pixdim: Sequence[float]) -> ValTransformMeta:
    """Host arithmetic of ``val_transform(return_meta=True)``: ``box`` is ``foreground_bbox``'s (start, end).  An
    all-background image, which ``crop_foreground`` leaves uncropped, has the whole volume as its box."""
    shape = tuple(int(n) for n in shape)
    start, end = (tuple(int(v) for v in b) for b in box)
    if end == (0, 0, 0):
        start, end = (0, 0, 0), shape
    box_shape = tuple(e - s for s, e in zip(start, end))
    return ValTransformMeta(shape, start, end, tuple(float(s) for s in spacing_in), tuple(float(p) for p in pixdim),
                            resampled_shape(box_shape, spacing_in, pixdim))


def val_transform(image: torch.Tensor, label: Optional[torch.Tensor], spacing_in: Sequence[float],
                  pixdim: Sequence[float] = (1.5, 1.5, 2.0), return_meta: bool = False):
    """The array part of ``transform["val"]`` (utils.py:165-181): intensity scaling, foreground crop, spacing resample.
    image: [in_channels, D, H, W] raw intensities; label: [L, D, H, W] or None.  Returns (image, label), and with
    ``return_meta=True`` (image, label, ValTransformMeta) for ``invert_labels``.  Every kernel
    here is channel-generic: the intensity window applies to every channel (as MONAI's ScaleIntensityRanged does), the
    foreground box is taken over all channels, and each channel is resampled on the same grid.  The CT window
    (-175, 250) HU is the reference's; other modalities need their own normalisation before the window driver."""
    image = scale_intensity_range(_chw(image, "image"))
    shape = tuple(image.shape[1:])
    if label is not None:
        image, label, box = crop_foreground(image, _chw(label, "label"))
        label = spacing_resample(label, spacing_in, pixdim, "nearest")
    else:
        image, box = crop_foreground(image)
    image = spacing_resample(image, spacing_in, pixdim, "bilinear")
    if not return_meta:
        return image, label
    return image, label, val_meta(shape, box, spacing_in, pixdim)
