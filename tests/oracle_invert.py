"""CPU restatement (test oracle) of the inverse of the val pre-pass: labels back on the grid of the array handed to
``val_transform``.  Helpers only, no tests; the package never imports it.

PARITY UNPINNED, like ``oracle/oracle_preprocess.py``'s forward transforms: MONAI's ``Invertd`` (undo ``Spacingd``, then
undo ``CropForegroundd`` with a zero ``BorderPad``) is restated from the published algorithm; there are no golden vectors.
"""
from typing import Sequence

import numpy as np
import torch


def invert_spacing_crop(blended: torch.Tensor, offset: Sequence[int], res_dims: Sequence[int], box_start: Sequence[int],
                        box_dims: Sequence[int], out_shape: Sequence[int], spacing_in: Sequence[float], pixdim: Sequence[float],
                        mode: str) -> torch.Tensor:
    """Inverse of ``oracle_preprocess.spacing_resample`` after ``foreground_bbox``'s crop.

    blended [C, *vol] fp32 holds the resampled volume [res_dims] at ``offset``.  Box voxel j samples it at
    clamp(j * spacing_in / pixdim, 0, res - 1) per axis -- coordinates in float64, "nearest" rint (half to even) or
    "bilinear" fp32 lerps along x, then y, then z, each as a + t * (b - a), as in ``spacing_resample``.  Returns the fp32
    logits [C, *out_shape], zero outside the box [box_start, box_start + box_dims)."""
    res = blended[:, offset[0]:offset[0] + res_dims[0], offset[1]:offset[1] + res_dims[1], offset[2]:offset[2] + res_dims[2]]
    coords = [np.clip(np.arange(n, dtype=np.float64) * (float(si) / float(so)), 0.0, float(r - 1))
              for n, r, si, so in zip(box_dims, res_dims, spacing_in, pixdim)]
    if mode == "nearest":
        iz, iy, ix = [torch.from_numpy(np.rint(c).astype(np.int64)) for c in coords]
        inner = res[:, iz][:, :, iy][:, :, :, ix]
    else:
        lo = [np.floor(c).astype(np.int64) for c in coords]
        hi = [np.minimum(l + 1, r - 1) for l, r in zip(lo, res_dims)]
        fr = [torch.from_numpy((c - l).astype(np.float32)) for c, l in zip(coords, lo)]
        lo = [torch.from_numpy(v) for v in lo]
        hi = [torch.from_numpy(v) for v in hi]

        def lerp(a, b, w):
            return a + w * (b - a)

        def take(zi, yi):
            plane = res[:, zi][:, :, yi]
            return lerp(plane[..., lo[2]], plane[..., hi[2]], fr[2][None, None, None, :])

        fy = fr[1][None, None, :, None]
        fz = fr[0][None, :, None, None]
        inner = lerp(lerp(take(lo[0], lo[1]), take(lo[0], hi[1]), fy), lerp(take(hi[0], lo[1]), take(hi[0], hi[1]), fy), fz)
    out = torch.zeros((blended.shape[0],) + tuple(out_shape), dtype=torch.float32)
    out[:, box_start[0]:box_start[0] + box_dims[0], box_start[1]:box_start[1] + box_dims[1],
        box_start[2]:box_start[2] + box_dims[2]] = inner
    return out
