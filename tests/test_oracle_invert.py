"""CPU pins of tests/oracle_invert.invert_spacing_crop (labels back onto the input grid) and of the host geometry of
val_transform(return_meta=True): known answers and round trips, no GPU."""
import numpy as np
import pytest
import torch

from diff_unet_amos_b200.inference import _pad_to_roi
from diff_unet_amos_b200.preprocess import val_meta
from oracle import oracle_preprocess as op
from tests.oracle_invert import invert_spacing_crop

PIXDIM = (1.5, 1.5, 2.0)


def test_identity_when_the_spacings_agree():
    torch.manual_seed(0)
    t = torch.randn(3, 7, 9, 11)
    for mode in ("nearest", "bilinear"):
        got = invert_spacing_crop(t, (0, 0, 0), t.shape[1:], (0, 0, 0), t.shape[1:], t.shape[1:], PIXDIM, PIXDIM, mode)
        assert torch.equal(got, t), mode


def test_trilinear_round_trip_of_a_linear_ramp():
    """A linear ramp resampled forward and back comes back wherever neither direction clamped a coordinate: linear
    interpolation of a linear function is exact up to fp32 rounding."""
    shape = (23, 31, 17)
    z, y, x = np.meshgrid(*[np.arange(n, dtype=np.float64) for n in shape], indexing="ij")
    ramp = torch.from_numpy((0.011 * z - 0.007 * y + 0.013 * x + 0.25).astype(np.float32))[None]
    for spacing_in in ((0.8, 0.8, 5.0), (2.2, 0.7, 1.0), (0.78, 0.78, 2.5)):
        res = op.spacing_resample(ramp, spacing_in, PIXDIM, "bilinear")
        back = invert_spacing_crop(res, (0, 0, 0), res.shape[1:], (0, 0, 0), shape, shape, spacing_in, PIXDIM, "bilinear")
        mask = np.ones(shape, dtype=bool)
        for d, (n, r, si, so) in enumerate(zip(shape, res.shape[1:], spacing_in, PIXDIM)):
            c = np.arange(n) * (si / so)                       # inverse coordinate on the resampled grid
            fwd_ok = np.ceil(c) * (so / si) <= n - 1           # the resampled samples it reads were not clamped either
            ok = (c <= r - 1) & fwd_ok
            mask &= ok.reshape([-1 if a == d else 1 for a in range(3)])
        assert mask.sum() > 0.5 * mask.size, spacing_in
        err = (back[0] - ramp[0]).abs().numpy()[mask]
        assert err.max() < 1e-5, (spacing_in, err.max())


def test_nearest_known_index_lists():
    """rint of clamp(j * spacing_in / pixdim, 0, res - 1), half to even: ratios 0.5, 2 and 0.78 / 1.5 on a ramp 0..5."""
    src = torch.arange(6.0).view(1, 6, 1, 1)
    cases = [
        ((0.75, 1.5, 2.0), 12, [0, 0, 1, 2, 2, 2, 3, 4, 4, 4, 5, 5]),  # 0.5, 1.5, 2.5, 3.5, 4.5 -> 0, 2, 2, 4, 4; 5.5 clamps
        ((3.0, 1.5, 2.0), 5, [0, 2, 4, 5, 5]),                          # 6 and 8 clamp to the border
        ((0.78, 1.5, 2.0), 12, [0, 1, 1, 2, 2, 3, 3, 4, 4, 5, 5, 5]),   # 0.52 j
    ]
    for spacing_in, n, want in cases:
        got = invert_spacing_crop(src, (0, 0, 0), (6, 1, 1), (0, 0, 0), (n, 1, 1), (n, 1, 1), spacing_in, PIXDIM, "nearest")
        assert got.flatten().tolist() == [float(v) for v in want], spacing_in


def test_zeros_outside_the_box_and_offset_read():
    torch.manual_seed(1)
    vol = torch.randn(2, 10, 12, 9) + 5.0                 # a padded driver volume; the resampled one sits at the offset
    offset, res = (2, 1, 0), (6, 10, 9)
    box_start, box_dims, out_shape = (3, 0, 4), (6, 10, 9), (11, 10, 15)
    for mode in ("nearest", "bilinear"):
        got = invert_spacing_crop(vol, offset, res, box_start, box_dims, out_shape, PIXDIM, PIXDIM, mode)
        assert got.shape == (2,) + out_shape
        inside = (slice(None),) + tuple(slice(s, s + n) for s, n in zip(box_start, box_dims))
        assert torch.equal(got[inside], vol[:, 2:8, 1:11, 0:9])
        outside = torch.ones(out_shape, dtype=torch.bool)
        outside[inside[1:]] = False
        assert int((got[:, outside] != 0).sum()) == 0 and int(outside.sum()) > 0


def test_val_meta_hand_worked_shapes():
    meta = val_meta((37, 45, 52), ((5, 0, 7), (37, 40, 52)), (0.8, 0.8, 5.0), PIXDIM)
    assert meta.orig_shape == (37, 45, 52) and meta.box_start == (5, 0, 7) and meta.box_end == (37, 40, 52)
    assert meta.box_shape == (32, 40, 45)
    # round((n - 1) * s_in / s_out) + 1: round(16.53) + 1, round(20.8) + 1, round(110) + 1
    assert meta.res_shape == (18, 22, 111)
    assert meta.spacing_in == (0.8, 0.8, 5.0) and meta.pixdim == PIXDIM
    # a 32^3 roi pads (18, 22, 111) to (32, 32, 111): floor of the symmetric pad on the low side
    assert meta.offset_in((32, 32, 111)) == (7, 5, 0)
    _, pad = _pad_to_roi(torch.zeros((1, 1) + meta.res_shape), (32, 32, 32))
    assert meta.offset_in((32, 32, 111)) == (pad[4], pad[2], pad[0])
    assert meta.offset_in(meta.res_shape) == (0, 0, 0)
    with pytest.raises(ValueError):
        meta.offset_in((32, 21, 111))  # smaller than the resampled volume


def test_val_meta_all_background_is_the_whole_volume():
    """crop_foreground leaves an all-background image uncropped; the box is then the whole volume."""
    meta = val_meta((20, 30, 40), ((0, 0, 0), (0, 0, 0)), (1.5, 0.75, 2.0), PIXDIM)
    assert meta.box_start == (0, 0, 0) and meta.box_end == (20, 30, 40) and meta.box_shape == (20, 30, 40)
    assert meta.res_shape == (20, 15, 40)  # round(19) + 1, round(14.5) + 1 = 15 (half to even), round(39) + 1
