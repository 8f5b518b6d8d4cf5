"""dunet_invert_labels (labels on the input grid: inverse spacing resample + inverse foreground crop + binarisation, one
kernel) against the composed path it replaces, against the oracle, and through predict_original / EngineB200."""
import ctypes
import math

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import diff_unet_amos_b200 as pkg
from diff_unet_amos_b200 import _lib
from oracle import oracle_preprocess as op
from tests.oracle_invert import invert_spacing_crop
from tests.realistic import ct_phantom_hu
from tests.util import SMALL, seeded_noise

pytestmark = pytest.mark.gpu

PIXDIM = (1.5, 1.5, 2.0)
SPACINGS = [(0.8, 0.8, 5.0), (1.5, 1.5, 2.0), (2.2, 0.7, 1.0)]
MODES = {"nearest": 0, "bilinear": 1}   # dunet_invert_labels modes
FWD_MODES = {"nearest": 1, "bilinear": 0}  # dunet_resample_spacing modes
INVALID = -1


def _p(t):
    return ctypes.c_void_p(None if t is None else t.data_ptr())


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _ratio(spacing_in):
    return (ctypes.c_double * 3)(*[si / so for si, so in zip(spacing_in, PIXDIM)])


def _kernel(blended, offset, res, box_start, box_dims, out, spacing_in, mode, binary=True, argmax=True):
    C = blended.shape[0]
    b = torch.full((C,) + tuple(out), 7, dtype=torch.uint8, device="cuda") if binary else None
    a = torch.full(tuple(out), 7, dtype=torch.uint8, device="cuda") if argmax else None
    _lib.check(_lib.load().dunet_invert_labels(_p(blended), C, _lib.i32x3(blended.shape[1:]), _lib.i32x3(offset), _lib.i32x3(res),
                                               _ratio(spacing_in), _lib.i32x3(box_start), _lib.i32x3(box_dims), _lib.i32x3(out),
                                               MODES[mode], _p(b), _p(a), _stream()))
    return b, a


def _finalize_unit(logits):
    """dunet_finalize with unit coverage counts: the binarisation and argmax of fp32 logits [C, D, H, W] on the GPU."""
    C, dims = logits.shape[0], logits.shape[1:]
    logits = logits.cuda().contiguous()
    ones = [torch.ones(n, dtype=torch.int32, device="cuda") for n in dims]
    b = torch.empty((C,) + tuple(dims), dtype=torch.uint8, device="cuda")
    a = torch.empty(tuple(dims), dtype=torch.uint8, device="cuda")
    _lib.check(_lib.load().dunet_finalize(_p(logits), _lib.i32x3(dims), C, _p(ones[0]), _p(ones[1]), _p(ones[2]), _p(b), _p(a),
                                          _stream()))
    return b, a


def _composed(blended, offset, res, box_start, box_dims, out, spacing_in, mode):
    """What a user composes by hand today: resample to the box in fp32, zero-pad to the original grid, dunet_finalize."""
    C = blended.shape[0]
    src = blended[:, offset[0]:offset[0] + res[0], offset[1]:offset[1] + res[1], offset[2]:offset[2] + res[2]].contiguous()
    boxed = torch.empty((C,) + tuple(box_dims), dtype=torch.float32, device="cuda")
    _lib.check(_lib.load().dunet_resample_spacing(_p(src), C, _lib.i32x3(res), _p(boxed), _lib.i32x3(box_dims), _ratio(spacing_in),
                                                  FWD_MODES[mode], _stream()))
    pad = []
    for d in (2, 1, 0):
        pad += [box_start[d], out[d] - box_start[d] - box_dims[d]]
    full = F.pad(boxed, pad)
    del boxed
    return _finalize_unit(full)


def _logits(C, vol, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return (torch.randn((C,) + tuple(vol), generator=g, device="cuda") * 2.0).contiguous()


def _case(spacing_in, box_dims):
    return op.resampled_shape(box_dims, spacing_in, PIXDIM)


@pytest.mark.parametrize("mode", list(MODES))
@pytest.mark.parametrize("C", [1, 3, 16])
@pytest.mark.parametrize("spacing_in", SPACINGS)
def test_kernel_equals_the_composed_path(spacing_in, C, mode):
    """Interior box on an odd original grid; the driver volume is padded around the resampled one (non-zero offset)."""
    out, box_start, box_dims = (41, 37, 29), (3, 5, 2), (33, 27, 25)
    res = _case(spacing_in, box_dims)
    vol = tuple(max(r, 32) + 1 for r in res)           # odd padding: floor on the low side
    offset = tuple((v - r) // 2 for v, r in zip(vol, res))
    assert any(offset)
    blended = _logits(C, vol, seed=C)
    kb, ka = _kernel(blended, offset, res, box_start, box_dims, out, spacing_in, mode)
    cb, ca = _composed(blended, offset, res, box_start, box_dims, out, spacing_in, mode)
    assert torch.equal(kb, cb) and torch.equal(ka, ca)
    assert 0 < int(kb.sum()) < kb.numel()
    # one output at a time: the same bytes
    assert torch.equal(_kernel(blended, offset, res, box_start, box_dims, out, spacing_in, mode, argmax=False)[0], cb)
    assert torch.equal(_kernel(blended, offset, res, box_start, box_dims, out, spacing_in, mode, binary=False)[1], ca)


@pytest.mark.parametrize("mode", list(MODES))
def test_whole_volume_box_without_padding(mode):
    spacing_in, out = (0.8, 0.8, 5.0), (23, 19, 9)
    res = _case(spacing_in, out)
    blended = _logits(3, res, seed=5)
    kb, ka = _kernel(blended, (0, 0, 0), res, (0, 0, 0), out, out, spacing_in, mode)
    cb, ca = _composed(blended, (0, 0, 0), res, (0, 0, 0), out, out, spacing_in, mode)
    assert torch.equal(kb, cb) and torch.equal(ka, ca)


def test_binary_output_beyond_2_to_the_31_bytes():
    """C * D0 * H0 * W0 > 2^31: the 64-bit indexing of the binary planes and of the argmax plane."""
    C, spacing_in, mode = 16, (0.78, 0.78, 2.5), "bilinear"
    out, box_start, box_dims = (512, 512, 520), (20, 30, 8), (460, 380, 500)
    assert C * out[0] * out[1] * out[2] > 2 ** 31
    res = _case(spacing_in, box_dims)
    blended = _logits(C, res, seed=11)
    kb, ka = _kernel(blended, (0, 0, 0), res, box_start, box_dims, out, spacing_in, mode)
    cb, ca = _composed(blended, (0, 0, 0), res, box_start, box_dims, out, spacing_in, mode)
    assert torch.equal(ka, ca)
    assert torch.equal(kb, cb)
    assert int(kb[-1, box_start[0]:box_start[0] + box_dims[0]].sum()) > 0  # the last plane was written


@pytest.mark.parametrize("mode", list(MODES))
def test_kernel_matches_the_oracle(mode):
    """The GPU labels equal dunet_finalize applied to tests/oracle_invert.invert_spacing_crop's fp32 logits."""
    for spacing_in in SPACINGS:
        out, box_start, box_dims = (30, 26, 35), (4, 0, 6), (21, 26, 24)
        res = _case(spacing_in, box_dims)
        vol = tuple(max(r, 32) for r in res)
        offset = tuple((v - r) // 2 for v, r in zip(vol, res))
        blended = _logits(4, vol, seed=3)
        ref = invert_spacing_crop(blended.cpu(), offset, res, box_start, box_dims, out, spacing_in, PIXDIM, mode)
        rb, ra = _finalize_unit(ref)
        kb, ka = _kernel(blended, offset, res, box_start, box_dims, out, spacing_in, mode)
        assert torch.equal(kb, rb) and torch.equal(ka, ra), spacing_in


def test_argument_checks():
    lib = _lib.load()
    blended = _logits(3, (12, 12, 12), seed=1)
    b = torch.zeros((3, 10, 10, 10), dtype=torch.uint8, device="cuda")
    a = torch.zeros((10, 10, 10), dtype=torch.uint8, device="cuda")
    good = dict(C=3, vol=(12, 12, 12), offset=(1, 1, 1), res=(10, 10, 10), ratio=(1.0, 1.0, 1.0), box_start=(0, 0, 0),
                box_dims=(10, 10, 10), out=(10, 10, 10), mode=0, binary=b, argmax=a)

    def call(**kw):
        k = dict(good, **kw)
        return lib.dunet_invert_labels(_p(blended), k["C"], _lib.i32x3(k["vol"]), _lib.i32x3(k["offset"]), _lib.i32x3(k["res"]),
                                       (ctypes.c_double * 3)(*k["ratio"]), _lib.i32x3(k["box_start"]), _lib.i32x3(k["box_dims"]),
                                       _lib.i32x3(k["out"]), k["mode"], _p(k["binary"]), _p(k["argmax"]), _stream())

    assert call() == 0
    assert call(binary=None, argmax=None) == INVALID
    assert call(C=0) == INVALID
    assert call(C=257, binary=None) == INVALID                       # argmax labels are uint8
    assert call(mode=2) == INVALID
    for bad in ((0.0, 1.0, 1.0), (1.0, -0.5, 1.0), (1.0, 1.0, float("inf")), (float("nan"), 1.0, 1.0)):
        assert call(ratio=bad) == INVALID, bad
    assert call(offset=(3, 1, 1)) == INVALID                         # offset + res > vol
    assert call(offset=(-1, 1, 1)) == INVALID
    assert call(box_start=(1, 0, 0)) == INVALID                      # box outside the output grid
    assert call(box_start=(0, -1, 0)) == INVALID
    for dims in ("vol", "res", "box_dims", "out"):
        bad = list(good[dims])
        bad[1] = 0
        assert call(**{dims: tuple(bad)}) == INVALID, dims
    torch.cuda.synchronize()
    # the C ABI allows more than 256 classes when only the binary planes are written
    big = _logits(257, (2, 2, 2), seed=2)
    bb = torch.empty((257, 2, 2, 2), dtype=torch.uint8, device="cuda")
    assert lib.dunet_invert_labels(_p(big), 257, _lib.i32x3((2, 2, 2)), _lib.i32x3((0, 0, 0)), _lib.i32x3((2, 2, 2)),
                                   (ctypes.c_double * 3)(1.0, 1.0, 1.0), _lib.i32x3((0, 0, 0)), _lib.i32x3((2, 2, 2)),
                                   _lib.i32x3((2, 2, 2)), 0, _p(bb), None, _stream()) == 0
    assert torch.equal(bb, _finalize_unit(big)[0])
    meta = pkg.val_meta((10, 10, 10), ((0, 0, 0), (10, 10, 10)), PIXDIM, PIXDIM)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        pkg.invert_labels(blended[:, 1:11, 1:11, 1:11].contiguous().cpu(), (10, 10, 10), meta)
    with pytest.raises(ValueError):
        pkg.invert_labels(blended, (12, 12, 12), meta, mode="cubic")


# ---- predict_original / EngineB200(space="original")

ROI, C, OVERLAP, SW = 32, 3, 0.25, 2


def _model(k):
    torch.manual_seed(0)
    return pkg.DiffUNetB200(in_channels=k, out_channels=C, image_size=ROI, spatial_size=ROI, features=SMALL).cuda().eval()


def _scan(k, shape=(44, 46, 40), radii=(15.0, 16.0), seed=3):
    """[k, D, H, W] HU: a body cylinder with air around it in D and H, plus air slabs at both ends of W."""
    chans = []
    for c in range(k):
        hu = ct_phantom_hu(shape, (shape[0] / 2, shape[1] / 2), radii, seed + c)
        hu[:, :, :3] = -1000.0
        hu[:, :, -2:] = -1000.0
        chans.append(hu)
    return torch.stack(chans).cuda()


_NOISE = []


def _nf(w, b):
    """Explicit initial noise of window w.. (the same windows get the same noise in every path compared)."""
    if not _NOISE:
        _NOISE.append(seeded_noise((64, C, ROI, ROI, ROI)).cuda())
    return _NOISE[0][w:w + b]


@pytest.mark.parametrize("interp", list(MODES))
@pytest.mark.parametrize("k", [1, 2])
def test_predict_original_end_to_end(k, interp):
    spacing_in = (0.8, 0.8, 2.5)
    m = _model(k)
    scan = _scan(k)
    got, lab = pkg.predict_original(m, scan, spacing_in, sw_batch_size=SW, overlap=OVERLAP, interp=interp, argmax=True, noise_fn=_nf)
    assert got.shape == (C,) + tuple(scan.shape[1:]) and got.dtype == torch.uint8 and lab.shape == scan.shape[1:]
    img, _, meta = pkg.val_transform(scan, None, spacing_in, return_meta=True)
    assert meta.box_start != (0, 0, 0) and meta.box_end != tuple(scan.shape[1:])
    inside = torch.zeros(scan.shape[1:], dtype=torch.bool, device="cuda")
    inside[tuple(slice(s, e) for s, e in zip(meta.box_start, meta.box_end))] = True
    assert int(got[:, ~inside].sum()) == 0 and int(lab[~inside].sum()) == 0 and int(got.sum()) > 0
    # the same pipeline composed step by step, inverted by the oracle and binarised by dunet_finalize
    (buf,) = pkg.sliding_window_inference(img[None], (ROI,) * 3, SW, m, OVERLAP, finalize=False, noise_fn=_nf, pred_type="ddim_sample")
    blended, _, _ = buf.finalize()
    assert any(v > r for v, r in zip(buf.vol, meta.res_shape))  # the driver padded: a non-zero offset was exercised
    ref = invert_spacing_crop(blended.cpu(), meta.offset_in(buf.vol), meta.res_shape, meta.box_start, meta.box_shape,
                                 meta.orig_shape, spacing_in, PIXDIM, interp)
    rb, ra = _finalize_unit(ref)
    assert torch.equal(got, rb) and torch.equal(lab, ra)


@pytest.mark.parametrize("k", [1, 2])
def test_predict_original_is_the_engine_when_nothing_is_cropped_or_resampled(k):
    """spacing_in == pixdim and a scan without air: the inverse is the identity, so the labels are EngineB200's on the
    transformed image, bit for bit."""
    m = _model(k)
    scan = _scan(k, shape=(36, 40, 34), radii=(100.0, 100.0))[:, :, :, 4:30].contiguous()  # drop the air slabs
    got = pkg.predict_original(m, scan, PIXDIM, sw_batch_size=SW, overlap=OVERLAP, noise_fn=_nf)
    img, _, meta = pkg.val_transform(scan, None, PIXDIM, return_meta=True)
    assert meta.box_shape == meta.orig_shape == meta.res_shape
    eng = pkg.EngineB200(m, sw_batch_size=SW, overlap=OVERLAP)
    ref = eng._infer_binary(img[None], noise_fn=_nf)[0]
    assert torch.equal(got, ref)


def _same(got, exp):
    return math.isnan(got) if math.isnan(exp) else got == exp


def test_engine_original_space_dice_and_hd95():
    spacing = (0.75, 0.75, 2.5)  # squares exact in fp64: HD95 bit-identical to any exact evaluation
    m = _model(1)
    names = {0: "bg", 1: "liver", 2: "spleen"}
    eng = pkg.EngineB200(m, class_names=names, sw_batch_size=SW, overlap=OVERLAP, metrics=("dice", "hd95"), space="original")
    scan = _scan(1)
    torch.manual_seed(9)
    label = (torch.rand((1, C) + tuple(scan.shape[1:])) > 0.6).float()
    label[:, 2, :20] = 0.0
    batch = {"image": scan[None].cpu(), "label": label, "spacing": torch.tensor(spacing)}
    mean = eng.validation_step(batch, noise_fn=_nf)
    pred = pkg.predict_original(m, scan, spacing, sw_batch_size=SW, overlap=OVERLAP, noise_fn=_nf)
    lab = label[0].cuda()
    dices = pkg.dice_from_counts(pkg.dice_counts(pred.flatten(1), lab.flatten(1)).cpu().tolist())
    assert list(eng.dices[-1].values()) == dices and mean == float(np.mean(dices))
    hd = pkg.hd95(pred, lab, spacing)
    assert len(eng.hd95s) == 1 and all(_same(g, e) for g, e in zip(eng.hd95s[0].values(), hd))
    unit = pkg.hd95(pred, lab, (1.0, 1.0, 1.0))  # the constructor's default spacing, which this engine must not use
    assert any(not math.isnan(e) and e != u for e, u in zip(hd, unit))
    _, outputs, _ = eng.infer({"image": scan[None], "label": label, "spacing": [list(spacing)]}, noise_fn=_nf)
    assert torch.equal(outputs[0], pred.float())
    with pytest.raises(ValueError, match="spacing"):
        eng.validation_step({"image": scan[None], "label": label}, noise_fn=_nf)
    with pytest.raises(ValueError, match="space"):
        pkg.EngineB200(m, space="resampled")
