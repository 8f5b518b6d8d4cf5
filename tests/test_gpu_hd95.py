"""dunet_hd95 (per-class HD95 surface distance on the GPU) against the scipy / numpy oracle, oracle/oracle_hd95.hd95.
Bit-identical wherever the squared spacing terms are exact in fp64; within 1e-12 relative otherwise."""
import ctypes
import math

import numpy as np
import pytest
import torch
from scipy.ndimage import gaussian_filter

import diff_unet_amos_b200 as pkg
from diff_unet_amos_b200 import _lib
from oracle import oracle_hd95
from tests.util import SMALL, seeded_image, seeded_noise

pytestmark = pytest.mark.gpu

EXACT_SPACINGS = [(1.0, 1.0, 1.0), (2.0, 1.5, 1.5)]
INEXACT_SPACING = (0.7, 0.8, 2.5)


def _p(t, offset=0):
    return ctypes.c_void_p(t.data_ptr() + offset)


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _same(got, exp, rel=0.0):
    if math.isnan(exp):
        return math.isnan(got)
    return got == exp if rel == 0.0 else abs(got - exp) <= rel * abs(exp)


def _oracle_cropped(a, b, spacing):
    """The oracle on the bounding box of a | b grown by one voxel (clipped to the volume).  Inside that crop both
    borders are the same voxels as in the whole volume, and every distance between them is the same, so the result
    equals the whole-volume oracle; it keeps the 512 x 512 x 160 comparisons affordable on the host."""
    fg = np.argwhere(a | b)
    if len(fg) == 0:
        return float("nan")
    lo = np.maximum(fg.min(0) - 1, 0)
    hi = np.minimum(fg.max(0) + 2, a.shape)
    sl = tuple(slice(int(l), int(h)) for l, h in zip(lo, hi))
    return oracle_hd95.hd95(a[sl], b[sl], spacing)


def _blobs(shape=(37, 53, 29), seed=0):
    """4 classes of seeded smooth blobs: 0 touches the volume edge, 1 is a single voxel, 2 is a shell with a cavity,
    3 is a generic blob.  Returns (pred, label) bool [4, D, H, W]."""
    rng = np.random.default_rng(seed)
    C = 4
    label, pred = np.zeros((C,) + shape, dtype=bool), np.zeros((C,) + shape, dtype=bool)
    field = lambda: gaussian_filter(rng.standard_normal(shape), 3.0)
    f0 = field()
    label[0] = f0 > 0.05
    label[0, 0, :, :] |= f0[0] > -0.02  # reaches the face z = 0
    pred[0] = (f0 + 0.3 * field()) > 0.04
    label[1, 20, 30, 10] = True
    pred[1, 22, 27, 14] = True
    zz, yy, xx = np.meshgrid(*[np.arange(s) for s in shape], indexing="ij")
    r = np.sqrt(((zz - 18) / 1.0) ** 2 + ((yy - 26) / 1.3) ** 2 + ((xx - 14) / 0.9) ** 2)
    label[2] = (r < 11) & (r > 5)
    pred[2] = ((r + 2.0 * field()) < 11.5) & (r > 4)
    f3 = field()
    label[3] = f3 > 0.1
    pred[3] = (f3 + 0.4 * field()) > 0.12
    return pred, label


def _gpu(pred, label, dtype):
    return (torch.from_numpy(pred.astype(np.uint8)).cuda(), torch.from_numpy(label).to(dtype).cuda())


@pytest.mark.parametrize("label_dtype", [torch.uint8, torch.float32])
@pytest.mark.parametrize("spacing", EXACT_SPACINGS + [INEXACT_SPACING])
def test_blobs_match_the_oracle(spacing, label_dtype):
    pred, label = _blobs()
    got = pkg.hd95(*_gpu(pred, label, label_dtype), spacing=spacing)
    rel = 0.0 if spacing in EXACT_SPACINGS else 1e-12
    for c in range(pred.shape[0]):
        exp = oracle_hd95.hd95(pred[c], label[c], spacing)
        assert not math.isnan(exp)
        assert _same(got[c], exp, rel), (c, got[c], exp)


def test_empty_classes_give_nan_and_leave_their_neighbours_alone():
    pred, label = _blobs()
    full = pkg.hd95(*_gpu(pred, label, torch.uint8), spacing=(2.0, 1.5, 1.5))
    pred[1], label[2] = False, False        # class 1: empty prediction; class 2: empty label
    pred = np.concatenate([pred, np.zeros_like(pred[:1])])  # class 4: both empty
    label = np.concatenate([label, np.zeros_like(label[:1])])
    got = pkg.hd95(*_gpu(pred, label, torch.float32), spacing=(2.0, 1.5, 1.5))
    assert math.isnan(got[1]) and math.isnan(got[2]) and math.isnan(got[4])
    assert got[0] == full[0] and got[3] == full[3]


def test_worst_case_box_opposite_corners():
    shape = (512, 512, 160)
    spacing = (1.5, 1.5, 2.0)
    pred = torch.zeros((1,) + shape, dtype=torch.uint8, device="cuda")
    label = torch.zeros_like(pred)
    pred[0, 0, 0, 0] = 1
    label[0, -1, -1, -1] = 1
    t = np.array([511 * 1.5, 511 * 1.5, 159 * 2.0]) ** 2
    exp = float(np.sqrt((t[0] + t[1]) + t[2]))
    assert pkg.hd95(pred, label, spacing) == [exp]


def _ellipsoid(shape, centre, radii):
    g = [(np.arange(s, dtype=np.float32) - c) / r for s, c, r in zip(shape, centre, radii)]
    return (g[0][:, None, None] ** 2 + g[1][None, :, None] ** 2 + g[2][None, None, :] ** 2) <= 1.0


def _amos_like(shape, n, seed):
    """n organ-sized ellipsoid labels with perturbed predictions (shifted, resized, a few flipped voxels)."""
    rng = np.random.default_rng(seed)
    label = np.zeros((n,) + shape, dtype=bool)
    pred = np.zeros_like(label)
    for c in range(n):
        radii = rng.uniform([15, 15, 8], [60, 60, 30])
        centre = [rng.uniform(r + 2, s - r - 2) for s, r in zip(shape, radii)]
        label[c] = _ellipsoid(shape, centre, radii)
        pred[c] = _ellipsoid(shape, centre + rng.uniform(-3, 3, 3), radii * rng.uniform(0.9, 1.1, 3))
        idx = np.argwhere(pred[c])
        flip = idx[rng.integers(0, len(idx), 40)]
        pred[c][tuple(flip.T)] = False  # holes inside the prediction: extra inner surface
    return pred, label


def test_full_size_amos_like_classes_match_the_oracle():
    shape, spacing = (512, 512, 160), (1.5, 1.5, 2.0)
    pred, label = _amos_like(shape, 3, seed=11)
    got = pkg.hd95(*_gpu(pred, label, torch.uint8), spacing=spacing)
    for c in range(3):
        assert got[c] == _oracle_cropped(pred[c], label[c], spacing), c


def _workspace(C, dims, fill):
    n = ctypes.c_size_t()
    _lib.check(_lib.load().dunet_hd95_workspace_bytes(C, _lib.i32x3(dims), ctypes.byref(n)))
    return torch.full((n.value,), fill, dtype=torch.uint8, device="cuda"), n.value


def _call(pred, label, spacing, ws, nbytes, out, label_is_float=0, C=None, dims=None, pred_p=None, label_p=None,
          out_p=None, ws_p=None, spacing_p=None):
    C = pred.shape[0] if C is None else C
    dims = tuple(pred.shape[1:]) if dims is None else dims
    sp = (ctypes.c_double * 3)(*spacing) if spacing_p is None else spacing_p
    return _lib.load().dunet_hd95(_p(pred) if pred_p is None else pred_p, _p(label) if label_p is None else label_p,
                                  label_is_float, C, _lib.i32x3(dims), sp, _p(out) if out_p is None else out_p,
                                  _p(ws) if ws_p is None else ws_p, nbytes, _stream())


def test_deterministic_and_independent_of_workspace_contents():
    pred, label = _blobs(seed=4)
    p, l = _gpu(pred, label, torch.uint8)
    runs = []
    for fill in (0x00, 0xFF, 0x00):  # 0xFF bytes: NaN as fp64, -1 as every integer
        ws, nbytes = _workspace(p.shape[0], p.shape[1:], fill)
        out = torch.full((p.shape[0],), -1.0, dtype=torch.float64, device="cuda")
        _lib.check(_call(p, l, (2.0, 1.5, 1.5), ws, nbytes, out))
        runs.append(out.cpu())
    assert torch.equal(runs[0], runs[1]) and torch.equal(runs[0], runs[2])
    assert not torch.isnan(runs[0]).any()


def test_argument_checks():
    lib = _lib.load()
    pred, label = _blobs()
    p, l = _gpu(pred, label, torch.uint8)
    lf = l.float()
    ws, nbytes = _workspace(p.shape[0], p.shape[1:], 0)
    out = torch.empty(p.shape[0], dtype=torch.float64, device="cuda")
    sp = (1.0, 1.0, 1.0)
    INVALID, UNSUPPORTED = -1, -4
    n = ctypes.c_size_t()
    assert lib.dunet_hd95_workspace_bytes(0, _lib.i32x3((4, 4, 4)), ctypes.byref(n)) == INVALID
    assert lib.dunet_hd95_workspace_bytes(1, None, ctypes.byref(n)) == INVALID
    assert lib.dunet_hd95_workspace_bytes(1, _lib.i32x3((4, 0, 4)), ctypes.byref(n)) == INVALID
    assert lib.dunet_hd95_workspace_bytes(1, _lib.i32x3((4, 4, 4)), None) == INVALID
    assert lib.dunet_hd95_workspace_bytes(1, _lib.i32x3((4, 40000, 4)), ctypes.byref(n)) == UNSUPPORTED
    assert lib.dunet_hd95_workspace_bytes(3, _lib.i32x3((37, 53, 29)), ctypes.byref(n)) == 0 and n.value == nbytes  # class count free
    null = ctypes.c_void_p(None)
    assert _call(p, l, sp, ws, nbytes, out, pred_p=null) == INVALID
    assert _call(p, l, sp, ws, nbytes, out, label_p=null) == INVALID
    assert _call(p, l, sp, ws, nbytes, out, out_p=null) == INVALID
    assert _call(p, l, sp, ws, nbytes, out, ws_p=null) == INVALID
    assert _call(p, l, sp, ws, nbytes, out, spacing_p=ctypes.POINTER(ctypes.c_double)()) == INVALID
    assert _call(p, lf, sp, ws, nbytes, out, label_is_float=1, label_p=_p(lf, 2)) == INVALID  # fp32 label off 4 bytes
    assert _call(p, l, sp, ws, nbytes, out, out_p=_p(out, 4)) == INVALID
    assert _call(p, l, sp, ws, nbytes - 256, out, ws_p=_p(ws, 128)) == INVALID                 # workspace off 256 bytes
    assert _call(p, l, sp, ws, nbytes - 1, out) == INVALID                                       # workspace too small
    assert _call(p, l, sp, ws, nbytes, out, C=0) == INVALID
    assert _call(p, l, sp, ws, nbytes, out, dims=(37, 0, 29)) == INVALID
    assert _call(p, l, sp, ws, nbytes, out, dims=(37, 53, -29)) == INVALID
    for bad in ((0.0, 1.0, 1.0), (1.0, -1.5, 1.0), (1.0, 1.0, float("inf")), (float("nan"), 1.0, 1.0)):
        assert _call(p, l, bad, ws, nbytes, out) == INVALID, bad
    assert b"spacing" in lib.dunet_last_error()
    torch.cuda.synchronize()
    # nothing was launched by the rejected calls: the output is still what a valid call writes
    _lib.check(_call(p, l, sp, ws, nbytes, out))
    assert out.cpu().tolist() == pkg.hd95(p, l, sp)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        pkg.hd95(p.cpu(), l.cpu())
    with pytest.raises(ValueError):
        pkg.hd95(p, l[:, :-1])


def _build(cout, S, feats, **kw):
    torch.manual_seed(0)
    m = pkg.DiffUNetB200(in_channels=1, out_channels=cout, image_size=S, spatial_size=S, features=feats, **kw)
    return m.to("cuda").eval()


def test_engine_hd95_beside_dice():
    """EngineB200(metrics=("dice", "hd95")) on the volume of test_engine_dropin_dice_matches_oracle: Dice and the return
    value are those of the default engine, and self.hd95s holds the oracle's HD95 of the same binarised outputs."""
    cout, S, vol = 3, 32, (40, 48, 32)
    spacing = (2.0, 1.5, 1.5)
    src = _build(cout, S, SMALL)
    sd = {k: v.detach().clone() for k, v in src.state_dict().items()}
    names = {0: "bg", 1: "liver", 2: "spleen"}
    engines = []
    for metrics in (("dice",), ("dice", "hd95")):
        m = _build(cout, S, SMALL)
        m.load_state_dict(sd)
        engines.append(pkg.EngineB200(m, class_names=names, sw_batch_size=2, overlap=0.25, metrics=metrics, spacing=spacing))
    with pytest.raises(ValueError):
        pkg.EngineB200(_build(cout, S, SMALL), metrics=("hd95",))
    image = seeded_image((1, 1) + vol)
    torch.manual_seed(9)
    label = (torch.rand(1, cout, *vol) > 0.6).float()
    label[:, 2] = 0  # empty label: HD95 NaN for that class, Dice 1 (prediction non-empty)
    n_win = len(pkg.window_starts(vol, (S, S, S), 0.25))
    noise = seeded_noise((n_win, cout, S, S, S)).cuda()
    nf = lambda w, b: noise[w:w + b]
    base, both = engines
    mean0 = base.validation_step({"image": image, "label": label}, noise_fn=nf)
    mean1 = both.validation_step({"image": image, "label": label}, noise_fn=nf)
    assert mean1 == mean0 and list(both.dices[-1].items()) == list(base.dices[-1].items())
    assert base.hd95s == [] and len(both.hd95s) == 1 and list(both.hd95s[0].keys()) == list(names.values())
    _, outputs, _ = both.infer({"image": image, "label": label}, noise_fn=nf)
    o, l = outputs[0].cpu().numpy() > 0, label[0].numpy() > 0
    for c, got in enumerate(both.hd95s[0].values()):
        assert _same(got, oracle_hd95.hd95(o[c], l[c], spacing)), c
    assert math.isnan(both.hd95s[0]["spleen"])
