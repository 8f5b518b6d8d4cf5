"""Multi-channel images (1 < in_channels <= 10, num_classes + in_channels <= 32) through the B200 path, against the oracle.

The packed denoiser input is [x_0 .. x_{C-1}, image_0 .. image_{k-1}, 0 ..] in 8-channel groups; the final kernel re-packs
the class groups (channels < 8 * ceil(C / 8), rounded to 1, 2 or 4 groups) every DDIM step and leaves later groups as the
initialisation wrote them.  The (C, k) cases put the image channels in every position that distinguishes:
  (3, 4)   channels 3-6 inside class group 0            (6, 4)   6-7 in group 0, 8-9 in a group past the classes
  (14, 3)  14-15 in class group 1, 16 past the classes  (16, 4)  all past the classes
  (2, 10)  the upper bound of in_channels
Every channel of an image is a different seeded volume, so a dropped, duplicated or misplaced channel cannot pass."""
import ctypes

import pytest
import torch

import diff_unet_amos_b200 as pkg
from diff_unet_amos_b200 import _lib
from oracle import oracle_model, oracle_sliding
from tests import realistic
from tests.realistic import amp_oracle
from tests.util import SMALL, rel_l2, seeded_image, seeded_noise

pytestmark = pytest.mark.gpu

TOL = {"bf16": 2e-2, "fp16": 4e-3, "fp32x3": 1e-4}
E_UNSUPPORTED = -4  # include/dunet.h DUNET_E_UNSUPPORTED
LABEL_GATE = 0.999
DEFAULT = oracle_model.DEFAULT_FEATURES
CASES = [(3, 4), (6, 4), (14, 3), (16, 4), (2, 10)]
CASE_IDS = [f"C{c}_k{k}" for c, k in CASES]


def _model(C, k, S, feats, precision="fp16", batch_max=1, **kw):
    torch.manual_seed(0)
    return pkg.DiffUNetB200(in_channels=k, out_channels=C, image_size=S, spatial_size=S, features=feats, batch_max=batch_max,
                            precision=precision, **kw).cuda().eval()


def _image(B, k, shape, seed=1):
    """[B, k, *shape]: channel c is seeded_image with seed ``seed + 10 c``"""
    return torch.cat([seeded_image((B, 1) + tuple(shape), seed=seed + 10 * c) for c in range(k)], 1)


def _sd(m):
    return {key: v.detach() for key, v in m.state_dict().items()}


@pytest.mark.parametrize("C,k", CASES, ids=CASE_IDS)
@pytest.mark.parametrize("precision", ["fp16", "bf16", "fp32x3"])
def test_encoder_and_denoiser_vs_fp64_oracle(C, k, precision):
    """Level-0 embedding (embed_model(image)) and one model(x, t, image=, embeddings=) call at 32^3, narrow features."""
    S = 32
    m = _model(C, k, S, SMALL, precision)
    sd = _sd(m)
    image = _image(1, k, (S, S, S)).cuda()
    x = seeded_noise((1, C, S, S, S)).cuda()
    t = torch.tensor([999])
    ref_emb = amp_oracle(torch.float64, "encoder", sd, image)
    ref = amp_oracle(torch.float64, "denoise", sd, x, t.cuda(), image, ref_emb)
    with torch.no_grad():
        emb = m.embed_model(image)
        logits = m.model(x, t, image=image, embeddings=emb)
    e0, e1 = rel_l2(emb[0], ref_emb[0]), rel_l2(logits, ref)
    print(f"C={C} k={k} {precision}: emb0 {e0:.3e}  logits {e1:.3e}")
    assert e0 < TOL[precision] and e1 < TOL[precision]


@pytest.mark.parametrize("S", [32, 48])
@pytest.mark.parametrize("C,k", CASES, ids=CASE_IDS)
def test_ddim_window_on_ct_channels_with_trained_like_parameters(C, k, S):
    """Whole DDIM-10 window, CT-phantom channels (tissue / boundary windows of different seeds), trained-like parameters,
    narrow features: fp32x3 within 1e-4 of the fp64 oracle, fp16 within 4e-3 or twice the fp16-AMP oracle's own error
    (the gate of the single-channel realistic-input tests)."""
    image = torch.cat([realistic.ct_phantom_window(("tissue", "boundary")[c % 2], S, seed=c) for c in range(k)], 1).cuda()
    noise = seeded_noise((1, C, S, S, S), seed=4).cuda()
    ref = amp16 = None
    for precision in ("fp16", "fp32x3"):
        m = _model(C, k, S, SMALL, precision)
        sd = realistic.model_state_dict(m)
        if ref is None:
            ref = amp_oracle(torch.float64, "window", sd, image, noise)
            amp16 = amp_oracle(torch.float16, "window", sd, image, noise)
        with torch.no_grad():
            acc = m(image=image, pred_type="ddim_sample", noise=noise)
        err, amp_err = rel_l2(acc, ref), rel_l2(amp16, ref)
        print(f"window {S}^3 C={C} k={k} {precision}: rel-l2 {err:.3e} (fp16-AMP oracle {amp_err:.3e})")
        if precision == "fp32x3":
            assert err < TOL["fp32x3"]
        else:
            assert err <= max(TOL["fp16"], 2.0 * amp_err)
        del m


def _label_gates(acc, ref):
    sign = ((acc > 0) == (ref > 0)).float().mean().item()
    am = (acc.argmax(1) == ref.argmax(1)).float().mean().item()
    return sign, am


def test_full_size_window_four_channels_vs_oracle_on_gpu():
    """96^3, C = 16, in_channels = 4, default features, fp16: rel-l2 and both label gates (the reference's binarisation
    and argmax) vs the oracle in fp32 with TF32 off."""
    C, k, S = 16, 4, 96
    m = _model(C, k, S, DEFAULT)
    image = _image(1, k, (S, S, S)).cuda()
    noise = seeded_noise((1, C, S, S, S)).cuda()
    with torch.no_grad():
        acc = m(image=image, pred_type="ddim_sample", noise=noise)
    ref = amp_oracle(None, "window", _sd(m), image, noise)
    err = rel_l2(acc, ref)
    sign, am = _label_gates(acc, ref)
    print(f"96^3 C=16 k=4 fp16: rel-l2 {err:.3e}  sign agreement {sign:.5f}  argmax agreement {am:.5f}")
    assert err < TOL["fp16"] and sign >= LABEL_GATE and am >= LABEL_GATE


def test_reference_default_constructor_runs_ddim_sample():
    """DiffUNetB200() is the reference signature's defaults (in_channels=3, out_channels=1, 96^3, default features)."""
    m = pkg.DiffUNetB200().cuda().eval()
    assert m.in_channels == 3 and m.num_classes == 1
    S = 96
    image = _image(1, 3, (S, S, S)).cuda()
    noise = seeded_noise((1, 1, S, S, S)).cuda()
    with torch.no_grad():
        acc = m(image=image, pred_type="ddim_sample", noise=noise)
    ref = amp_oracle(None, "window", _sd(m), image, noise)
    err = rel_l2(acc, ref)
    sign = ((acc > 0) == (ref > 0)).float().mean().item()
    print(f"DiffUNetB200(): rel-l2 {err:.3e}  sign agreement {sign:.5f}")
    assert acc.shape == (1, 1, S, S, S)
    assert err < TOL["fp16"] and sign >= LABEL_GATE


def test_batching_is_bit_transparent_with_four_channels():
    """A batch of 4 (two half batches on the plan's internal streams) == four batch-1 calls, bit for bit."""
    C, k, S = 6, 4, 32
    m = _model(C, k, S, SMALL, batch_max=4)
    image, noise = _image(4, k, (S, S, S)).cuda(), seeded_noise((4, C, S, S, S)).cuda()
    with torch.no_grad():
        full = m(image=image, pred_type="ddim_sample", noise=noise)
        for j in range(4):
            one = m(image=image[j:j + 1], pred_type="ddim_sample", noise=noise[j:j + 1])
            assert torch.equal(one[0], full[j]), j


@pytest.mark.parametrize("mode", ["constant", "gaussian"])
def test_fused_window_loop_equals_generic_driver_with_three_channels(mode):
    """dunet_infer_windows (crop of all channels + encoder + DDIM + stitch) == crop_windows + forward + `out[slices] +=
    pred`, bit for bit, on a 48x56x24 volume (smaller than the 32^3 roi on one axis: padded and cropped back)."""
    C, k, S, vol, batch = 3, 3, 32, (48, 56, 24), 4
    m = _model(C, k, S, SMALL, batch_max=batch)
    image = _image(1, k, vol).cuda()
    n_win = len(pkg.window_starts(tuple(max(v, S) for v in vol), (S, S, S), 0.25))
    noise = seeded_noise((n_win, C, S, S, S)).cuda()
    nf = lambda w, b: noise[w:w + b]
    cursor = {"w": 0}

    def predictor(b, pred_type=None):
        assert b.shape[1] == k
        nz = nf(cursor["w"], b.shape[0])
        cursor["w"] += b.shape[0]
        return m(image=b, pred_type=pred_type, noise=nz)

    with torch.no_grad():
        generic = pkg.sliding_window_inference(image, (S, S, S), batch, predictor, 0.25, mode=mode, pred_type="ddim_sample")
        fused = pkg.sliding_window_inference(image, (S, S, S), batch, m, 0.25, mode=mode, noise_fn=nf, pred_type="ddim_sample")
    assert fused.shape == generic.shape == (1, C) + vol
    assert torch.equal(fused, generic)


def test_sliding_window_vs_oracle_driver_and_model():
    """The whole volume (fused window loop) vs the restated MONAI driver running the fp64 oracle window per window."""
    C, k, S, vol = 3, 2, 32, (48, 48, 40)
    m = _model(C, k, S, SMALL, batch_max=4)
    sd = _sd(m)
    image = _image(1, k, vol, seed=3)
    n_win = len(pkg.window_starts(vol, (S, S, S), 0.25))
    noise = seeded_noise((n_win, C, S, S, S)).cuda()

    def oracle_predictor(b, window_indices=None):
        nz = noise[window_indices[0]:window_indices[-1] + 1]
        return amp_oracle(torch.float64, "window", sd, b.cuda(), nz).float().cpu()

    ref = oracle_sliding.sliding_window_inference(image, (S, S, S), 4, oracle_predictor, 0.25)
    with torch.no_grad():
        got = pkg.sliding_window_inference(image.cuda(), (S, S, S), 4, m, 0.25, noise_fn=lambda w, b: noise[w:w + b],
                                           pred_type="ddim_sample").cpu()
    err = rel_l2(got, ref)
    agree = (oracle_sliding.engine_infer_labels(got) == oracle_sliding.engine_infer_labels(ref)).float().mean().item()
    print(f"sliding window C={C} k={k}: rel-l2 {err:.3e}  binarisation agreement {agree:.5f}")
    assert err < TOL["fp16"] and agree >= LABEL_GATE


def test_denoise_training_seam_with_per_sample_timesteps():
    """forward(image=, x=, step=, pred_type="denoise") with one timestep per sample (on and off the respaced schedule)."""
    C, k, S = 2, 2, 32
    m = _model(C, k, S, SMALL, batch_max=3)
    sd = _sd(m)
    image, x = _image(3, k, (S, S, S)).cuda(), seeded_noise((3, C, S, S, S)).cuda()
    emb = amp_oracle(torch.float64, "encoder", sd, image)
    for steps in ([999, 500, 37], [888, 888, 888]):
        t = torch.tensor(steps).cuda()
        with torch.no_grad():
            got = m(image=image, x=x, step=t, pred_type="denoise")
        ref = amp_oracle(torch.float64, "denoise", sd, x, t, image, emb)
        err = rel_l2(got, ref)
        print(f"denoise k={k} t={steps}: rel-l2 {err:.3e}")
        assert err < TOL["fp16"], steps


def _plan_create(C, k):
    cfg = _lib.DunetCfg()
    cfg.num_classes, cfg.in_channels, cfg.batch_max, cfg.num_steps, cfg.flags = C, k, 1, 10, 0
    cfg.patch = (ctypes.c_int32 * 3)(32, 32, 32)
    cfg.features = (ctypes.c_int32 * 6)(*SMALL)
    lib = _lib.load()
    plan = ctypes.c_void_p()
    rc = lib.dunet_plan_create(ctypes.byref(plan), ctypes.byref(cfg))
    if rc == 0:
        lib.dunet_plan_destroy(plan)
        return rc, ""
    return rc, lib.dunet_last_error().decode()


def test_out_of_range_channel_counts_are_refused():
    for k in (0, 11):
        rc, msg = _plan_create(2, k)
        assert rc == E_UNSUPPORTED and f"in_channels = {k} outside [1, {_lib.MAX_IN_CHANNELS}]" in msg, msg
    rc, msg = _plan_create(23, 10)
    assert rc == E_UNSUPPORTED and "num_classes + in_channels = 33 exceeds 32" in msg, msg
    assert _plan_create(22, 10)[0] == 0 and _plan_create(2, 10)[0] == 0
    m = _model(2, 11, 32, SMALL)
    with pytest.raises(pkg.DunetError, match=r"in_channels = 11 outside \[1, 10\]"):
        m(image=torch.rand(1, 11, 32, 32, 32, device="cuda"), pred_type="ddim_sample")


def test_fused_call_with_the_wrong_channel_count_raises():
    m = _model(2, 3, 32, SMALL)
    with pytest.raises(ValueError, match="in_channels = 3"):
        pkg.sliding_window_inference(torch.rand(1, 2, 40, 40, 40, device="cuda"), (32, 32, 32), 1, m, 0.25, pred_type="ddim_sample")
    out = torch.zeros(2, 40, 40, 40, device="cuda")
    for vol in (torch.rand(2, 40, 40, 40, device="cuda"), torch.rand(40, 40, 40, device="cuda")):
        with pytest.raises(ValueError, match=r"volume must be \[3, D, H, W\]"):
            m.infer_windows(vol, [(0, 0, 0)], out, seed=0, noise_ids=[0])
