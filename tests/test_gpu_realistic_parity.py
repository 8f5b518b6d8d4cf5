"""GPU parity on realistic inputs and parameters (tests/realistic.py): CT-like windows (clipped air / bone, soft tissue with
a faint texture) and trained-like parameters (distinct InstanceNorm gamma / beta per channel, large conv biases), against
the oracle in fp64 on the GPU.  (With an N(0, 2) conv bias in front of every InstanceNorm the fp32 oracle's own error
reaches 3e-4 on an all-air window: b - mean(b) is a few ulps instead of 0, and rstd = 1/sqrt(eps) amplifies it.  The kernels
drop that bias and get it exactly.)  With the seeded init (gamma = 1, beta = 0) a gamma / beta read at the wrong
channel, swapped or dropped gives bit-identical results; here it cannot.  The 16-bit modes are also held against the
reference's own AMP path (the oracle under torch.autocast): 16-bit storage of a raw conv output whose mean is several times
its std costs the same there, so a kernel error above twice the AMP oracle's is a bug, not the design limit.

Kernels reached at the production 96^3 level shapes (encoder, denoiser and window cases; launch counts per mode in
profiles/r3_launch_families.txt): conv3d_tc64 with normalise-on-load (in_affine_kernel) at 96^3 / 48^3 in fp16 and bf16, the
flattened-plane conv with splitk_norm_kernel at 24^3 / 12^3 / 6^3, splitk_reduce_stats_kernel in fp32x3,
norm_act(_pool)_kernel in all three modes (out_single_h: the split-precision encoder of the fp16 mode), final_ddim_kernel."""
import pytest
import torch

import diff_unet_amos_b200 as pkg
from diff_unet_amos_b200 import _lib
from oracle import oracle_model
from tests import realistic
from tests.realistic import amp_oracle
from tests.util import SMALL, rel_l2, seeded_noise

pytestmark = pytest.mark.gpu

TOL = {"bf16": 2e-2, "fp16": 4e-3, "fp32x3": 1e-4}
AMP = {"bf16": torch.bfloat16, "fp16": torch.float16}
ENC_FP16_TOL = 1e-3  # fp16 mode: split-precision encoder, each map rounded once to fp16
DEFAULT = oracle_model.DEFAULT_FEATURES
T3 = [999, 500, 40]


def _model(cout, S, feats, precision="fp16", batch_max=3, seed=0, **kw):
    torch.manual_seed(0)
    m = pkg.DiffUNetB200(in_channels=1, out_channels=cout, image_size=S, spatial_size=S, features=feats, batch_max=batch_max,
                         precision=precision, **kw).cuda().eval()
    sd = realistic.model_state_dict(m, seed)
    return m, sd


def _images(kinds, S):
    return torch.cat([realistic.ct_phantom_window(k, S, seed=i) for i, k in enumerate(kinds)]).cuda()


def _x_t(cout, S, t):
    """q_sample of a +-1 block label volume per sample (seeded), at timesteps t"""
    x0 = torch.cat([realistic.label_volume(cout, S, seed=10 + i) for i in range(len(t))])
    return realistic.q_sample(x0, t, seeded_noise(x0.shape, seed=3)).cuda()


def _gate(precision, err, amp_err):
    if precision == "fp32x3":
        return err < TOL["fp32x3"]
    return err <= max(TOL[precision], 2.0 * amp_err)


# ---------------------------------------------------------------------------------------------------------------------
def test_encoder_all_levels_on_ct_windows():
    """Every level of the embeddings, 96^3, default features, batch [tissue, boundary, air], per sample: fp16 (split-precision
    encoder, rounded once to fp16) < 1e-3, bf16 within 2x of the bf16-AMP oracle, fp32x3 < 1e-4 or within 2x of the fp64
    oracle with the fp32x3 number format (bf16 hi + lo operands, three products, raw conv outputs stored as pairs), whichever
    is larger.  The fp64 oracle with fp32 statistics rows instead is printed next to it: which rounding the error comes from."""
    S = 96
    image = _images(("tissue", "boundary", "air"), S)
    ref = None
    failed = []
    for precision in ("fp16", "bf16", "fp32x3"):
        m, sd = _model(16, S, DEFAULT, precision)
        if ref is None:
            ref = amp_oracle(torch.float64, "encoder", sd, image)
            amp = amp_oracle(torch.bfloat16, "encoder", sd, image)
            fmt = amp_oracle(torch.float64, "encoder", sd, image, variant="storage")
            stats = amp_oracle(torch.float64, "encoder", sd, image, variant="stats")
        with torch.no_grad():
            emb = m.embed_model(image)
        for lvl in range(5):
            for b, kind in enumerate(("tissue", "boundary", "air")):
                err = rel_l2(emb[lvl][b], ref[lvl][b])
                line = f"encoder {precision:6s} level {lvl} {kind:8s}: rel-l2 {err:.3e}"
                if precision == "fp32x3":
                    fmt_err, stats_err = rel_l2(fmt[lvl][b], ref[lvl][b]), rel_l2(stats[lvl][b], ref[lvl][b])
                    line += f"  (fp32x3 format oracle {fmt_err:.3e}, fp32 statistics rows oracle {stats_err:.3e})"
                    # the format alone reaches ~1e-4 at the deeper levels of the tissue window (DESIGN section 2)
                    ok = err < max(TOL["fp32x3"], 2.0 * fmt_err)
                elif precision == "fp16":
                    ok = err < ENC_FP16_TOL
                else:
                    amp_err = rel_l2(amp[lvl][b], ref[lvl][b])
                    line += f"  (bf16-AMP oracle {amp_err:.3e})"
                    # above the 2e-2 of a whole window at the deeper levels (up to 4.8e-2 measured), but 4-6x below the
                    # bf16-AMP oracle: the cost of 8 mantissa bits on these inputs, not a kernel error (DESIGN section 2)
                    ok = err <= 2.0 * amp_err
                print(line)
                if not ok:
                    failed.append(line)
        del m
    assert not failed, failed


@pytest.mark.parametrize("S,cout,feats", [(96, 16, DEFAULT), (32, 13, SMALL)], ids=["96_C16_default", "32_C13_small"])
def test_denoiser_call_on_ct_windows(S, cout, feats):
    """One denoiser call, batch [tissue, boundary, tissue] at t = 999 / 500 / 40 (x_t = q_sample of a block label volume:
    at t = 40 the input is nearly piecewise constant), every mode, vs the fp64 oracle and the AMP oracles."""
    image = _images(("tissue", "boundary", "tissue"), S)
    x = _x_t(cout, S, T3)
    t = torch.tensor(T3)
    ref = amps = None
    for precision in ("fp16", "bf16", "fp32x3"):
        m, sd = _model(cout, S, feats, precision)
        if ref is None:
            e = amp_oracle(torch.float64, "encoder", sd, image)
            ref = amp_oracle(torch.float64, "denoise", sd, x, t.cuda(), image, e)
            amps = {}
            for p, dt in AMP.items():
                ea = amp_oracle(dt, "encoder", sd, image)
                amps[p] = amp_oracle(dt, "denoise", sd, x, t.cuda(), image, ea)
        with torch.no_grad():
            got = m.model(x, t, image=image, embeddings=m.embed_model(image))
        for b, tb in enumerate(T3):
            err = rel_l2(got[b], ref[b])
            amp_err = {p: rel_l2(a[b], ref[b]) for p, a in amps.items()}
            line = (f"denoise {S}^3 C={cout} {precision:6s} t={tb:3d}: rel-l2 {err:.3e}  "
                    f"(fp16-AMP {amp_err['fp16']:.3e}, bf16-AMP {amp_err['bf16']:.3e})")
            print(line)
            assert _gate(precision, err, amp_err.get(precision, 0.0)), line
        del m


def test_ddim_window_on_ct_windows():
    """Whole DDIM-10 window, 96^3, C = 16, tissue and boundary windows; fp32x3 also holds the label gates."""
    S, cout = 96, 16
    image = _images(("tissue", "boundary"), S)
    noise = seeded_noise((2, cout, S, S, S), seed=4).cuda()
    ref = amp16 = None
    for precision in ("fp16", "fp32x3"):
        m, sd = _model(cout, S, DEFAULT, precision, batch_max=2)
        if ref is None:
            ref = torch.cat([amp_oracle(torch.float64, "window", sd, image[b:b + 1], noise[b:b + 1]) for b in range(2)])
            amp16 = torch.cat([amp_oracle(torch.float16, "window", sd, image[b:b + 1], noise[b:b + 1]) for b in range(2)])
        with torch.no_grad():
            acc = m(image=image, pred_type="ddim_sample", noise=noise)
        for b, kind in enumerate(("tissue", "boundary")):
            err, amp_err = rel_l2(acc[b], ref[b]), rel_l2(amp16[b], ref[b])
            sign = ((acc[b] > 0) == (ref[b] > 0)).float().mean().item()
            am = (acc[b].argmax(0) == ref[b].argmax(0)).float().mean().item()
            sign_a = ((amp16[b] > 0) == (ref[b] > 0)).float().mean().item()
            am_a = (amp16[b].argmax(0) == ref[b].argmax(0)).float().mean().item()
            line = (f"ddim window {kind:8s} {precision:6s}: rel-l2 {err:.3e} sign {sign:.5f} argmax {am:.5f} | "
                    f"fp16-AMP oracle: rel-l2 {amp_err:.3e} sign {sign_a:.5f} argmax {am_a:.5f}")
            print(line)
            assert _gate(precision, err, amp_err), line
            if precision == "fp32x3":
                assert sign >= 0.999 and am >= 0.999, line
        del m


@pytest.mark.parametrize("name,feats,flags", [("wide", (64, 128, 256, 512, 1024, 64), 0),
                                              ("generic_conv", DEFAULT, _lib.DUNET_FLAG_GENERIC_CONV),
                                              ("tc64_cb64", DEFAULT, _lib.DUNET_FLAG_TC64_CB64),
                                              ("plain_encoder", DEFAULT, _lib.DUNET_FLAG_PLAIN_ENCODER)])
def test_kernel_path_variants_on_ct_windows(name, feats, flags):
    """The other kernel paths, one fp16 denoiser call each at 32^3 (C = 13), same gate as the denoiser case."""
    S, cout = 32, 13
    image = _images(("tissue", "boundary", "tissue"), S)
    x, t = _x_t(cout, S, T3), torch.tensor(T3)
    m, sd = _model(cout, S, feats, "fp16", debug_flags=flags)
    ref = amp_oracle(torch.float64, "denoise", sd, x, t.cuda(), image, amp_oracle(torch.float64, "encoder", sd, image))
    amp = amp_oracle(torch.float16, "denoise", sd, x, t.cuda(), image, amp_oracle(torch.float16, "encoder", sd, image))
    with torch.no_grad():
        got = m.model(x, t, image=image, embeddings=m.embed_model(image))
    for b, tb in enumerate(T3):
        err, amp_err = rel_l2(got[b], ref[b]), rel_l2(amp[b], ref[b])
        line = f"{name:13s} fp16 t={tb:3d}: rel-l2 {err:.3e} (fp16-AMP {amp_err:.3e})"
        print(line)
        assert _gate("fp16", err, amp_err), line


@pytest.mark.parametrize("precision", ["fp16", "bf16"])
def test_normalise_on_load_and_batching_stay_bit_identical(precision):
    """Under real gamma / beta: normalise-on-load (default) == the materialised norm_act tensor (DUNET_FLAG_NO_FUSED_NORM),
    and the mixed batch [air, tissue, boundary] == three batch-1 calls, bit for bit."""
    S, cout = 96, 3
    image = _images(("air", "tissue", "boundary"), S)
    noise = seeded_noise((3, cout, S, S, S), seed=5).cuda()
    m, _ = _model(cout, S, DEFAULT, precision, num_steps=2)
    m2, _ = _model(cout, S, DEFAULT, precision, num_steps=2, debug_flags=_lib.DUNET_FLAG_NO_FUSED_NORM)
    with torch.no_grad():
        a = m(image=image, pred_type="ddim_sample", noise=noise)
        assert torch.equal(a, m2(image=image, pred_type="ddim_sample", noise=noise))
        for b in range(3):
            assert torch.equal(m(image=image[b:b + 1], pred_type="ddim_sample", noise=noise[b:b + 1])[0], a[b]), b


def test_conv_bias_in_front_of_instance_norm_has_no_effect():
    """Re-drawing every InstanceNorm-followed conv bias leaves the library's output bit-identical (the kernels drop it)
    and moves the fp64 oracle by rounding only: the mean subtraction removes a per-channel constant."""
    S, cout = 32, 13
    image = _images(("tissue", "boundary", "tissue"), S)
    x, t = _x_t(cout, S, T3), torch.tensor(T3)
    m, sd = _model(cout, S, SMALL, "fp16")
    sd2 = dict(sd)
    g = torch.Generator().manual_seed(99)
    for k in sd:
        if k.endswith(".conv.bias"):
            sd2[k] = (5.0 * torch.randn(sd[k].shape, generator=g)).cuda()
    with torch.no_grad():
        a = m.model(x, t, image=image, embeddings=m.embed_model(image))
        m.load_state_dict({k: v.cpu() for k, v in sd2.items()})
        b = m.model(x, t, image=image, embeddings=m.embed_model(image))
        assert torch.equal(a, b)
    outs = [amp_oracle(torch.float64, "denoise", s, x, t.cuda(), image, amp_oracle(torch.float64, "encoder", s, image))
            for s in (sd, sd2)]
    moved = rel_l2(outs[1], outs[0])
    print(f"conv bias re-drawn: library bit-identical, oracle moved {moved:.2e}")
    assert moved < 1e-5


@pytest.mark.parametrize("cout", [13, 16])
def test_final_conv_bias_shifts_the_logits(cout):
    """Shifting model.final_conv.bias by delta_c shifts logit channel c by delta_c, to fp32 rounding of the logits."""
    S = 32
    image = _images(("tissue", "boundary", "tissue"), S)
    x, t = _x_t(cout, S, T3), torch.tensor(T3)
    m, sd = _model(cout, S, SMALL, "fp16")
    delta = torch.linspace(-3.0, 2.0, cout)
    with torch.no_grad():
        emb = m.embed_model(image)
        a = m.model(x, t, image=image, embeddings=emb)
        m.model_params.final_conv.bias.add_(delta.cuda())
        b = m.model(x, t, image=image, embeddings=m.embed_model(image))
    err = float(((b - a) - delta.cuda().view(1, -1, 1, 1, 1)).abs().max())
    top = max(float(a.abs().max()), float(b.abs().max()))
    print(f"final conv bias C={cout}: max |shift - delta| = {err:.2e}, max |logits| = {top:.2f}")
    assert err <= 1e-6 * top
