"""GPU parity of the two bench.py configurations whose plans run conv classes that the 96^3 and 32^3 cases of
tests/test_gpu_realistic_parity.py do not reach: msd128_ddim25 (128^3 windows, C = 3, DDIM-25) and wide (features
64-128-256-512-1024(+64) at 96^3, C = 16).  Same CT-like windows, trained-like parameters, fp64 oracle and gates as that file.
The classes (tests/test_plan_coverage.py checks the list on the CPU):
* 128^3: the generic voxel-as-M kernel at ZT 4, unsplit, writing the InstanceNorm statistics rows itself (32^3 level);
  the flattened-plane kernel at ZT 2, K split 2 on 16^3 and K split 3 on 8^3 (uneven over 4 or 8 blocks in the 16-bit modes);
* wide 96^3: the generic kernel at ZT 4 on 48^3; the flattened-plane kernel at ZT 6, K split 6 on 6^3 (uneven over 8 or 16
  blocks in the 16-bit modes)."""
import pytest
import torch

from tests.realistic import amp_oracle
from tests.test_gpu_realistic_parity import (DEFAULT, T3, TOL, _gate, _images, _model, _x_t, check_denoiser_call,
                                             check_encoder_levels)
from tests.test_plan_coverage import WIDE, window_classes
from tests.test_realistic_inputs import _roll
from tests.util import rel_l2, seeded_noise

pytestmark = pytest.mark.gpu

CONFIGS = {"msd128": (128, DEFAULT, 3), "wide96": (96, WIDE, 16)}  # window edge, features, classes


@pytest.mark.parametrize("name", list(CONFIGS))
def test_encoder_all_levels(name):
    """Every embedding level of a [tissue, boundary] batch in every mode, with the per-level gates of the 96^3 encoder case."""
    S, feats, _ = CONFIGS[name]
    check_encoder_levels(name, S, feats, ("tissue", "boundary"))


@pytest.mark.parametrize("name", list(CONFIGS))
def test_denoiser_call(name):
    """One denoiser call on [tissue, boundary, tissue] at t = 999 / 500 / 40 in every mode, with the 96^3 case's gates."""
    S, feats, C = CONFIGS[name]
    check_denoiser_call(name, S, C, feats)


# layers whose gamma / beta are rolled by one channel, with the plan class (fp32x3) each stands for
ROLLED = {"msd128": [("model.down_2.convs.conv_0", ("generic", 4, 1, 1, False)),  # 32^3
                     ("model.down_3.convs.conv_1", ("flat", 2, 2, 1, False))],   # 16^3
          "wide96": [("model.down_4.convs.conv_1", ("flat", 6, 6, 1, False))]}   # 6^3


@pytest.mark.parametrize("name", list(ROLLED))
def test_rolled_gamma_beta_misses_the_fp32x3_gate(name):
    """gamma / beta read one channel off at exactly the layers these cases exist for, loaded into the model only (the oracle
    keeps the original parameters): the fp32x3 denoiser call, within its 1e-4 gate before, must miss it by >= 10x."""
    S, feats, C = CONFIGS[name]
    image = _images(("tissue", "boundary", "tissue"), S)
    x, t = _x_t(C, S, T3), torch.tensor(T3)
    m, sd = _model(C, S, feats, "fp32x3")
    ref = amp_oracle(torch.float64, "denoise", sd, x, t.cuda(), image, amp_oracle(torch.float64, "encoder", sd, image))

    def worst():
        with torch.no_grad():
            got = m.model(x, t, image=image, embeddings=m.embed_model(image))
        return max(rel_l2(got[b], ref[b]) for b in range(len(T3)))

    base = worst()
    print(f"rolled gamma/beta {name}: unchanged parameters rel-l2 {base:.3e}")
    assert base < TOL["fp32x3"]
    for layer, cls in ROLLED[name]:
        assert layer in window_classes(S, feats, C, "fp32x3").get(cls, []), (layer, cls)
        m.load_state_dict({k: v.cpu() for k, v in _roll(sd, layer).items()})
        err = worst()
        print(f"rolled gamma/beta {name} {layer} {cls}: rel-l2 {err:.3e} = {err / TOL['fp32x3']:.0f}x the fp32x3 gate")
        assert err >= 10 * TOL["fp32x3"], (layer, err)
    del m


def test_ddim25_window_128():
    """One whole DDIM-25 window of msd128_ddim25 (tissue, C = 3) in fp16 and fp32x3 against the fp64 oracle, with the gate of
    the DDIM-10 case (fp16 within max(4e-3, 2x the fp16-AMP oracle)); fp32x3 also holds the label gates."""
    S, feats, C = CONFIGS["msd128"]
    image = _images(("tissue",), S)
    noise = seeded_noise((1, C, S, S, S), seed=4).cuda()
    ref = amp16 = None
    for precision in ("fp16", "fp32x3"):
        m, sd = _model(C, S, feats, precision, batch_max=1, num_steps=25)
        if ref is None:
            ref = amp_oracle(torch.float64, "window", sd, image, noise, num_steps=25)[0]
            amp16 = amp_oracle(torch.float16, "window", sd, image, noise, num_steps=25)[0]
        with torch.no_grad():
            acc = m(image=image, pred_type="ddim_sample", noise=noise)[0]
        err, amp_err = rel_l2(acc, ref), rel_l2(amp16, ref)
        sign = ((acc > 0) == (ref > 0)).float().mean().item()
        am = (acc.argmax(0) == ref.argmax(0)).float().mean().item()
        sign_a = ((amp16 > 0) == (ref > 0)).float().mean().item()
        am_a = (amp16.argmax(0) == ref.argmax(0)).float().mean().item()
        line = (f"ddim-25 window 128^3 tissue {precision:6s}: rel-l2 {err:.3e} sign {sign:.5f} argmax {am:.5f} | "
                f"fp16-AMP oracle: rel-l2 {amp_err:.3e} sign {sign_a:.5f} argmax {am_a:.5f}")
        print(line)
        assert _gate(precision, err, amp_err), line
        if precision == "fp32x3":
            assert sign >= 0.999 and am >= 0.999, line
        del m


@pytest.mark.parametrize("precision", ["fp16", "bf16"])
def test_btcv_batch8_is_bit_identical_to_single_windows(precision):
    """btcv_b8_ens3's window batch under trained-like parameters: 8 mixed windows, run as two half batches of 4 on two
    streams, == eight batch-1 calls, bit for bit."""
    S, C = 96, 14
    image = _images(("air", "tissue", "boundary", "tissue", "boundary", "air", "tissue", "boundary"), S)
    noise = seeded_noise((8, C, S, S, S), seed=6).cuda()
    m, _ = _model(C, S, DEFAULT, precision, batch_max=8, num_steps=2)
    with torch.no_grad():
        a = m(image=image, pred_type="ddim_sample", noise=noise)
        for b in range(8):
            assert torch.equal(m(image=image[b:b + 1], pred_type="ddim_sample", noise=noise[b:b + 1])[0], a[b]), b
    del m
