"""CPU checks of the realistic inputs and parameters (tests/realistic.py) that the GPU parity tests in
tests/test_gpu_realistic_parity.py run on: the phantoms are what they claim to be, the trained-like parameters load into
the product and round-trip, and every kernel mistake those tests are meant to catch moves the oracle's output by at
least ten times the tolerance of the mode whose test claims to catch it."""
import pytest
import torch
import torch.nn.functional as F

import diff_unet_amos_b200 as pkg
from oracle import oracle_model
from tests import realistic
from tests.util import SMALL, rel_l2, seeded_image

FP32X3_TOL = 1e-4  # precision="fp32x3" gate of tests/test_gpu_parity.py (rel-l2)


def test_phantoms_are_deterministic_and_have_the_expected_composition():
    for kind in realistic.KINDS:
        a, b = realistic.ct_phantom_window(kind, 48, seed=3), realistic.ct_phantom_window(kind, 48, seed=3)
        assert a.shape == (1, 1, 48, 48, 48) and torch.equal(a, b)
        assert float(a.min()) >= 0.0 and float(a.max()) <= 1.0
    assert not torch.equal(realistic.ct_phantom_window("tissue", 48, 3), realistic.ct_phantom_window("tissue", 48, 4))
    frac = {k: ((float((im == 0).float().mean()), float((im == 1).float().mean())))
            for k, im in ((k, realistic.ct_phantom_window(k, 96, 0)) for k in realistic.KINDS)}
    print("fractions exact 0 / exact 1:", frac)
    assert frac["tissue"][0] == 0.0 and 1e-3 < frac["tissue"][1] < 0.05          # no air, a clipped bone rod
    assert 0.4 < frac["boundary"][0] < 0.6 and 1e-3 < frac["boundary"][1] < 0.05  # half air, the rod
    assert frac["air"] == (1.0, 0.0)
    tissue = realistic.ct_phantom_window("tissue", 96, 0)
    soft = tissue[(tissue > 0.3) & (tissue < 0.7)]
    assert 0.45 < float(soft.median()) < 0.6 and 0.02 < float(soft.std()) < 0.08
    body = realistic.ct_phantom((128, 128, 40), "body", 0)
    assert 0.3 < float((body == 0).float().mean()) < 0.8


def _first_conv_ratio(image, sd):
    y = F.conv3d(image, sd["embed_model.conv_0.conv_0.conv.weight"], sd["embed_model.conv_0.conv_0.conv.bias"], padding=1)
    return (y.mean((2, 3, 4)).abs() / y.std((2, 3, 4)))[0]


def test_tissue_window_reaches_a_large_mean_to_std_ratio():
    """The first encoder conv of the tissue window (seeded init, 96^3) has per-channel |mean| / std several times that of
    a torch.rand image.  A whole-window median of 10 is out of reach for any 96^3 window: the conv's zero padding makes the
    border voxels a step of about a third of the mean off the interior, and a noise-free constant window -- no texture, no
    organs, no bone, only that border -- already has a median of only ~4.2.  Away from the border the tissue window's
    channels do reach the higher ratios."""
    sd = oracle_model.init_state_dict(1, 16)
    tissue = realistic.ct_phantom_window("tissue", 96, 0)
    r = _first_conv_ratio(tissue, sd)
    r_rand = _first_conv_ratio(seeded_image((1, 1, 96, 96, 96)), sd)
    r_const = _first_conv_ratio(torch.full_like(tissue, float(tissue.median())), sd)
    y = F.conv3d(tissue, sd["embed_model.conv_0.conv_0.conv.weight"], sd["embed_model.conv_0.conv_0.conv.bias"])  # interior
    r_in = (y.mean((2, 3, 4)).abs() / y.std((2, 3, 4)))[0]
    print(f"first-conv |mean|/std (median, max): tissue phantom {float(r.median()):.2f}, {float(r.max()):.2f}; "
          f"its interior {float(r_in.median()):.2f}, {float(r_in.max()):.2f}; constant window {float(r_const.median()):.2f}; "
          f"torch.rand image {float(r_rand.median()):.2f}, {float(r_rand.max()):.2f}")
    assert float(r.median()) >= 3.0 * float(r_rand.median())
    assert float(r.max()) >= 10.0
    assert float(r_const.median()) < 5.0                                 # the border alone caps the whole-window ratio
    assert float(r_in.median()) >= 6.0 and float(r_in.max()) >= 15.0


def test_trained_like_state_dict_shapes_and_values():
    sd = oracle_model.init_state_dict(1, 13, SMALL)
    tl = realistic.trained_like_state_dict(sd, seed=5)
    assert list(tl) == list(sd) and all(tl[k].shape == sd[k].shape and tl[k].dtype == torch.float32 for k in sd)
    assert torch.equal(realistic.trained_like_state_dict(sd, seed=5)["model.final_conv.bias"], tl["model.final_conv.bias"])
    n_neg = n_all = 0
    for k in sd:
        if k.endswith(".adn.N.weight"):
            g = tl[k]
            assert len(torch.unique(g)) == g.numel(), k               # distinct per channel
            assert float(g.abs().min()) >= 0.3 and float(g.abs().max()) <= 2.5
            n_neg, n_all = n_neg + int((g < 0).sum()), n_all + g.numel()
        elif k.endswith(".adn.N.bias"):
            assert bool((tl[k] != 0).all()) and len(torch.unique(tl[k])) == tl[k].numel(), k
        elif k.endswith(".conv.bias"):
            assert float(tl[k].abs().max()) > 1.0, k
        elif ".temb_proj." in k and k.endswith(".weight"):
            assert torch.allclose(tl[k], 3.0 * sd[k]), k
        elif k.endswith("deconv.bias") or k == "model.final_conv.bias":
            assert not torch.equal(tl[k], sd[k]), k
        else:
            assert torch.equal(tl[k], sd[k]), k
    assert 0.1 < n_neg / n_all < 0.3


def test_product_loads_trained_like_parameters():
    """DiffUNetB200.load_state_dict accepts them under the reference's keys and returns them unchanged."""
    torch.manual_seed(0)
    m = pkg.DiffUNetB200(in_channels=1, out_channels=13, image_size=32, spatial_size=32, features=SMALL)
    tl = realistic.trained_like_state_dict(m.state_dict(), seed=1)
    m.load_state_dict(tl)
    got = m.state_dict()
    assert list(got) == list(tl)
    assert all(torch.equal(got[k], tl[k]) for k in tl)


# ---------------------------------------------------------------------------------------------------------------------
# sensitivity: how far each kernel mistake moves the oracle's output on these inputs
# ---------------------------------------------------------------------------------------------------------------------
def _conv_in_act_unbiased(sd, prefix, x):
    x = F.conv3d(x, sd[prefix + ".conv.weight"], sd[prefix + ".conv.bias"], padding=1)
    mean = x.mean((2, 3, 4), keepdim=True)
    var = x.var((2, 3, 4), keepdim=True, unbiased=True)
    g = sd[prefix + ".adn.N.weight"].view(1, -1, 1, 1, 1)
    b = sd[prefix + ".adn.N.bias"].view(1, -1, 1, 1, 1)
    return F.leaky_relu((x - mean) / torch.sqrt(var + oracle_model.IN_EPS) * g + b, oracle_model.LEAKY_SLOPE)


def _roll(sd, prefix):
    sd = dict(sd)
    for k in (prefix + ".adn.N.weight", prefix + ".adn.N.bias"):
        sd[k] = sd[k].roll(1)
    return sd


def _swap(sd, prefix):
    sd = dict(sd)
    sd[prefix + ".adn.N.weight"], sd[prefix + ".adn.N.bias"] = sd[prefix + ".adn.N.bias"], sd[prefix + ".adn.N.weight"]
    return sd


def _drop_beta(sd, prefix):
    sd = dict(sd)
    sd[prefix + ".adn.N.bias"] = torch.zeros_like(sd[prefix + ".adn.N.bias"])
    return sd


# name, what it changes.  Each is claimed for the fp32x3 cases of the GPU tests: their gates (1e-4 on
# logits, max(1e-4, 2x the fp32x3 format oracle) per embedding level) are the tight ones; the 16-bit gates are
# max(tolerance, 2x the AMP oracle), up to ~2e-2 for fp16 logits, too loose to claim a 10x margin for every mistake.
MUTATIONS = [
    ("gamma/beta rolled by one channel", lambda sd: (_roll(sd, "model.down_2.convs.conv_0"), {})),
    ("gamma and beta swapped", lambda sd: (_swap(sd, "embed_model.down.1.convs.conv_1"), {})),
    ("unbiased variance", lambda sd: (sd, {"_conv_in_act": lambda s, p, x: _conv_in_act_unbiased(s, p, x)})),
    ("eps 1e-6", lambda sd: (sd, {"IN_EPS": 1e-6})),
    ("LeakyReLU slope 0.01", lambda sd: (sd, {"LEAKY_SLOPE": 0.01})),
    ("beta missing before final_conv", lambda sd: (_drop_beta(sd, "model.upcat_1.convs.conv_1"), {})),
]


@pytest.fixture(scope="module")
def sensitivity_case():
    # the tissue and boundary windows at 96^3, as in the GPU encoder case (narrow features keep it quick on the CPU)
    S, C = 96, 13
    sd = realistic.trained_like_state_dict(oracle_model.init_state_dict(1, C, SMALL), seed=0)
    image = torch.cat([realistic.ct_phantom_window(k, S, seed=0) for k in ("tissue", "boundary")])
    torch.manual_seed(7)
    t = torch.tensor([500, 500])
    x = realistic.q_sample(torch.cat([realistic.label_volume(C, S, seed=s) for s in (0, 1)]), t.numpy(), torch.randn(2, C, S, S, S))
    # the per-sample, per-level gate of the GPU encoder case: max(1e-4, 2x the fp64 oracle in the fp32x3 number format)
    ref = realistic.amp_oracle(torch.float64, "encoder", sd, image)
    fmt = realistic.amp_oracle(torch.float64, "encoder", sd, image, variant="storage")
    gates = [[max(FP32X3_TOL, 2.0 * rel_l2(f[b], r[b])) for f, r in zip(fmt, ref)] for b in range(2)]
    return sd, image, x, t, gates


def _outputs(sd, image, x, t):
    with torch.no_grad():
        e = oracle_model.encoder_forward(sd, image)
        return e, oracle_model.denoiser_forward(sd, x, t, image, e)


@pytest.mark.parametrize("name,mutate", MUTATIONS, ids=[m[0] for m in MUTATIONS])
def test_mutation_moves_the_output_far_beyond_the_gate(sensitivity_case, monkeypatch, name, mutate):
    """The GPU tests compare every embedding level (encoder case) and the logits (denoiser case) per window, and fail when
    any of them exceeds its gate, so the margin is the largest move / gate over those tensors; each is printed."""
    sd, image, x, t, gates = sensitivity_case
    e0, l0 = _outputs(sd, image, x, t)
    sd_m, patches = mutate(sd)
    for attr, val in patches.items():
        monkeypatch.setattr(oracle_model, attr, val)
    e1, l1 = _outputs(sd_m, image, x, t)
    ratios = []
    for b, kind in enumerate(("tissue", "boundary")):
        moves = [rel_l2(a[b], c[b]) for a, c in zip(e1, e0)] + [rel_l2(l1[b], l0[b])]
        g = gates[b] + [FP32X3_TOL]
        ratios += [m / q for m, q in zip(moves, g)]
        per = "  ".join(f"{n} {m:.1e}/{q:.1e}" for n, m, q in zip(["L0", "L1", "L2", "L3", "L4", "logits"], moves, g))
        print(f"{name}, {kind}: move / fp32x3 gate  {per}")
    print(f"{name}: margin {max(ratios):.0f}x")
    assert max(ratios) >= 10
