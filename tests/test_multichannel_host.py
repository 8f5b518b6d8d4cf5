"""Multi-channel images (in_channels > 1) on the host side: parameter layout and seeded initialisation (CPU only).

The AMOS reference builds its denoiser for ``out_channels + 1`` input channels (models/diff_unet.py:34), which is the
``cat([image, x])`` width only for one image channel; the multi-modal Diff-UNet builds ``in_channels + out_channels``,
and so does DiffUNetB200.  The oracle's ``init_state_dict(k, C)`` therefore matches DiffUNetB200's encoder and time
embedding, and ``init_state_dict(k, C + k - 1)`` -- whose denoiser input is also C + k wide -- matches every denoiser
tensor up to the final 1x1 conv (the last one created, so the random stream agrees until there)."""
import pytest
import torch

import diff_unet_amos_b200 as pkg
from oracle import oracle_model
from tests.util import SMALL


@pytest.mark.parametrize("k", [2, 3, 4])
def test_state_dict_layout_and_seeded_values_follow_the_oracle(k):
    C, f = 3, SMALL
    torch.manual_seed(0)
    sd = pkg.DiffUNetB200(in_channels=k, out_channels=C, image_size=32, spatial_size=32, features=f).state_dict()
    ref = oracle_model.init_state_dict(k, C, f, seed=0)
    wide = oracle_model.init_state_dict(k, C + k - 1, f, seed=0)
    assert list(sd) == list(ref)
    assert tuple(sd["embed_model.conv_0.conv_0.conv.weight"].shape) == (f[0], k, 3, 3, 3)
    assert tuple(sd["model.conv_0.conv_0.conv.weight"].shape) == (f[0], k + C, 3, 3, 3)
    assert tuple(sd["model.final_conv.weight"].shape) == (C, f[5], 1, 1, 1)
    fp, fp_ref, fp_wide = (oracle_model.state_dict_fingerprint(d) for d in (sd, ref, wide))
    enc = lambda key: key.startswith("embed_model.") or key.startswith("model.temb.")
    for key in sd:
        if enc(key):
            assert fp[key] == fp_ref[key], key
        elif not key.startswith("model.final_conv."):
            assert fp[key] == fp_wide[key], key


def test_reference_default_constructor_round_trips_its_state_dict():
    """DiffUNetB200() takes the reference signature's defaults: in_channels=3, out_channels=1, 96^3."""
    torch.manual_seed(0)
    m = pkg.DiffUNetB200()
    assert m.in_channels == 3 and m.num_classes == 1 and tuple(m.patch) == (96, 96, 96)
    sd = m.state_dict()
    assert tuple(sd["embed_model.conv_0.conv_0.conv.weight"].shape) == (64, 3, 3, 3, 3)
    assert tuple(sd["model.conv_0.conv_0.conv.weight"].shape) == (64, 4, 3, 3, 3)
    torch.manual_seed(1)
    other = pkg.DiffUNetB200()
    assert not torch.equal(other.state_dict()["model.conv_0.conv_0.conv.weight"], sd["model.conv_0.conv_0.conv.weight"])
    other.load_state_dict(sd)
    got = other.state_dict()
    assert list(got) == list(sd)
    assert all(torch.equal(got[key], sd[key]) for key in sd)
