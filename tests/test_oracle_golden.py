"""Pin the oracle (oracle/) against goldens produced by running the UNMODIFIED reference
(oracle/make_golden.py)."""
import json
import os

import numpy as np
import pytest
import torch

from oracle import oracle_ddim, oracle_model
from tests.util import GOLDEN, SMALL, load_golden, rel_l2, seeded_image, seeded_noise

FP32_TOL = 2e-5  # same fp32 algorithm, different summation order across CPU kernels


def test_ddim_tables_match_reference():
    gold = json.load(open(os.path.join(GOLDEN, "ddim_tables.json")))
    for n in (10, 25):
        s = oracle_ddim.SpacedSchedule(n)
        g = gold[str(n)]
        assert s.timestep_map == g["timestep_map"]
        for key in ("alphas_cumprod", "alphas_cumprod_prev", "sqrt_recip_alphas_cumprod", "sqrt_recipm1_alphas_cumprod"):
            ref = np.array([float.fromhex(h) for h in g[key]])
            assert np.array_equal(getattr(s, key), ref), key  # bit-exact float64
    assert oracle_ddim.SpacedSchedule(10).timestep_map == [0, 111, 222, 333, 444, 555, 666, 777, 888, 999]


@pytest.mark.parametrize("name,cout,feats", [("C16_default", 16, None), ("C3_default", 3, None),
                                             ("C2_small", 2, SMALL), ("C16_wide", 16, (64, 128, 256, 512, 1024, 64))])
def test_weight_init_matches_reference(name, cout, feats):
    gold = json.load(open(os.path.join(GOLDEN, "weights_fingerprint.json")))[name]
    sd = oracle_model.init_state_dict(1, cout, feats or oracle_model.DEFAULT_FEATURES, seed=0)
    assert len(sd) == gold["n_tensors"]
    assert sum(v.numel() for v in sd.values()) == gold["n_params"]
    fp = oracle_model.state_dict_fingerprint(sd)
    assert list(fp.keys()) == list(gold["fingerprint"].keys())
    for k, v in fp.items():
        assert v == gold["fingerprint"][k], k
    if name == "C16_default":
        assert gold["n_params"] == 38405520 and gold["n_tensors"] == 144  # SURVEY 3.4


def _oracle_window(cout, S, feats):
    sd = oracle_model.init_state_dict(1, cout, feats, seed=0)
    image = seeded_image((1, 1, S, S, S))
    noise = seeded_noise((1, cout, S, S, S))
    with torch.no_grad():
        emb = oracle_model.encoder_forward(sd, image)
        fn = lambda x, t: oracle_model.denoiser_forward(sd, x, t, image, emb)
        res = oracle_ddim.ddim_sample_window(fn, noise, oracle_ddim.SpacedSchedule(10), collect=True)
        logits999 = fn(noise, torch.tensor([999]))
    return emb, res, logits999


@pytest.mark.parametrize("tag,cout,S,feats", [("S32_C2_small", 2, 32, SMALL), ("S48_C16_small", 16, 48, SMALL),
                                              ("S32_C3_default", 3, 32, oracle_model.DEFAULT_FEATURES)])
def test_window_matches_reference_golden(tag, cout, S, feats):
    g = load_golden(f"window_{tag}.npz")
    sub = int(g["sub"])
    s = slice(None, None, sub)
    emb, res, logits999 = _oracle_window(cout, S, feats)
    assert rel_l2(logits999[:, :, s, s, s], g["logits999"]) < FP32_TOL
    assert rel_l2(res["sample_return"][:, :, s, s, s], g["acc"]) < 1e-4
    assert rel_l2(res["final_x"][:, :, s, s, s], g["final_x"]) < 1e-4
    for i, e in enumerate(emb):
        assert abs(float(e.double().abs().sum()) - g["emb_abs"][i]) <= 1e-5 * g["emb_abs"][i]
    assert rel_l2(emb[0][:, ::8, ::4, ::4, ::4], g["emb0"]) < FP32_TOL
    for k, o in enumerate(res["model_outputs"]):
        assert abs(float(o.double().abs().sum()) - g["step_out_abs"][k]) <= 1e-4 * g["step_out_abs"][k]
    acc = res["sample_return"]
    assert float(acc.min()) >= -10.0 and float(acc.max()) <= 10.0  # sum of 10 clamped x0 (diffusion.py:94-98)


def test_oracle_matches_reference_outputs_tight():
    """The S32_C2_small case against the reference's own outputs at full resolution (window_S32_C2_small.npz stores every
    voxel), at the tolerances of a same-machine comparison: the same fp32 graph, only CPU kernel choice may differ.  The
    weights are pinned bit-exactly by test_weight_init_matches_reference[C2_small]."""
    cout, S = 2, 32
    g = load_golden("window_S32_C2_small.npz")
    assert int(g["sub"]) == 1
    emb, res, logits999 = _oracle_window(cout, S, SMALL)
    assert rel_l2(emb[0][:, ::8, ::4, ::4, ::4], g["emb0"]) < 1e-6
    assert rel_l2(emb[4], g["emb4"]) < 1e-6
    for i, e in enumerate(emb):
        assert abs(float(e.double().sum()) - g["emb_sum"][i]) <= 1e-6 * g["emb_abs"][i]
    assert rel_l2(logits999, g["logits999"]) < 1e-6
    for k, o in enumerate(res["model_outputs"]):
        assert abs(float(o.double().sum()) - g["step_out_sum"][k]) <= 1e-5 * g["step_out_abs"][k]
    assert rel_l2(res["sample_return"], g["acc"]) < 1e-5
    assert rel_l2(res["final_x"], g["final_x"]) < 1e-5
