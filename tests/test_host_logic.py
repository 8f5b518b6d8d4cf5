"""CPU tests of the product's host logic: window grid, schedule tables, parameter init / checkpoint keys, and the
C-ABI library exporting every symbol include/dunet.h declares (no compute calls: there is no GPU here)."""
import ctypes
import json
import os
import re

import numpy as np
import pytest
import torch

import diff_unet_amos_b200 as pkg
from diff_unet_amos_b200 import _lib, windows
from diff_unet_amos_b200.schedule import DdimSchedule
from oracle import oracle_ddim, oracle_model, oracle_sliding
from tests.util import GOLDEN, SMALL

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("vol,roi,ov", [((512, 512, 160), (96, 96, 96), 0.25), ((512, 512, 160), (96, 96, 96), 0.8),
                                        ((512, 512, 160), (128, 128, 128), 0.25), ((48, 48, 40), (32, 32, 32), 0.25),
                                        ((96, 200, 96), (96, 96, 96), 0.5), ((97, 131, 33), (32, 48, 32), 0.1),
                                        ((32, 32, 32), (32, 32, 32), 0.25)])
def test_window_grid_bit_exact_vs_oracle(vol, roi, ov):
    ours = windows.window_starts(vol, roi, ov)
    ref = oracle_sliding.window_grid(vol, roi, ov)
    assert ours.dtype == np.int64 and np.array_equal(ours, ref)
    cnt = oracle_sliding.count_map(vol, roi, ref)
    cd, ch, cw = windows.axis_counts(vol, roi, ov)
    assert np.array_equal(cd[:, None, None] * ch[None, :, None] * cw[None, None, :], cnt)


def test_known_answers():
    assert len(windows.window_starts((512, 512, 160), (96, 96, 96), 0.25)) == 98
    assert len(windows.window_starts((512, 512, 160), (96, 96, 96), 0.8)) == 2645
    assert windows.scan_intervals((512, 512, 160), (96, 96, 96), 0.8) == (19, 19, 19)


def test_shard_ranges_cover_and_balance():
    for n in (98, 2645, 8, 1, 50):
        for world in (1, 2, 4, 8):
            spans = [windows.shard_range(n, r, world) for r in range(world)]
            assert spans[0][0] == 0 and spans[-1][1] == n
            assert all(a[1] == b[0] for a, b in zip(spans, spans[1:]))
            sizes = [hi - lo for lo, hi in spans]
            assert max(sizes) - min(sizes) <= 1
    assert max(hi - lo for lo, hi in (windows.shard_range(98, r, 8) for r in range(8))) == 13  # 94 % ceiling


@pytest.mark.parametrize("n", [10, 25])
def test_schedule_matches_reference_tables(n):
    gold = json.load(open(os.path.join(GOLDEN, "ddim_tables.json")))[str(n)]
    s = DdimSchedule.build(n)
    assert s.timestep_map == gold["timestep_map"]
    for key in ("alphas_cumprod", "alphas_cumprod_prev", "sqrt_recip_alphas_cumprod", "sqrt_recipm1_alphas_cumprod"):
        ref = np.array([float.fromhex(h) for h in gold[key]])
        assert np.array_equal(getattr(s, key), ref), key
    o = oracle_ddim.SpacedSchedule(n)
    assert np.array_equal(o.alphas_cumprod, s.alphas_cumprod)


def test_closed_form_constants():
    a, b = DdimSchedule.build(10).closed_form()
    assert np.allclose(a, [1.0, 0.97365769, 0.50212764, 0.33832169, 0.24135542, 0.16651885, 0.10488461, 0.05837202,
                           0.02833401, 0.01197097], atol=5e-6)  # SURVEY Appendix C
    assert np.allclose(b[1:3], [0.02813009, 0.55989865], atol=5e-6) and abs(b[0]) < 1e-12


@pytest.mark.parametrize("name,cout,feats", [("C16_default", 16, None), ("C2_small", 2, SMALL)])
def test_parameter_init_and_keys_match_reference(name, cout, feats):
    gold = json.load(open(os.path.join(GOLDEN, "weights_fingerprint.json")))[name]
    torch.manual_seed(0)
    m = pkg.DiffUNetB200(in_channels=1, out_channels=cout, **({"features": feats} if feats else {}))
    sd = m.state_dict()
    assert list(sd.keys()) == list(gold["fingerprint"].keys())
    for k, v in oracle_model.state_dict_fingerprint(sd).items():
        assert v == gold["fingerprint"][k], k
    # round trip through the reference's key names
    m2 = pkg.DiffUNetB200(in_channels=1, out_channels=cout, **({"features": feats} if feats else {}))
    m2.load_state_dict(sd)
    assert all(torch.equal(a, b) for a, b in zip(m2.state_dict().values(), sd.values()))


def test_forward_dispatch_errors():
    m = pkg.DiffUNetB200(in_channels=1, out_channels=2, features=SMALL, image_size=32, spatial_size=32)
    with pytest.raises(NotImplementedError):
        m(image=torch.zeros(1, 1, 32, 32, 32), pred_type="nope")
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m(image=torch.zeros(1, 1, 32, 32, 32), pred_type="ddim_sample")
    with pytest.raises(RuntimeError, match="no CPU fallback"):  # q_sample is a CUDA kernel too (round 2)
        m(x=torch.zeros(2, 2, 8, 8, 8), pred_type="q_sample")
    with pytest.raises(NotImplementedError):
        pkg.model_hub("swin_unetr")


def test_library_exports_every_declared_symbol_at_the_header_version():
    lib = _lib.load()
    header = open(os.path.join(ROOT, "include", "dunet.h")).read()
    declared = set(re.findall(r"\b(dunet_[a-z0-9_]+)\s*\(", header))
    assert declared == set(_lib.SIGNATURES), declared ^ set(_lib.SIGNATURES)
    for name in declared:
        assert hasattr(lib, name), name
    header_version = int(re.search(r"#define DUNET_VERSION (\d+)", header).group(1))
    assert header_version == _lib.DUNET_VERSION == lib.dunet_version()
    assert ctypes.sizeof(_lib.DunetCfg) == 4 * 14


def test_product_fails_loudly_without_a_gpu():
    """No CPU fallback anywhere on the product path: without a CUDA device plan creation returns a negative code with a
    message (nothing throws across the ABI), compute calls on CPU tensors raise, and nothing under the package imports
    oracle/."""
    if torch.cuda.is_available():
        pytest.skip("this is the no-GPU behaviour test")
    lib = _lib.load()
    cfg = _lib.DunetCfg()
    cfg.num_classes, cfg.in_channels, cfg.batch_max, cfg.num_steps, cfg.flags = 2, 1, 1, 10, 0
    cfg.patch = (ctypes.c_int32 * 3)(32, 32, 32)
    cfg.features = (ctypes.c_int32 * 6)(*SMALL)
    plan = ctypes.c_void_p()
    assert lib.dunet_plan_create(ctypes.byref(plan), ctypes.byref(cfg)) < 0
    assert len(lib.dunet_last_error()) > 0
    m = pkg.DiffUNetB200(in_channels=1, out_channels=2, image_size=32, spatial_size=32, features=SMALL)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m(image=torch.rand(1, 1, 32, 32, 32), pred_type="ddim_sample")
    with pytest.raises(RuntimeError, match="GPU only"):
        pkg.sliding_window_inference(torch.rand(1, 1, 40, 40, 40), (32, 32, 32), 1, lambda b: b)
    pkg_dir = os.path.join(ROOT, "diff-unet-amos_b200")
    for fn in os.listdir(pkg_dir):
        if fn.endswith(".py"):
            src = open(os.path.join(pkg_dir, fn)).read()
            assert not re.search(r"^\s*(from|import)\s+oracle", src, re.M), fn


def test_window_grid_property_random_shapes():
    """Property test (hypothesis): for random volumes / windows / overlaps the product's integer grid equals the restated
    MONAI driver's, every voxel is covered, the last window ends at the border, and the count map is the outer product of
    the per-axis counts."""
    from hypothesis import given, settings, strategies as st

    dim = st.integers(min_value=1, max_value=6).map(lambda k: 16 * k)

    @settings(max_examples=60, deadline=None)
    @given(roi=st.tuples(dim, dim, dim), extra=st.tuples(st.integers(0, 70), st.integers(0, 70), st.integers(0, 70)),
           ov=st.sampled_from([0.0, 0.1, 0.25, 0.5, 0.8, 0.9]))
    def check(roi, extra, ov):
        vol = tuple(r + e for r, e in zip(roi, extra))
        ours = windows.window_starts(vol, roi, ov)
        ref = oracle_sliding.window_grid(vol, roi, ov)
        assert np.array_equal(ours, ref)
        cnt = oracle_sliding.count_map(vol, roi, ref)
        assert cnt.min() >= 1
        cd, ch, cw = windows.axis_counts(vol, roi, ov)
        assert np.array_equal(cd[:, None, None] * ch[None, :, None] * cw[None, None, :], cnt)
        assert all(int(ours[:, d].max()) + roi[d] == vol[d] for d in range(3))
        for world in (2, 3, 8):
            spans = [windows.shard_range(len(ours), r, world) for r in range(world)]
            assert spans[0][0] == 0 and spans[-1][1] == len(ours) and all(a[1] == b[0] for a, b in zip(spans, spans[1:]))

    check()


def test_bench_reference_arm_prints_one_valid_json_line():
    """`bench.py --impl reference` (the reference's CPU path = oracle port on the host cores) prints exactly one JSON line
    with the contract's keys; this is the only bench leg that may run without a GPU."""
    import subprocess
    import sys

    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stderr[-2000:]
    lines = [l for l in res.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "patches/s" and d["higher_is_better"] is True and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "patches/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and "model" not in d["config"]


def test_window_queue_shares_balance_and_cover():
    """Throughput-mode sharding (dist.py): G consecutive volumes form one queue that splits evenly; every window of every
    volume is owned by exactly one rank, shares are contiguous in MONAI order."""
    from diff_unet_amos_b200 import queue_group_size, queue_shares

    assert queue_group_size(98, 8) == 4 and queue_group_size(98, 4) == 2 and queue_group_size(98, 2) == 1
    assert queue_group_size(98, 1) == 1 and queue_group_size(2645, 8) == 8 and queue_group_size(50, 8) == 4
    for n_win, world in ((98, 8), (98, 4), (98, 3), (50, 8), (7, 2)):
        G = queue_group_size(n_win, world)
        owner = np.full((G, n_win), -1)
        per_rank = []
        for r in range(world):
            tot = 0
            for v, lo, hi in queue_shares(n_win, G, r, world):
                assert 0 <= lo < hi <= n_win and (owner[v, lo:hi] == -1).all()
                owner[v, lo:hi] = r
                tot += hi - lo
            per_rank.append(tot)
        assert (owner >= 0).all() and max(per_rank) - min(per_rank) <= 1
        if (n_win * G) % world == 0:
            assert max(per_rank) == min(per_rank)
        flat = owner.reshape(-1)
        assert (np.diff(flat) >= 0).all()  # contiguous, rank order = queue order


def _conv_geometry(dims, cin, cout, flags=0):
    out = (ctypes.c_int32 * 16)()
    _lib.check(_lib.load().dunet_debug_conv_geometry(_lib.i32x3(dims), cin, cout, flags, out))
    keys = ["kernel", "zt", "tiles_x", "tiles_y", "tiles_z", "ksplit", "ksub", "hx", "ty", "npos", "a_slots", "w_slots", "smem",
            "items", "n_tiles", "ncb"]
    return dict(zip(keys, list(out)))


def test_deep_level_conv_geometry_known_answers():
    """The tiling of the deep U-Net levels of a 96^3 window (host logic of csrc/conv3d_flat.cuh, DESIGN.md section 4):
    flattened-plane kernel, N = positions of a (ty x W+2) halo-plane strip, smallest ZT with >= 160 accumulator columns,
    split-K until a sample has ~48 items.  No GPU needed: the decision is a pure function of per-sample shapes."""
    g = _conv_geometry((24, 24, 24), 128, 128)
    assert (g["kernel"], g["hx"], g["ty"], g["npos"], g["zt"], g["tiles_y"], g["tiles_z"], g["ksplit"]) == (2, 26, 8, 208, 1, 3, 24, 1)
    assert g["items"] == 72
    g = _conv_geometry((12, 12, 12), 256, 256)
    assert (g["kernel"], g["hx"], g["ty"], g["npos"], g["zt"], g["ksplit"], g["ksub"], g["items"]) == (2, 14, 12, 176, 1, 2, 1, 24)
    g = _conv_geometry((12, 12, 12), 128, 256)  # 24 items per sample: split in two, one 64-channel block each
    assert (g["kernel"], g["ksplit"], g["ksub"]) == (2, 2, 1)
    g = _conv_geometry((6, 6, 6), 512, 512)
    assert (g["kernel"], g["hx"], g["ty"], g["npos"], g["zt"], g["ksplit"], g["ksub"], g["items"]) == (2, 8, 6, 48, 6, 12, 3, 4)
    # not on the flattened-plane kernel: Cout = 64 layers (z-stacked kernel), rows longer than 30 voxels, debug flags
    assert _conv_geometry((96, 96, 96), 64, 64)["kernel"] == 0
    assert _conv_geometry((48, 48, 48), 64, 128)["kernel"] == 1
    assert _conv_geometry((24, 24, 24), 128, 128, flags=_lib.DUNET_FLAG_GENERIC_CONV)["kernel"] == 1
    # Cout = 64 with too few items per sample: a plan splits K over the generic kernel (8 tiles, 3 hi/lo input blocks);
    # only the stand-alone dunet_op_conv3x3x3, which never splits K, runs such a layer on the z-stacked kernel
    g = _conv_geometry((16, 16, 16), 17, 64, flags=_lib.DUNET_FLAG_FP32X3)
    assert (g["kernel"], g["ksplit"], g["items"], g["ncb"]) == (1, 3, 8, 3)


@pytest.mark.parametrize("cin,cout", [(64, 128), (128, 128), (256, 128), (256, 256), (512, 256), (512, 512), (1024, 1024), (96, 384)])
def test_flat_conv_geometry_invariants(cin, cout):
    """For every level shape the flattened-plane kernel accepts: the strip covers the volume, N and the accumulators fit the
    instruction / TMEM limits, the rings hold one K unit, the shared memory fits, the split leaves every K slice non-empty."""
    for D in (2, 3, 4, 6, 8, 9, 12, 16, 20, 24, 30):
        for H in (2, 5, 6, 8, 12, 16, 24, 30, 48, 96):
            for W in (2, 3, 6, 8, 12, 16, 24, 30):
                g = _conv_geometry((D, H, W), cin, cout)
                assert g["kernel"] == 2, (D, H, W)
                assert g["hx"] == W + 2 and g["hx"] * 8 <= 256                      # TMA box: inner dimension <= 256 elements
                assert g["npos"] % 16 == 0 and 16 <= g["npos"] <= 256              # tcgen05 N at M = 128
                assert g["ty"] * g["hx"] - 2 <= g["npos"] < g["ty"] * g["hx"] - 2 + 16
                assert g["ty"] + 2 <= 256                                          # TMA box rows
                assert g["tiles_y"] * g["ty"] >= H > (g["tiles_y"] - 1) * g["ty"]  # strips cover H, none is empty
                assert g["zt"] in (1, 2, 3, 4, 6) and D % g["zt"] == 0 and g["tiles_z"] * g["zt"] == D
                assert g["zt"] * g["npos"] <= 512                                  # TMEM columns
                assert g["a_slots"] >= g["zt"] + 2 and g["w_slots"] >= 2 and g["smem"] <= 232448
                assert g["smem"] > 116 * 1024                                      # one CTA per SM (each allocates all of TMEM)
                assert g["ksub"] in (1, 3) and 1 <= g["ksplit"] <= g["ncb"] * g["ksub"] and g["ksplit"] <= 16
                assert g["items"] == g["tiles_y"] * g["tiles_z"] * g["n_tiles"]
    # rows of more than 30 voxels stay on the voxel-as-M kernels
    assert _conv_geometry((8, 8, 31), cin, cout)["kernel"] != 2
