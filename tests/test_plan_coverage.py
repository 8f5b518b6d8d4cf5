"""Every conv plan class that a bench.py configuration runs is held to the fp64 oracle by a GPU parity test.

A class is what picks the kernel code and the reduction a 3x3x3 conv layer runs: (kernel, ZT, K split, K units per
64-channel block, whether the split leaves the K slices uneven).  dunet_debug_conv_geometry returns the plan's own decision
on the host, so this runs without a GPU.  A planner change that gives a benchmark configuration a class that no GPU case
runs in the same mode fails here, naming the configuration, mode and layer, before anyone benchmarks it."""
import ctypes
import re
from functools import lru_cache

import torch

from diff_unet_amos_b200 import _lib
from oracle import oracle_model

DEFAULT = oracle_model.DEFAULT_FEATURES
WIDE = (64, 128, 256, 512, 1024, 64)
MODES = ("fp16", "bf16", "fp32x3")

# bench.py's CONFIGS, restated: name -> (window edge, features, classes)
BENCH = {"amos98": (96, DEFAULT, 16), "amos2645": (96, DEFAULT, 16), "btcv_b8_ens3": (96, DEFAULT, 14),
         "msd128_ddim25": (128, DEFAULT, 3), "wide": (96, WIDE, 16)}

# GPU cases that run every conv layer of a window (encoder and denoiser) in every mode against the fp64 oracle on CT-like
# windows with trained-like parameters: name -> (window edge, features, classes)
REALISTIC_96 = "test_gpu_realistic_parity.py::test_denoiser_call_on_ct_windows[96_C16_default]"
MSD_128 = "test_gpu_bench_config_parity.py::test_denoiser_call[msd128]"
WIDE_96 = "test_gpu_bench_config_parity.py::test_denoiser_call[wide96]"
GPU_CASES = {REALISTIC_96: (96, DEFAULT, 16), MSD_128: (128, DEFAULT, 3), WIDE_96: (96, WIDE, 16)}

# (kernel, ZT, ksplit, ksub, uneven split) -> the GPU case that runs it
COVERED = {
    ("tc64", 4, 1, 1, False): REALISTIC_96,      # Cout = 64 layers at 96^3 / 48^3
    ("flat", 1, 1, 1, False): REALISTIC_96,      # 24^3
    ("flat", 1, 2, 1, False): REALISTIC_96,      # 12^3
    ("flat", 6, 12, 1, False): REALISTIC_96,     # 6^3, split precision: 12 or 24 blocks
    ("flat", 6, 12, 3, False): REALISTIC_96,     # 6^3, 4 or 8 blocks cut in thirds
    ("generic", 4, 1, 1, False): MSD_128,        # 32^3 of the 128^3 window (and 48^3 of the wide network)
    ("flat", 2, 2, 1, False): MSD_128,           # 16^3
    ("flat", 2, 3, 1, False): MSD_128,           # 8^3, split precision
    ("flat", 2, 3, 1, True): MSD_128,            # 8^3, 4 or 8 blocks over 3 slices
    ("flat", 6, 6, 1, False): WIDE_96,           # 6^3 of the wide network, split precision
    ("flat", 6, 6, 1, True): WIDE_96,            # 6^3 of the wide network, 8 or 16 blocks over 6 slices
}


def _level(name):
    """U-Net level of a conv from its state-dict name"""
    m = re.match(r"(embed_model\.conv_0|model\.conv_0)\.|embed_model\.down\.(\d)\.|model\.down_(\d)\.|model\.upcat_(\d)\.", name)
    assert m, name
    if m[1]:
        return 0
    return int(m[2]) + 1 if m[2] else int(m[3]) if m[3] else int(m[4]) - 1


@lru_cache(maxsize=None)
def conv_layers(C, feats):
    """(name, level, cin, cout) of every 3x3x3 conv of the encoder and the denoiser, from the reference's weight shapes (the
    denoiser's first conv reads [x_t, image]: 1 + C channels; an up-block's first conv reads cat([skip, up]))."""
    with torch.device("meta"):  # shapes only
        sd = oracle_model.init_state_dict(1, C, feats, seed=None)
    return tuple((k[:-len(".conv.weight")], _level(k), w.shape[1], w.shape[0]) for k, w in sd.items() if k.endswith(".conv.weight"))


def plan_class(mode, name, dims, cin, cout):
    # Split-precision convs walk three times the input blocks (hi*hi, hi*lo, lo*hi): every conv in fp32x3 mode and the
    # encoder's in fp16 mode, except the encoder's first conv, whose three products share one block (DESIGN section 2).
    split = (mode == "fp32x3" or (mode == "fp16" and name.startswith("embed_model."))) and name != "embed_model.conv_0.conv_0"
    flags = _lib.DUNET_FLAG_FP32X3 if split else _lib.DUNET_FLAG_FP16 if mode == "fp16" else 0
    out = (ctypes.c_int32 * 16)()
    _lib.check(_lib.load().dunet_debug_conv_geometry(_lib.i32x3(dims), cin, cout, flags, out))
    kernel, zt, ksplit, ksub, ncb = out[0], out[1], out[5], out[6], out[15]
    return ({0: "tc64", 1: "generic", 2: "flat"}[kernel], zt, ksplit, ksub, ksplit > 1 and ncb * ksub % ksplit != 0)


def window_classes(S, feats, C, mode):
    """{class: [layer names]} of one S^3 window"""
    # the probe pads cin as one tensor; an up-block conv pads skip and up separately: the same when both are multiples of 64
    assert all(f % 64 == 0 for f in feats)
    out = {}
    for name, lvl, cin, cout in conv_layers(C, feats):
        out.setdefault(plan_class(mode, name, (S >> lvl,) * 3, cin, cout), []).append(name)
    return out


def test_every_bench_config_class_has_a_gpu_parity_case():
    reached = {case: {(mode, k) for mode in MODES for k in window_classes(S, f, C, mode)} for case, (S, f, C) in GPU_CASES.items()}
    missing = []
    for cfg, (S, feats, C) in BENCH.items():
        for mode in MODES:
            for k, names in window_classes(S, feats, C, mode).items():
                case = COVERED.get(k)
                if case is None or (mode, k) not in reached[case]:
                    missing += [f"{cfg} {mode} {name}: class {k} " + ("is in no GPU case" if case is None else f"is not run by {case}")
                                for name in names]
    assert not missing, "\n".join(missing)


def test_every_table_row_is_used():
    """A row no benchmark configuration needs is stale: the planner moved and the table did not."""
    used = {k for S, f, C in BENCH.values() for mode in MODES for k in window_classes(S, f, C, mode)}
    assert set(COVERED) == used, set(COVERED) ^ used

