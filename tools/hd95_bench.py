"""Time dunet_hd95 on one AMOS-sized volume: 15 organ-like classes at 512 x 512 x 160, spacing (1.5, 1.5, 2.0).

Prints the GPU time per volume (CUDA events over --calls calls after a warm-up), the kernel launches per call, the
workspace size, the card's name and power limit, and the host oracle (scipy / numpy, oracle/oracle_hd95.hd95) for
one class of the same volume.  Every class's GPU result is checked against the oracle on its one-voxel-grown bounding
box (which gives the whole-volume answer, see tests/test_gpu_hd95.py) and the timed class against the whole volume.
Writes the JSON result line to --out as well when given.

usage: python tools/hd95_bench.py [--calls 20] [--classes 15] [--out FILE]
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SHAPE = (512, 512, 160)
SPACING = (1.5, 1.5, 2.0)


def _card():
    import torch

    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        limit = q.stdout.strip() or q.stderr.strip()
    except (OSError, subprocess.SubprocessError) as e:
        limit = f"unavailable ({e})"
    return name, limit


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--classes", type=int, default=15)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import numpy as np
    import torch

    from diff_unet_amos_b200 import _lib
    from oracle import oracle_hd95
    from tests.test_gpu_hd95 import _amos_like, _oracle_cropped

    if not torch.cuda.is_available():
        raise SystemExit("hd95_bench needs a CUDA device")
    name, limit = _card()
    lib = _lib.load()
    pred_np, label_np = _amos_like(SHAPE, args.classes, seed=7)
    pred = torch.from_numpy(pred_np.astype(np.uint8)).cuda()
    label = torch.from_numpy(label_np.astype(np.uint8)).cuda()
    C, dims = args.classes, _lib.i32x3(SHAPE)
    nbytes = ctypes.c_size_t()
    _lib.check(lib.dunet_hd95_workspace_bytes(C, dims, ctypes.byref(nbytes)))
    ws = torch.empty(nbytes.value, dtype=torch.uint8, device="cuda")
    out = torch.empty(C, dtype=torch.float64, device="cuda")
    sp = (ctypes.c_double * 3)(*SPACING)
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    p = lambda t: ctypes.c_void_p(t.data_ptr())
    call = lambda: _lib.check(lib.dunet_hd95(p(pred), p(label), 0, C, dims, sp, p(out), p(ws), nbytes.value, st))

    for _ in range(3):
        call()
    torch.cuda.synchronize()
    n0 = lib.dunet_launch_count()
    call()
    launches = lib.dunet_launch_count() - n0
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(args.calls):
        call()
    ev1.record()
    torch.cuda.synchronize()
    ms = ev0.elapsed_time(ev1) / args.calls
    got = out.cpu().tolist()

    mismatches = [c for c in range(C) if got[c] != _oracle_cropped(pred_np[c], label_np[c], SPACING)]
    t0 = time.perf_counter()
    host = oracle_hd95.hd95(pred_np[0], label_np[0], SPACING)  # the whole volume, as a user computes it today
    host_s = time.perf_counter() - t0
    res = {
        "metric": "hd95_ms_per_volume", "ms_per_volume": round(ms, 3), "classes": C, "shape": list(SHAPE),
        "spacing": list(SPACING), "calls": args.calls, "launches_per_call": int(launches),
        "workspace_bytes": int(nbytes.value), "host_oracle_s_one_class": round(host_s, 2),
        "host_oracle_equal": host == got[0], "mismatching_classes": mismatches,
        "foreground_fraction": [round(float(label_np[c].mean()), 5) for c in range(C)],
        "card": name, "power_limit_and_max_sm_clock": limit,
    }
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")
    if mismatches or host != got[0]:
        raise SystemExit("GPU HD95 differs from the oracle")


if __name__ == "__main__":
    main()
