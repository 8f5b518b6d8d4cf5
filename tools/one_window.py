"""Run ONE 96^3 window (C=16, default features, DDIM-10) through the B200 path: the ncu / timing target.
usage: python tools/one_window.py [--batch B] [--reps R] [--ddim N] [--in-channels K]"""
import argparse
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import diff_unet_amos_b200 as pkg

ap = argparse.ArgumentParser()
ap.add_argument("--batch", type=int, default=1)
ap.add_argument("--reps", type=int, default=1)
ap.add_argument("--S", type=int, default=96)
ap.add_argument("--C", type=int, default=16)
ap.add_argument("--in-channels", type=int, default=1, help="image channels (1 .. 10)")
ap.add_argument("--ddim", type=int, default=10)
ap.add_argument("--prof", action="store_true")
ap.add_argument("--flags", type=int, default=0)
ap.add_argument("--dump", action="store_true")
ap.add_argument("--precision", default="fp16", choices=["fp16", "bf16", "fp32x3"])
ap.add_argument("--features", default="64,64,128,256,512,64")
a = ap.parse_args()
torch.manual_seed(0)
m = pkg.DiffUNetB200(in_channels=a.in_channels, out_channels=a.C, image_size=a.S, spatial_size=a.S, batch_max=a.batch, num_steps=a.ddim, features=tuple(int(v) for v in a.features.split(",")), debug_flags=a.flags, precision=a.precision).cuda().eval()
image = torch.rand(a.batch, a.in_channels, a.S, a.S, a.S, device="cuda")
noise = torch.randn(a.batch, a.C, a.S, a.S, a.S, device="cuda")
with torch.no_grad():
    m(image=image, pred_type="ddim_sample", noise=noise)  # warm-up: packs weights, allocates the workspace
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record()
    for _ in range(a.reps):
        out = m(image=image, pred_type="ddim_sample", noise=noise)
    e1.record()
    torch.cuda.synchronize()
    t1 = time.perf_counter()
ms = e0.elapsed_time(e1) / a.reps
if a.prof:
    import ctypes
    from diff_unet_amos_b200 import _lib
    lib = _lib.load()
    plan = m._rt.plan
    lib.dunet_profile_enable(plan, 1)
    with torch.no_grad():
        m(image=image, pred_type="ddim_sample", noise=noise)
    torch.cuda.synchronize()
    msb = (ctypes.c_double * 12)(); cnt = (ctypes.c_uint64 * 12)(); byt = (ctypes.c_double * 12)()
    _lib.check(lib.dunet_profile_read_all(plan, msb, cnt, byt))
    lib.dunet_profile_enable(plan, 0)
    names = ["conv3x3x3", "normalise", "final+ddim", "deconv", "splitk-reduce", "affine-map", "norm-small", "glue", "conv-split-enc", "deconv-small", "-", "-"]
    tot = sum(msb)
    print("in-situ CUDA-event time per kernel family (one call, batch %d):" % a.batch)
    for i, nme in enumerate(names):
        bw = (f"  {byt[i] / msb[i] / 1e9:7.0f} TFLOP/s algorithmic" if i in (0, 8) else f"  {byt[i] / msb[i] / 1e6:7.0f} GB/s algorithmic") if byt[i] > 0 and msb[i] > 0 else ""
        print(f"  {nme:14s} {msb[i]:8.3f} ms  {100 * msb[i] / tot:5.1f}%  launches {cnt[i]}{bw}")
    print(f"  sum {tot:.3f} ms")
    if a.dump:
        cap = 4096
        dms = (ctypes.c_double * cap)(); dtg = (ctypes.c_int32 * cap)(); dn = ctypes.c_int32()
        lib.dunet_profile_enable(plan, 1)
        with torch.no_grad():
            m(image=image, pred_type="ddim_sample", noise=noise)
        torch.cuda.synchronize()
        _lib.check(lib.dunet_profile_dump(plan, dms, dtg, cap, ctypes.byref(dn)))
        lib.dunet_profile_enable(plan, 0)
        seq = [(dtg[i], dms[i] * 1e3) for i in range(dn.value)]
        # one denoiser step = the launches between the 2nd and 3rd final kernel
        fin = [i for i, (tg, _) in enumerate(seq) if tg == 2]
        print("one DDIM step, in issue order (us):")
        for tg, us in seq[fin[1] + 1:fin[2] + 1]:
            print(f"   {names[tg]:14s} {us:8.1f}")
print(f"window batch {a.batch}, in_channels {a.in_channels}: {ms:.2f} ms per call ({ms / a.batch:.2f} ms/window, {1e3 * a.batch / ms:.1f} patches/s), "
      f"host wall {1e3 * (t1 - t0) / a.reps:.2f} ms, out range [{out.min().item():.2f}, {out.max().item():.2f}]")
