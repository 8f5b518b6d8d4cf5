"""Time dunet_invert_labels (labels back on the input grid) on an AMOS-like case against the path a user composes by hand.

Case: a 512 x 512 x 120 scan at spacing (0.78, 0.78, 2.5) whose foreground box is 460 x 380 x 120, 16 classes, resampled
to (1.5, 1.5, 2.0): the finalised fp32 volume the window driver leaves is [16, 240, 198, 150] (seeded N(0, 4) logits).
For both interpolation modes, with and without the argmax labels, it prints:

  * the fused kernel's ms per volume (CUDA events over --calls calls after a warm-up; outputs preallocated), its
    algorithmic bytes (4 C V_res read + C V_orig written, + V_orig with argmax) and the GB/s they give;
  * the same for the composed path: dunet_resample_spacing in fp32 to the box, torch zero pad to the scan,
    dunet_finalize with unit counts (its bytes: every fp32 intermediate written once and read once, finalize's
    in-place divide written back, the uint8 labels);
  * the growth of torch.cuda.max_memory_allocated of one call of each path, outputs included;
  * whether the two paths' labels are equal (bit for bit);

and the card's name and power limit.  The working set (~1 GB) is far beyond the 126 MB L2, so no pass reads from a warm
cache.  Writes the JSON result line to --out as well when given.

usage: python tools/invert_bench.py [--calls 20] [--out FILE]
"""
import argparse
import ctypes
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SHAPE = (512, 512, 120)
SPACING = (0.78, 0.78, 2.5)
BOX_START, BOX_END = (26, 66, 0), (486, 446, 120)
PIXDIM = (1.5, 1.5, 2.0)
CLASSES = 16


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    import torch.nn.functional as F

    import diff_unet_amos_b200 as pkg
    from diff_unet_amos_b200 import _lib
    from diff_unet_amos_b200.invert import INTERP_MODES
    from tools.hd95_bench import _card

    if not torch.cuda.is_available():
        raise SystemExit("invert_bench needs a CUDA device")
    name, limit = _card()
    lib = _lib.load()
    meta = pkg.val_meta(SHAPE, (BOX_START, BOX_END), SPACING, PIXDIM)
    C, res, box, out = CLASSES, meta.res_shape, meta.box_shape, meta.orig_shape
    v_res, v_box, v_orig = (int(torch.tensor(s).prod()) for s in (res, box, out))
    g = torch.Generator(device="cuda").manual_seed(0)
    blended = torch.randn((C,) + res, generator=g, device="cuda") * 2.0
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    p = lambda t: ctypes.c_void_p(None if t is None else t.data_ptr())
    i3 = _lib.i32x3
    inv_ratio = (ctypes.c_double * 3)(*[si / so for si, so in zip(SPACING, PIXDIM)])
    ones = [torch.ones(n, dtype=torch.int32, device="cuda") for n in out]

    def composed(mode, argmax):
        boxed = torch.empty((C,) + box, dtype=torch.float32, device="cuda")
        _lib.check(lib.dunet_resample_spacing(p(blended), C, i3(res), p(boxed), i3(box), inv_ratio, 1 if mode == "nearest" else 0, st))
        pad = []
        for d in (2, 1, 0):
            pad += [meta.box_start[d], out[d] - meta.box_end[d]]
        full = F.pad(boxed, pad)
        del boxed
        b = torch.empty((C,) + out, dtype=torch.uint8, device="cuda")
        a = torch.empty(out, dtype=torch.uint8, device="cuda") if argmax else None
        _lib.check(lib.dunet_finalize(p(full), i3(out), C, p(ones[0]), p(ones[1]), p(ones[2]), p(b), p(a), st))
        return b, a

    def timed(fn):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.calls):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / args.calls

    def growth(fn):
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        r = fn()
        torch.cuda.synchronize()
        return r, torch.cuda.max_memory_allocated() - base

    rows = []
    equal_all = True
    for mode in ("nearest", "bilinear"):
        for argmax in (False, True):
            (fb, fa), fused_mem = growth(lambda: pkg.invert_labels(blended, res, meta, mode, binary=True, argmax=argmax))
            (cb, ca), comp_mem = growth(lambda: composed(mode, argmax))
            equal = bool(torch.equal(fb, cb)) and (not argmax or bool(torch.equal(fa, ca)))
            equal_all &= equal
            del cb, ca
            call = lambda: _lib.check(lib.dunet_invert_labels(p(blended), C, i3(res), i3((0, 0, 0)), i3(res), inv_ratio,
                                                               i3(meta.box_start), i3(box), i3(out), INTERP_MODES[mode],
                                                               p(fb), p(fa), st))
            fused_ms = timed(call)
            comp_ms = timed(lambda: composed(mode, argmax))
            lab = v_orig if argmax else 0
            fused_bytes = 4 * C * v_res + C * v_orig + lab
            comp_bytes = (4 * C * v_res + 4 * C * v_box) + (4 * C * v_box + 4 * C * v_orig) + (8 * C * v_orig + C * v_orig + lab)
            rows.append({
                "mode": mode, "argmax": argmax,
                "fused_ms": round(fused_ms, 4), "fused_bytes": fused_bytes, "fused_GBps": round(fused_bytes / fused_ms / 1e6, 1),
                "fused_mem_growth_bytes": int(fused_mem), "fused_output_bytes": C * v_orig + lab,
                "composed_ms": round(comp_ms, 4), "composed_bytes": comp_bytes, "composed_GBps": round(comp_bytes / comp_ms / 1e6, 1),
                "composed_mem_growth_bytes": int(comp_mem), "speedup": round(comp_ms / fused_ms, 2), "equal": equal,
            })
            del fb, fa
    res_line = {
        "metric": "invert_labels_ms_per_volume", "classes": C, "scan": list(SHAPE), "spacing": list(SPACING),
        "box_start": list(meta.box_start), "box": list(box), "pixdim": list(PIXDIM), "resampled": list(res), "calls": args.calls,
        "rows": rows, "equal": equal_all, "card": name, "power_limit_and_max_sm_clock": limit,
    }
    line = json.dumps(res_line)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")
    if not equal_all:
        raise SystemExit("the fused kernel's labels differ from the composed path")


if __name__ == "__main__":
    main()
