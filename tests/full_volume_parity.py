"""NOT a pytest test (run it by hand on a B200): BASELINE config 2 at FULL size -- AMOS 16-class sliding-window DDIM-10 on a
synthetic 512x512x160 volume (98 windows) -- the B200 path in all three precisions against the oracle restatement evaluated
in fp32 on the GPU (TF32 off), window by window with identical weights / image / noise, then stitched.  Reports the
north_star gates on the whole volume: per-patch rel-l2, label agreement of the reference's binarisation (out > 0) and of
argmax, raw and margin-filtered.  Lives under tests/ because only tests/ may import oracle/.

    python tests/full_volume_parity.py [--windows N] [--image {rand,phantom}]
        N < 98: only the first N windows, for a quick look
        phantom: a body-shaped CT phantom through the reference's intensity window (tests/realistic.py: air outside the
        body, soft tissue with a faint texture, organs, a clipped bone rod) and trained-like parameters (distinct
        InstanceNorm gamma / beta, large conv biases) instead of torch.rand and the seeded initialisation
"""
import argparse
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import diff_unet_amos_b200 as pkg
from oracle import oracle_ddim, oracle_model
from tests import realistic

ap = argparse.ArgumentParser()
ap.add_argument("--windows", type=int, default=98)
ap.add_argument("--image", choices=("rand", "phantom"), default="rand")
a = ap.parse_args()
torch.backends.cudnn.allow_tf32 = False
torch.backends.cuda.matmul.allow_tf32 = False
VOL, ROI, C = (512, 512, 160), (96, 96, 96), 16
PRECS = ("fp16", "bf16", "fp32x3")
GATED = ("fp16", "fp32x3")  # modes that must pass the raw >= 99.9 % label gates (fp16 is the default / benchmarked mode)
dev = "cuda"
torch.manual_seed(0)
models = {prec: pkg.DiffUNetB200(in_channels=1, out_channels=C, image_size=96, spatial_size=96, batch_max=2, precision=prec).to(dev).eval()
          for prec in PRECS}
if a.image == "phantom":
    models[PRECS[0]].load_state_dict(realistic.trained_like_state_dict(models[PRECS[0]].state_dict(), seed=0))
for prec in PRECS[1:]:
    models[prec].load_state_dict(models[PRECS[0]].state_dict())
sd = {k: v.detach() for k, v in models[PRECS[0]].state_dict().items()}
torch.manual_seed(1)
volume = torch.rand(1, 1, *VOL, device=dev) if a.image == "rand" else realistic.ct_phantom(VOL, "body", seed=1).to(dev)
starts = pkg.window_starts(VOL, ROI, 0.25)[:a.windows]
sched = oracle_ddim.SpacedSchedule(10)
gen = torch.Generator(device=dev)
gen.manual_seed(2)


def oracle_window(image, noise):
    e = oracle_model.encoder_forward(sd, image)
    x, acc = noise, torch.zeros_like(noise)
    for i in reversed(range(10)):
        t = torch.full((1,), sched.timestep_map[i], dtype=torch.int64, device=dev)
        x, x0 = oracle_ddim.ddim_step(sched, i, x, oracle_model.denoiser_forward(sd, x, t, image, e))
        acc = acc + x0
    return acc


bufs = {k: pkg.StitchBuffers(C, VOL, ROI, 0.25, dev) for k in ("oracle",) + PRECS}
worst = {k: 0.0 for k in PRECS}
with torch.no_grad():
    for w, s in enumerate(starts):
        img = volume[:, :, s[0]:s[0] + 96, s[1]:s[1] + 96, s[2]:s[2] + 96].contiguous()
        noise = torch.randn((1, C) + ROI, device=dev, generator=gen)
        ref = oracle_window(img, noise)
        bufs["oracle"].add(ref[0].contiguous(), s)
        for prec in PRECS:
            out = models[prec](image=img, pred_type="ddim_sample", noise=noise)
            worst[prec] = max(worst[prec], float((out - ref).norm() / ref.norm()))
            bufs[prec].add(out[0].contiguous(), s)
        if w % 10 == 0:
            print(f"window {w + 1}/{len(starts)}  worst per-patch rel-l2 so far: " + "  ".join(f"{k} {v:.3e}" for k, v in worst.items()), flush=True)
    covered = torch.zeros(VOL, dtype=torch.bool, device=dev)
    for s in starts:
        covered[s[0]:s[0] + 96, s[1]:s[1] + 96, s[2]:s[2] + 96] = True
    if a.windows < 98:  # uncovered voxels would divide by zero counts: restrict the comparison to the covered region
        for b in bufs.values():
            for c in b.counts:
                c.clamp_(min=1)
    ref_vol = bufs["oracle"].finalize()[0]
    print(f"\nfull volume {VOL} ({a.image}), {len(starts)} windows, oracle = fp32 torch on the GPU (TF32 off), "
          f"{torch.cuda.get_device_name()}")
    failed = []
    for prec in PRECS:
        out = bufs[prec].finalize()[0]
        m = covered.unsqueeze(0).expand_as(out)
        rel = float((out[m] - ref_vol[m]).norm() / ref_vol[m].norm())
        sign = ((out > 0) == (ref_vol > 0))[m].float().mean().item()
        am = (out.argmax(0) == ref_vol.argmax(0))[covered].float().mean().item()
        srt = ref_vol.sort(0, descending=True).values
        margin_am = ((srt[0] - srt[1]) > 0.05)[covered]
        am_f = (out.argmax(0) == ref_vol.argmax(0))[covered][margin_am].float().mean().item()
        margin_s = (ref_vol.abs() > 0.05)[m]
        sign_f = ((out > 0) == (ref_vol > 0))[m][margin_s].float().mean().item()
        print(f"  {prec:7s} worst per-patch rel-l2 {worst[prec]:.3e} | stitched rel-l2 {rel:.3e} | binarisation agreement {sign:.6f} "
              f"(|ref| > 0.05: {sign_f:.6f}) | argmax agreement {am:.6f} (top-2 margin > 0.05: {am_f:.6f})")
        if prec in GATED and (sign < 0.999 or am < 0.999):
            failed.append(prec)
    assert not failed, f"raw label agreement below 99.9 % in {failed}"
    print("north_star label gates (raw, >= 99.9 %): PASS for", ", ".join(GATED))
