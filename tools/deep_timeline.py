"""Per-CTA phase timeline (clock64 stamps) of ONE deep-level conv launch (conv3d_flat_kernel) inside a real batch-4 DDIM step.
usage: DUNET_DBG_LAUNCH=k python tools/deep_timeline.py   (k-th deep-level conv launch after the warm-up call;
per DDIM step the deep-level launches are, in order: down_2.a down_2.b down_3.a down_3.b down_4.a down_4.b upcat_4.a upcat_4.b
upcat_3.a upcat_3.b; the encoder contributes 6 first: down.1.a/b, down.2.a/b, down.3.a/b)"""
import ctypes
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import diff_unet_amos_b200 as pkg
from diff_unet_amos_b200 import _lib

B = int(os.environ.get("B", "4"))
lib = _lib.load()
torch.manual_seed(0)
m = pkg.DiffUNetB200(in_channels=1, out_channels=16, image_size=96, spatial_size=96, batch_max=B, num_steps=2).cuda().eval()
image = torch.rand(B, 1, 96, 96, 96, device="cuda")
noise = torch.randn(B, 16, 96, 96, 96, device="cuda")
with torch.no_grad():
    m(image=image, pred_type="ddim_sample", noise=noise)
    torch.cuda.synchronize()
    dbg = torch.zeros(8 * 256, dtype=torch.int64, device="cuda")
    lib.dunet_debug_set_conv_timeline(ctypes.c_void_p(dbg.data_ptr()))
    m(image=image, pred_type="ddim_sample", noise=noise)
    torch.cuda.synchronize()
    lib.dunet_debug_set_conv_timeline(None)
t = dbg.view(-1, 8).cpu()
t = t[t[:, 0] != 0].double()
if len(t) == 0:
    print("no stamps (launch index out of range?)")
    sys.exit(0)
rel = t[:, 1:6] - t[:, 0:1]
names = ["pdl_wait done", "MMA issue done", "first operands in smem", "first accumulators complete", "epilogue done"]
print(f"launch {os.environ.get('DUNET_DBG_LAUNCH')}: {len(t)} CTAs, items per CTA min/max {int(t[:, 6].min())}/{int(t[:, 6].max())}")
for i, n in enumerate(names):
    print(f"   {n:30s} mean {rel[:, i].mean():9.0f}  max {rel[:, i].max():9.0f} clk after kernel start")
