"""Window driver + Engine.infer equivalent for the B200 path.

``sliding_window_inference`` keeps the positional signature the reference uses at engine.py:173-177
(``(inputs, roi_size, sw_batch_size, predictor, overlap, **kwargs)``; MONAI constant blend, SURVEY Appendix B).
Grid / count map are integer host math (windows.py); crop, stitch (``out[slices] += pred`` in window order) and
``out /= count`` (+ sigmoid > 0.5, engine.py:179-180) run in CUDA kernels through the C ABI.
"""
from __future__ import annotations

import ctypes
from typing import Callable, Optional, Sequence, Tuple

import numpy as np
import torch
import torch.nn.functional as F

from . import _lib
from .windows import axis_counts, gaussian_importance_map, window_starts


def _ptr(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


class StitchBuffers:
    """Output accumulator of one volume: fp32 [C, D, H, W] sums + coverage: per-axis integer counts (constant blend, the
    count map is their outer product) or an accumulated fp32 weight volume (gaussian blend)."""

    def __init__(self, channels: int, vol: Sequence[int], roi: Sequence[int], overlap: float, device, mode: str = "constant",
                 sigma_scale: float = 0.125, out: Optional[torch.Tensor] = None):
        self.vol = tuple(int(v) for v in vol)
        self.roi = tuple(int(r) for r in roi)
        self.channels = channels
        self.mode = mode
        if out is not None:  # caller-provided (already zeroed) accumulator, e.g. a CUDA-IPC buffer of the peer exchange
            if tuple(out.shape) != (channels,) + self.vol or out.dtype != torch.float32 or not out.is_contiguous():
                raise ValueError(f"out must be contiguous fp32 {(channels,) + self.vol}")
            self.out = out
        else:
            self.out = torch.empty((channels,) + self.vol, dtype=torch.float32, device=device)
            self.zero_()
        self._finalized = False
        if mode == "constant":
            self.counts = [torch.from_numpy(c).to(device) for c in axis_counts(self.vol, self.roi, overlap)]
        elif mode == "gaussian":
            self.weights = gaussian_importance_map(self.roi, sigma_scale).to(device).contiguous()
            self.count_vol = torch.zeros(self.vol, dtype=torch.float32, device=device)
        else:
            raise NotImplementedError(f"blend mode {mode!r}: only 'constant' (the reference's) and 'gaussian' exist")

    def zero_(self) -> None:
        """Clear the accumulator (cudaMemsetAsync through the C ABI: no library kernel on the path)."""
        with torch.cuda.device(self.out.device):
            _lib.check(_lib.load().dunet_zero(_ptr(self.out), self.out.numel() * 4, _stream()))
        if self.mode == "gaussian" and hasattr(self, "count_vol"):
            self.count_vol.zero_()

    def add(self, patch: torch.Tensor, start) -> None:
        lib = _lib.load()
        if self.mode == "constant":
            _lib.check(lib.dunet_stitch_add(_ptr(self.out), _lib.i32x3(self.vol), self.channels, _ptr(patch),
                                            _lib.i32x3(self.roi), _lib.i32x3(start), _stream()))
        else:
            _lib.check(lib.dunet_stitch_add_weighted(_ptr(self.out), _ptr(self.count_vol), _lib.i32x3(self.vol), self.channels,
                                                     _ptr(patch), _ptr(self.weights), _lib.i32x3(self.roi), _lib.i32x3(start),
                                                     _stream()))

    def add_windows(self, model, volume: torch.Tensor, starts, **kw) -> None:
        """Fused crop + encoder + DDIM + ``out[slices] += pred`` for a batch of windows (model.infer_windows), ordered on the
        current stream."""
        if self.mode == "constant":
            model.infer_windows(volume, starts, self.out, **kw)
        else:
            model.infer_windows(volume, starts, self.out, count_volume=self.count_vol, weights=self.weights, **kw)

    def finalize(self, binary: bool = False, argmax: bool = False):
        if self._finalized:
            raise RuntimeError("StitchBuffers.finalize() was already called: the volume has been divided by the counts")
        self._finalized = True
        b = torch.empty((self.channels,) + self.vol, dtype=torch.uint8, device=self.out.device) if binary else None
        a = torch.empty(self.vol, dtype=torch.uint8, device=self.out.device) if argmax else None
        lib = _lib.load()
        if self.mode == "constant":
            _lib.check(lib.dunet_finalize(_ptr(self.out), _lib.i32x3(self.vol), self.channels, _ptr(self.counts[0]),
                                          _ptr(self.counts[1]), _ptr(self.counts[2]), _ptr(b), _ptr(a), _stream()))
        else:
            _lib.check(lib.dunet_finalize_weighted(_ptr(self.out), _ptr(self.count_vol), _lib.i32x3(self.vol), self.channels,
                                                   _ptr(b), _ptr(a), _stream()))
        return self.out, b, a


def scale_intensity_range(image: torch.Tensor, a_min: float = -175.0, a_max: float = 250.0, b_min: float = 0.0,
                          b_max: float = 1.0, clip: bool = True) -> torch.Tensor:
    """``ScaleIntensityRanged`` of the reference's val/test transforms (utils.py:167-170) as a GPU pre-pass."""
    if not image.is_cuda:
        raise RuntimeError("scale_intensity_range runs on the GPU only (no CPU fallback)")
    x = image.float().contiguous()
    out = torch.empty_like(x)
    with torch.cuda.device(x.device):
        _lib.check(_lib.load().dunet_scale_intensity(_ptr(x), _ptr(out), x.numel(), a_min, a_max, b_min, b_max, 1 if clip else 0,
                                                     _stream()))
    return out


def _pad_to_roi(inputs: torch.Tensor, roi) -> Tuple[torch.Tensor, list]:
    pad = []
    for k in range(inputs.dim() - 1, 1, -1):
        diff = max(roi[k - 2] - inputs.shape[k], 0)
        half = diff // 2
        pad.extend([half, diff - half])
    if any(pad):
        inputs = F.pad(inputs, pad=pad, mode="constant", value=0.0)
    return inputs, pad


def crop_windows(volume: torch.Tensor, starts, roi) -> torch.Tensor:
    """volume [c, D, H, W] fp32 -> [len(starts), c, *roi].  One launch of the batched crop kernel for c == 1; a
    multi-channel volume is cropped window by window and channel by channel straight into the batch."""
    lib = _lib.load()
    vol = tuple(volume.shape[-3:])
    b, c = len(starts), volume.shape[0]
    out = torch.empty((b, c) + tuple(roi), dtype=torch.float32, device=volume.device)
    if c == 1:
        st = (ctypes.c_int32 * (3 * b))(*[int(x) for s3 in starts for x in s3])
        _lib.check(lib.dunet_crop_windows(_ptr(volume), _lib.i32x3(vol), _ptr(out), _lib.i32x3(roi), st, b, _stream()))
        return out
    for j, s3 in enumerate(starts):
        for k in range(c):
            _lib.check(lib.dunet_crop_window(_ptr(volume[k]), _lib.i32x3(vol), _ptr(out[j, k]), _lib.i32x3(roi), _lib.i32x3(s3),
                                             _stream()))
    return out


def sliding_window_inference(inputs: torch.Tensor, roi_size, sw_batch_size: int, predictor: Callable[..., torch.Tensor],
                             overlap: float = 0.25, mode: str = "constant", sigma_scale: float = 0.125,
                             window_range: Optional[Tuple[int, int]] = None, finalize: bool = True,
                             out_channels: Optional[int] = None, noise_fn=None, seed: Optional[int] = None, ensemble: int = 1,
                             **kwargs):
    """Sliding window on the GPU, ``mode`` "constant" (what the reference uses) or "gaussian" (MONAI's other blend).
    ``predictor(window_batch, **kwargs)`` -> [b, C, *roi].

    When ``predictor`` is a DiffUNetB200 and the call is the reference's (``pred_type="ddim_sample"``, engine.py:173-177)
    the loop body runs fused in the library (crop + encoder + DDIM + ``out[slices] += pred``, no planar intermediates);
    results are bit-identical to the generic loop.  ``noise_fn(first_window_index, count)`` supplies explicit initial
    noise (parity runs); otherwise the noise of window w is the library's counter-based stream (seed, w) -- ``seed``
    defaults to a draw from torch's global generator, so ``torch.manual_seed`` makes runs repeatable.

    ``window_range=(lo, hi)`` restricts the run to a contiguous shard of the window list (multi-GPU); with
    ``finalize=False`` the un-normalised StitchBuffers is returned instead of the blended volume.
    """
    if mode not in ("constant", "gaussian"):
        raise NotImplementedError(f"blend mode {mode!r}: only 'constant' (the reference's) and 'gaussian' exist")
    if not inputs.is_cuda:
        raise RuntimeError("sliding_window_inference runs on the GPU only (no CPU fallback)")
    roi = tuple(int(r) for r in (roi_size if not isinstance(roi_size, int) else (roi_size,) * 3))
    inputs = inputs.float().contiguous()
    orig = tuple(inputs.shape[2:])
    inputs, pad = _pad_to_roi(inputs, roi)
    inputs = inputs.contiguous()
    vol = tuple(inputs.shape[2:])
    starts = window_starts(vol, roi, overlap)
    n_win = len(starts)
    lo, hi = (0, n_win) if window_range is None else window_range
    outs = []
    from .model import DiffUNetB200

    fused = isinstance(predictor, DiffUNetB200) and kwargs.get("pred_type") == "ddim_sample" and tuple(predictor.patch) == roi
    if fused and inputs.shape[1] != predictor.in_channels:
        raise ValueError(f"inputs have {inputs.shape[1]} channels, the model takes in_channels = {predictor.in_channels}")
    if fused and seed is None and noise_fn is None:
        seed = int(torch.randint(0, 2 ** 62, (1,)).item())
    with torch.cuda.device(inputs.device):
        for n in range(inputs.shape[0]):
            buf = None
            if fused:
                model = predictor
                step = min(int(sw_batch_size), model.batch_max)
                buf = StitchBuffers(model.num_classes, vol, roi, overlap, inputs.device, mode, sigma_scale)
                vol_n = inputs[n]  # [in_channels, D, H, W]
                if vol_n.data_ptr() % 16:
                    vol_n = vol_n.clone()
                for g in range(lo, hi, step):
                    g1 = min(g + step, hi)
                    if noise_fn is not None:
                        buf.add_windows(model, vol_n, starts[g:g1], noise=noise_fn(n * n_win + g, g1 - g), ensemble=ensemble)
                    else:
                        buf.add_windows(model, vol_n, starts[g:g1], seed=seed, noise_ids=range(n * n_win + g, n * n_win + g1),
                                        ensemble=ensemble)
                outs.append(buf)
                continue
            for g in range(lo, hi, sw_batch_size):
                grp = starts[g:min(g + sw_batch_size, hi)]
                batch = crop_windows(inputs[n], grp, roi)
                pred = predictor(batch, **kwargs)
                if pred.dtype != torch.float32 or not pred.is_contiguous():
                    pred = pred.float().contiguous()
                if buf is None:
                    buf = StitchBuffers(pred.shape[1], vol, roi, overlap, inputs.device, mode, sigma_scale)
                for j, s in enumerate(grp):
                    buf.add(pred[j], s)
            if buf is None:  # empty shard (more ranks than windows): contribute zeros to the reduction
                if out_channels is None:
                    raise ValueError("empty window range: pass out_channels")
                buf = StitchBuffers(out_channels, vol, roi, overlap, inputs.device, mode, sigma_scale)
            outs.append(buf)
    if not finalize:
        return outs
    res = torch.stack([b.finalize()[0] for b in outs])
    if any(pad):
        sl = [slice(None), slice(None)]
        for d in range(3):
            lo_ = pad[(2 - d) * 2]
            sl.append(slice(lo_, lo_ + orig[d]))
        res = res[tuple(sl)].contiguous()
    return res


@torch.no_grad()
def infer_volume(model, image: torch.Tensor, sw_batch_size: int = 4, overlap: float = 0.25, noise_fn=None, seed: Optional[int] = None,
                 ensemble: int = 1, mode: str = "constant"):
    """``Engine.infer`` for a diffusion model (engine.py:167-182): window driver with pred_type="ddim_sample", then
    ``(sigmoid(out) > 0.5).float()`` -- formed by the finalize kernel together with the division by the counts.
    Returns (blended fp32 volume [N, C, D, H, W], binary labels as float)."""
    bufs = sliding_window_inference(image, model.patch, sw_batch_size, model, overlap, mode=mode, finalize=False, noise_fn=noise_fn,
                                    seed=seed, ensemble=ensemble, pred_type="ddim_sample")
    outs, labs = [], []
    for b in bufs:
        blended, binary, _ = b.finalize(binary=True)
        outs.append(crop_to(blended, image.shape[2:], b.vol))
        labs.append(crop_to(binary, image.shape[2:], b.vol))
    return torch.stack(outs), torch.stack(labs).float()


def crop_to(t: torch.Tensor, orig, vol) -> torch.Tensor:
    """Undo the symmetric padding (floor on the low side) the driver applies to volumes smaller than the roi."""
    if tuple(orig) == tuple(vol):
        return t
    sl = [slice(None)]
    for o, v in zip(orig, vol):
        lo = (v - o) // 2
        sl.append(slice(lo, lo + o))
    return t[tuple(sl)].contiguous()
