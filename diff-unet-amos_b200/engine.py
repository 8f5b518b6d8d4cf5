"""``Tester`` / ``Engine.infer`` drop-in for the B200 path (SURVEY 8f-1).

Mirrors the evaluation seams of the reference:

  * ``load_checkpoint(path)``          -> test.py:85-91   (``torch.load(path)['model']``, optional ``epoch_{n}.pt``)
  * ``convert_labels(labels, phase)``  -> engine.py:158-166
  * ``infer(batch)``                   -> engine.py:167-182 (window driver + sigmoid + 0.5 threshold)
  * ``validation_step(batch)``         -> test.py:112-160  (per-class Dice with the reference's special cases)
  * ``test(batches)``                  -> test.py:101-110

The window driver, stitching, binarisation and the Dice reductions run in CUDA kernels through the C ABI; this file is
host sequencing only.  ``use_amp`` maps the reference's autocast switch (test.py:104,119: fp16 autocast when the config
sets ``use_amp``, plain fp32 otherwise) onto the kernels' arithmetic mode: True -> "fp16" operands, False -> "fp32x3"
(fp32-class split operands), None (default) -> keep the model's own ``precision``.
"""
from __future__ import annotations

import ctypes
import os
from collections import OrderedDict
from typing import Dict, Iterable, Optional, Sequence, Tuple

import numpy as np
import torch

from . import _lib
from .inference import StitchBuffers, crop_to, sliding_window_inference
from .invert import predict_original


def _ptr(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def dice_counts(pred_u8: torch.Tensor, label: torch.Tensor) -> torch.Tensor:
    """int64 [C, 3] = (|pred & label|, |pred|, |label|) per class, computed on the GPU.  pred_u8: uint8 [C, ...] in
    {0, 1}; label: one-hot [C, ...], uint8 / bool / fp32."""
    if not pred_u8.is_cuda or not label.is_cuda:
        raise RuntimeError("dice_counts runs on the GPU only (no CPU fallback)")
    if pred_u8.dtype != torch.uint8:
        raise TypeError("pred must be uint8")
    pred_u8 = pred_u8.contiguous()
    if label.dtype == torch.bool:
        label = label.to(torch.uint8)
    if label.dtype not in (torch.uint8, torch.float32):
        label = label.float()
    label = label.contiguous()
    C = pred_u8.shape[0]
    vox = pred_u8[0].numel()
    if label.shape[0] != C or label[0].numel() != vox:
        raise ValueError(f"label shape {tuple(label.shape)} does not match prediction {tuple(pred_u8.shape)}")
    counts = torch.empty((C, 3), dtype=torch.int64, device=pred_u8.device)
    with torch.cuda.device(pred_u8.device):
        _lib.check(_lib.load().dunet_dice_counts(_ptr(pred_u8), _ptr(label), 1 if label.dtype == torch.float32 else 0, C, vox,
                                                 _ptr(counts), _stream()))
    return counts


def hd95(pred_u8: torch.Tensor, label: torch.Tensor, spacing: Sequence[float] = (1.0, 1.0, 1.0)) -> list:
    """Per-class HD95 surface distance, computed on the GPU: medpy ``hd95(pred, label, voxelspacing=spacing,
    connectivity=1)`` for each class (the reference's medpy-based metric).  pred_u8: uint8 [C, D, H, W] in {0, 1}; label:
    one-hot [C, D, H, W], uint8 / bool / fp32, non-zero = foreground; spacing: per array axis (D, H, W).  A class whose
    prediction or label is empty gives NaN (medpy raises there); the other classes are unaffected."""
    if not pred_u8.is_cuda or not label.is_cuda:
        raise RuntimeError("hd95 runs on the GPU only (no CPU fallback)")
    if pred_u8.dtype != torch.uint8:
        raise TypeError("pred must be uint8")
    if pred_u8.dim() != 4:
        raise ValueError(f"pred must be [C, D, H, W], got {tuple(pred_u8.shape)}")
    pred_u8 = pred_u8.contiguous()
    if label.dtype == torch.bool:
        label = label.to(torch.uint8)
    if label.dtype not in (torch.uint8, torch.float32):
        label = label.float()
    label = label.contiguous()
    if label.shape != pred_u8.shape:
        raise ValueError(f"label shape {tuple(label.shape)} does not match prediction {tuple(pred_u8.shape)}")
    C, dims = pred_u8.shape[0], _lib.i32x3(pred_u8.shape[1:])
    lib = _lib.load()
    nbytes = ctypes.c_size_t()
    _lib.check(lib.dunet_hd95_workspace_bytes(C, dims, ctypes.byref(nbytes)))
    ws = torch.empty(nbytes.value, dtype=torch.uint8, device=pred_u8.device)
    out = torch.empty(C, dtype=torch.float64, device=pred_u8.device)
    with torch.cuda.device(pred_u8.device):
        _lib.check(lib.dunet_hd95(_ptr(pred_u8), _ptr(label), 1 if label.dtype == torch.float32 else 0, C, dims,
                                  (ctypes.c_double * 3)(*[float(s) for s in spacing]), _ptr(out), _ptr(ws), nbytes.value,
                                  _stream()))
    return out.cpu().tolist()


def dice_from_counts(counts: Sequence[Sequence[int]]) -> list:
    """The reference's per-class rule (test.py:143-151 + metric.py:38-47): prediction non-empty and label empty -> 1;
    otherwise 2|A&B| / (|A| + |B|), with 0/0 -> 0."""
    out = []
    for inter, n_pred, n_label in counts:
        if n_pred > 0 and n_label == 0:
            out.append(1.0)
        elif n_pred + n_label == 0:
            out.append(0.0)
        else:
            out.append(2.0 * inter / float(n_pred + n_label))
    return out


METRICS = ("dice", "hd95")
SPACES = ("transformed", "original")


class EngineB200:
    """``metrics``: "dice" (always: ``validation_step`` returns the mean Dice) and optionally "hd95", which appends one
    ``OrderedDict`` of per-class HD95 per sample to ``self.hd95s`` (NaN for a class with an empty prediction or label);
    ``spacing`` is the voxel spacing per array axis (D, H, W) that HD95 is measured in.

    ``space``: "transformed" (the reference's loop: batches hold the val-transformed image and label) or "original": a
    batch holds the raw-intensity ``"image"`` [N, in_channels, D, H, W], the ``"label"`` on that same grid and its voxel
    spacing ``"spacing"`` ((3,) or [N, 3]); each sample runs ``predict_original`` (val transform to ``pixdim``, window driver,
    labels inverted back onto the input grid), Dice is scored against the original label and HD95 in each sample's own
    ``"spacing"`` (the constructor's ``spacing`` is then unused) -- the way challenge evaluations such as AMOS score."""

    def __init__(self, model, class_names: Optional[Dict[int, str]] = None, sw_batch_size: int = 4, overlap: float = 0.25,
                 include_background: bool = True, use_amp: Optional[bool] = None, device="cuda", epoch: Optional[int] = None,
                 metrics: Sequence[str] = ("dice",), spacing: Sequence[float] = (1.0, 1.0, 1.0), space: str = "transformed",
                 pixdim: Sequence[float] = (1.5, 1.5, 2.0)):
        unknown = set(metrics) - set(METRICS)
        if unknown or "dice" not in metrics:
            raise ValueError(f"metrics must include 'dice' and be drawn from {METRICS}, got {tuple(metrics)}")
        if len(spacing) != 3:
            raise ValueError(f"spacing needs one value per axis (D, H, W), got {tuple(spacing)}")
        if space not in SPACES:
            raise ValueError(f"space must be one of {SPACES}, got {space!r}")
        if len(pixdim) != 3:
            raise ValueError(f"pixdim needs one value per axis (D, H, W), got {tuple(pixdim)}")
        self.metrics, self.spacing = tuple(metrics), tuple(float(s) for s in spacing)
        self.space, self.pixdim = space, tuple(float(p) for p in pixdim)
        self.hd95s = []
        if use_amp is not None:
            model.set_precision("fp16" if use_amp else "fp32x3")
        self.model = model.to(device).eval()
        self.device = torch.device(device)
        self.num_classes = model.num_classes
        self.class_names = class_names or {i: f"class_{i}" for i in range(self.num_classes)}
        self.sw_batch_size, self.overlap = int(sw_batch_size), float(overlap)
        self.include_background, self.use_amp, self.epoch = include_background, use_amp, epoch
        self.spatial_size, self.image_size = model.patch[0], model.patch[1]
        self.dices, self.patient_index, self.global_step = [], 0, 0

    # ---- test.py:85-91
    def load_checkpoint(self, model_path: str) -> None:
        if self.epoch is not None:
            model_path = os.path.join(os.path.dirname(model_path), f"epoch_{self.epoch}.pt")
        state_dict = torch.load(model_path, map_location="cpu")
        self.model.load_state_dict(state_dict["model"])
        self.model.to(self.device)

    # ---- engine.py:151-166
    def convert_labels(self, labels: torch.Tensor, phase: str = "val") -> torch.Tensor:
        if not self.include_background:
            new_labels = [labels == i for i in sorted(self.class_names.keys())]
            return torch.cat(new_labels, dim=1)
        return labels

    def get_input(self, batch: dict, phase: str = "val") -> Tuple[torch.Tensor, torch.Tensor]:
        image = batch["image"].to(self.device)
        label = self.convert_labels(batch["label"].to(self.device), phase).float()
        return image, label

    def _spacings(self, batch: dict, n: int) -> list:
        """Per-sample voxel spacing of an original-space batch: ``batch["spacing"]`` as (3,) or [N, 3]."""
        if "spacing" not in batch:
            raise ValueError('space="original" needs batch["spacing"], the voxel spacing (D, H, W) of the input grid')
        s = torch.as_tensor(batch["spacing"], dtype=torch.float64).cpu()
        if s.shape == (3,):
            s = s.expand(n, 3)
        if s.shape != (n, 3):
            raise ValueError(f'batch["spacing"] must be (3,) or [{n}, 3], got {tuple(s.shape)}')
        return [tuple(row) for row in s.tolist()]

    # ---- engine.py:167-182
    @torch.no_grad()
    def infer(self, batch: dict, noise_fn=None):
        image, labels = self.get_input(batch, phase="val")
        spacings = self._spacings(batch, image.shape[0]) if self.space == "original" else None
        outputs_u8 = self._infer_binary(image, noise_fn, spacings)
        return image, outputs_u8.float(), labels

    def _infer_binary(self, image: torch.Tensor, noise_fn=None, spacings=None) -> torch.Tensor:
        """[N, C, D, H, W] uint8: ``(sigmoid(sliding_window(...)) > 0.5)`` formed by the finalize kernel.  With per-sample
        ``spacings`` the image is raw and each sample runs ``predict_original``: labels on the image's own grid."""
        if spacings is not None:
            return torch.stack([predict_original(self.model, image[n], spacings[n], self.pixdim, self.sw_batch_size, self.overlap,
                                                 noise_fn=noise_fn) for n in range(image.shape[0])])
        roi = tuple(self.model.patch)
        # the reference's call, engine.py:173-177: sliding_window_inference(image, roi, sw_batch_size, self.model, overlap,
        # pred_type="ddim_sample") -- the driver recognises the model and runs the fused window loop
        bufs = sliding_window_inference(image, roi, self.sw_batch_size, self.model, self.overlap, finalize=False,
                                        noise_fn=noise_fn, pred_type="ddim_sample")
        outs = []
        for b in bufs:
            _, binary, _ = b.finalize(binary=True)
            outs.append(crop_to(binary, image.shape[2:], b.vol))
        return torch.stack(outs)

    _crop_to = staticmethod(crop_to)

    # ---- test.py:112-160
    @torch.no_grad()
    def validation_step(self, batch: dict, noise_fn=None, verbose: bool = False) -> float:
        image, labels = self.get_input(batch, phase="val")
        spacings = self._spacings(batch, image.shape[0]) if self.space == "original" else None
        outputs = self._infer_binary(image, noise_fn, spacings)
        classes = list(self.class_names.values())
        dices = OrderedDict()
        counts = dice_counts(outputs.transpose(0, 1).contiguous().flatten(1), labels.transpose(0, 1).contiguous().flatten(1))
        for i, d in enumerate(dice_from_counts(counts.cpu().tolist())):
            dices[classes[i]] = d
            if verbose:
                print(f"{classes[i]} : {d:.4f}")
        self.dices.append(dices)
        if "hd95" in self.metrics:
            for n in range(outputs.shape[0]):  # per sample: surfaces must not mix across the batch
                spacing = self.spacing if spacings is None else spacings[n]
                self.hd95s.append(OrderedDict(zip(classes, hd95(outputs[n], labels[n], spacing))))
        self.patient_index += 1
        return float(np.mean(list(dices.values())))

    # ---- test.py:101-110
    def test(self, batches: Iterable[dict], noise_fn=None) -> float:
        vals = []
        for batch in batches:
            vals.append(self.validation_step(batch, noise_fn))
            self.global_step += 1
        return float(np.mean(vals)) if vals else float("nan")
