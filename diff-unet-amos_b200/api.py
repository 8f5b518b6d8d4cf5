"""Public surface of the B200 Diff-UNet inference package."""
from ._lib import DunetError, load as load_library
from .dist import (PeerExchange, peer_exchange_for, exchange_and_finalize, gather_channel_chunks, infer_volume_distributed, infer_volumes_distributed, my_window_range,
                   queue_group_size, queue_shares, reduce_partial_volume, reduce_scatter_channels)
from .engine import EngineB200, dice_counts, dice_from_counts, hd95
from .inference import StitchBuffers, crop_to, crop_windows, infer_volume, scale_intensity_range, sliding_window_inference
from .invert import invert_labels, predict_original
from .model import DEFAULT_FEATURES, PRECISIONS, DiffUNetB200, SmoothUNetDenoiserB200
from .preprocess import ValTransformMeta, crop_box, crop_foreground, foreground_bbox, resampled_shape, spacing_resample, val_meta, val_transform
from .schedule import DdimSchedule
from .windows import axis_counts, gaussian_importance_map, scan_intervals, shard_range, window_starts


def model_hub(model_name: str, **kwargs):
    """Registration seam of the reference's string-keyed factory (models/utils/model_hub.py:15-50, utils.py:27-33):
    ``"diff_unet_b200"`` (any name containing "diff" maps to ModelType.Diffusion there)."""
    if model_name in ("diff_unet_b200", "diff_unet"):
        return DiffUNetB200(**kwargs)
    raise NotImplementedError(f"No such model : {model_name}")


__all__ = ["DiffUNetB200", "EngineB200", "PeerExchange", "peer_exchange_for", "SmoothUNetDenoiserB200", "crop_box", "crop_foreground", "foreground_bbox", "resampled_shape", "spacing_resample", "val_transform", "ValTransformMeta", "val_meta", "invert_labels", "predict_original", "PRECISIONS", "crop_to", "crop_windows", "exchange_and_finalize", "infer_volumes_distributed", "queue_group_size", "queue_shares", "gather_channel_chunks", "reduce_scatter_channels", "gaussian_importance_map", "scale_intensity_range", "dice_counts", "dice_from_counts", "hd95", "DEFAULT_FEATURES", "DdimSchedule", "DunetError", "StitchBuffers", "axis_counts",
           "infer_volume", "infer_volume_distributed", "load_library", "my_window_range", "reduce_partial_volume", "model_hub", "scan_intervals", "shard_range", "sliding_window_inference",
           "window_starts"]
