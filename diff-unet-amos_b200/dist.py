"""Multi-GPU sliding-window inference: one process per GPU, windows sharded contiguously, ONE exchange per volume.

The reference runs inference on a single GPU (engine.py:172-177); its only distributed idiom on the evaluation side is a
contiguous per-rank shard followed by a gather (light_training/sampler.py:5-48).  Windows are independent units, so the
same idea applies.  Rank r processes a contiguous range of MONAI's window order into its own partial fp32 sum volume;
then the partial volumes are exchanged ONCE per volume:

  * ``ncclReduceScatter`` by channel (rank r keeps the summed logits of C/N channels),
  * every rank divides its channels by the analytic coverage counts and binarises them (finalize kernel),
  * the uint8 labels (4x smaller than the logits) are gathered on rank 0.

(``ncclReduce`` of the whole volume to rank 0 when C is not divisible by N.)  No collective touches the per-window data
path.  Two schedules:

  * latency mode   (``infer_volume_distributed``): the windows of ONE volume are split over all ranks.  With 98 windows
    on 8 ranks somebody owns ceil(98 / 8) = 13: scaling ceiling 98 / (8 * 13) = 0.942.
  * throughput mode (``infer_volumes_distributed``): G consecutive volumes form one window queue, G the smallest count
    with G * n_windows divisible by the world size (98 windows, 8 ranks: G = 4, 49 windows per rank), so every rank does
    exactly the same work between two exchange points.  The exchanges of a group run back to back once all its windows
    are done (never concurrently with the convolutions: a spinning NCCL kernel would take SMs away from the persistent
    one-CTA-per-SM conv kernels).

In throughput mode the exchange itself is NOT an NCCL collective: ``PeerExchange`` maps every rank's partial-sum buffers
into every other rank through CUDA IPC, and one kernel per (rank, volume) -- ``dunet_finalize_peers`` -- reads the
contributing ranks' partial sums of its channels directly over NVLink (only the slabs their windows touched), adds them,
divides by the counts, binarises and stores the uint8 labels straight into rank 0's volume.  The fp32 sums cross NVLink
once, only where they are non-zero (a volume of a 4-volume queue is covered by 2-3 of the 8 ranks), instead of an 8-rank
reduce-scatter of mostly-zero 2.7 GB buffers followed by a gather.  NCCL is used for two 4-byte all-reduces per group
that order the streams of the ranks (all partial sums written before / all peer reads done after).
"""
from __future__ import annotations

import ctypes
import math
from typing import Callable, Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch
import torch.distributed as dist

from . import _lib
from .windows import axis_counts, shard_range, window_starts


def _world() -> int:
    return dist.get_world_size() if dist.is_initialized() else 1


def _rank() -> int:
    return dist.get_rank() if dist.is_initialized() else 0


def my_window_range(n_windows: int, rank: Optional[int] = None, world: Optional[int] = None) -> Tuple[int, int]:
    if world is None:
        world = _world()
    if rank is None:
        rank = _rank()
    return shard_range(n_windows, rank, world)


def queue_group_size(n_windows: int, world: int, cap: int = 8) -> int:
    """Smallest number of volumes G (<= cap) whose combined window queue splits evenly over ``world`` ranks."""
    g = world // math.gcd(n_windows, world)
    return g if g <= cap else 1


def queue_shares(n_windows: int, group: int, rank: int, world: int) -> List[Tuple[int, int, int]]:
    """Rank ``rank``'s share of the window queue of ``group`` consecutive volumes: a list of (volume index in the group,
    first window, one past the last window), contiguous in the concatenated MONAI order."""
    lo, hi = shard_range(n_windows * group, rank, world)
    out = []
    for v in range(group):
        a, b = max(lo, v * n_windows), min(hi, (v + 1) * n_windows)
        if a < b:
            out.append((v, a - v * n_windows, b - v * n_windows))
    return out


def reduce_partial_volume(partial: torch.Tensor, dst: int = 0) -> torch.Tensor:
    """Sum the per-rank partial stitched volumes onto ``dst`` (in place on ``dst``).  Works with NCCL (CUDA tensors) and
    gloo (CPU tensors, used by the CPU tests)."""
    if _world() > 1:
        dist.reduce(partial, dst=dst, op=dist.ReduceOp.SUM)
    return partial


def reduce_scatter_channels(partial: torch.Tensor) -> torch.Tensor:
    """Sum the per-rank partial stitched volumes [C, D, H, W] and leave rank r with channels [r*C/N, (r+1)*C/N) of the
    sum (C must be divisible by the world size).  NCCL: one reduce-scatter over NVLink -- every rank then divides /
    binarises its own channels, so the fp32 volume is never gathered.  gloo (CPU tests) has no reduce-scatter: all-reduce
    then slice."""
    world = _world()
    if world == 1:
        return partial
    C = partial.shape[0]
    if C % world:
        raise ValueError(f"{C} channels cannot be split over {world} ranks")
    per = C // world
    rank = dist.get_rank()
    if partial.is_cuda:
        out = torch.empty((per,) + tuple(partial.shape[1:]), dtype=partial.dtype, device=partial.device)
        dist.reduce_scatter_tensor(out, partial.contiguous(), op=dist.ReduceOp.SUM)
        return out
    dist.all_reduce(partial, op=dist.ReduceOp.SUM)
    return partial[rank * per:(rank + 1) * per].clone()


def gather_channel_chunks(chunk: torch.Tensor, dst: int = 0):
    """Concatenate every rank's channel chunk (in rank order) on ``dst``; returns None elsewhere."""
    world = _world()
    if world == 1:
        return chunk
    chunk = chunk.contiguous()
    if dist.get_rank() == dst:
        parts = [torch.empty_like(chunk) for _ in range(world)]
        dist.gather(chunk, gather_list=parts, dst=dst)
        return torch.cat(parts, dim=0)
    dist.gather(chunk, gather_list=None, dst=dst)
    return None


def exchange_and_finalize(buf, dst: int = 0, want_blended: bool = True):
    """The one exchange of a volume: partial StitchBuffers of every rank -> (blended fp32 volume or None, uint8 binary
    labels) on ``dst``, (None, None) elsewhere.  Constant blend with C divisible by the world size: reduce-scatter by
    channel + local finalize + gather of the results; otherwise reduce to ``dst`` (the gaussian count volume included)."""
    from .inference import StitchBuffers

    world = _world()
    if world > 1 and buf.channels % world == 0 and buf.mode == "constant":
        mine = StitchBuffers.__new__(StitchBuffers)
        mine.vol, mine.roi, mine.mode, mine.counts, mine._finalized = buf.vol, buf.roi, buf.mode, buf.counts, False
        mine.channels = buf.channels // world
        mine.out = reduce_scatter_channels(buf.out)
        blended_c, binary_c, _ = mine.finalize(binary=True)
        blended = gather_channel_chunks(blended_c, dst) if want_blended else None
        binary = gather_channel_chunks(binary_c, dst)
        return (blended, binary) if _rank() == dst else (None, None)
    reduce_partial_volume(buf.out, dst)
    if buf.mode == "gaussian":
        reduce_partial_volume(buf.count_vol, dst)
    if _rank() == dst:
        blended, binary, _ = buf.finalize(binary=True)
        return (blended if want_blended else None), binary
    return None, None


class _RawCuda:
    """__cuda_array_interface__ view of a raw device pointer (memory owned by the library / another process)."""

    def __init__(self, ptr: int, nbytes: int):
        self.__cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (ptr, False), "version": 2}


class PeerExchange:
    """Peer-memory exchange of the partial stitched volumes (see the module docstring).  Every rank owns ``slots`` partial
    buffers [C, D, H, W] fp32 and (on ``dst``) ``label_slots`` label volumes [C, D, H, W] uint8, all allocated with
    ``dunet_ipc_alloc`` and mapped into every other rank with ``dunet_ipc_open`` (one exchange of 64-byte handles through
    torch.distributed at construction).  ``channels`` must be divisible by the world size, the volume width by 4."""

    def __init__(self, channels: int, vol: Sequence[int], roi: Sequence[int], overlap: float, device, slots: int = 3,
                 label_slots: int = 8, dst: int = 0):
        self.world, self.rank, self.dst = _world(), _rank(), dst
        self.channels, self.vol, self.roi, self.overlap = int(channels), tuple(int(v) for v in vol), tuple(roi), overlap
        if self.channels % self.world or self.vol[2] % 4:
            raise ValueError("PeerExchange needs channels % world == 0 and a volume width that is a multiple of 4")
        self.device = torch.device(device)
        self.lib = _lib.load()
        self.vox = self.vol[0] * self.vol[1] * self.vol[2]
        self.counts = [torch.from_numpy(c).to(self.device) for c in axis_counts(self.vol, self.roi, overlap)]
        self._owned, self._opened = [], []
        pbytes, lbytes = self.channels * self.vox * 4, self.channels * self.vox
        n_lab = label_slots if self.rank == dst else 0
        handles = np.zeros((slots + label_slots, 64), dtype=np.uint8)
        self.partial_ptr: List[List[int]] = [[0] * slots for _ in range(self.world)]
        self.label_ptr: List[int] = [0] * label_slots
        # Every rank goes through the SAME sequence of collectives whether or not its local CUDA-IPC calls succeed (a rank
        # that raised between two collectives would leave the others hanging); the outcome is agreed on at the end.
        err = None
        with torch.cuda.device(self.device):
            try:
                for i in range(slots + n_lab):
                    ptr = ctypes.c_void_p()
                    h = (ctypes.c_uint8 * 64)()
                    _lib.check(self.lib.dunet_ipc_alloc(ctypes.byref(ptr), pbytes if i < slots else lbytes, h))
                    self._owned.append(ptr.value)
                    handles[i] = np.frombuffer(bytes(h), dtype=np.uint8)
                    if i < slots:
                        self.partial_ptr[self.rank][i] = ptr.value
                    else:
                        self.label_ptr[i - slots] = ptr.value
            except Exception as e:  # noqa: BLE001
                err = e
            gathered = [None] * self.world
            dist.all_gather_object(gathered, None if err is not None else handles.tobytes())
            if err is None and any(g is None for g in gathered):
                err = RuntimeError("another rank could not allocate its CUDA-IPC buffers")
            if err is None:
                try:
                    for r in range(self.world):
                        if r == self.rank:
                            continue
                        hs = np.frombuffer(gathered[r], dtype=np.uint8).reshape(slots + label_slots, 64)
                        rng = list(range(slots)) + (list(range(slots, slots + label_slots)) if r == dst else [])
                        for i in rng:
                            ptr = ctypes.c_void_p()
                            h = (ctypes.c_uint8 * 64).from_buffer_copy(hs[i].tobytes())
                            _lib.check(self.lib.dunet_ipc_open(h, ctypes.byref(ptr)))
                            self._opened.append(ptr.value)
                            if i < slots:
                                self.partial_ptr[r][i] = ptr.value
                            else:
                                self.label_ptr[i - slots] = ptr.value
                except Exception as e:  # noqa: BLE001
                    err = e
            ok = torch.tensor([0.0 if err is not None else 1.0], device=self.device)
            dist.all_reduce(ok, op=dist.ReduceOp.MIN)
            if float(ok) == 0.0:
                self._release()
                raise RuntimeError(f"peer-memory exchange unavailable on this system: {err or 'another rank failed'}")
            # torch views of this rank's own buffers
            self.partial = [torch.as_tensor(_RawCuda(self.partial_ptr[self.rank][i], pbytes), device=self.device).view(torch.float32)
                            .view((self.channels,) + self.vol) for i in range(slots)]
            self.labels = ([torch.as_tensor(_RawCuda(self.label_ptr[i], lbytes), device=self.device).view((self.channels,) + self.vol)
                            for i in range(label_slots)] if self.rank == dst else [])
        self._flag = torch.zeros(1, device=self.device)
        self.slots, self.label_slots = slots, label_slots

    def barrier(self) -> None:
        """Stream-ordered barrier across the ranks: everything enqueued before it on every rank's current stream is
        complete (and visible to peers) before anything enqueued after it on any rank starts."""
        dist.all_reduce(self._flag)

    def finalize(self, sources: Sequence[Tuple[int, int, int, int]], label_slot: int) -> None:
        """sources: (rank, partial slot, first dim-0 row, one past the last row) of every rank that contributed to the
        volume, in rank order.  This rank reduces + finalizes its channel range into rank ``dst``'s label slot."""
        per = self.channels // self.world
        n = len(sources)
        ptrs = (ctypes.c_void_p * n)(*[self.partial_ptr[r][s] for r, s, _, _ in sources])
        lo = (ctypes.c_int32 * n)(*[a for _, _, a, _ in sources])
        hi = (ctypes.c_int32 * n)(*[b for _, _, _, b in sources])
        with torch.cuda.device(self.device):
            _lib.check(self.lib.dunet_finalize_peers(ptrs, lo, hi, n, _lib.i32x3(self.vol), self.rank * per, (self.rank + 1) * per,
                                                     ctypes.c_void_p(self.counts[0].data_ptr()), ctypes.c_void_p(self.counts[1].data_ptr()),
                                                     ctypes.c_void_p(self.counts[2].data_ptr()), ctypes.c_void_p(self.label_ptr[label_slot]),
                                                     None, ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)))

    def _release(self) -> None:
        for p in self._opened:
            self.lib.dunet_ipc_close(ctypes.c_void_p(p))
        self._opened = []
        for p in self._owned:
            self.lib.dunet_ipc_free(ctypes.c_void_p(p))
        self._owned = []

    def close(self) -> None:
        """Collective: unmap the peers' buffers, then free the own ones."""
        torch.cuda.synchronize(self.device)
        if dist.is_initialized():
            dist.barrier()
        for p in self._opened:
            self.lib.dunet_ipc_close(ctypes.c_void_p(p))
        self._opened = []
        if dist.is_initialized():
            dist.barrier()
        self._release()


_PEER_CACHE: Dict[tuple, Optional[PeerExchange]] = {}


def peer_exchange_for(channels: int, vol, roi, overlap: float, device, dst: int = 0) -> Optional[PeerExchange]:
    """The process-wide PeerExchange for this geometry (created on first use, collectively), or None when the fused
    peer-memory path does not apply (single rank, CPU / gloo tests, channels not divisible by the world size, ...)."""
    if _world() == 1 or torch.device(device).type != "cuda" or channels % _world() or vol[2] % 4 or dist.get_backend() != "nccl":
        return None
    key = (channels, tuple(vol), tuple(roi), float(overlap), str(device), dst, _world())
    if key not in _PEER_CACHE:
        try:  # the constructor is collective and fails on ALL ranks together (e.g. CUDA IPC not permitted in this container)
            _PEER_CACHE[key] = PeerExchange(channels, vol, roi, overlap, device, dst=dst)
        except RuntimeError as e:
            import warnings

            warnings.warn(f"{e}; falling back to the NCCL exchange")
            _PEER_CACHE[key] = None
    return _PEER_CACHE[key]


@torch.no_grad()
def infer_volume_distributed(model, image: torch.Tensor, sw_batch_size: int = 4, overlap: float = 0.25,
                             noise_fn: Optional[Callable[[int, int], torch.Tensor]] = None, dst: int = 0,
                             seed: Optional[int] = 0, mode: str = "constant"):
    """Engine.infer (engine.py:167-182) with the window list of every volume sharded over the process group (latency mode).

    Every rank holds the full input volume and the same weights.  Returns (blended volume, binary labels) on ``dst``
    and (None, None) elsewhere, cropped back to the input shape like the single-GPU driver.  ``noise_fn(first_window_index,
    count)`` supplies explicit noise (parity runs), window indices numbered ``n * n_windows + w`` like ``infer_volume``;
    otherwise window w draws from the library's counter-based stream (``seed``, w): the result does not depend on the
    number of ranks."""
    from .inference import crop_to, sliding_window_inference

    roi = model.patch
    vol = tuple(max(int(i), int(r)) for i, r in zip(image.shape[2:], roi))
    n_win = len(window_starts(vol, roi, overlap))
    lo, hi = my_window_range(n_win)
    bufs = sliding_window_inference(image, roi, sw_batch_size, model, overlap, mode=mode, window_range=(lo, hi), finalize=False,
                                    out_channels=model.num_classes, noise_fn=noise_fn, seed=seed, pred_type="ddim_sample")
    outs = []
    for b in bufs:
        blended, binary = exchange_and_finalize(b, dst)
        if _rank() == dst:
            outs.append((crop_to(blended, image.shape[2:], b.vol), crop_to(binary, image.shape[2:], b.vol)))
    if _rank() != dst:
        return None, None
    blended = torch.stack([o[0] for o in outs])
    labels = torch.stack([o[1] for o in outs]).float()
    return blended, labels


@torch.no_grad()
def infer_volumes_distributed(model, images: Sequence[torch.Tensor], sw_batch_size: int = 4, overlap: float = 0.25, dst: int = 0,
                              seed: int = 0, on_result: Optional[Callable[[int, torch.Tensor], None]] = None,
                              noise_fn: Optional[Callable[[int, int], torch.Tensor]] = None, exchange: str = "auto",
                              volume_shape: Optional[Sequence[int]] = None, device=None):
    """Throughput mode: ``images`` (a sequence of [1, in_channels, D, H, W] volumes of ONE shape, already >= the roi on every axis,
    available on every rank; an entry may also be a zero-argument callable returning the volume, which is then only called
    on the ranks whose queue share touches that volume -- e.g. a host-to-device copy that the other ranks can skip; pass
    ``volume_shape=`` in that case) are processed as window queues of G volumes (``queue_group_size``) so that every rank does the
    same number of windows between two exchange points.  ``on_result(volume_index, binary_labels_uint8)`` is called on
    ``dst`` as results become available (e.g. to start the D2H copy); returns the list of label volumes on ``dst``.
    Window w of volume i draws its noise from the stream (``seed``, i * n_windows + w): identical to running the volumes
    one by one through ``infer_volume_distributed`` / ``infer_volume`` with the same seed.
    ``exchange``: "p2p" = fused peer-memory reduce + finalize + gather (``PeerExchange``), "nccl" = reduce-scatter +
    finalize + gather collectives, "auto" = p2p whenever it applies."""
    from .inference import StitchBuffers

    world, rank = _world(), _rank()
    roi = model.patch
    if not images:
        return []
    if volume_shape is None:
        first = images[0]() if callable(images[0]) else images[0]
        images = [first] + list(images[1:])
        volume_shape = first.shape[2:]
        device = first.device
    vol = tuple(int(v) for v in volume_shape)
    if any(v < r for v, r in zip(vol, roi)):
        raise ValueError("throughput mode needs volumes that are at least the window size on every axis")
    starts = window_starts(vol, roi, overlap)
    n_win = len(starts)
    G = queue_group_size(n_win, world)
    step = min(int(sw_batch_size), model.batch_max)
    results = []
    dev = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
    px = peer_exchange_for(model.num_classes, vol, roi, overlap, dev, dst) if exchange in ("auto", "p2p") else None
    if exchange == "p2p" and px is None and world > 1:
        raise ValueError("the peer-memory exchange needs NCCL ranks on CUDA, channels % world == 0 and a width % 4 == 0")
    if px is not None and px.label_slots < G:
        px = None
    for g0 in range(0, len(images), G):
        grp = list(range(g0, min(g0 + G, len(images))))
        shares = queue_shares(n_win, len(grp), rank, world)
        bufs = {}
        for slot, (v, lo, hi) in enumerate(shares):
            img = images[grp[v]]
            if callable(img):
                img = img()  # materialised only on the ranks that need it
            if tuple(img.shape[2:]) != vol:
                raise ValueError("all volumes of a queue must have the same shape")
            if px is not None:
                if slot >= px.slots:
                    raise RuntimeError("a rank's queue share spans more volumes than the peer exchange has partial buffers")
                buf = bufs[v] = StitchBuffers(model.num_classes, vol, roi, overlap, dev, out=px.partial[slot])
                buf.zero_()
            else:
                buf = bufs[v] = StitchBuffers(model.num_classes, vol, roi, overlap, dev)
            bounds = list(range(lo, hi, step)) + [hi]
            if len(bounds) > 2 and bounds[-1] - bounds[-2] == 1 and step + 1 <= model.batch_max:
                del bounds[-2]  # a single left-over window joins the previous batch instead of running alone
            for a, b in zip(bounds[:-1], bounds[1:]):
                base = grp[v] * n_win
                if noise_fn is not None:
                    buf.add_windows(model, img[0], starts[a:b], noise=noise_fn(base + a, b - a))
                else:
                    buf.add_windows(model, img[0], starts[a:b], seed=seed, noise_ids=range(base + a, base + b))
        if px is not None:
            # ---- fused peer-memory exchange: every rank finalizes its channels of every volume of the group
            px.barrier()  # all partial sums of the group are complete on every rank
            for v in range(len(grp)):
                sources = []
                for r in range(world):
                    for slot, (vv_, lo, hi) in enumerate(queue_shares(n_win, len(grp), r, world)):
                        if vv_ == v:
                            sources.append((r, slot, int(starts[lo][0]), int(starts[hi - 1][0]) + roi[0]))
                px.finalize(sources, v)
            px.barrier()  # all peer reads and label stores are complete: buffers may be reused, labels consumed
            if rank == dst:
                for v in range(len(grp)):
                    binary = px.labels[v].clone()
                    if on_result is not None:
                        on_result(grp[v], binary)
                    results.append(binary)
            continue
        zero = None
        for v in range(len(grp)):  # the exchanges of the group, back to back, every rank takes part in every one
            buf = bufs.get(v)
            if buf is None:
                if zero is None:
                    zero = StitchBuffers(model.num_classes, vol, roi, overlap, dev)
                else:
                    zero.zero_()
                    zero._finalized = False
                buf = zero
            _, binary = exchange_and_finalize(buf, dst, want_blended=False)
            if rank == dst:
                if on_result is not None:
                    on_result(grp[v], binary)
                results.append(binary)
    return results if rank == dst else None
