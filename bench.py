#!/usr/bin/env python
"""bench.py -- Diff-UNet DDIM sliding-window inference throughput (BASELINE.json metric: 96^3 patches/s, DDIM-10).

    python bench.py --gpus N --steps K --warmup W                     # B200 path (this repo), default config amos98
    python bench.py --config {amos98|amos2645|btcv_b8_ens3|msd128_ddim25|wide} ...
    python bench.py --impl reference --gpus N --steps K ...           # the reference's CPU path (oracle port), host cores
    python bench.py ... --dump-outputs DIR                            # also write the last timed step's labels to DIR/labels.npy

One "step" = one pass of the hot path over one synthetic CT volume: window crop, encoder + N DDIM steps per window,
stitching, division by the coverage counts, binarisation.  Legs of the B200 arm (each bracketed by barrier + synchronize,
timed with CUDA events, max over ranks):

  value    K volumes resident in HBM, the PRODUCT configuration (fp16 operands, dual-stream batches, fused window loop,
           library noise generator).  N > 1: throughput mode -- G consecutive volumes form one window queue sharded
           evenly over the ranks (dist.py), one NCCL exchange per volume at the group boundary.
  e2e      the same through host buffers: every volume's H2D copy from pinned memory and the D2H copy of its label volume
           are inside the timed region (side streams, the D2H of volume i overlaps the windows of volume i + 1).
  latency  (N > 1) ONE volume sharded over all ranks (infer_volume_distributed): per-volume latency.
  profile  one short pass with CUDA events around every kernel launch (dual stream off so kernels do not overlap):
           roofline of the conv family, per-family HBM figures and time shares.  Not part of `value`.

Outside the timed regions, rank 0 also reports: `parity` (one window of the benchmarked mode against the fp32 oracle on
the GPU), `library_bar` (the oracle port = the reference's PyTorch graph, eager torch/cuDNN bf16 autocast on the same
GPU), `cpu_baseline` (the oracle port on the host cores, bounded sample), `checksum` of the label volume and, for N > 1,
`multi_gpu_check` (labels of the sharded run against a single-GPU run of the same volume on rank 0).
Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

DEFAULT_FEATURES = (64, 64, 128, 256, 512, 64)
METRIC = "96^3 patches/s (DDIM-10)"
# BASELINE.json configs (SURVEY 8d).  amos98 is the configuration the metric is quoted on (config 2/3); the others are
# selectable so that every named configuration has a measured line under profiles/.
CONFIGS = {
    "amos98": dict(volume=(512, 512, 160), roi=96, classes=16, features=DEFAULT_FEATURES, overlap=0.25, sw_batch=4, ddim=10, ensemble=1,
                   workload="AMOS 16-class sliding-window DDIM-10 inference, synthetic 512x512x160 CT volume, roi 96^3, overlap 0.25 (98 windows)"),
    "amos2645": dict(volume=(512, 512, 160), roi=96, classes=16, features=DEFAULT_FEATURES, overlap=0.8, sw_batch=4, ddim=10, ensemble=1,
                     workload="AMOS 16-class sliding-window DDIM-10 inference, synthetic 512x512x160 CT volume, roi 96^3, overlap 0.8 (2645 windows; cfg/btcv, cfg/msd)"),
    "btcv_b8_ens3": dict(volume=(512, 512, 160), roi=96, classes=14, features=DEFAULT_FEATURES, overlap=0.25, sw_batch=8, ddim=10, ensemble=3,
                         workload="BTCV 14-class, 96^3 patches, window batch 8, DDIM-10, 3-sample ensemble averaging, synthetic 512x512x160 volume, overlap 0.25 (98 windows)"),
    "msd128_ddim25": dict(volume=(512, 512, 160), roi=128, classes=3, features=DEFAULT_FEATURES, overlap=0.25, sw_batch=4, ddim=25, ensemble=1,
                          workload="MSD 3-class, 128^3 patches, window batch 4, DDIM-25, synthetic 512x512x160 volume, overlap 0.25 (50 windows)"),
    "wide": dict(volume=(96, 96, 96), roi=96, classes=16, features=(64, 128, 256, 512, 1024, 64), overlap=0.25, sw_batch=1, ddim=10, ensemble=1,
                 workload="BasicUNet feat 64-128-256-512-1024(+64), single 96^3 patch, 1+16 ch, DDIM-10, batch 1 (BASELINE config 1 on the GPU)"),
}


def algorithmic_gflop(features, classes, S, n_steps):
    """ALGORITHMIC GFLOP of one window: 2*M*N*K per layer, real channels only (SURVEY 8d / Appendix A).  Returns
    (encoder, one denoiser step, conv3x3x3-only part of a denoiser step)."""
    f = list(features)
    V = [(S >> l) ** 3 for l in range(5)]
    conv = lambda v, cin, cout: 2.0 * v * cout * 27 * cin
    enc = conv(V[0], 1, f[0]) + conv(V[0], f[0], f[0])
    den3 = conv(V[0], 1 + classes, f[0]) + conv(V[0], f[0], f[0])
    for l in range(1, 5):
        enc += conv(V[l], f[l - 1], f[l]) + conv(V[l], f[l], f[l])
        den3 += conv(V[l], f[l - 1], f[l]) + conv(V[l], f[l], f[l])
    other = 0.0
    for l in range(4, 0, -1):  # UpCat l: deconv f[l] -> up, cat([f[l-1], up]) -> out
        up = f[1] if l == 1 else f[l] // 2
        out = f[5] if l == 1 else f[l - 1]
        other += 2.0 * V[l - 1] * f[l] * up
        den3 += conv(V[l - 1], f[l - 1] + up, out) + conv(V[l - 1], out, out)
    other += 2.0 * V[0] * f[5] * classes
    return enc / 1e9, (den3 + other) / 1e9, den3 / 1e9


DUMP_MAX_VALUES = 1 << 23  # 32 MB of float32: the largest array --dump-outputs writes whole


def dump_outputs(out_dir, arrays):
    """Write each tensor of ``arrays`` as out_dir/<name>.npy in float32: whole when it has at most DUMP_MAX_VALUES
    elements, otherwise the elements at DUMP_MAX_VALUES flat indices drawn from numpy default_rng(0) (with repetition,
    sorted), the same for every run of the same configuration.  Returns what was written, for the JSON line."""
    import numpy as np
    import torch

    os.makedirs(out_dir, exist_ok=True)
    info = {}
    for name, t in arrays.items():
        entry = {"shape": list(t.shape), "dtype": str(t.dtype).replace("torch.", "")}
        if t.numel() > DUMP_MAX_VALUES:
            idx = np.sort(np.random.default_rng(0).integers(0, t.numel(), DUMP_MAX_VALUES))
            t = t.reshape(-1)[torch.from_numpy(idx).to(t.device)]
            entry["sample"] = f"{DUMP_MAX_VALUES} flat indices, numpy default_rng(0).integers(0, numel, n), sorted"
        np.save(os.path.join(out_dir, name + ".npy"), t.float().cpu().numpy())
        info[name] = entry
    return {"dir": out_dir, "arrays": info}


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"], "bf16_tflops_sustained": d["bf16_tflops_sustained"],
                "source": "measured (MEASURED_PEAKS.json)"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    """nvidia-smi SM clocks / throttle reasons sampled every 200 ms during the timed region."""

    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index: int):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thr = threading.Thread(target=self._read, daemon=True)
            self.thr.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm = sorted(int(r[0]) for r in self.rows if r and r[0].isdigit())
        mx = [int(r[1]) for r in self.rows if len(r) > 1 and r[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 2 + i and r[2 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm)}


# ----------------------------------------------------------------------------------------------------------------
# reference arm / cpu_baseline: the oracle port of the reference's CPU path on the host cores
# ----------------------------------------------------------------------------------------------------------------
def cpu_window_sample(cfg, threads: int):
    """Bounded sample of one window of the reference path at the config's own width / classes / window size: the encoder
    once + ONE of the N denoiser/DDIM steps, fp32, torch CPU.  Returns (seconds_encoder, seconds_step)."""
    import torch

    from oracle import oracle_ddim, oracle_model

    torch.set_num_threads(threads)
    S, C = cfg["roi"], cfg["classes"]
    sd = oracle_model.init_state_dict(1, C, cfg["features"], seed=0)
    torch.manual_seed(1)
    image = torch.rand(1, 1, S, S, S)
    torch.manual_seed(2)
    x = torch.randn(1, C, S, S, S)
    sched = oracle_ddim.SpacedSchedule(cfg["ddim"])
    with torch.no_grad():
        t0 = time.perf_counter()
        emb = oracle_model.encoder_forward(sd, image)
        t1 = time.perf_counter()
        out = oracle_model.denoiser_forward(sd, x, torch.tensor([sched.timestep_map[-1]]), image, emb)
        oracle_ddim.ddim_step(sched, sched.num_timesteps - 1, x, out)
        t2 = time.perf_counter()
    return t1 - t0, t2 - t1


def cpu_sample_text(cfg):
    return (f"encoder + 1 of {cfg['ddim']} DDIM steps of one {cfg['roi']}^3 window (C={cfg['classes']}, features {list(cfg['features'])}, "
            f"x{cfg['ensemble']} ensemble draws), fp32 torch CPU oracle port; patches/s = 1/(t_enc + {cfg['ddim'] * cfg['ensemble']}*t_step)")


def run_reference(args, cfg):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    n_steps = cfg["ddim"] * cfg["ensemble"]
    cpu_window_sample(cfg, threads) if args.warmup > 0 else None  # one warm-up sample (allocator, oneDNN primitives)
    t_all, vals = time.perf_counter(), []
    for _ in range(max(args.steps, 1)):
        te, ts = cpu_window_sample(cfg, threads)
        vals.append(1.0 / (te + n_steps * ts))
    elapsed = time.perf_counter() - t_all
    v = sum(vals) / len(vals)
    print_json({
        "impl": "reference", "metric": METRIC, "value": v, "unit": "patches/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * elapsed / max(args.steps, 1), "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": cfg["workload"], "name": args.config,
                   "note": "reference CPU path (oracle port of the reference's PyTorch code; the reference is pure Python and cannot travel to the GPU box)"},
        "cpu_baseline": {"value": v, "unit": "patches/s", "cores": threads, "kind": "port", "sample": "per step: " + cpu_sample_text(cfg)},
        "e2e": {"value": v, "unit": "patches/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    })


# ----------------------------------------------------------------------------------------------------------------
# B200 arm
# ----------------------------------------------------------------------------------------------------------------
def oracle_window_gpu(sd, image, noise, n_steps):
    """the oracle port evaluated with torch on the GPU (fp32, TF32 off): the checker of the `parity` block"""
    import numpy as np
    import torch

    from oracle import oracle_ddim, oracle_model

    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    sched = oracle_ddim.SpacedSchedule(n_steps)
    e = oracle_model.encoder_forward(sd, image)
    x, ref = noise, torch.zeros_like(noise)
    for i in reversed(range(n_steps)):
        t = torch.full((image.shape[0],), sched.timestep_map[i], dtype=torch.int64, device=image.device)
        x, x0 = oracle_ddim.ddim_step(sched, i, x, oracle_model.denoiser_forward(sd, x, t, image, e))
        ref = ref + x0
    return ref


def library_bar(sd, cfg, batch, dev):
    """SURVEY 8d "library bar": the reference's network (oracle port of its PyTorch graph) run eagerly with torch/cuDNN on
    this GPU under bf16 autocast (TF32 allowed), one batch of windows, same window size / classes / steps."""
    import torch

    from oracle import oracle_ddim, oracle_model

    S, C, n = cfg["roi"], cfg["classes"], cfg["ddim"]
    torch.backends.cudnn.allow_tf32 = True
    torch.backends.cuda.matmul.allow_tf32 = True
    torch.backends.cudnn.benchmark = True
    image = torch.rand(batch, 1, S, S, S, device=dev)
    noise = torch.randn(batch, C, S, S, S, device=dev)
    sched = oracle_ddim.SpacedSchedule(n)

    def window():
        with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16):
            emb = oracle_model.encoder_forward(sd, image)
            for _ in range(cfg["ensemble"]):
                x, acc = noise, torch.zeros_like(noise)
                for i in reversed(range(n)):
                    t = torch.full((batch,), sched.timestep_map[i], dtype=torch.int64, device=dev)
                    x, x0 = oracle_ddim.ddim_step(sched, i, x, oracle_model.denoiser_forward(sd, x, t, image, emb).float())
                    acc = acc + x0
        return acc

    window()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 2
    e0.record()
    for _ in range(reps):
        window()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    torch.backends.cudnn.benchmark = False
    return {"value": 1e3 * batch / ms, "unit": "patches/s", "ms_per_call": ms, "windows_per_call": batch,
            "what": "oracle port of the reference's PyTorch network, eager torch + cuDNN/cuBLAS on this GPU, bf16 autocast (TF32 allowed), "
                    "window compute only (no crop / stitch), device-resident"}


def run_b200(args, cfg):
    import numpy as np
    import torch
    import torch.distributed as dist

    import diff_unet_amos_b200 as pkg
    from diff_unet_amos_b200 import _lib

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    lib = pkg.load_library()

    VOLUME, S, C, FEATURES = tuple(cfg["volume"]), cfg["roi"], cfg["classes"], tuple(cfg["features"])
    ROI = (S, S, S)
    sw_batch = args.sw_batch or cfg["sw_batch"]
    ens = cfg["ensemble"]
    torch.manual_seed(0)
    model = pkg.DiffUNetB200(in_channels=1, out_channels=C, image_size=S, spatial_size=S, features=FEATURES, num_steps=cfg["ddim"],
                             batch_max=sw_batch + 1, precision=args.precision, dual_stream=bool(args.dual_stream)).to(dev).eval()
    torch.manual_seed(1)
    host_vol = torch.rand(1, 1, *VOLUME).pin_memory()
    dev_vol = host_vol.to(dev)
    starts = pkg.window_starts(VOLUME, ROI, cfg["overlap"])
    n_win = len(starts)
    G = pkg.queue_group_size(n_win, world)
    lo, hi = pkg.shard_range(n_win, rank, world)
    SEED = 2
    host_labels = [torch.empty((C,) + VOLUME, dtype=torch.uint8).pin_memory() for _ in range(2)] if rank == 0 else None
    enc_gf, step_gf, step_conv_gf = algorithmic_gflop(FEATURES, C, S, cfg["ddim"])
    gflop_per_window = enc_gf + ens * cfg["ddim"] * step_gf

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def run_queue(volumes, on_result=None):
        return pkg.infer_volumes_distributed(model, volumes, sw_batch_size=sw_batch, overlap=cfg["overlap"], seed=SEED, on_result=on_result,
                                             exchange=args.exchange, volume_shape=VOLUME, device=dev)

    def my_windows_only(volume):
        """this rank's latency-mode shard of one volume, no exchange (profiled pass)"""
        buf = pkg.StitchBuffers(C, VOLUME, ROI, cfg["overlap"], dev)
        for g in range(lo, hi, sw_batch):
            g1 = min(g + sw_batch, hi)
            buf.add_windows(model, volume[0, 0], starts[g:g1], seed=SEED, noise_ids=range(g, g1), ensemble=ens)
        return buf

    if ens > 1:  # ensemble draws ride on the single-volume driver (the queue driver is R = 1)
        def run_queue(volumes, on_result=None):  # noqa: F811
            outs = []
            for i, v in enumerate(volumes):
                bufs = pkg.sliding_window_inference(v, ROI, sw_batch, model, cfg["overlap"], finalize=False, seed=SEED, ensemble=ens,
                                                    window_range=(lo, hi), out_channels=C, pred_type="ddim_sample")
                _, binary = pkg.exchange_and_finalize(bufs[0], 0, want_blended=False)
                if rank == 0:
                    if on_result is not None:
                        on_result(i, binary)
                    outs.append(binary)
            return outs if rank == 0 else None

    with torch.no_grad():
        for _ in range(args.warmup):
            run_queue([dev_vol])
        # ---------------- device-resident leg: `value` (product configuration, nothing profiled) ----------------
        clocks = ClockSampler(local) if rank == 0 else None  # started BEFORE the barrier: spawning nvidia-smi takes ~0.1 s on rank 0
        if n_win * cfg["ddim"] * ens < 200:
            # a step of a few tens of ms (the single-window config): the GPU idled while nvidia-smi was spawned and the clocks
            # dropped -- one more untimed step right before the timed region (the long configs re-ramp within 1 % of a step)
            run_queue([dev_vol])
        barrier()
        l0 = lib.dunet_launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        labels = run_queue([dev_vol] * args.steps)
        e1.record()
        barrier()
        launches = lib.dunet_launch_count() - l0
        clk = clocks.stop() if clocks else None
        ms = e0.elapsed_time(e1)
        last_labels = labels[0] if rank == 0 else None  # volume 0 of the queue: its windows draw the noise streams (seed, 0 .. n_win - 1)
        final_labels = labels[-1] if rank == 0 and args.dump_outputs else None  # what the last timed step returned
        del labels
        # ---------------- end-to-end leg: host volume in, host labels out, every step ----------------
        barrier()
        copy_stream, d2h_stream = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)
        main = torch.cuda.current_stream()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        keep = []

        def to_host(i, binary):
            d2h_stream.wait_stream(main)
            with torch.cuda.stream(d2h_stream):
                host_labels[i % 2].copy_(binary, non_blocking=True)  # D2H of the step's result (binary label volume)
            binary.record_stream(d2h_stream)

        h2d_count = [0]

        def upload():
            """H2D of one step's input from pinned memory, on the copy stream; the compute stream waits for it"""
            with torch.cuda.stream(copy_stream):
                v = host_vol.to(dev, non_blocking=True)
            main.wait_stream(copy_stream)
            v.record_stream(main)
            h2d_count[0] += 1
            return v

        f0.record()
        if world == 1 or ens > 1:
            for _ in range(args.steps):
                keep.append(run_queue([upload()], on_result=to_host))
        else:
            # window queues: a rank uploads only the volumes its share of the queue touches (2 of the 4 volumes of a group at N = 8)
            run_queue([upload] * args.steps, on_result=to_host)
        main.wait_stream(d2h_stream)
        f1.record()
        barrier()
        ms_e2e = f0.elapsed_time(f1)
        del keep
        # ---------------- latency leg (N > 1): one volume sharded over all ranks ----------------
        ms_lat = None
        if world > 1:
            barrier()
            g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            reps = 3
            for it in range(reps + 1):  # first repetition untimed (first NCCL collectives of this shape)
                if it == 1:
                    barrier()
                    g0.record()
                bufs = pkg.sliding_window_inference(dev_vol, ROI, sw_batch, model, cfg["overlap"], finalize=False, seed=SEED,
                                                    window_range=(lo, hi), out_channels=C, pred_type="ddim_sample")
                _, lat_labels = pkg.exchange_and_finalize(bufs[0], 0, want_blended=False)
            g1.record()
            barrier()
            ms_lat = g0.elapsed_time(g1) / reps
        # ---------------- profiled pass: this rank's shard of one volume, events around every launch ----------------
        plan = model._rt.plan
        _lib.check(lib.dunet_profile_enable(plan, 1))
        barrier()
        p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        p0.record()
        my_windows_only(dev_vol)
        p1.record()
        torch.cuda.synchronize()
        ms_prof = p0.elapsed_time(p1)
        conv_ms, conv_n, conv_fl = ctypes.c_double(), ctypes.c_uint64(), ctypes.c_double()
        _lib.check(lib.dunet_profile_read(plan, ctypes.byref(conv_ms), ctypes.byref(conv_n), ctypes.byref(conv_fl)))
        fam_ms, fam_n, fam_b = (ctypes.c_double * 12)(), (ctypes.c_uint64 * 12)(), (ctypes.c_double * 12)()
        _lib.check(lib.dunet_profile_read_all(plan, fam_ms, fam_n, fam_b))
        _lib.check(lib.dunet_profile_enable(plan, 0))
    if world > 1:
        t = torch.tensor([ms, ms_e2e, ms_lat, float(launches)], device=dev, dtype=torch.float64)
        tmax = t.clone()
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        ms, ms_e2e, ms_lat, launches = float(tmax[0]), float(tmax[1]), float(tmax[2]), int(t[3])
    # ---------------- correctness evidence outside the timed regions ----------------
    check = None
    if world > 1:
        with torch.no_grad():
            if rank == 0:  # the same volume on ONE GPU (all windows, MONAI order): labels must match the sharded run
                _, single = pkg.infer_volume(model, dev_vol, sw_batch_size=sw_batch, overlap=cfg["overlap"], seed=SEED, ensemble=ens)
                single = single[0].to(torch.uint8)
                diff = single != last_labels
                n_diff = int(diff.sum())
                check = {"label_mismatch_voxels": n_diff, "of": int(single.numel()), "labels_equal_to_single_gpu_run": n_diff == 0,
                         "note": "a sharded run sums the per-rank partial volumes in a different fp32 order than one GPU does; voxels whose "
                                 "stitched logit is within ~1e-6 of 0 may binarise differently"}
                del single, diff
            barrier()
    if rank == 0:
        from oracle import oracle_model  # checker only: parity block, library bar, cpu baseline

        peaks = measured_peaks()
        peak = peaks["bf16_tflops_sustained"]
        value = n_win * args.steps / (ms / 1e3)
        e2e = n_win * args.steps / (ms_e2e / 1e3)
        conv_tflops = conv_fl.value / (conv_ms.value / 1e3) / 1e12 if conv_ms.value > 0 else 0.0
        # checksum of the label volume of the value leg (noise is a function of (seed, window index): identical at every N up
        # to the fp32 summation order of the exchange, see multi_gpu_check)
        lab_host = host_labels[0]
        lab_host.copy_(last_labels)
        torch.cuda.synchronize()
        arr = lab_host.numpy().reshape(-1)
        pad = (-arr.size) % 8
        words = np.concatenate([arr, np.zeros(pad, np.uint8)]).view(np.uint64)
        checksum = {"positive_voxels": int(arr.sum(dtype=np.int64)), "xor64": f"{int(np.bitwise_xor.reduce(words)):016x}",
                    "voxels": int(arr.size), "noise": f"library Philox stream (seed {SEED}, global window index)"}
        # parity of the benchmarked mode: window 0 of the volume, fixed noise, against the fp32 oracle on this GPU
        sd = {k: v.detach() for k, v in model.state_dict().items()}
        with torch.no_grad():
            s0 = starts[0]
            img = dev_vol[:, :, s0[0]:s0[0] + S, s0[1]:s0[1] + S, s0[2]:s0[2] + S].contiguous()
            gen = torch.Generator(device=dev)
            gen.manual_seed(2)
            nz = torch.randn((1, C) + ROI, device=dev, generator=gen)
            got = model(image=img, pred_type="ddim_sample", noise=nz)
            ref = oracle_window_gpu(sd, img, nz, cfg["ddim"])
            parity = {"window": "window 0 of the volume, fixed noise, vs the fp32 oracle port on this GPU (TF32 off)",
                      "rel_l2": float((got - ref).norm() / ref.norm()),
                      "binarisation_agreement_raw": float(((got > 0) == (ref > 0)).float().mean()),
                      "argmax_agreement_raw": float((got.argmax(1) == ref.argmax(1)).float().mean()) if C > 1 else None,
                      "gates": "north_star: rel-l2 <= 2e-2 (reduced precision), label agreement >= 0.999"}
            del got, ref
            bar = library_bar(sd, cfg, sw_batch, dev) if not args.no_library_bar else None
        dtype = {"fp16": "fp16 (fp32 accumulate; encoder in split-bf16)", "bf16": "bf16", "fp32x3": "bf16x3 (fp32-class split operands)"}[args.precision]
        out = {
            "metric": METRIC, "value": value, "unit": "patches/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": dtype, "data": "synthetic",
            "config": {"workload": cfg["workload"], "name": args.config, "features": list(FEATURES), "classes": C, "sw_batch": sw_batch,
                       "ddim_steps": cfg["ddim"], "ensemble": ens, "windows_per_step": n_win, "volumes_per_s": value / n_win,
                       "schedule": (f"throughput mode: window queues of {G} volume(s) sharded evenly over {world} ranks, one exchange per volume at the "
                                    "group boundary") if world > 1 else "single GPU, windows in batches of sw_batch",
                       "exchange": (("fused peer-memory kernel over NVLink (dunet_finalize_peers: reduce + divide + binarise + gather; NCCL only for two "
                                     "4-byte stream barriers per group)" if (args.exchange != "nccl" and ens == 1 and C % world == 0 and VOLUME[2] % 4 == 0)
                                     else "NCCL reduce-scatter by channel + local finalize + gather") if world > 1 else None),
                       "dual_stream": "on (half batches on two internal streams)" if args.dual_stream else "off",
                       "l2": "inputs larger than L2 (each window streams > 1 GB of activations; no flush needed)",
                       "algorithmic_tflop_per_window": gflop_per_window / 1e3,
                       "whole_path_tflops": value * gflop_per_window / 1e3,
                       "whole_path_frac_of_bf16_peak": value * gflop_per_window / 1e3 / world / peak},
            "clocks": clk,
            "e2e": {"value": e2e, "unit": "patches/s", "h2d_bytes_per_step": host_vol.numel() * 4 * h2d_count[0] / args.steps,
                    "d2h_bytes_per_step": host_labels[0].numel(), "ms_per_step": ms_e2e / args.steps,
                    "note": "h2d bytes: rank 0's uploads per step (N > 1: every rank uploads the volumes its queue share touches)"},
            "gpu_launches": int(launches),
            "parity": parity,
            "checksum": checksum,
            "roofline": {"bound": "tensor", "kernel": "conv3d_tc64_kernel + conv3d_flat_kernel (+ conv3d_tc_kernel): every 16-bit-operand 3x3x3 conv launch of rank 0 in the profiled pass (CUDA events "
                                                      "around each launch); the encoder's split-precision convs (fp16 mode: 3 MMAs per product, 2.6 % of the FLOPs) are listed under split_precision_convs",
                         "achieved": conv_tflops, "peak": peak, "unit": "TFLOP/s", "frac": conv_tflops / peak,
                         "peak_source": peaks["source"] + ", sustained cuBLAS bf16 (kind::f16 MMAs run fp16 and bf16 at the same rate)",
                         "launches": int(conv_n.value), "avg_launch_ms": conv_ms.value / max(conv_n.value, 1),
                         "conv_share_of_profiled_pass": (fam_ms[0] + fam_ms[8]) / ms_prof,
                         "frac_of_burst_peak": conv_tflops / peaks["bf16_tflops"],
                         "split_precision_convs": ({"algorithmic_tflops": fam_b[8] / fam_ms[8] / 1e9, "executed_mma_tflops": 3 * fam_b[8] / fam_ms[8] / 1e9,
                                                    "launches": int(fam_n[8]), "share_of_profiled_pass": fam_ms[8] / ms_prof} if fam_ms[8] > 0 else None),
                         "all_convs_algorithmic_tflops": (fam_b[0] + fam_b[8]) / (fam_ms[0] + fam_ms[8]) / 1e9 if fam_ms[0] + fam_ms[8] > 0 else None,
                         "traffic": None, "traffic_source": "profiles/ (ncu --set full captures per kernel: dram__bytes_read.sum + dram__bytes_write.sum); not read live"},
            "roofline_hbm": {name: {"bound": "hbm", "achieved": fam_b[i] / fam_ms[i] / 1e6, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                                    "frac": fam_b[i] / fam_ms[i] / 1e6 / peaks["hbm_gbs"], "launches": int(fam_n[i]),
                                    "share_of_profiled_pass": fam_ms[i] / ms_prof}
                             for i, name in ((1, "normalise (IN+LeakyReLU+bias+residual+pool), launches >= 64 MB"), (2, "final 1x1 conv + DDIM update + accumulate"),
                                             (3, "transposed conv k2s2, launches >= 64 MB"), (9, "transposed conv k2s2, launches < 64 MB (launch-latency bound)"),
                                             (4, "split-K reduce (split-precision encoder only; the denoiser's is fused into the normalise pass)"),
                                             (6, "normalise, launches < 64 MB (launch-latency bound)"),
                                             (7, "glue: window crop, noise + state init, stitch from the voxel-major accumulator")) if fam_ms[i] > 0},
            "kernel_time_share": dict({n: fam_ms[i] / ms_prof for i, n in enumerate(["conv3x3x3", "normalise_large", "final_ddim", "deconv", "splitk_reduce", "affine_map", "normalise_small", "glue",
                                                                                     "conv3x3x3_split_precision_encoder", "deconv_small"])},
                                      sum=sum(fam_ms) / ms_prof, profiled_pass_ms=ms_prof,
                                      note="profiled pass: single stream, events around every launch; shares are of that pass's own elapsed time"),
        }
        if ms_lat is not None:
            out["volume_latency_ms"] = ms_lat
            out["config"]["latency_mode"] = f"one volume sharded over {world} ranks (max {-(-n_win // world)} windows per rank): {ms_lat:.1f} ms per volume"
        if check is not None:
            out["multi_gpu_check"] = check
        if bar is not None:
            out["library_bar"] = bar
        if world == 1 and not args.no_cpu_baseline:
            threads = os.cpu_count() or 1
            te, ts = cpu_window_sample(cfg, threads)
            out["cpu_baseline"] = {"value": 1.0 / (te + cfg["ddim"] * ens * ts), "unit": "patches/s", "cores": threads, "kind": "port",
                                   "sample": cpu_sample_text(cfg)}
        if final_labels is not None:
            out["dump_outputs"] = dump_outputs(args.dump_outputs, {"labels": final_labels})
        print_json(out)
    if world > 1:
        dist.destroy_process_group()


def _claim_stdout():
    """Libraries (NCCL prints its version banner) write to fd 1; the contract is ONE JSON line on stdout.  Route fd 1 to
    stderr for the duration of the run and return a writer bound to the real stdout."""
    sys.stdout.flush()
    real = os.dup(1)
    os.dup2(2, 1)
    return os.fdopen(real, "w")


def main():
    out_stream = _claim_stdout()
    global print_json

    def print_json(obj):
        out_stream.write(json.dumps(obj) + "\n")
        out_stream.flush()

    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="amos98", choices=sorted(CONFIGS), help="BASELINE.json configuration (default: the one the metric is quoted on)")
    ap.add_argument("--sw-batch", type=int, default=0, help="windows per launch (default: the config's)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-library-bar", action="store_true")
    ap.add_argument("--precision", default="fp16", choices=["fp16", "bf16", "fp32x3"],
                    help="fp16 (default, passes every north_star gate), bf16 (misses the 99.9 %% label gate), fp32x3 (fp32-class)")
    ap.add_argument("--exchange", default="auto", choices=["auto", "p2p", "nccl"],
                    help="N > 1: how the per-rank partial volumes are combined: p2p = one fused kernel over NVLink peer memory (reduce + "
                         "finalize + gather, dist.PeerExchange), nccl = reduce-scatter + finalize + gather collectives; auto = p2p when it applies")
    ap.add_argument("--dual-stream", type=int, default=1, help="DUNET_FLAG_DUAL_STREAM: two half batches on two internal streams (the product default)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the label volume the last timed step returned as DIR/labels.npy (float32; "
                         "volumes over 2^23 voxels as a fixed seeded sample) so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs needs the B200 path (the reference arm times a sample of one window and returns no volume)")
    cfg = CONFIGS[args.config]
    if args.impl == "reference":
        run_reference(args, cfg)
    else:
        run_b200(args, cfg)


if __name__ == "__main__":
    main()
