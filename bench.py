#!/usr/bin/env python
"""bench.py -- MC-dropout tiles/sec of the B200-native Xception-UQ + UQ-thresholding hot path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl native|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is one pass of the hot path over one synthetic whole-slide image per GPU (BASELINE.json
configs[1]: 10,000 uint8 299x299x3 tiles, T = 30): tile standardisation + Xception backbone (once per
tile) + 30 dropout-head samples + per-tile mean/std, then the per-slide reduction and `threshold.apply`.
Weak scaling: every rank processes its own slide(s); only per-slide aggregates are all-gathered (NCCL).

Prints ONE JSON line (rank 0):
  value     tiles/s with the tiles already resident in HBM (whole job, all GPUs, max time over ranks)
  e2e       the same through the public API with HOST (pinned) tiles: H2D of every tile and D2H of the
            per-tile results inside the timed region
  roofline  dominant kernel family: algorithmic FLOPs of its launches / their summed CUDA-event time
            (events on the library's own stream), against MEASURED_PEAKS.json
  cpu_baseline  the restated reference schedule (T full forward passes, fp32, oracle/xception_uq.py)
            on the host cores over a bounded sample -- a reported baseline, not the target
`--impl reference` times that CPU path alone (TensorFlow/Slideflow cannot be installed: no wheel, no
network -- DESIGN.md), same metric / unit / config.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "MC-dropout tiles/sec (Xception-UQ, T=30, 299^2)"
TILE_PX = 299
TILE_BYTES = TILE_PX * TILE_PX * 3
BACKBONE_GFLOP = 16.7107          # SURVEY.md 8d, checked by biscuit_b200.weights.backbone_macs_per_tile
HEAD_MFLOP_PER_SAMPLE = 2 * (1024 * 1024 + 1024 * 2) / 1e6
HEAD_ONCE_MFLOP = 2 * 2048 * 1024 / 1e6


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--tiles", type=int, default=10000, help="tiles per slide (per GPU per step)")
    ap.add_argument("--slides", type=int, default=1, help="slides per GPU per step")
    ap.add_argument("--T", type=int, default=30)
    ap.add_argument("--max-batch", type=int, default=503, help="micro-batch (biscuit_b200.uq.BENCH_MICRO_BATCH)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--cpu-seconds", type=float, default=15.0, help="target size of the CPU-baseline sample")
    ap.add_argument("--workload", default="wsi", choices=["wsi", "cohort"],
                    help="wsi: BASELINE configs[1] (headline, weak scaling); cohort: configs[2], --slides x --tiles sharded by "
                         "whole slides over the ranks (strong scaling), slide-level thresholding through apply_sharded")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step returned (per-tile mean / std, apply "
                         "results, kept-slide table) as DIR/<name>.npy, to compare two builds output for output")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "native":
        ap.error("--dump-outputs needs --impl native")
    return args


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return {"hbm_gbs": d["hbm_gbs"], "tflops_burst": d["bf16_tflops"],
                "tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]), "source": "measured"}
    return {"hbm_gbs": 6650.0, "tflops_burst": 1590.0, "tflops_sustained": 1400.0, "source": "fallback"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.device = device
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                       "-lms", "200", "-i", str(self.device)], stdout=self.f, stderr=subprocess.DEVNULL)
        except OSError:
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.f.read().splitlines():
            parts = [x.strip() for x in line.split(",")]
            if len(parts) < 9:
                continue
            try:
                sm.append(float(parts[1]))
                mx.append(float(parts[2]))
            except ValueError:
                continue
            for nm, val in zip(names, parts[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        try:
            os.unlink(self.f.name)
        except OSError:
            pass
        busy = [c for c in sm if c > 0]
        return {"sm_mhz": float(np.median(busy)) if busy else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# --------------------------------------------------------------------------------------------------
# CPU arm: the restated reference schedule (oracle) on the host cores
# --------------------------------------------------------------------------------------------------
def cpu_reference_step(oracle, tiles, T, seed):
    """one bounded sample: T FULL forward passes per tile (what Slideflow does), fp32, then mean/std"""
    t0 = time.perf_counter()
    oracle.predict_uq(tiles, T=T, seed=seed, reference_schedule=True)
    return time.perf_counter() - t0


def make_cpu_oracle():
    import torch
    try:                      # torchrun pins OMP_NUM_THREADS=1: the CPU arm uses every core this process may run on
        torch.set_num_threads(max(1, len(os.sched_getaffinity(0))))
    except (AttributeError, RuntimeError):
        pass
    from biscuit_b200.weights import random_init
    from oracle import xception_uq as X          # CPU-baseline leg: the one place bench.py may touch oracle/
    return X.XceptionUQOracle(random_init(seed=1), emulate_bf16=False), torch.get_num_threads()


def cpu_sample_tiles(n, seed=0):
    from oracle import synth
    return synth.tiles_u8(n, seed=seed, n_slides=1)


def run_reference_arm(args, rank, world):
    if rank != 0:
        return None
    oracle, threads = make_cpu_oracle()
    # calibrate: one tile, one pass
    probe = cpu_sample_tiles(1)
    t0 = time.perf_counter()
    oracle.predict_uq(probe, T=1, seed=0, reference_schedule=True)
    per_pass = time.perf_counter() - t0
    budget = 120.0 / max(1, args.steps + args.warmup)            # whole run within a few minutes
    n = int(max(1, min(8, budget / max(per_pass * args.T, 1e-6))))
    tiles = cpu_sample_tiles(n)
    for _ in range(args.warmup):
        cpu_reference_step(oracle, tiles, args.T, 0)
    t = [cpu_reference_step(oracle, tiles, args.T, 1 + i) for i in range(args.steps)]
    total = float(sum(t))
    value = n * args.steps / total
    sample = f"{n} synthetic tiles x T={args.T} full forward passes (fp32, torch CPU ops) per step"
    return {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "tiles/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "fp32", "data": "synthetic",
        "config": {"workload": "configs[1]: one synthetic WSI, 10k tiles, T=30 -- bounded sample of it on the host CPU",
                   "tiles_per_step": n, "T": args.T,
                   "note": "restated TF-CPU path (TensorFlow/Slideflow not installable; parity with TF unpinned)"},
        "cpu_baseline": {"value": value, "unit": "tiles/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "tiles/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }


# --------------------------------------------------------------------------------------------------
# native arm
# --------------------------------------------------------------------------------------------------
DUMP_BYTES = 60_000_000          # array payload of --dump-outputs: under 64 MB with the .npy headers


def dump_outputs(out_dir, rank, world, mean, std, results, s_df):
    """--dump-outputs: the arrays a caller of one step receives, as float32 / float64 .npy files.  Rank 0 writes the
    apply results that are defined (apply returns None, or NaN for an empty confusion cell, where a result has no value:
    on a single slide, for one, there is no slide-level ROC) and the kept-slide table (identical on every rank); each
    rank writes its own per-tile mean / std, suffixed `_rank<r>` when there are several.  Everything stays within
    DUMP_BYTES: past that the tile arrays are a fixed seeded sample of rows, whose indices go to tile_sample_index."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {}
    if rank == 0:
        for k, v in results.items():
            if v is not None and np.isfinite(v):
                arrays[f"apply_{k}"] = np.float64(v)
        if s_df is not None:
            for c in s_df.columns:
                if s_df[c].dtype.kind in "biuf":
                    arrays[f"slide_{c}"] = s_df[c].to_numpy(np.float64)
    budget = (DUMP_BYTES - sum(a.nbytes for a in arrays.values())) // world
    sfx = "" if world == 1 else f"_rank{rank}"
    rows = np.arange(len(mean))
    if mean.nbytes + std.nbytes > budget:
        k = budget // (mean[:1].nbytes + std[:1].nbytes + 8)
        rows = np.sort(np.random.default_rng(0).choice(len(mean), k, replace=False))
        arrays["tile_sample_index" + sfx] = rows.astype(np.float64)
    arrays["tile_mean" + sfx] = mean[rows]
    arrays["tile_std" + sfx] = std[rows]
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def synth_tiles_device(n, device, seed):
    """uint8 NHWC tiles generated on the device: per-tile colour bias + gaussian texture"""
    import torch
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    out = torch.empty((n, TILE_PX, TILE_PX, 3), dtype=torch.uint8, device=device)
    chunk = 500
    for i in range(0, n, chunk):
        m = min(chunk, n - i)
        bias = torch.rand((m, 1, 1, 3), generator=g, device=device) * 110 + 70
        amp = torch.rand((m, 1, 1, 1), generator=g, device=device) * 35 + 10
        x = bias + amp * torch.randn((m, TILE_PX, TILE_PX, 3), generator=g, device=device)
        out[i:i + m] = x.clamp_(0, 255).to(torch.uint8)
    return out


def run_native_arm(args, rank, world, local_rank):
    import pandas as pd
    import torch
    import torch.distributed as dist
    from biscuit_b200 import _ffi, threshold
    from biscuit_b200.uq import UncertaintyInterface
    from biscuit_b200.weights import random_init

    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    ctx = _ffi.default_context(local_rank)
    iface = UncertaintyInterface(random_init(seed=1), max_batch=args.max_batch, ctx=ctx)
    n = args.tiles * args.slides
    tiles_dev = synth_tiles_device(n, device, seed=1000 + rank)
    torch.cuda.synchronize()
    slide_names = np.repeat([f"r{rank:02d}s{j:03d}" for j in range(args.slides)], args.tiles)
    y_true = np.repeat((np.arange(args.slides) + rank) % 2, args.tiles).astype(np.int64)
    mean = np.empty((n, 2), np.float32)
    std = np.empty((n, 2), np.float32)
    thresholds = dict(tile_uq=0.06, slide_uq=0.08, tile_pred=0.5, slide_pred=0.5)
    ext_stream = torch.cuda.ExternalStream(ctx.stream, device=device)

    def one_step(tiles, step):
        iface.predict(tiles, T=args.T, seed=step, tile_index_base=rank * n, out_mean=mean, out_std=std)
        df = pd.DataFrame({"slide": slide_names, "y_true": y_true, "y_pred": mean[:, 1], "uncertainty": std[:, 1]})
        if world > 1:
            return threshold.apply_sharded(df, **thresholds)
        return threshold.apply(df, **thresholds)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        ctx.sync()

    def timed(tiles, steps, first_step):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        w0 = time.perf_counter()
        with torch.cuda.stream(ext_stream):
            e0.record()
        for s in range(steps):
            last = one_step(tiles, first_step + s)
        with torch.cuda.stream(ext_stream):
            e1.record()
        barrier()
        wall = time.perf_counter() - w0
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms, wall * 1e3], dtype=torch.float64, device=device)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms, wall = float(t[0]), float(t[1]) / 1e3
        return ms, wall, last

    # ---- warm-up, then the timed region on HBM-resident tiles
    for s in range(args.warmup):
        res = one_step(tiles_dev, s)
    sampler = ClockSampler(local_rank)
    launches0 = ctx.launches
    if rank == 0:
        sampler.start()
    ms, wall, last = timed(tiles_dev, args.steps, args.warmup)
    clocks = sampler.stop() if rank == 0 else None
    launches = ctx.launches - launches0
    if args.dump_outputs:                                    # before the steps below overwrite mean / std
        dump_outputs(args.dump_outputs, rank, world, mean, std, *last)
    total_tiles = n * args.steps * world
    value = total_tiles / (ms / 1e3)

    # ---- roofline of the dominant kernel family: one more step with an event pair around every launch
    iface.set_profiling(2)
    iface.predict(tiles_dev, T=args.T, seed=99, tile_index_base=rank * n, out_mean=mean, out_std=std)
    prof = iface.kernel_profile()
    iface.set_profiling(0)

    # ---- e2e: HOST (pinned) tiles through the public API, H2D + D2H inside the timed region
    e2e = None
    if not args.no_e2e:
        host = torch.empty((n, TILE_PX, TILE_PX, 3), dtype=torch.uint8, pin_memory=True)
        host.copy_(tiles_dev)
        torch.cuda.synchronize()
        host_np = host.numpy()
        one_step(host_np, 0)
        ems, _, _ = timed(host_np, args.steps, 100)
        h2d = n * TILE_BYTES + n * (4 + 4 + 1 + 4)            # tiles + (y_pred, uncertainty, y_true, codes) table
        d2h = n * 2 * 4 * 2 + n * (8 + 1 + 1) + 64 * args.slides
        e2e = {"value": total_tiles / (ems / 1e3), "unit": "tiles/s", "h2d_bytes_per_step": h2d,
               "d2h_bytes_per_step": d2h, "ms_per_step": ems / args.steps, "host_memory": "pinned"}
        # what a NumPy / DataFrame caller passes is PAGEABLE memory: the same call on a plain ndarray
        pageable = np.array(host_np, copy=True)
        one_step(pageable, 0)
        pms, _, _ = timed(pageable, args.steps, 100)
        e2e["pageable_value"] = n * args.steps * world / (pms / 1e3)
        del host, host_np, pageable

    if rank != 0:
        return None
    peaks = measured_peaks()
    fam = max(prof, key=lambda k: prof[k]["ms"])
    dom = prof[fam]
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    if os.path.exists(tpath):
        with open(tpath) as f:
            traffic = json.load(f).get(fam, {}).get("dram_bytes_per_launch")
    tensor_bound = fam.startswith("gemm") or fam in ("head_gemm", "sepconv_mid")
    if tensor_bound:
        achieved = dom["flops"] / (dom["ms"] * 1e-3) / 1e12
        roof = {"kernel": fam, "bound": "tensor", "achieved": achieved, "peak": peaks["tflops_sustained"],
                "unit": "TFLOP/s", "frac": achieved / peaks["tflops_sustained"], "traffic": traffic,
                "peak_source": peaks["source"] + " (sustained: kernel timed inside a long step)",
                "launches": dom["launches"], "avg_launch_ms": dom["ms"] / max(1, dom["launches"])}
    else:
        achieved = dom["bytes"] / (dom["ms"] * 1e-3) / 1e9
        roof = {"kernel": fam, "bound": "hbm", "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                "frac": achieved / peaks["hbm_gbs"], "traffic": traffic, "peak_source": peaks["source"],
                "launches": dom["launches"], "avg_launch_ms": dom["ms"] / max(1, dom["launches"])}
    flop_per_tile = BACKBONE_GFLOP * 1e9 + (HEAD_ONCE_MFLOP + HEAD_MFLOP_PER_SAMPLE * args.T) * 1e6
    out = {
        "metric": METRIC, "value": value, "unit": "tiles/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": f"configs[1]: {args.slides} synthetic WSI x {args.tiles} tiles per GPU per step, T={args.T}, "
                               "tile mean/std + slide UQ (threshold.apply)",
                   "tiles_per_gpu_per_step": n, "T": args.T, "max_batch": args.max_batch,
                   "cache": f"inputs {n * TILE_BYTES / 1e9:.2f} GB per step >> 126 MB L2", "weights": "random init seed 1"},
        "slides_per_sec": value / args.tiles,
        "wall_ms_per_step": wall * 1e3 / args.steps,
        "model_tflops": value * flop_per_tile / 1e12,
        "model_tensor_frac_of_sustained_peak": value * flop_per_tile / 1e12 / peaks["tflops_sustained"] / world,
        "roofline": roof,
        "kernels": {k: {"ms": round(v["ms"], 3), "launches": v["launches"],
                        "tflops": round(v["flops"] / max(v["ms"], 1e-9) / 1e9, 2),
                        "gbs": round(v["bytes"] / max(v["ms"], 1e-9) / 1e6, 1)} for k, v in prof.items() if v["launches"]},
        "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks,
        "apply_results": {k: (None if v is None or v != v else float(v)) for k, v in res[0].items()},
    }
    return out


def run_cohort_arm(args, rank, world, local_rank):
    """BASELINE configs[2]: a cohort of `--slides` slides x `--tiles` tiles sharded over the ranks by WHOLE slides
    (dist.shard_bounds), MC-dropout inference on each rank's slides, then ONE exchange of per-slide aggregates and the
    replicated slide-level thresholding (threshold.apply_sharded).  Strong scaling: the cohort is fixed, ranks split it.
    Tiles are synthetic and generated on the device: a pool of distinct slides is cycled (2 M real tiles would be 536 GB);
    every slide still draws its own dropout masks (Philox counters carry the global tile index)."""
    import pandas as pd
    import torch
    import torch.distributed as dist
    from biscuit_b200 import _ffi, threshold
    from biscuit_b200 import dist as bdist
    from biscuit_b200.uq import UncertaintyInterface
    from biscuit_b200.weights import random_init

    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    ctx = _ffi.default_context(local_rank)
    iface = UncertaintyInterface(random_init(seed=1), max_batch=args.max_batch, ctx=ctx)
    S, Tn = args.slides, args.tiles
    lo, hi = bdist.shard_bounds([Tn] * S, world)[rank]
    pool_n = min(8, max(1, hi - lo))
    pool = [synth_tiles_device(Tn, device, seed=5000 + j) for j in range(pool_n)]
    torch.cuda.synchronize()
    names = np.array([f"slide{j:05d}" for j in range(S)], dtype=object)
    labels = (np.random.default_rng(7).random(S) < 0.5).astype(np.int64)
    n_local = (hi - lo) * Tn
    mean = np.empty((n_local, 2), np.float32)
    std = np.empty((n_local, 2), np.float32)
    thresholds = dict(tile_uq=0.06, slide_uq=0.055, tile_pred=0.5, slide_pred=0.5)
    ext_stream = torch.cuda.ExternalStream(ctx.stream, device=device)

    def one_step(step):
        for k, sl in enumerate(range(lo, hi)):
            iface.predict(pool[k % pool_n], T=args.T, seed=step, tile_index_base=sl * Tn,
                          out_mean=mean[k * Tn:(k + 1) * Tn], out_std=std[k * Tn:(k + 1) * Tn])
        df = pd.DataFrame({"slide": np.repeat(names[lo:hi], Tn), "y_true": np.repeat(labels[lo:hi], Tn),
                           "y_pred": mean[:, 1], "uncertainty": std[:, 1]})
        if world > 1:
            return threshold.apply_sharded(df, **thresholds), df
        return threshold.apply(df, **thresholds), df

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        ctx.sync()

    for s_ in range(args.warmup):
        one_step(s_)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    launches0 = ctx.launches
    w0 = time.perf_counter()
    with torch.cuda.stream(ext_stream):
        e0.record()
    for s_ in range(args.steps):
        (res, s_df), df_local = one_step(args.warmup + s_)
    with torch.cuda.stream(ext_stream):
        e1.record()
    barrier()
    wall = time.perf_counter() - w0
    ms = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms, wall * 1e3], dtype=torch.float64, device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, wall = float(t[0]), float(t[1]) / 1e3
    clocks = sampler.stop() if rank == 0 else None
    launches = ctx.launches - launches0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, rank, world, mean, std, res, s_df)
    # sharded decisions == single-process apply on the concatenated table (bit for bit), checked on rank 0
    same = None
    if world > 1:
        meta = bdist.all_gather_meta([len(df_local)])
        parts = bdist.all_gather_bytes(bdist.pack_tiles(df_local["y_pred"].to_numpy(), df_local["uncertainty"].to_numpy(),
                                                        df_local["y_true"].to_numpy().astype(np.uint8)),
                                       [int(m[0]) * 9 for m in meta], device=f"cuda:{local_rank}")
        if rank == 0:
            cols = [bdist.unpack_tiles(p_, int(m[0]), np.float32) for m, p_ in zip(meta, parts)]
            full = pd.DataFrame({"slide": np.repeat(names, Tn), "y_true": np.concatenate([c[2] for c in cols]).astype(np.int64),
                                 "y_pred": np.concatenate([c[0] for c in cols]), "uncertainty": np.concatenate([c[1] for c in cols])})
            r1, s1 = threshold.apply(full, **thresholds)
            same = bool(all((r1[k] == res[k]) or (r1[k] != r1[k] and res[k] != res[k]) for k in r1) and
                        ((s1 is None and s_df is None) or (s1 is not None and s_df is not None and s1.equals(s_df))))
    if rank != 0:
        return None
    total_tiles = S * Tn * args.steps
    value = total_tiles / (ms / 1e3)
    return {
        "metric": METRIC, "value": value, "unit": "tiles/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "bf16",
        "data": "synthetic",
        "config": {"workload": f"configs[2]: cohort of {S} synthetic slides x {Tn} tiles, T={args.T}, tiles sharded by whole slides "
                               f"over {world} GPU(s), per-slide aggregates all-gathered, threshold.apply_sharded",
                   "slides": S, "tiles_per_slide": Tn, "T": args.T, "max_batch": args.max_batch,
                   "cache": f"a pool of {pool_n} distinct slides ({pool_n * Tn * TILE_BYTES / 1e9:.2f} GB) cycled per rank >> 126 MB L2"},
        "slides_per_sec": value / Tn, "wall_ms_per_step": wall * 1e3 / args.steps,
        "sharded_equals_single_process_apply": same, "slides_included": None if s_df is None else int(len(s_df)),
        "apply_results": {k: (None if v is None or v != v else float(v)) for k, v in res.items()},
        "gpu_launches": int(launches), "clocks": clocks,
        "e2e": None, "roofline": None,
        "cpu_baseline": {"value": None, "unit": "tiles/s", "cores": 0, "kind": "port",
                         "sample": "not measured in the cohort workload (see the headline wsi line)"},
    }


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        out = run_reference_arm(args, rank, world)
        if out is not None:
            print(json.dumps(out))
        return
    import torch
    import torch.distributed as dist
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", local_rank))
    if args.workload == "cohort":
        out = run_cohort_arm(args, rank, world, local_rank)
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        if rank == 0:
            print(json.dumps(out))
        return
    out = run_native_arm(args, rank, world, local_rank)
    if rank == 0 and world > 1:
        # the CPU baseline is a rank-0, N = 1 measurement (torchrun pins OMP_NUM_THREADS=1 and the other ranks would
        # spin in a barrier for its duration): not repeated on the multi-GPU lines
        out["cpu_baseline"] = {"value": None, "unit": "tiles/s", "cores": 0, "kind": "port",
                               "sample": "not measured at N > 1 (rank-0, N = 1 measurement: see the N = 1 line)"}
    elif rank == 0 and not args.no_cpu_baseline:
        oracle, threads = make_cpu_oracle()
        probe = cpu_sample_tiles(1)
        t0 = time.perf_counter()
        oracle.predict_uq(probe, T=1, seed=0, reference_schedule=True)
        per_pass = time.perf_counter() - t0
        ns = int(max(1, min(8, args.cpu_seconds / max(per_pass * args.T, 1e-6))))
        dt = cpu_reference_step(oracle, cpu_sample_tiles(ns), args.T, 1)
        out["cpu_baseline"] = {"value": ns / dt, "unit": "tiles/s", "cores": threads, "kind": "port",
                               "sample": f"{ns} synthetic tiles x T={args.T} FULL forward passes, fp32 torch CPU ops "
                                         f"(restated Slideflow schedule; TF not installable), {dt:.1f} s"}
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank == 0:
        print(json.dumps(out))


if __name__ == "__main__":
    main()
