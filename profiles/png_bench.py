"""Compressed-tile input on one GPU, PNG: decode kernel times and end-to-end MC-dropout throughput of
`predict(PngBatch)` against `predict(uint8)`, plus the host's own Pillow decode rate over all its cores.

    python profiles/png_bench.py [--tiles 10000] [--big-tiles 100000] [--T 30] [--reps 3] [--out results.json]

Two encodings: Pillow `compress_level` 1 and 6 (Pillow's default).  The inputs cycle 503 distinct `synth.tiles_u8`
tiles (about 200 KB of PNG each), so the 10 k-tile pass already reads about 2 GB, far more than the 126 MB L2.  The
uint8 and PNG inputs alternate within one run, pinned and pageable, and their outputs must be equal.  One extra run at
--big-tiles tiles reads both inputs from device memory, to show the rate holds over a long stream.
"""
from __future__ import annotations

import argparse
import json
import multiprocessing as mp
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

LEVELS = (1, 6)


def _pil_worker(files):
    from oracle import png_synth
    t = time.perf_counter()
    for b in files:
        png_synth.pil_decode(b)
    return len(files), time.perf_counter() - t


def host_pil_rate(files, procs):
    chunks = [files[i::procs] for i in range(procs)]
    with mp.get_context("spawn").Pool(procs) as pool:
        pool.map(_pil_worker, [c[:4] for c in chunks])          # warm the workers
        t = time.perf_counter()
        pool.map(_pil_worker, chunks)
        return len(files) / (time.perf_counter() - t)


def kernel_split(batch, ctx, reps=5):
    """per-kernel device time of one decode of `batch` (device bytes, device output), from torch.profiler, and the
    call's time from CUDA events in a separate loop"""
    import torch
    from torch.profiler import ProfilerActivity, profile

    from biscuit_b200 import png
    out = torch.empty((len(batch), 299, 299, 3), dtype=torch.uint8, device="cuda")
    for _ in range(2):
        png.decode(batch, ctx=ctx, out=out)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            png.decode(batch, ctx=ctx, out=out)
    names = {"dechunk": "png_dechunk_kernel", "inflate": "png_inflate_kernel", "unfilter": "png_unfilter_kernel"}
    ms = {k: 0.0 for k in names}
    for ev in prof.key_averages():
        for k, n in names.items():
            if n in ev.key:
                ms[k] += ev.device_time_total / 1e3 / reps
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    s.record()
    for _ in range(reps):
        png.decode(batch, ctx=ctx, out=out)
    e.record()
    torch.cuda.synchronize()
    ms["call"] = s.elapsed_time(e) / reps
    return ms


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--tiles", type=int, default=10000)
    ap.add_argument("--big-tiles", type=int, default=100000)
    ap.add_argument("--T", type=int, default=30)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--pil-tiles", type=int, default=4000)
    ap.add_argument("--out", default=None, help="also write the result JSON to this file")
    a = ap.parse_args()

    import torch

    from biscuit_b200 import _ffi, uq
    from biscuit_b200.png import PngBatch
    from biscuit_b200.weights import random_init
    from oracle import png_synth, synth

    if not torch.cuda.is_available():
        raise SystemExit("png_bench needs a GPU")
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True).stdout.strip()
    res = dict(gpu=q or torch.cuda.get_device_name(0), tiles=a.tiles, T=a.T, micro_batch=uq.BENCH_MICRO_BATCH,
               host_cpus=os.cpu_count(), configs={})
    ctx = _ffi.default_context(0)
    base = synth.tiles_u8(uq.BENCH_MICRO_BATCH, seed=7, n_slides=8)
    iface = uq.UncertaintyInterface(random_init(seed=1), max_batch=uq.BENCH_MICRO_BATCH, ctx=ctx)
    for level in LEVELS:
        name = f"pil_level{level}"
        files = [png_synth.pil_encode(t, level) for t in base]
        mb = PngBatch.from_bytes(files)
        r = dict(bytes_per_tile=mb.nbytes / len(mb))
        split = kernel_split(mb.cuda(), ctx)
        r["decode_ms_per_503"] = split
        r["decode_tiles_per_s"] = len(mb) / (split["call"] / 1e3)
        r["decode_compressed_GBps"] = mb.nbytes / (split["call"] / 1e3) / 1e9

        idx = np.arange(a.tiles) % len(files)
        big = PngBatch.from_bytes([files[i] for i in idx])
        pixels = base[idx]
        pin_px = torch.empty(pixels.shape, dtype=torch.uint8).pin_memory().numpy()
        pin_px[...] = pixels
        pin_data = torch.empty(big.data.shape, dtype=torch.uint8).pin_memory().numpy()
        pin_data[...] = big.data
        inputs = {"uint8_pinned": pin_px, "png_pinned": PngBatch(pin_data, big.offsets),
                  "uint8_pageable": pixels, "png_pageable": big}
        for k, x in inputs.items():                     # warm-up: every shape / route once
            iface.predict(x[:uq.BENCH_MICRO_BATCH] if k.startswith("uint8") else
                          PngBatch(x.data, x.offsets[:uq.BENCH_MICRO_BATCH + 1]), T=a.T, seed=0)
        times = {k: [] for k in inputs}
        outs = {}
        for _ in range(a.reps):
            for k, x in inputs.items():
                torch.cuda.synchronize()
                t = time.perf_counter()
                outs[k] = iface.predict(x, T=a.T, seed=3)
                times[k].append(time.perf_counter() - t)
        r["e2e_tiles_per_s"] = {k: a.tiles / float(np.median(v)) for k, v in times.items()}
        r["e2e_spread"] = {k: [round(a.tiles / t) for t in v] for k, v in times.items()}
        for kind in ("pinned", "pageable"):
            r[f"png_over_uint8_{kind}"] = r["e2e_tiles_per_s"][f"png_{kind}"] / r["e2e_tiles_per_s"][f"uint8_{kind}"]
            assert np.array_equal(outs[f"png_{kind}"][0], outs[f"uint8_{kind}"][0])
            assert np.array_equal(outs[f"png_{kind}"][1], outs[f"uint8_{kind}"][1])
        del pin_px, pin_data, inputs, outs

        if a.big_tiles and level == 6:
            reps = -(-a.big_tiles // len(files))
            dev = mb.cuda().data.repeat(reps)
            lens = np.tile(np.diff(mb.offsets), reps)[:a.big_tiles]
            big_dev = PngBatch(dev, np.concatenate([[0], np.cumsum(lens)]))
            px_dev = torch.from_numpy(base).cuda().repeat(reps, 1, 1, 1)[:a.big_tiles].contiguous()
            bt, ref_big = {}, None
            for k, x in (("uint8_device", px_dev), ("png_device", big_dev)) * 2:
                torch.cuda.synchronize()
                t = time.perf_counter()
                o = iface.predict(x, T=a.T, seed=3)
                bt.setdefault(k, []).append(time.perf_counter() - t)
                if k == "uint8_device":
                    ref_big = o
                else:
                    assert np.array_equal(o[0], ref_big[0]) and np.array_equal(o[1], ref_big[1])
            r["big_run"] = dict(tiles=a.big_tiles, compressed_GB=float(big_dev.nbytes) / 1e9,
                                e2e_tiles_per_s={k: a.big_tiles / min(v) for k, v in bt.items()})
            del dev, big_dev, px_dev
            torch.cuda.empty_cache()

        pil_files = [files[i % len(files)] for i in range(a.pil_tiles)]
        r["host_pil_tiles_per_s"] = host_pil_rate(pil_files, os.cpu_count() or 1)
        r["decode_over_host_pil"] = r["decode_tiles_per_s"] / r["host_pil_tiles_per_s"]
        res["configs"][name] = r
        print(name, json.dumps(r, indent=1), flush=True)
    if a.out:
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
