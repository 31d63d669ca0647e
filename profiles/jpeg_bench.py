"""Compressed-tile input on one GPU: decode kernel times, subsequence statistics and end-to-end MC-dropout throughput of
`predict(JpegBatch)` against `predict(uint8)`, plus the host's own Pillow decode rate.

    python profiles/jpeg_bench.py [--tiles 10000] [--T 30] [--reps 3] [--out results.json]

Two encodings: quality 90 4:2:0 (Pillow's default sampling) and quality 100 4:4:4 (the synthetic worst case).  The
10 k-tile inputs cycle 503 distinct `synth.tiles_u8` tiles, so one pass reads more bytes than the 126 MB L2 holds at
quality 100 (and 0.34 GB at quality 90).  The two inputs kinds alternate within one run, pinned and pageable.
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

CONFIGS = [("q90_420", 90, "4:2:0"), ("q100_444", 100, "4:4:4")]


def _pil_worker(files):
    from oracle import jpeg_synth
    t = time.perf_counter()
    for b in files:
        jpeg_synth.pil_decode(b)
    return len(files), time.perf_counter() - t


def host_pil_rate(files, procs):
    chunks = [files[i::procs] for i in range(procs)]
    with mp.get_context("spawn").Pool(procs) as pool:
        pool.map(_pil_worker, [c[:4] for c in chunks])          # warm the workers
        t = time.perf_counter()
        pool.map(_pil_worker, chunks)
        return len(files) / (time.perf_counter() - t)


def kernel_split(batch, ctx, reps=5):
    """per-kernel device time of one decode of `batch` (device bytes, device output), from torch.profiler"""
    import torch
    from torch.profiler import ProfilerActivity, profile

    from biscuit_b200 import jpeg
    out = torch.empty((len(batch), 299, 299, 3), dtype=torch.uint8, device="cuda")
    for _ in range(2):
        jpeg.decode(batch, ctx=ctx, out=out)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            jpeg.decode(batch, ctx=ctx, out=out)
    names = {"unstuff": "jpeg_unstuff_kernel", "huffman": "jpeg_huffman_kernel", "idct": "jpeg_idct_kernel",
             "color": "jpeg_color_kernel"}
    ms = {k: 0.0 for k in names}
    for ev in prof.key_averages():
        for k, n in names.items():
            if n in ev.key:
                ms[k] += ev.device_time_total / 1e3 / reps
    # wall time of the decode call on device-resident input, CUDA events around it
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    s.record()
    for _ in range(reps):
        jpeg.decode(batch, ctx=ctx, out=out)
    e.record()
    torch.cuda.synchronize()
    ms["call"] = s.elapsed_time(e) / reps
    return ms


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--tiles", type=int, default=10000)
    ap.add_argument("--T", type=int, default=30)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--pil-tiles", type=int, default=4000)
    ap.add_argument("--out", default=None, help="also write the result JSON to this file")
    a = ap.parse_args()

    import torch

    from biscuit_b200 import _ffi, jpeg, uq
    from biscuit_b200.jpeg import JpegBatch
    from biscuit_b200.weights import random_init
    from oracle import jpeg_synth, synth

    if not torch.cuda.is_available():
        raise SystemExit("jpeg_bench needs a GPU")
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True).stdout.strip()
    res = dict(gpu=q or torch.cuda.get_device_name(0), tiles=a.tiles, T=a.T, micro_batch=uq.BENCH_MICRO_BATCH,
               host_cpus=os.cpu_count(), configs={})
    ctx = _ffi.default_context(0)
    base = synth.tiles_u8(uq.BENCH_MICRO_BATCH, seed=7, n_slides=8)
    iface = uq.UncertaintyInterface(random_init(seed=1), max_batch=uq.BENCH_MICRO_BATCH, ctx=ctx)
    for name, quality, ss in CONFIGS:
        files = [jpeg_synth.jpeg_encode(t, quality, ss) for t in base]
        mb = JpegBatch.from_bytes(files)
        r = dict(bytes_per_tile=mb.nbytes / len(mb))
        split = kernel_split(mb.cuda(), ctx)
        st = jpeg.last_stats(ctx)
        r["decode_ms_per_503"] = split
        r["huffman_ms"] = split["unstuff"] + split["huffman"]
        r["idct_color_ms"] = split["idct"] + split["color"]
        r["decode_tiles_per_s"] = len(mb) / (split["call"] / 1e3)
        r["decode_compressed_GBps"] = mb.nbytes / (split["call"] / 1e3) / 1e9
        r["sync"] = dict(st, subsequences_per_tile=st["subsequences"] / max(1, st["tiles"]),
                         redecoded_share=st["redecoded"] / max(1, st["subsequences"]))

        idx = np.arange(a.tiles) % len(files)
        big = JpegBatch.from_bytes([files[i] for i in idx])
        pixels = np.stack([jpeg_synth.pil_decode(b) for b in files])[idx]
        pin_px = torch.empty(pixels.shape, dtype=torch.uint8).pin_memory().numpy()
        pin_px[...] = pixels
        pin_data = torch.empty(big.data.shape, dtype=torch.uint8).pin_memory().numpy()
        pin_data[...] = big.data
        inputs = {"uint8_pinned": pin_px, "jpeg_pinned": JpegBatch(pin_data, big.offsets),
                  "uint8_pageable": pixels, "jpeg_pageable": big}
        for k, x in inputs.items():                     # warm-up: every shape / route once
            iface.predict(x[:uq.BENCH_MICRO_BATCH] if k.startswith("uint8") else
                          JpegBatch(x.data, x.offsets[:uq.BENCH_MICRO_BATCH + 1]), T=a.T, seed=0)
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
            r[f"jpeg_over_uint8_{kind}"] = r["e2e_tiles_per_s"][f"jpeg_{kind}"] / r["e2e_tiles_per_s"][f"uint8_{kind}"]
            assert np.array_equal(outs[f"jpeg_{kind}"][0], outs[f"uint8_{kind}"][0])
            assert np.array_equal(outs[f"jpeg_{kind}"][1], outs[f"uint8_{kind}"][1])
        pil_files = [files[i % len(files)] for i in range(a.pil_tiles)]
        r["host_pil_tiles_per_s"] = host_pil_rate(pil_files, os.cpu_count() or 1)
        res["configs"][name] = r
        print(name, json.dumps(r, indent=1), flush=True)
    if a.out:
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
