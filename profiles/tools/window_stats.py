"""Timings of the per-instant window statistics (dcdf_superchunk_window_stats) on the GPU; prints JSON lines and, when OUT
is given, writes them there as well.

(a) C2-shaped raster: Superchunk.window_stats_batch against window_batch on the same 1024 windows (side uniform in
    [8, 256], 64 instants).  Kernels: dcdf_ctx_last_kernel_ms(ctx, 6) against (ctx, 3) with the window written into a CUDA
    tensor.  End to end: window_stats_batch against window_batch to host memory followed by numpy nan-reductions.
(b) Variable.window_stats against Variable.window + numpy on a CPC-sized un-rounded variable with a NaN ocean, for the
    full grid and a sub-region; (c) the same on the nested [2, 4, 6] C5 grid.
Every leg reports whether the outputs agreed (count, min, max equal; sums within 1e-11 of sum |v| / v^2).  Warm-up
first, then three rounds in which the two routes alternate.

    python profiles/tools/window_stats.py [OUT]
"""
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import numpy as np

from dcdf_b200 import Context, Superchunk, Variable, _ffi, synth

OUT = sys.argv[1] if len(sys.argv) > 1 else None
lines = []


def emit(d):
    print(json.dumps(d), flush=True)
    lines.append(d)


def gpu():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, power, clock = [x.strip() for x in q.split(",")]
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def numpy_stats(w):
    """The host route: per-instant count / nanmin / nanmax / sums of a decoded [T, R, C] window."""
    x = w.reshape(w.shape[0], -1).astype(np.float64)
    ok = ~np.isnan(x)
    cnt = ok.sum(axis=1)
    z = np.where(ok, x, 0.0)
    with np.errstate(all="ignore"):
        mn = np.where(cnt > 0, np.nanmin(np.where(ok, x, np.inf), axis=1), np.nan)
        mx = np.where(cnt > 0, np.nanmax(np.where(ok, x, -np.inf), axis=1), np.nan)
    return cnt, mn, mx, z.sum(axis=1), (z * z).sum(axis=1), np.abs(z).sum(axis=1)


def agree(rec, host):
    cnt, mn, mx, s, q, a = host
    same_nan = lambda u, v: np.array_equal(np.asarray(u, np.float64), v, equal_nan=True)
    return bool(np.array_equal(rec["count"].astype(np.int64), cnt) and same_nan(rec["min"], mn) and same_nan(rec["max"], mx)
                and (np.abs(rec["sum"] - s) <= 1e-11 * a).all() and (np.abs(rec["sum_sq"] - q) <= 1e-11 * q).all())


def leg_a(ctx):
    import torch
    T, R, C, cs = 256, 1024, 1024, 64
    data = synth.raster_slice(0, T, R, C, noise_every=1).numpy()
    sc = Superchunk.build(ctx, data, [4, 6], compute_bits=True, chunk_size=cs)
    del data
    rng = np.random.default_rng(21)
    n = 1024
    side = rng.integers(8, 257, n)
    top, left = rng.integers(0, R - 8, n), rng.integers(0, C - 8, n)
    t0s = rng.integers(0, T - cs + 1, n)
    cubes = np.stack([t0s, t0s + cs, top, np.minimum(top + side, R), left, np.minimum(left + side, C)], axis=1)
    sizes = (cubes[:, 1] - cubes[:, 0]) * (cubes[:, 3] - cubes[:, 2]) * (cubes[:, 5] - cubes[:, 4])
    dev = torch.empty(int(sizes.sum()), dtype=torch.float32, device="cuda:0")

    def stats():
        return sc.window_stats_batch(cubes)

    def window_dev():
        sc.window_batch(cubes, out=dev)

    def window_host():
        w, off = sc.window_batch(cubes)
        return [numpy_stats(w[int(off[i]):int(off[i + 1])].reshape(c[1] - c[0], c[3] - c[2], c[5] - c[4])) for i, c in enumerate(cubes)]

    stats(); window_dev(); window_host()     # warm-up
    res = {"stats_kernel_ms": [], "window_kernel_ms": [], "stats_e2e_ms": [], "window_host_numpy_e2e_ms": []}
    same = True
    for _ in range(3):
        t = time.perf_counter(); rec, off = stats(); res["stats_e2e_ms"].append((time.perf_counter() - t) * 1e3)
        res["stats_kernel_ms"].append(ctx.last_kernel_ms(_ffi.KT_REDUCE))
        window_dev(); res["window_kernel_ms"].append(ctx.last_kernel_ms(_ffi.KT_WINDOW))
        t = time.perf_counter(); host = window_host(); res["window_host_numpy_e2e_ms"].append((time.perf_counter() - t) * 1e3)
        same = same and all(agree(rec[int(off[i]):int(off[i + 1])], h) for i, h in enumerate(host))
    emit({"leg": "a", "workload": f"C2-shaped synth {T}x{R}x{C} f32 (noise_every=1), k2_levels [4, 6], chunk_size {cs}; {n} windows, "
                                 f"side 8..256, {cs} instants", "cells": int(sizes.sum()), "outputs_agree": same, **res})
    sc.close()


def leg_v(ctx, name, data, levels, chunk_size, span_size, queries):
    v = Variable(ctx, {}, levels, chunk_size=chunk_size, span_size=span_size)
    v.append(data)
    for q in queries:                      # warm-up (cache loads, buffers)
        v.window_stats(*q); numpy_stats(v.window(*q))
    res = {"window_numpy_ms": [], "window_stats_ms": []}
    same = True
    for _ in range(3):
        t = time.perf_counter()
        a = [numpy_stats(v.window(*q)) for q in queries]
        res["window_numpy_ms"].append((time.perf_counter() - t) * 1e3)
        t = time.perf_counter()
        b = [v.window_stats(*q) for q in queries]
        res["window_stats_ms"].append((time.perf_counter() - t) * 1e3)
        same = same and all(agree(y, x) for x, y in zip(a, b))
    emit({"workload": name, "queries": [list(q) for q in queries], "outputs_agree": bool(same), **res})
    v.close()


def main():
    ctx = Context(0)
    emit(gpu())
    leg_a(ctx)
    T, R, C = 128, 360, 720
    d3 = synth.raster_slice(0, T, R, C, nan_ocean=True, scale=1.37).numpy()
    leg_v(ctx, f"(b) CPC-sized {T}x{R}x{C} f32 un-rounded (x1.37), NaN ocean, k2_levels [4, 6], chunk_size 32, span 2", d3, [4, 6], 32, 2,
          [(0, T, 0, R, 0, C), (5, 120, 50, 300, 100, 600)])
    T, R, C = 16, 1801, 3600
    d5 = synth.raster_slice(0, T, R, C, nan_ocean=True, scale=1.37).numpy()
    leg_v(ctx, f"(c) nested {T}x{R}x{C} f32 un-rounded (x1.37), NaN ocean, k2_levels [2, 4, 6], chunk_size 16, span 2", d5, [2, 4, 6], 16, 2,
          [(0, T, 0, R, 0, C), (3, 13, 500, 1600, 200, 3100)])
    ctx.close()
    if OUT is None:
        return
    os.makedirs(os.path.dirname(os.path.abspath(OUT)), exist_ok=True)
    with open(OUT, "w") as f:
        for d in lines:
            f.write(json.dumps(d) + "\n")


if __name__ == "__main__":
    main()
