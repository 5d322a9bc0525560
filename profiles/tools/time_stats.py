"""Timings of the per-cell time statistics (dcdf_superchunk_time_stats) on the GPU; prints JSON lines and, when OUT is
given, writes them there as well.  The first line names the GPU and its power limit, read in the same run.

(1) C2-shaped synthetic raster (synth.raster 721x1440 f32, k2_levels [5, 6], chunk_size 64, 512 instants), one
    full-extent window: Superchunk.time_stats_batch.  Kernel ms (dcdf_ctx_last_kernel_ms(ctx, 7)), cell-instants per
    second over that time, slice groups and scratch bytes of partials.
(2) The route it replaces: the same window decoded by Superchunk.window_batch into a CUDA tensor, then torch
    reductions over time (isnan count, nansum, masked min / max, sum of squares).  Timed with CUDA events around decode
    plus reductions; the decode kernel alone is dcdf_ctx_last_kernel_ms(ctx, 3).  Counts, min and max must agree
    exactly; the sums are summed in another order, so their largest relative difference is reported.
(3) 10^4 windows of 16x16 cells over all 512 instants in one batch, both routes as in (1) and (2).
Warm-up first, then three rounds in which the two routes alternate.

    python profiles/tools/time_stats.py [OUT]
"""
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import numpy as np
import torch

from dcdf_b200 import Context, Superchunk, _ffi, synth

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


def torch_stats(w):
    """The dense route: per-cell statistics over dim 1 of a decoded [n, T, cells] CUDA tensor."""
    ok = ~torch.isnan(w)
    z = torch.where(ok, w, torch.zeros((), dtype=w.dtype, device=w.device)).double()
    mn = torch.where(ok, w, torch.full((), float("inf"), dtype=w.dtype, device=w.device)).amin(dim=1)
    mx = torch.where(ok, w, torch.full((), float("-inf"), dtype=w.dtype, device=w.device)).amax(dim=1)
    return ok.sum(dim=1), mn, mx, z.sum(dim=1), (z * z).sum(dim=1)


def compare(rec, dense):
    cnt, mn, mx, s, q = [x.cpu().numpy().ravel() for x in dense]
    empty = cnt == 0
    mn, mx = np.where(empty, np.nan, mn), np.where(empty, np.nan, mx)
    same = (np.array_equal(rec["count"].astype(np.int64), cnt) and np.array_equal(rec["min"], mn.astype(np.float32), equal_nan=True)
            and np.array_equal(rec["max"], mx.astype(np.float32), equal_nan=True))
    rel = lambda a, b: float(np.max(np.abs(a - b) / np.maximum(np.abs(b), 1e-300), initial=0.0))
    return bool(same), rel(rec["sum"], s), rel(rec["sum_sq"], q)


def leg(ctx, sc, name, cubes, T, cells):
    n = len(cubes)
    dense = torch.empty(n * T * cells, dtype=torch.float32, device="cuda:0")
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def fused():
        return sc.time_stats_batch(cubes)

    def unfused():
        ev0.record()
        sc.window_batch(cubes, out=dense)
        res = torch_stats(dense.view(n, T, cells))
        ev1.record()
        torch.cuda.synchronize()
        return res

    fused(); unfused()                       # warm-up
    res = {"fused_kernel_ms": [], "fused_call_ms": [], "dense_decode_kernel_ms": [], "dense_decode_plus_torch_ms": []}
    agree, d_sum, d_sq = True, 0.0, 0.0
    for _ in range(3):
        t = time.perf_counter()
        rec, _ = fused()
        res["fused_call_ms"].append((time.perf_counter() - t) * 1e3)
        res["fused_kernel_ms"].append(ctx.last_kernel_ms(_ffi.KT_TIME_STATS))
        groups, scratch = ctx.get_stat("time_stats_groups"), ctx.get_stat("time_stats_scratch_bytes")
        d = unfused()
        res["dense_decode_kernel_ms"].append(ctx.last_kernel_ms(_ffi.KT_WINDOW))
        res["dense_decode_plus_torch_ms"].append(ev0.elapsed_time(ev1))
        a, s, q = compare(rec, d)
        agree, d_sum, d_sq = agree and a, max(d_sum, s), max(d_sq, q)
    best = min(res["fused_kernel_ms"])
    emit({"leg": name, "windows": n, "cell_instants": n * T * cells, "groups": groups, "scratch_bytes": scratch,
          "dense_window_bytes": n * T * cells * 4, "fused_cell_instants_per_s": n * T * cells / (best * 1e-3),
          "count_min_max_agree": agree, "max_rel_diff_sum": d_sum, "max_rel_diff_sum_sq": d_sq, **res})
    del dense
    torch.cuda.empty_cache()


def main():
    emit(gpu())
    ctx = Context(0)
    T, R, Cc = 512, 721, 1440
    data = synth.raster(T, R, Cc, device="cuda:0")
    sc = Superchunk.build(ctx, data, [5, 6], compute_bits=True, chunk_size=64)
    del data
    torch.cuda.empty_cache()
    leg(ctx, sc, f"(1)+(2) C2-shaped synth {T}x{R}x{Cc} f32, k2_levels [5, 6], chunk_size 64; one full-extent window",
        np.array([[0, T, 0, R, 0, Cc]], np.int64), T, R * Cc)
    rng = np.random.default_rng(51)
    n = 10000
    top, left = rng.integers(0, R - 16, n), rng.integers(0, Cc - 16, n)
    cubes = np.stack([np.zeros(n, np.int64), np.full(n, T), top, top + 16, left, left + 16], axis=1)
    leg(ctx, sc, f"(3) {n} windows of 16x16 cells, all {T} instants, one batch", cubes, T, 256)
    sc.close()
    ctx.close()
    if OUT is None:
        return
    os.makedirs(os.path.dirname(os.path.abspath(OUT)), exist_ok=True)
    with open(OUT, "w") as f:
        for d in lines:
            f.write(json.dumps(d) + "\n")


if __name__ == "__main__":
    main()
