"""Timings of the value-bound search (dcdf_superchunk_search_values) on the GPU; prints JSON lines and, when OUT is
given, writes them there as well.

(a) Superchunk.search_values_batch against search_batch with the same bounds converted to fixed point on the host, C4-style
    batches (2048 windows with cells, 10^5 windows count-only) over a uniform-bit C2-shaped raster.  Kernel time from
    dcdf_ctx_last_kernel_ms(ctx, 5) and the call end to end; the two routes alternate, three rounds each.
(b) Variable.search (one device search per span group) against the route it replaced, written out here:
    Superchunk.window of the slice range followed by np.argwhere on the host.  On a C3-shaped un-rounded variable with
    mixed bits and a NaN ocean, and on a nested [2, 4, 6] one.

    python profiles/tools/search_values.py [OUT]
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


def timed(ctx, fn):
    t0 = time.perf_counter()
    r = fn()
    return r, (time.perf_counter() - t0) * 1e3, ctx.last_kernel_ms(_ffi.KT_SEARCH)


def leg_a(ctx):
    T, R, C, cs = 256, 1024, 1024, 64
    data = synth.raster_slice(0, T, R, C, noise_every=1).numpy()   # q * 2^-4 with per-cell noise
    sc = Superchunk.build(ctx, data, [4, 6], compute_bits=True, chunk_size=cs)
    bits = set()
    for s in range(sc.n_slices):
        kinds, _, _, cbits = sc.refs(s)
        bits |= {int(b) for k, b in zip(kinds, cbits) if k == _ffi.REF_EXTERNAL}
    rng = np.random.default_rng(9)
    n = 100000
    side = rng.integers(8, 257, n)
    top, left = rng.integers(0, R - 8, n), rng.integers(0, C - 8, n)
    t0s = rng.integers(0, T - cs, n)
    cubes = np.stack([t0s, t0s + cs, top, np.minimum(top + side, R), left, np.minimum(left + side, C)], axis=1)
    vals = data[np.isfinite(data)]
    lo = rng.uniform(float(vals.min()), float(vals.max()), n)
    hi = lo + 0.05 * float(vals.max() - vals.min())
    fb = 4
    flo = 2 * np.ceil(lo * 2 ** fb).astype(np.int64) + 1
    fhi = 2 * np.floor(hi * 2 ** fb).astype(np.int64) + 1
    ns = 2048
    routes = {"search_values_batch": lambda m, cells: sc.search_values_batch(cubes[:m], lo[:m], hi[:m], want_cells=cells),
              "search_batch": lambda m, cells: sc.search_batch(cubes[:m], flo[:m], fhi[:m], want_cells=cells)}
    for f in routes.values():   # warm-up at full size
        f(n, False)
        f(ns, True)
    res = {k: {"count_kernel_ms": [], "count_e2e_ms": [], "cells_kernel_ms": [], "cells_e2e_ms": []} for k in routes}
    same = True
    for _ in range(3):
        outs = {}
        for k, f in routes.items():
            (c1, _), e1, k1 = timed(ctx, lambda: f(n, False))
            (c2, x2), e2, k2 = timed(ctx, lambda: f(ns, True))
            outs[k] = (c1, c2, x2)
            res[k]["count_kernel_ms"].append(k1); res[k]["count_e2e_ms"].append(e1)
            res[k]["cells_kernel_ms"].append(k2); res[k]["cells_e2e_ms"].append(e2)
        a, b = outs.values()
        same = same and np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]) and np.array_equal(a[2], b[2])
    emit({"leg": "a", "workload": f"C2-shaped synth {T}x{R}x{C} f32, k2_levels [4, 6], chunk_size {cs}; {n} windows count-only, "
                                 f"{ns} with cells; 5% bands", "subchunk_bits": sorted(bits), "matches": int(outs["search_batch"][0].sum()),
          "identical_results": bool(same), **res})
    sc.close()


def old_search(v, start, stop, top, bottom, left, right, lower, upper):
    """The route Variable.search took for slices with mixed bits or nested superchunks: decode, copy out, filter."""
    hits = []
    for sc, t0, a, b in v._groups(start, stop):
        w = sc.window(a, b, top, bottom, left, right)
        idx = np.argwhere((w >= lower) & (w <= upper))
        idx[:, 0] += t0 + a
        idx[:, 1] += top
        idx[:, 2] += left
        hits.append(idx.astype(np.int64))
    return np.concatenate(hits) if hits else np.zeros((0, 3), np.int64)


def leg_b(ctx, name, data, levels, chunk_size, span_size, queries):
    v = Variable(ctx, {}, levels, chunk_size=chunk_size, span_size=span_size)
    v.append(data)
    for q in queries:                      # warm-up (cache loads, buffers)
        old_search(v, *q); v.search(*q)
    res = {"old_ms": [], "new_ms": []}
    same = True
    for _ in range(3):
        t0 = time.perf_counter()
        a = [old_search(v, *q) for q in queries]
        res["old_ms"].append((time.perf_counter() - t0) * 1e3)
        t0 = time.perf_counter()
        b = [v.search(*q) for q in queries]
        res["new_ms"].append((time.perf_counter() - t0) * 1e3)
        for x, y in zip(a, b):
            same = same and len(x) == len(y) and np.array_equal(x[np.lexsort(x.T[::-1])], y[np.lexsort(y.T[::-1])])
    emit({"leg": "b", "workload": name, "queries": len(queries), "matches": int(sum(len(x) for x in b)), "identical_sets": bool(same), **res})
    v.close()


def main():
    ctx = Context(0)
    emit(gpu())
    leg_a(ctx)
    # C3-shaped: a CPC-sized daily grid, un-rounded (scaled by a non-power-of-two), NaN ocean, 128 instants
    T, R, C = 128, 360, 720
    d3 = synth.raster_slice(0, T, R, C, nan_ocean=True, scale=1.37).numpy()
    q3 = [(5, 120, 0, R, 0, C, 280.0, 290.0), (0, 128, 50, 300, 100, 600, 250.0, 400.0), (10, 40, 0, 180, 0, 360, -1e9, 1e9)]
    leg_b(ctx, f"C3-shaped {T}x{R}x{C} f32 un-rounded (x1.37), NaN ocean, k2_levels [4, 6], chunk_size 32, span 2", d3, [4, 6], 32, 2, q3)
    # nested [2, 4, 6]: the C5 (ERA5-Land) grid 1801x3600, 16 instants
    T, R, C = 16, 1801, 3600
    d5 = synth.raster_slice(0, T, R, C, nan_ocean=True, scale=1.37).numpy()
    p = np.nanpercentile(d5, [40, 42, 60, 61])                  # bands that hold cells of this field
    q5 = [(0, 16, 0, R, 0, C, float(p[0]), float(p[1])), (3, 13, 500, 1600, 200, 3100, float(p[2]), float(p[3]))]
    leg_b(ctx, f"nested {T}x{R}x{C} f32 un-rounded (x1.37), NaN ocean, k2_levels [2, 4, 6], chunk_size 16, span 2", d5, [2, 4, 6], 16, 2, q5)
    ctx.close()
    if OUT is None:
        return
    os.makedirs(os.path.dirname(os.path.abspath(OUT)), exist_ok=True)
    with open(OUT, "w") as f:
        for d in lines:
            f.write(json.dumps(d) + "\n")


if __name__ == "__main__":
    main()
