#!/usr/bin/env python
"""bench.py -- BASELINE.json's metric on BASELINE.json's configs.

  metric  : encode raw-input GB/s (+ window-decode cells/s, cell-series cells/s, search windows/s) on N B200s,
            each with its fraction of the HBM roofline and the CPU path (the oracle) timed beside it
  workload: configs[1] -- ERA5-shaped 721x1440 grid, 8760 hourly f32 instants, full Superchunk encode
            (k2_levels [5,6], chunk_size 64: 137 time slices x 276 in-bounds 64x64 subchunks), synthetic data
  step    : one pass of the hot path over the whole raster:
            compute_fractional_bits + Superchunk::build for every 64-instant slice (dataset.rs:834-851)

`value` is measured with the raster resident in HBM; `e2e` runs the same call with pinned HOST buffers (H2D of the
raster and D2H of every encoded byte inside the timed region).  N > 1: every rank encodes its own year of the same
grid (independent time spans, no collective; weak scaling).

Beside the main line's keys the JSON carries:
  decode    full-extent window decode of the encoded slices (cells/s, roofline S_in + 4 N_out)
  queries   configs[2]-style batched cell time series and configs[3]-style value-range search over the C2 chunks
            (10^5 series / 10^5 windows by default), each with a sector-model roofline (SURVEY 8d) and checked against
            the input / the oracle
  cpu_baseline  the oracle (a line-faithful C++ port of the reference's Rust path; Rust cannot be built in this image)
            on ONE host core -- the reference never spawns its futures -- for encode, window decode, cell series, search
  extras    configs[0] (256x256x100 Chunk build + get_window), configs[2] (621x1405 daily, NaN ocean: encode + cell
            series), the int64-path and per-cell-noise variants of configs[1] on a reduced span, node assembly + CIDs
`--config c5` runs configs[4] instead: ONE 1801x3600 hourly year, k2_levels [2,4,6], dealt to the N ranks as
contiguous time spans (strong scaling: the whole job is fixed), encode + full-tile window decode.

--impl reference times the oracle on all host cores (one full 64-instant slice of the 721x1440 grid per worker).

--dump-outputs DIR writes a seeded sample of the last timed step's result as .npy files (see dump_outputs); the inputs
are the same on every run with the same arguments, so two builds of the project can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

GRID = (721, 1440)
INSTANTS = 8760
LEVELS = [5, 6]
CHUNK_SIZE = 64
METRIC = "encode_raw_input_GBps"
WORKLOAD = (f"ERA5-shaped {GRID[0]}x{GRID[1]} f32, {INSTANTS} hourly instants per GPU, Superchunk encode k2_levels {LEVELS} "
            f"chunk_size {CHUNK_SIZE} (configs[1])")
L2_NOTE = "inputs larger than L2 (no flush needed)"


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured"
        except Exception:
            pass
    return 6650.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""

    def __init__(self, index):
        self.index, self.samples, self.reasons, self.max_mhz = index, [], set(), None
        self._stop = threading.Event()
        self._t = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip().split(",")
                self.samples.append(float(out[0]))
                self.max_mhz = float(out[1])
                for n, v in zip(names, out[2:]):
                    if v.strip().lower().startswith("active"):
                        self.reasons.add(n)
            except Exception:
                pass
            self._stop.wait(0.2)

    def __enter__(self):
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._t.join(timeout=6)

    def summary(self):
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


def _dist_init(args):
    import torch
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl" if args.impl == "ours" else "gloo", rank=rank, world_size=world)
    if args.impl == "ours":
        torch.cuda.set_device(local)
    return rank, world, local


def _bind_to_gpu_numa_node(local):
    """Pin this rank's host threads (and so its first-touch pinned buffers) to the CPUs NVML lists as local to the GPU."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(local)
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
        cpus = [64 * i + b for i, w in enumerate(words) for b in range(64) if (int(w) >> b) & 1]
        allowed = os.sched_getaffinity(0)
        cpus = [c for c in cpus if c in allowed]
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        pass
    return 0


def _barrier(world):
    if world > 1:
        import torch.distributed as dist
        dist.barrier()


def _reduce(x, world, device, op):
    if world == 1:
        return x
    import torch
    import torch.distributed as dist
    t = torch.tensor([x], dtype=torch.float64, device=device)
    dist.all_reduce(t, op=getattr(dist.ReduceOp, op))
    return float(t.item())


def _max_over_ranks(x, world, device):
    return _reduce(x, world, device, "MAX")


def _sum_over_ranks(x, world, device):
    return _reduce(x, world, device, "SUM")


# ------------------------------------------------------------------------------------------ CPU side (the oracle)
def _oracle_slice_worker(job):
    """One full 64-instant slice of the grid through the oracle's Superchunk::build (reference arm: one per host core)."""
    import numpy as np
    import oracle_lib as orc
    path, levels = job
    a = np.ascontiguousarray(np.load(path))
    sec, nbytes = orc.bench_superchunk(a, levels, repeats=1)
    return sec, nbytes, a.nbytes


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return  # the other ranks exit 0 without work
    import tempfile

    import numpy as np
    import oracle_lib as orc
    from dcdf_b200 import synth
    orc.build_oracle()
    workers = os.cpu_count() or 1
    rows, cols = GRID
    a = synth.raster_slice(0, CHUNK_SIZE, rows, cols, device="cpu").numpy()
    import multiprocessing as mp
    times, gbps = [], []
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "slice.npy")
        np.save(path, a)
        with mp.get_context("fork").Pool(workers) as pool:
            for step in range(args.warmup + args.steps):
                t0 = time.perf_counter()
                res = pool.map(_oracle_slice_worker, [(path, LEVELS)] * workers)
                wall = time.perf_counter() - t0
                if step >= args.warmup:
                    times.append(wall)
                    gbps.append(sum(r[2] for r in res) / wall / 1e9)
    value = sum(gbps) / len(gbps)
    sample = (f"{workers} workers x one full {CHUNK_SIZE}-instant slice of the {rows}x{cols} grid per step "
              f"(Superchunk::build, k2_levels {LEVELS}; {1e3 * sum(times) / len(times):.0f} ms per step)")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "GB/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * sum(times) / len(times), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "i64", "data": "synthetic",
        "config": {"workload": WORKLOAD, "l2": L2_NOTE, "parallelism": f"{args.gpus} independent time spans"},
        "cpu_baseline": {"value": value, "unit": "GB/s", "cores": workers, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def cpu_baselines(host_slice, levels, n_series, n_windows, rng_seed=11):
    """The oracle on ONE host core over one 64-instant slice of the workload: encode, full-extent window decode, cell
    series, value-range search; plus the sector-model densities (SURVEY 8d) the random-access rooflines use."""
    import numpy as np
    import oracle_lib as orc
    orc.build_oracle()
    T, R, Cc = host_slice.shape
    out = {}
    t0 = time.perf_counter()
    ref = orc.superchunk_build(host_slice, levels)
    t_enc = time.perf_counter() - t0
    out["encode"] = {"value": host_slice.nbytes / t_enc / 1e9, "unit": "GB/s", "cores": 1, "kind": "port",
                     "sample": f"one {T}-instant slice of the {R}x{Cc} grid, single thread ({t_enc:.1f} s)"}
    t0 = time.perf_counter()
    raw = ref.window_raw(0, T, 0, R, 0, Cc)
    t_win = time.perf_counter() - t0
    out["decode"] = {"value": raw.size / t_win, "unit": "cells/s", "cores": 1, "kind": "port",
                     "sample": f"full-extent fill_window of that slice, {raw.size} cells ({t_win:.1f} s)"}
    rng = np.random.default_rng(rng_seed)
    q = np.stack([np.zeros(n_series, np.int64), np.full(n_series, T, np.int64), rng.integers(0, R, n_series), rng.integers(0, Cc, n_series)], axis=1)
    t0 = time.perf_counter()
    ref.cell_batch(q, want_values=True)
    t_cell = time.perf_counter() - t0
    _, cell_sectors = ref.cell_batch(q, sectors=True, want_values=False)
    out["cell"] = {"value": n_series * T / t_cell, "unit": "cells/s", "cores": 1, "kind": "port",
                   "sample": f"{n_series} full-slice cell series ({T} instants each) of that slice ({t_cell:.2f} s)",
                   "sectors_per_series_slice": cell_sectors / n_series}
    side = rng.integers(8, 257, n_windows)
    top = rng.integers(0, R - 8, n_windows)
    left = rng.integers(0, Cc - 8, n_windows)
    cubes = np.stack([np.zeros(n_windows, np.int64), np.full(n_windows, T, np.int64), top, np.minimum(top + side, R), left,
                      np.minimum(left + side, Cc)], axis=1)
    vals = raw[raw != 0]
    lo_v = rng.integers(int(vals.min()), int(vals.max()), n_windows) if vals.size else np.zeros(n_windows, np.int64)
    band = max(1, int((int(vals.max()) - int(vals.min())) * 0.05)) if vals.size else 1
    t0 = time.perf_counter()
    counts, cells, _ = ref.search_batch(cubes, lo_v, lo_v + band)
    t_search = time.perf_counter() - t0
    _, _, search_sectors = ref.search_batch(cubes, lo_v, lo_v + band, sectors=True, want_cells=False)
    vol = int(((cubes[:, 1] - cubes[:, 0]) * (cubes[:, 3] - cubes[:, 2]) * (cubes[:, 5] - cubes[:, 4])).sum())
    out["search"] = {"value": n_windows / t_search, "unit": "windows/s", "cores": 1, "kind": "port",
                     "cells_scanned_per_s": vol / t_search, "matches": int(counts.sum()),
                     "sample": f"{n_windows} windows (side 8..256, {T} instants, 5 % band) inside that slice ({t_search:.2f} s)",
                     "sectors_per_window": search_sectors / n_windows}
    return out, ref, (cubes, lo_v, band, counts, cells)


# ------------------------------------------------------------------------------------------ GPU legs
def encode_leg(ctx, data, levels, steps, warmup, world, dev, stream, clock_index=None):
    """W warm-ups + K timed steps of compute_fractional_bits + Superchunk::build over `data` (resident in HBM)."""
    import torch
    from dcdf_b200 import Superchunk, _ffi
    enc_ms, stat_ms, gather_ms = [], [], []
    sc = None
    for _ in range(warmup):
        sc = Superchunk.build(ctx, data, levels, compute_bits=True, chunk_size=CHUNK_SIZE)
        sc.close()
    torch.cuda.synchronize()
    _barrier(world)
    launches0 = ctx.launch_count
    sampler = ClockSampler(clock_index) if clock_index is not None else None
    if sampler:
        sampler.__enter__()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    ev0.record(stream)
    for i in range(steps):
        sc = Superchunk.build(ctx, data, levels, compute_bits=True, chunk_size=CHUNK_SIZE)
        enc_ms.append(ctx.last_kernel_ms(_ffi.KT_ENCODE))
        stat_ms.append(ctx.last_kernel_ms(_ffi.KT_STATS))
        gather_ms.append(ctx.last_kernel_ms(_ffi.KT_GATHER))
        if i < steps - 1:
            sc.close()  # the last result is kept for the decode / query legs
    ev1.record(stream)
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    _barrier(world)
    if sampler:
        sampler.__exit__()
    dev_ms = ev0.elapsed_time(ev1)
    return {"sc": sc, "step_ms": max(dev_ms, wall * 1e3) / steps, "dev_ms": dev_ms / steps, "wall_ms": wall * 1e3 / steps,
            "enc_ms": sum(enc_ms) / len(enc_ms), "stat_ms": sum(stat_ms) / len(stat_ms), "gather_ms": sum(gather_ms) / len(gather_ms),
            "launches": ctx.launch_count - launches0, "s_out": sc.total_bytes(), "fast_units": ctx.get_stat("encode_units_fast"),
            "general_units": ctx.get_stat("encode_units_general"), "wide_units": ctx.get_stat("encode_units_wide"),
            "clocks": sampler.summary() if sampler else None}


def dump_outputs(sc, out_dir, n_bytes=8192, n_cells=1 << 18, seed=0xDCDF0D):
    """Writes what the last timed Superchunk.build returned as .npy files, so that two builds of the project can be
    compared output for output: every slice's info and root-node references, a sample of its stored bytes, and the
    values decoded at a sample of cells.  Sample positions depend on `seed` and the sizes alone; about 25 MB for the
    workload's 137 slices."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    rng = np.random.default_rng(seed)
    info, refs, sample = [], [], []
    for s in range(sc.n_slices):
        i = sc.info(s)
        st = i.stats
        info.append([*i.shape, i.sidelen, i.chunks_sidelen, i.subsidelen, i.levels, i.encoding, i.fractional_bits, i.n_refs,
                     i.max_dac_bytes, i.min_dac_bytes, i.chunk_bytes, st.size, st.elided, st.local, st.external, st.snapshots, st.logs])
        refs.append(np.stack(sc.refs(s), axis=1))  # per subchunk slot: kind, offset, size, fractional bits
        for which in range(3):  # the slice's stored Chunks back to back, its max DAC, its min DAC
            blob = np.frombuffer(sc.bytes(s, which), np.uint8)
            at = (rng.random(n_bytes) * len(blob)).astype(np.int64)
            sample.append(blob[at] if len(blob) else np.zeros(n_bytes, np.uint8))
    T, rows, cols = sc.shape
    irc = np.stack([rng.integers(0, n, n_cells) for n in (T, rows, cols)], axis=1)
    outputs = {"slice_info": np.array(info, np.float64), "root_refs": np.stack(refs).astype(np.float64),
               "stored_bytes_sample": np.stack(sample).reshape(sc.n_slices, 3, n_bytes).astype(np.float32),
               "cells_sample_irc": irc.astype(np.float64), "cells_sample_values": sc.get_batch(irc).astype(np.float32)}
    for name, a in outputs.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a)
    return {"dir": out_dir, "bytes": int(sum(a.nbytes for a in outputs.values()))}


def decode_leg(ctx, sc, data, tspan, stream, s_out_total, T_total, peak, reps=3):
    """Full-extent window decode of the first `tspan` instants, f32 output resident in HBM, checked against the input."""
    import torch
    from dcdf_b200 import _ffi
    rows, cols = data.shape[1], data.shape[2]
    out = torch.empty((tspan, rows, cols), device=data.device, dtype=data.dtype)
    sc.window(0, tspan, 0, rows, 0, cols, out=out)
    torch.cuda.synchronize()
    d0, d1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    d0.record(stream)
    for _ in range(reps):
        sc.window(0, tspan, 0, rows, 0, cols, out=out)
    d1.record(stream)
    torch.cuda.synchronize()
    dms = d0.elapsed_time(d1) / reps
    kms = ctx.last_kernel_ms(_ffi.KT_WINDOW)
    a, b = out, data[:tspan]
    ok = bool(torch.equal(torch.nan_to_num(a, nan=-7.0), torch.nan_to_num(b, nan=-7.0)))
    cells = tspan * rows * cols
    algo = s_out_total * tspan / T_total + out.element_size() * cells
    del out
    return {"ms": dms, "kernel_ms": kms, "cells": cells, "round_trip_equal": ok, "algorithmic_bytes": int(algo),
            "achieved": algo / (kms * 1e-3) / 1e9, "frac": algo / (kms * 1e-3) / 1e9 / peak}


def cell_leg(ctx, sc, data, n_series, peak, sectors_per_series_slice, rng_seed=7, verify=64):
    import numpy as np
    from dcdf_b200 import _ffi
    T, rows, cols = data.shape
    rng = np.random.default_rng(rng_seed)
    q = np.stack([np.zeros(n_series, np.int64), np.full(n_series, T, np.int64), rng.integers(0, rows, n_series), rng.integers(0, cols, n_series)], axis=1)
    import torch
    host_out = torch.empty(n_series * T, dtype=data.dtype).pin_memory()  # results land in pinned host memory
    sc.cell_batch(q, out=host_out, flat=True)  # warm-up at full size: staging buffers grow here, not inside the timed call
    t0 = time.perf_counter()
    flat, off = sc.cell_batch(q, out=host_out, flat=True)
    t_e2e = time.perf_counter() - t0
    kms = ctx.last_kernel_ms(_ffi.KT_CELL)
    ok = True
    res_np = flat.numpy()
    for i in np.linspace(0, n_series - 1, verify).astype(int):
        want = data[:, int(q[i, 2]), int(q[i, 3])].cpu().numpy()
        ok = ok and bool(np.array_equal(res_np[int(off[i]):int(off[i + 1])], want, equal_nan=True))
    n_slices = (T + CHUNK_SIZE - 1) // CHUNK_SIZE
    res = {"series": n_series, "cells": int(n_series * T), "cells_per_s_kernel": n_series * T / (kms * 1e-3), "cells_per_s_e2e": n_series * T / t_e2e,
           "kernel_ms": kms, "verified_series": int(verify), "matches_input": ok}
    if sectors_per_series_slice:
        # Bytes that have to move: per series the distinct sectors its walks touch (SURVEY 8d's sector model) -- but never more
        # than every encoded byte once, which is what the tile path reads when a batch puts many series into each tile.
        out_bytes = 4.0 * n_series * T
        sector_bytes = 32.0 * sectors_per_series_slice * n_series * n_slices
        once_bytes = float(sc.total_bytes())
        algo = min(sector_bytes, once_bytes) + out_bytes
        res["roofline"] = {"bound": "hbm", "achieved": algo / (kms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                           "frac": algo / (kms * 1e-3) / 1e9 / peak, "traffic": None, "algorithmic_bytes": int(algo),
                           "kernel": "k_cell_tiles4 (tiles with >= 64 series of the batch: decoded once per instant) + k_cell_batch (per-cell walks)",
                           "model": f"min(sector model, every encoded byte once) + 4 B per cell; sector model = 32 B x {sectors_per_series_slice:.1f} distinct "
                                    f"sectors per (series, 64-instant slice), measured by the oracle on a sample slice, x {n_series} series x {n_slices} "
                                    f"slices = {sector_bytes / 1e9:.1f} GB; every encoded byte once = {once_bytes / 1e9:.1f} GB",
                           "frac_sector_model": (sector_bytes + out_bytes) / (kms * 1e-3) / 1e9 / peak}
    return res


def search_leg(ctx, sc, T, rows, cols, n_windows, peak, sectors_per_window, value_range, rng_seed=9):
    import numpy as np
    from dcdf_b200 import _ffi
    rng = np.random.default_rng(rng_seed)
    side = rng.integers(8, 257, n_windows)
    top = rng.integers(0, rows - 8, n_windows)
    left = rng.integers(0, cols - 8, n_windows)
    t0s = rng.integers(0, max(T - CHUNK_SIZE, 1), n_windows)
    cubes = np.stack([t0s, np.minimum(t0s + CHUNK_SIZE, T), top, np.minimum(top + side, rows), left, np.minimum(left + side, cols)], axis=1)
    vmin, vmax = value_range
    band = max(1, int((vmax - vmin) * 0.05))
    lo_v = rng.integers(vmin, vmax, n_windows)
    sc.search_batch(cubes, lo_v, lo_v + band, want_cells=False)  # warm-up at full size: the per-job count buffers grow here, not inside the timed call
    t0 = time.perf_counter()
    counts, _ = sc.search_batch(cubes, lo_v, lo_v + band, want_cells=False)  # counting pass: 10^5 windows hold ~10^9 matches
    t_count = time.perf_counter() - t0
    k_count = ctx.last_kernel_ms(_ffi.KT_SEARCH)
    vol = int(((cubes[:, 1] - cubes[:, 0]) * (cubes[:, 3] - cubes[:, 2]) * (cubes[:, 5] - cubes[:, 4])).sum())
    # both passes (count + write) on a subset whose matches fit comfortably
    ns = min(n_windows, 2048)
    sc.search_batch(cubes[:ns], lo_v[:ns], lo_v[:ns] + band)
    t0 = time.perf_counter()
    c2, cells = sc.search_batch(cubes[:ns], lo_v[:ns], lo_v[:ns] + band)
    t_full = time.perf_counter() - t0
    k_full = ctx.last_kernel_ms(_ffi.KT_SEARCH)
    vol_s = int(((cubes[:ns, 1] - cubes[:ns, 0]) * (cubes[:ns, 3] - cubes[:ns, 2]) * (cubes[:ns, 5] - cubes[:ns, 4])).sum())
    res = {"windows": n_windows, "cells_scanned": vol, "matches": int(counts.sum()), "count_pass_kernel_ms": k_count,
           "windows_per_s_count_e2e": n_windows / t_count, "cells_scanned_per_s_count_kernel": vol / (k_count * 1e-3),
           "with_cells": {"windows": ns, "matches": int(c2.sum()), "kernel_ms_both_passes": k_full, "windows_per_s_e2e": ns / t_full,
                          "windows_per_s_kernel": ns / (k_full * 1e-3), "cells_scanned_per_s_kernel": vol_s / (k_full * 1e-3)}}
    if sectors_per_window:
        # count-only leg: the windows overlap, so the bytes that have to move are every encoded byte once at most
        algo_c = min(32.0 * sectors_per_window * n_windows, float(sc.total_bytes())) + 8.0 * n_windows
        res["count_roofline"] = {"bound": "hbm", "achieved": algo_c / (k_count * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                                 "frac": algo_c / (k_count * 1e-3) / 1e9 / peak, "traffic": None, "algorithmic_bytes": int(algo_c),
                                 "kernel": "k_count_tiles4<int> + the scan of the per-job counts",
                                 "model": "min(sector model x windows, every encoded byte once) + 8 B per window"}
        algo = 32.0 * sectors_per_window * ns + 24.0 * float(c2.sum())
        res["roofline"] = {"bound": "hbm", "achieved": algo / (k_full * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                           "frac": algo / (k_full * 1e-3) / 1e9 / peak, "traffic": None, "algorithmic_bytes": int(algo),
                           "kernel": "k_search_tiles4<int> (count + write passes of the windows whose cells are wanted; the count-only leg runs k_count_tiles4)",
                           "model": f"sector model: 32 B x {sectors_per_window:.0f} distinct sectors per window (oracle, sample slice) x {ns} windows + 24 B per match"}
    return res


def run_ours(args):
    import numpy as np
    import torch
    from dcdf_b200 import Chunk, Context, Superchunk, _ffi, synth
    rank, world, local = _dist_init(args)
    numa_cpus = _bind_to_gpu_numa_node(local) if world > 1 else 0
    dev = torch.device("cuda", local)
    rows, cols = GRID
    T = args.instants
    free, total = torch.cuda.mem_get_info(dev)
    need = 4 * T * rows * cols * 2.2
    if need > free:
        if args.dump_outputs:  # a shorter raster would make the outputs incomparable with another run's
            raise SystemExit(f"--dump-outputs: {T} instants need {need / 1e9:.0f} GB, {free / 1e9:.0f} GB free on {dev}")
        T = int(free / (4 * rows * cols * 2.2)) // CHUNK_SIZE * CHUNK_SIZE
    raw_bytes = 4 * T * rows * cols
    data = torch.empty((T, rows, cols), device=dev, dtype=torch.float32)
    synth.raster(T, rows, cols, out=data, device=dev, seed=0xDCDF0002 + rank)  # every rank its own year
    torch.cuda.synchronize()
    ctx = Context(local)
    stream = torch.cuda.current_stream(dev)
    ctx.set_stream(stream.cuda_stream)
    peak, peak_kind = _peaks()
    extras = {} if (rank == 0) else None
    sections = set(args.sections.split(",")) if args.sections else set()

    # ---- configs[1]: device-resident encode
    enc = encode_leg(ctx, data, LEVELS, args.steps, args.warmup, world, dev, stream, clock_index=local)
    sc = enc["sc"]
    s_out = enc["s_out"]
    step_ms = _max_over_ranks(enc["step_ms"], world, dev)
    total_raw = _sum_over_ranks(raw_bytes, world, dev)
    value = total_raw / (step_ms * 1e-3) / 1e9
    dumped = dump_outputs(sc, args.dump_outputs) if args.dump_outputs and rank == 0 else None

    # ---- CPU path beside it (rank 0, N == 1): one slice through the oracle, all four legs + sector densities
    cpu, oracle_ref, oracle_search = None, None, None
    sample_slice = 2
    if rank == 0 and world == 1 and "cpu" in sections:
        try:
            host_slice = data[sample_slice * CHUNK_SIZE:(sample_slice + 1) * CHUNK_SIZE].cpu().numpy()
            cpu, oracle_ref, oracle_search = cpu_baselines(host_slice, LEVELS, args.cpu_series, args.cpu_windows)
        except Exception as e:
            cpu = {"error": str(e)}
    sect_cell = cpu["cell"]["sectors_per_series_slice"] if cpu and "cell" in cpu else None
    sect_win = cpu["search"]["sectors_per_window"] if cpu and "search" in cpu else None

    # ---- window decode of every unit (full extent), device-resident output
    dec = None
    try:
        tspan = min(CHUNK_SIZE * 8, T)
        d = decode_leg(ctx, sc, data, tspan, stream, s_out, T, peak)
        dec = {"metric": "window_decode_cells_per_s", "value": _sum_over_ranks(d["cells"], world, dev) / (_max_over_ranks(d["ms"], world, dev) * 1e-3),
               "unit": "cells/s", "ms": d["ms"], "cells": d["cells"], "round_trip_equal": d["round_trip_equal"],
               "roofline": {"bound": "hbm", "achieved": d["achieved"], "peak": peak, "unit": "GB/s", "frac": d["frac"],
                            "traffic": None, "frac_of_nominal_8TBps": d["achieved"] / 8000.0,
                            "kernel": "k_window_tiles4<int> (one launch: every 64x64 tile of 8 slices, f32 output resident in HBM)",
                            "algorithmic_bytes": d["algorithmic_bytes"], "kernel_ms": d["kernel_ms"]}}
        try:
            dec["roofline"]["traffic"] = json.load(open(os.path.join(ROOT, "profiles", "r1_decode_traffic.json")))["dram_bytes_per_cell"] * d["cells"]
        except Exception:
            pass
    except Exception as e:  # decode is the second half of the metric; never hide an encode number behind it
        dec = {"error": str(e)}

    # ---- configs[2]-style cell series and configs[3]-style search over the same chunks
    queries = None
    try:
        cellr = cell_leg(ctx, sc, data, args.series, peak, sect_cell)
        vr = (270 * 32, 300 * 32)  # fixed point with 4 fractional bits: value * 32 + 1
        if oracle_search is not None:
            vals = oracle_ref.window_raw(0, 4, 0, rows, 0, cols)
            vr = (int(vals.min()), int(vals.max()))
        searchr = search_leg(ctx, sc, T, rows, cols, args.windows, peak, sect_win, vr)
        if oracle_search is not None:
            # results (order included) of the oracle's sample windows, shifted to the sample slice's instants
            ocubes, olo, oband, ocounts, ocells = oracle_search
            gc = ocubes.copy()
            gc[:, 0] += sample_slice * CHUNK_SIZE
            gc[:, 1] += sample_slice * CHUNK_SIZE
            counts_g, cells_g = sc.search_batch(gc, olo, olo + oband)
            want = ocells.copy()
            want[:, 0] += sample_slice * CHUNK_SIZE
            searchr["verified_windows"] = int(len(gc))
            searchr["matches_oracle"] = bool(np.array_equal(counts_g, ocounts) and np.array_equal(cells_g, want))
        cellr["cells_per_s_kernel"] = _sum_over_ranks(cellr["cells"], world, dev) / (_max_over_ranks(cellr["kernel_ms"], world, dev) * 1e-3)
        queries = {"cell_series": cellr, "search": searchr}
    except Exception as e:
        queries = {"error": str(e)}

    # ---- node assembly + content addressing (SURVEY 8f1) on the encoded year
    if rank == 0 and "store" in sections:
        try:
            t0 = time.perf_counter()
            nodes, stats = sc.save(0)          # first call hashes every chunk of every slice on the device
            t_first = time.perf_counter() - t0
            t0 = time.perf_counter()
            for s in range(1, min(sc.n_slices, 9)):
                sc.save(s)
            t_rest = (time.perf_counter() - t0) / max(1, min(sc.n_slices, 9) - 1)
            extras["store"] = {"sha256_all_chunks_plus_slice0_s": t_first, "hashed_bytes": int(s_out), "hash_GBps": s_out / t_first / 1e9,
                               "assemble_slice_s": t_rest, "slice0_objects": len(nodes), "slice0_stats": stats}
        except Exception as e:
            extras["store"] = {"error": str(e)}
    sc.close()

    # ---- end to end through host buffers (pinned): H2D raster + encode + D2H of all encoded bytes
    e2e = None
    if "e2e" in sections:
        Te = min(T, args.e2e_instants)
        try:
            host = torch.empty((Te, rows, cols), dtype=torch.float32).pin_memory()
            host.copy_(data[:Te])
            torch.cuda.synchronize()
            host_np = host.numpy()
            # Two contexts on two host threads work on alternate groups of slices, so the H2D copy of one group
            # overlaps the kernels and the D2H copies of the other (the public API, used the way a caller would).
            group = 8 * CHUNK_SIZE
            spans = [(g, min(g + group, Te)) for g in range(0, Te, group)]
            workers = [Context(local) for _ in range(2)]
            out_bufs = [None, None]
            done = [0, 0]

            def work(w):
                cw = workers[w]
                nbytes = 0
                for gi in range(w, len(spans), 2):
                    a0, a1 = spans[gi]
                    sc_ = Superchunk.build(cw, host_np[a0:a1], LEVELS, compute_bits=True, chunk_size=CHUNK_SIZE)
                    for s in range(sc_.n_slices):
                        info = sc_.info(s)
                        for which, n in ((0, info.chunk_bytes), (1, info.max_dac_bytes), (2, info.min_dac_bytes)):
                            if out_bufs[w] is None or out_bufs[w].numel() < n:
                                out_bufs[w] = torch.empty(int(n * 1.5) + 1024, dtype=torch.uint8).pin_memory()
                            cw.check(cw._lib.dcdf_superchunk_bytes(cw._h, sc_._h, s, which, out_bufs[w].data_ptr(), n, 0))
                            nbytes += n
                    sc_.close()
                done[w] = nbytes

            def e2e_step():
                th = [threading.Thread(target=work, args=(w,)) for w in range(2)]
                for t_ in th:
                    t_.start()
                for t_ in th:
                    t_.join()
                return done[0] + done[1]

            e2e_step()
            torch.cuda.synchronize()
            _barrier(world)
            t0 = time.perf_counter()
            n_e2e = max(1, min(args.steps, 2))
            d2h = 0
            for _ in range(n_e2e):
                d2h = e2e_step()
            torch.cuda.synchronize()
            t_e2e = _max_over_ranks((time.perf_counter() - t0) / n_e2e, world, dev)
            raw_e = 4 * Te * rows * cols
            e2e = {"value": _sum_over_ranks(raw_e, world, dev) / t_e2e / 1e9, "unit": "GB/s", "h2d_bytes_per_step": raw_e,
                   "d2h_bytes_per_step": int(d2h), "instants": Te, "ms_per_step": t_e2e * 1e3,
                   "how": "pinned host raster -> Superchunk.build on 2 contexts / host threads over alternate 512-instant groups -> every encoded byte copied back to pinned host memory"}
            for cw in workers:
                cw.close()
            del host
        except Exception as e:
            e2e = {"error": str(e)}

    # ---- extras (rank 0, N == 1): the other configs and the stress variants of SURVEY 8d
    if rank == 0 and world == 1:
        if "variants" in sections:
            try:
                Tv = min(T, args.variant_instants)
                var = {}
                for name, kw in (("per_cell_noise", dict(noise_every=1)), ("unrounded_int64_path", dict(nan_ocean=True, scale=0.1))):
                    v = synth.raster(Tv, rows, cols, device=dev, **kw)
                    r = encode_leg(ctx, v, LEVELS, 2, 2, 1, dev, stream)
                    dd = decode_leg(ctx, r["sc"], v, min(Tv, 256), stream, r["s_out"], Tv, peak, reps=2)
                    algo = 4 * Tv * rows * cols + r["s_out"]
                    var[name] = {"instants": Tv, "encode_GBps": 4 * Tv * rows * cols / (r["step_ms"] * 1e-3) / 1e9, "ratio": r["s_out"] / (4 * Tv * rows * cols),
                                 "encode_kernel_ms": r["enc_ms"], "encode_roofline_frac": algo / (r["enc_ms"] * 1e-3) / 1e9 / peak,
                                 "fast_units": r["fast_units"], "general_units": r["general_units"], "wide_units": r["wide_units"],
                                 "decode_cells_per_s": dd["cells"] / (dd["kernel_ms"] * 1e-3), "decode_roofline_frac": dd["frac"],
                                 "round_trip_equal": dd["round_trip_equal"]}
                    r["sc"].close()
                    del v
                extras["variants"] = var
            except Exception as e:
                extras["variants"] = {"error": str(e)}
        if "c1" in sections:
            try:
                c1 = synth.raster_slice(0, 100, 256, 256, device=dev)
                ck = Chunk.build(ctx, c1, fractional_bits=4)
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                ck2 = Chunk.build(ctx, c1, fractional_bits=4)
                t_build = time.perf_counter() - t0
                k_build = ctx.last_kernel_ms(_ffi.KT_ENCODE)
                out1 = torch.empty_like(c1)
                ck2.window(0, 100, 0, 256, 0, 256, out=out1)
                ck2.window(0, 100, 0, 256, 0, 256, out=out1)
                kw = ctx.last_kernel_ms(_ffi.KT_WINDOW)
                extras["c1"] = {"workload": "256x256x100 f32 Chunk::build + full-extent get_window (configs[0])", "build_ms": t_build * 1e3,
                                "build_GBps": c1.numel() * 4 / t_build / 1e9, "build_encode_phase_ms": k_build, "size": ck2.size(),
                                "window_kernel_ms": kw, "window_cells_per_s": c1.numel() / (kw * 1e-3),
                                "round_trip_equal": bool(torch.equal(out1, c1))}
                ck.close()
                ck2.close()
            except Exception as e:
                extras["c1"] = {"error": str(e)}
        if "c3" in sections:
            try:
                del data
                torch.cuda.empty_cache()
                data = None
                r3, c3c = 621, 1405
                T3 = args.c3_instants
                d3 = torch.empty((T3, r3, c3c), device=dev, dtype=torch.float32)
                synth.raster(T3, r3, c3c, out=d3, device=dev, seed=0xDCDF0003, hourly=False, nan_ocean=True)
                r = encode_leg(ctx, d3, LEVELS, 2, 2, 1, dev, stream)
                algo = 4 * T3 * r3 * c3c + r["s_out"]
                cpu3 = None
                sect3 = None
                if "cpu" in sections:
                    h3 = d3[128:192].cpu().numpy()
                    cpu3, _, _ = cpu_baselines(h3, LEVELS, args.cpu_series, 64)
                    sect3 = cpu3["cell"]["sectors_per_series_slice"]
                cellr = cell_leg(ctx, r["sc"], d3, args.series, peak, sect3)
                dd = decode_leg(ctx, r["sc"], d3, 512, stream, r["s_out"], T3, peak, reps=2)
                extras["c3"] = {"workload": f"PRISM/CPC-shaped {r3}x{c3c} daily f32 with a NaN ocean, {T3} instants, k2_levels {LEVELS} (configs[2])",
                                "encode_GBps": 4 * T3 * r3 * c3c / (r["step_ms"] * 1e-3) / 1e9, "ms_per_step": r["step_ms"], "ratio": r["s_out"] / (4 * T3 * r3 * c3c),
                                "encode_kernel_ms": r["enc_ms"], "encode_roofline_frac": algo / (r["enc_ms"] * 1e-3) / 1e9 / peak,
                                "fast_units": r["fast_units"], "general_units": r["general_units"], "cell_series": cellr,
                                "decode_cells_per_s": dd["cells"] / (dd["kernel_ms"] * 1e-3), "decode_roofline_frac": dd["frac"],
                                "round_trip_equal": dd["round_trip_equal"], "cpu_baseline": cpu3}
                r["sc"].close()
                del d3
            except Exception as e:
                extras["c3"] = {"error": str(e)}

    if rank == 0:
        k_ms = enc["enc_ms"]
        algo = raw_bytes + s_out
        line = {
            "metric": METRIC, "value": value, "unit": "GB/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": step_ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "i64",
            "data": "synthetic",
            "config": {"workload": WORKLOAD, "l2": L2_NOTE, "parallelism": f"{world} independent time spans"},
            "instants": T, "encoded_bytes": int(s_out), "ratio": s_out / raw_bytes,
            "host_binding": f"rank threads pinned to the {numa_cpus} CPUs local to their GPU (NVML)" if numa_cpus else "none",
            "roofline": {"bound": "hbm", "achieved": algo / (k_ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                         "frac": algo / (k_ms * 1e-3) / 1e9 / peak, "traffic": None, "peak_kind": peak_kind,
                         "frac_of_nominal_8TBps": algo / (k_ms * 1e-3) / 1e9 / 8000.0,
                         "kernel": "encode kernels, one timed region: k_encode_v5 (full f32 tiles, fast path: "
                                   f"{enc['fast_units']} units) with k_encode_v4 / k_encode_tiles for the clipped ring and everything not eligible "
                                   f"({enc['general_units']} units) on a second stream",
                         "kernel_ms": k_ms, "stats_kernel_ms": enc["stat_ms"], "gather_ms": enc["gather_ms"], "algorithmic_bytes": int(algo),
                         "frac_of_whole_step": algo / (step_ms * 1e-3) / 1e9 / peak},
            "cpu_baseline": (dict(cpu["encode"], decode=cpu.get("decode"), cell=cpu.get("cell"), search=cpu.get("search")) if cpu and "encode" in cpu else cpu),
            "e2e": e2e, "decode": dec, "queries": queries, "extras": extras, "gpu_launches": int(enc["launches"]), "clocks": enc["clocks"],
            "wall_ms_per_step": enc["wall_ms"], "device_ms_per_step": enc["dev_ms"], "dumped_outputs": dumped,
        }
        try:  # DRAM traffic of the dominant kernel from the committed ncu capture (bytes per (unit, instant)), scaled to this launch
            tj = json.load(open(os.path.join(ROOT, "profiles", "r2_traffic.json")))
            line["roofline"]["traffic"] = tj["dram_bytes_per_unit_instant"] * enc["fast_units"] * CHUNK_SIZE * (T / (((T + CHUNK_SIZE - 1) // CHUNK_SIZE) * CHUNK_SIZE))
            line["roofline"]["traffic_note"] = "ncu dram bytes of k_encode_v5 per (unit, instant) x fast-path units of this launch (profiles/r2_traffic.json)"
        except Exception:
            pass
        print(json.dumps(line))
    ctx.close()
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------ configs[4]
def _c5_span(n_slices, world, rank):
    """Slices [s0, s1) of the year that `rank` encodes and decodes: contiguous spans of ceil(n_slices / world) slices, so
    every slice belongs to exactly one rank (the last ranks may get fewer, or none when world does not divide)."""
    per = (n_slices + world - 1) // world
    return min(n_slices, rank * per), min(n_slices, (rank + 1) * per)


def run_c5(args):
    """One 1801x3600 hourly year, k2_levels [2,4,6], as contiguous time spans over the N ranks (strong scaling).  A rank
    walks its span slab by slab (a slab = up to 17 slices, 28 GB raw, generated on the device, untimed): encode, then
    full-tile window decode of every unit; throughput = whole-year bytes / cells over the slowest rank's summed time."""
    import torch
    from dcdf_b200 import Context, Superchunk, _ffi, synth
    rank, world, local = _dist_init(args)
    dev = torch.device("cuda", local)
    rows, cols, levels = 1801, 3600, [2, 4, 6]
    T_year = args.instants
    n_slices = (T_year + CHUNK_SIZE - 1) // CHUNK_SIZE
    s0, s1 = _c5_span(n_slices, world, rank)
    ctx = Context(local)
    stream = torch.cuda.current_stream(dev)
    ctx.set_stream(stream.cuda_stream)
    peak, _ = _peaks()
    slab = args.c5_slab_slices
    enc_ms = dec_ms = 0.0
    enc_k = dec_k = 0.0
    raw = out_bytes = cells = 0
    ok = True
    warmed = False
    buf = None
    for a in range(s0, s1, slab):
        b = min(a + slab, s1)
        t0i, t1i = a * CHUNK_SIZE, min(b * CHUNK_SIZE, T_year)
        data = synth.raster(t1i - t0i, rows, cols, device=dev, seed=0xDCDF0005, t_start=t0i)
        torch.cuda.synchronize()
        if not warmed:
            for _ in range(max(1, args.warmup)):  # full-size: scratch, arena and result pools reach their final sizes here
                Superchunk.build(ctx, data, levels, compute_bits=True, chunk_size=CHUNK_SIZE).close()
            warmed = True
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        sc = Superchunk.build(ctx, data, levels, compute_bits=True, chunk_size=CHUNK_SIZE)
        e1.record(stream)
        torch.cuda.synchronize()
        enc_ms += e0.elapsed_time(e1)
        enc_k += ctx.last_kernel_ms(_ffi.KT_ENCODE)
        raw += data.numel() * 4
        out_bytes += sc.total_bytes()
        if buf is None or buf.shape[0] < data.shape[0]:
            buf = torch.empty_like(data)
        o = buf[:data.shape[0]]
        sc.window(0, data.shape[0], 0, rows, 0, cols, out=o)  # warm
        d0, d1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        d0.record(stream)
        sc.window(0, data.shape[0], 0, rows, 0, cols, out=o)
        d1.record(stream)
        torch.cuda.synchronize()
        dec_ms += d0.elapsed_time(d1)
        dec_k += ctx.last_kernel_ms(_ffi.KT_WINDOW)
        cells += data.numel()
        ok = ok and bool(torch.equal(o, data))
        sc.close()
        del data
    _barrier(world)
    t_enc = _max_over_ranks(enc_ms, world, dev)
    t_dec = _max_over_ranks(dec_ms, world, dev)
    tot_raw = _sum_over_ranks(raw, world, dev)
    tot_out = _sum_over_ranks(out_bytes, world, dev)
    tot_cells = _sum_over_ranks(cells, world, dev)
    all_ok = _sum_over_ranks(0 if ok else 1, world, dev) == 0
    k_enc = _max_over_ranks(enc_k, world, dev)
    k_dec = _max_over_ranks(dec_k, world, dev)
    if rank == 0:
        line = {"metric": METRIC, "value": tot_raw / (t_enc * 1e-3) / 1e9, "unit": "GB/s", "n_gpus": world, "steps": 1, "warmup": args.warmup,
                "ms_per_step": t_enc, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "i64", "data": "synthetic",
                "config": {"workload": f"0.1-degree global {rows}x{cols} f32, {T_year} hourly instants, k2_levels {levels} chunk_size {CHUNK_SIZE}, "
                                       f"time spans dealt to the ranks (configs[4])", "l2": L2_NOTE, "parallelism": f"{world} contiguous time spans of one year"},
                "encoded_bytes": int(tot_out), "ratio": tot_out / tot_raw,
                "roofline": {"bound": "hbm", "achieved": (tot_raw + tot_out) / world / (k_enc * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                             "frac": (tot_raw + tot_out) / world / (k_enc * 1e-3) / 1e9 / peak, "traffic": None, "kernel": "encode kernels (per GPU, slowest rank)"},
                "decode": {"metric": "window_decode_cells_per_s", "value": tot_cells / (t_dec * 1e-3), "unit": "cells/s", "ms": t_dec, "round_trip_equal": all_ok,
                           "roofline_frac_per_gpu": (tot_out + 4 * tot_cells) / world / (k_dec * 1e-3) / 1e9 / peak},
                "cpu_baseline": None, "e2e": None, "gpu_launches": int(ctx.launch_count)}
        print(json.dumps(line))
    ctx.close()
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="c2", choices=["c2", "c5"])
    ap.add_argument("--instants", type=int, default=INSTANTS)
    ap.add_argument("--e2e-instants", type=int, default=INSTANTS)
    ap.add_argument("--sections", default="cpu,e2e,store,variants,c1,c3", help="comma list of: cpu, e2e, store, variants, c1, c3")
    ap.add_argument("--series", type=int, default=100000, help="cell time series of the query leg (configs[2]: 10^5)")
    ap.add_argument("--windows", type=int, default=100000, help="search windows of the query leg (configs[3]: 10^5)")
    ap.add_argument("--cpu-series", type=int, default=2000)
    ap.add_argument("--cpu-windows", type=int, default=192)
    ap.add_argument("--variant-instants", type=int, default=512)
    ap.add_argument("--c3-instants", type=int, default=14610)
    ap.add_argument("--c5-slab-slices", type=int, default=18)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write a seeded sample of what the last "
                    "step's Superchunk.build returned (rank 0) to DIR/<name>.npy; default config and impl only")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.config != "c2"):
        ap.error("--dump-outputs applies to the default --impl ours --config c2 run")
    if args.no_e2e:
        args.sections = ",".join(s for s in args.sections.split(",") if s != "e2e")
    if args.no_cpu:
        args.sections = ",".join(s for s in args.sections.split(",") if s != "cpu")
    if args.impl == "reference":
        run_reference(args)
    elif args.config == "c5":
        run_c5(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
