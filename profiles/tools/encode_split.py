"""Where the encode region of one C2 build goes: per-kernel time of the encoder lists under torch.profiler.

Builds the bench's C2 raster (721x1440 f32, 8760 hourly instants, seed 0xDCDF0002), runs warm-up builds, then traces
a few `Superchunk.build(..., [5, 6], compute_bits=True, chunk_size=64)` calls.  Prints one JSON line per kernel name
(calls, total and per-call device time), one line per encode kernel of the last traced build with its start and end
inside the encode region (the span from the first encode kernel's start to the last one's end), and one line with the
card's name, power limit and the units per encoder list.

  python profiles/tools/encode_split.py [OUT_DIR] [--instants T] [--builds N]

OUT_DIR gets the same lines in encode_split.jsonl.
"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", ".."))

import torch  # noqa: E402
from torch.profiler import ProfilerActivity, profile  # noqa: E402

from dcdf_b200 import Context, Superchunk, synth  # noqa: E402

ENCODE_KERNELS = ("k_encode_v5", "k_encode_v4", "k_encode_tiles")


def card():
    q = "name,power.limit,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", "--id=0", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=10).stdout.strip()
    except Exception as e:  # the line still says what was not available
        out = f"unavailable: {e}"
    return {"card": out, "torch_name": torch.cuda.get_device_name(0)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out", nargs="?")
    ap.add_argument("--instants", type=int, default=8760)
    ap.add_argument("--builds", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=2)
    a = ap.parse_args()
    lines = []

    def emit(d):
        print(json.dumps(d), flush=True)
        lines.append(d)

    dev = torch.device("cuda", 0)
    ctx = Context(0)
    data = synth.raster(a.instants, 721, 1440, device=dev, seed=0xDCDF0002)
    torch.cuda.synchronize()
    build = lambda: Superchunk.build(ctx, data, [5, 6], compute_bits=True, chunk_size=64).close()  # noqa: E731
    for _ in range(a.warmup):
        build()
    torch.cuda.synchronize()
    stats = {}
    for k in ("encode_units_fast", "encode_units_edge", "encode_units_general", "encode_units_clipped"):
        try:
            stats[k] = ctx.get_stat(k)
        except Exception:  # a build without that counter
            stats[k] = None
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(a.builds):
            build()
            torch.cuda.synchronize()

    kernels = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA and e.time_range.elapsed_us() > 0]
    per = {}
    for e in kernels:
        d = per.setdefault(e.name, [0, 0.0])
        d[0] += 1
        d[1] += e.time_range.elapsed_us()
    for name, (n, us) in sorted(per.items(), key=lambda kv: -kv[1][1]):
        emit({"kernel": name, "calls_per_build": n / a.builds, "ms_per_build": us / a.builds / 1e3, "us_per_call": us / n})

    # the last build's encode region: from the first encode kernel's start to the last one's end
    enc = sorted((e for e in kernels if e.name.startswith(ENCODE_KERNELS)), key=lambda e: e.time_range.start)
    per_build = len(enc) // a.builds
    last = enc[-per_build:] if per_build else []
    if last:
        t0 = min(e.time_range.start for e in last)
        t1 = max(e.time_range.end for e in last)
        emit({"encode_region_ms": (t1 - t0) / 1e3, "encode_kernels_per_build": per_build})
        for e in last:
            emit({"timeline": e.name, "start_ms": (e.time_range.start - t0) / 1e3, "end_ms": (e.time_range.end - t0) / 1e3,
                  "ms": e.time_range.elapsed_us() / 1e3})
    emit({**card(), "instants": a.instants, "builds": a.builds, "units": stats})
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "encode_split.jsonl"), "w") as f:
            for d in lines:
                f.write(json.dumps(d) + "\n")


if __name__ == "__main__":
    main()
