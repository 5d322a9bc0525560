"""world_size-2 gloo test of the N > 1 host logic of bench.py (no GPU): every rank owns an independent time
span, nothing is exchanged on the data path, and only the timing / byte totals are reduced."""
import os
import socket
import sys

import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _worker(rank, world, port, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    sys.path.insert(0, ROOT)
    import bench
    from dcdf_b200 import synth
    dist.init_process_group("gloo", rank=rank, world_size=world)
    dev = torch.device("cpu")
    # each rank generates its own span (seed differs per rank, as in bench.run_ours)
    a = synth.raster_slice(0, 4, 40, 50, seed=0xDCDF0002 + rank)
    b = synth.raster_slice(0, 4, 40, 50, seed=0xDCDF0002)
    assert (rank == 0) == bool(torch.equal(a, b))
    step_ms = bench._max_over_ranks(10.0 + 5.0 * rank, world, dev)
    total = bench._sum_over_ranks(float(a.numel() * 4), world, dev)
    bench._barrier(world)
    out[rank] = (step_ms, total)
    dist.destroy_process_group()


def test_two_rank_reduction_of_timings_and_totals():
    world = 2
    with socket.socket() as s:  # a free port chosen by the OS: a fixed one may be taken on a shared machine
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    with mp.Manager() as m:
        out = m.dict()
        mp.spawn(_worker, args=(world, port, out), nprocs=world, join=True)
        res = dict(out)
    assert res[0] == res[1] == (15.0, 2 * 4 * 40 * 50 * 4.0)   # max over ranks, whole-job bytes


def test_reference_arm_extra_ranks_exit_without_work(monkeypatch, capsys):
    sys.path.insert(0, ROOT)
    import bench
    monkeypatch.setenv("RANK", "1")
    bench.run_reference(type("A", (), dict(gpus=2, steps=1, warmup=0, ref_rows=8))())
    assert capsys.readouterr().out == ""


def test_c5_time_spans_cover_the_year_exactly_once():
    """bench.py --config c5 (north_star's multi-GPU statement): the 137 slices of one year dealt as contiguous spans."""
    sys.path.insert(0, ROOT)
    import bench
    for n_slices in (1, 7, 8, 137, 229):
        for world in (1, 2, 4, 8):
            spans = [bench._c5_span(n_slices, world, r) for r in range(world)]
            covered = [s for a, b in spans for s in range(a, b)]
            assert covered == list(range(n_slices)), (n_slices, world)
            assert max(b - a for a, b in spans) == -(-n_slices // world)        # the slowest rank's share sets the time
            assert all(0 <= a <= b <= n_slices for a, b in spans)
