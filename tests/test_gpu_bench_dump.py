"""bench.py --dump-outputs: the files are float arrays, the same on every call, and hold what the Superchunk holds."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

pytestmark = pytest.mark.gpu


def test_dump_outputs_samples_what_the_build_returned(tmp_path):
    sys.path.insert(0, ROOT)
    import bench
    from dcdf_b200 import Context, Superchunk, synth
    ctx = Context(0)
    data = synth.raster_slice(0, 150, 100, 130).numpy()                 # three slices, the last one 22 instants
    sc = Superchunk.build(ctx, data, [2, 6], chunk_size=64)
    kw = dict(n_bytes=512, n_cells=4096, seed=5)
    first = bench.dump_outputs(sc, str(tmp_path / "a"), **kw)
    bench.dump_outputs(sc, str(tmp_path / "b"), **kw)
    names = sorted(os.listdir(tmp_path / "a"))
    assert names == sorted(os.listdir(tmp_path / "b")) and len(names) == 5
    out = {}
    for n in names:
        a, b = np.load(tmp_path / "a" / n), np.load(tmp_path / "b" / n)
        assert a.dtype in (np.float32, np.float64) and np.array_equal(a, b)
        out[n[:-4]] = a
    assert first["bytes"] == sum(a.nbytes for a in out.values())
    info = out["slice_info"]
    assert info.shape == (3, 19) and list(info[:, 0]) == [64, 64, 22]
    assert out["root_refs"].shape == (3, 16, 4)
    rng = np.random.default_rng(kw["seed"])                              # the positions dump_outputs draws
    for s in range(3):
        for which in range(3):
            blob = np.frombuffer(sc.bytes(s, which), np.uint8)
            at = (rng.random(kw["n_bytes"]) * len(blob)).astype(np.int64)
            assert np.array_equal(out["stored_bytes_sample"][s, which], blob[at]), (s, which)
    irc = out["cells_sample_irc"].astype(np.int64)
    assert np.array_equal(out["cells_sample_values"], data[irc[:, 0], irc[:, 1], irc[:, 2]])
    sc.close()
    ctx.close()
