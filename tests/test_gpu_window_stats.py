"""Per-instant window statistics reduced on the device (dcdf_superchunk_window_stats, Superchunk.window_stats_batch,
Variable.window_stats).  Truth is numpy over the decoded window: the oracle's window_f32 for f32, Superchunk.window
(parity-tested elsewhere) otherwise.  count exactly, min / max by equality, sum / sum_sq within 1e-11 of the sum of
|v| / v^2 (math.fsum), under the default 32-bit expansion and with "window_wide"."""
import ctypes as C
import math

import numpy as np
import pytest

import oracle_lib as orc

pytestmark = pytest.mark.gpu
OPTIONS = {"default": {}, "window_wide": {"window_wide": 1}}


def _context(opts):
    from dcdf_b200 import Context
    c = Context(0)
    for k, v in opts.items():
        c.set_option(k, v)
    return c


@pytest.fixture(scope="module", params=list(OPTIONS))
def ctx(request):
    c = _context(OPTIONS[request.param])
    yield c
    c.close()


def _truth_check(rec, w):
    """rec: the window's records; w: its decoded [T, R, C] window."""
    assert len(rec) == w.shape[0]
    for t in range(w.shape[0]):
        x = w[t].ravel()
        r = rec[t]
        if np.issubdtype(w.dtype, np.floating):
            x = x[~np.isnan(x)]
        assert int(r["count"]) == x.size, t
        if x.size == 0:
            assert r["sum"] == 0.0 and r["sum_sq"] == 0.0
            if np.issubdtype(w.dtype, np.floating):
                assert np.isnan(r["min"]) and np.isnan(r["max"])
            else:
                assert r["min"] == 0 and r["max"] == 0
            continue
        assert r["min"] == x.min() and r["max"] == x.max(), (t, r["min"], x.min(), r["max"], x.max())
        v = [float(a) for a in x.tolist()]
        s, a, q = math.fsum(v), math.fsum(abs(e) for e in v), math.fsum(e * e for e in v)
        assert abs(float(r["sum"]) - s) <= 1e-11 * a, (t, float(r["sum"]), s)
        assert abs(float(r["sum_sq"]) - q) <= 1e-11 * q, (t, float(r["sum_sq"]), q)


def _check(sc, values, cubes):
    recs, off = sc.window_stats_batch(cubes)
    assert recs.dtype["min"] == np.dtype(sc.window(0, 1, 0, 1, 0, 1).dtype)
    for i, c in enumerate(cubes):
        _truth_check(recs[int(off[i]):int(off[i + 1])], values(c))
    return recs, off


def _mixed_bits(T=10):
    rng = np.random.default_rng(31)
    R, Cc = 192, 192
    data = np.empty((T, R, Cc), np.float32)
    data[:, 0:64, 0:64] = rng.integers(-20, 40, (T, 64, 64))                               # 0 bits
    data[:, 0:64, 64:128] = rng.integers(-300, 300, (T, 64, 64)) / 16.0                   # 4 bits
    data[:, 0:64, 128:192] = 1.0 + rng.integers(0, 1 << 20, (T, 64, 64)) * 2.0 ** -22     # 22 bits
    data[:, 64:128, 0:64] = np.nan                                                        # elided, all NaN
    data[:, 64:128, 64:128] = 3.25                                                        # elided, constant
    tile = rng.integers(0, 40, (T, 64, 64)) / 4.0
    tile[:, rng.random((64, 64)) < 0.5] = np.nan                                          # NaN ocean
    data[:, 64:128, 128:192] = tile
    data[:, 128:, :] = rng.integers(-50, 50, (T, 64, 192)) / 8.0
    return data


def test_mixed_bits_nan_ocean_and_elided_subchunks(ctx):
    from dcdf_b200 import Superchunk
    data = _mixed_bits()
    T, R, Cc = data.shape
    sc, ref = Superchunk.build(ctx, data, [2, 6]), orc.superchunk_build(data, [2, 6])
    kinds, _, _, bits = sc.refs(0)
    assert {int(b) for k, b in zip(kinds, bits) if k == 2} >= {0, 4, 22} and 0 in set(int(k) for k in kinds)
    cubes = [[0, T, 0, R, 0, Cc], [1, T - 1, 5, R - 7, 3, Cc - 2], [2, 7, 100, 101, 0, Cc], [4, 5, 150, 151, 77, 78],
             [0, T, 70, 90, 5, 50], [0, T, 64, 128, 64, 128]]
    recs, off = _check(sc, lambda c: ref.window_f32(*c), cubes)
    empty = recs[int(off[4]):int(off[5])]
    assert (empty["count"] == 0).all() and np.isnan(empty["min"]).all() and (empty["sum"] == 0).all()
    assert (recs[int(off[5]):int(off[6])]["sum"] == 3.25 * 64 * 64).all()
    sc.close()


def test_slices_and_windows_starting_inside_a_block(ctx):
    """chunk_size 8: windows crossing slice boundaries that start on Log instants (the snapshot is expanded first)."""
    from dcdf_b200 import Superchunk, synth
    data = synth.raster_slice(0, 40, 130, 200, nan_ocean=True).numpy()
    sc = Superchunk.build(ctx, data, [2, 6], chunk_size=8)
    assert sc.n_slices == 5
    cubes = [[3, 37, 0, 130, 0, 200], [5, 18, 17, 99, 33, 180], [9, 10, 0, 130, 0, 200], [15, 33, 64, 128, 0, 64],
             [1, 40, 129, 130, 199, 200]]
    _check(sc, lambda c: sc.window(*c), cubes)
    sc.close()


@pytest.mark.parametrize("levels", [[1, 1, 6], [1, 1, 1, 5]])
def test_nested_superchunk_with_elided_upper_level(ctx, levels):
    from dcdf_b200 import Superchunk
    rng = np.random.default_rng(33)
    T, R, Cc = 9, 256, 224
    data = (rng.integers(-400, 400, (T, R, Cc)) / 16.0).astype(np.float32)
    data[:, 0:128, 128:224] = 7.5                                     # a whole inner node is constant
    data[:, 128:192, 0:64] = np.nan
    data[:, 192:256, 64:128] = rng.integers(-9, 9, (T, 64, 64))       # 0 bits
    data[:, 128:192, 128:192] = (5.0 + rng.integers(0, 1 << 18, (T, 64, 64)) * 2.0 ** -20).astype(np.float32)
    sc, ref = Superchunk.build(ctx, data, levels), orc.superchunk_build(data, levels)
    assert sc.node_count() > 1
    cubes = [[0, T, 0, R, 0, Cc], [1, 8, 3, 250, 100, 220], [0, T, 10, 120, 130, 220], [2, 3, 130, 190, 1, 63]]
    _check(sc, lambda c: ref.window_f32(*c), cubes)
    sc.close()


def test_nested_2_4_6_with_an_elided_1024_node(ctx):
    """k2_levels [2, 4, 6] (the C5 layout): the second 1024-wide node of the root is constant, so the root elides it."""
    from dcdf_b200 import Superchunk, synth
    T, R, Cc = 3, 600, 2600                                           # every 1024-wide node's part needs 10 levels
    data = synth.raster_slice(0, T, R, Cc, nan_ocean=True, scale=1.37).numpy()
    data[:, :, 1024:2048] = 2.5
    sc = Superchunk.build(ctx, data, [2, 4, 6])
    kinds, _, _, _ = sc.refs(0)
    assert 0 in set(int(k) for k in kinds)
    cubes = [[0, T, 0, R, 0, Cc], [1, 3, 17, 590, 1000, 2590], [0, T, 100, 200, 1100, 1200]]
    recs, off = _check(sc, lambda c: sc.window(*c), cubes)
    assert (recs[int(off[2]):int(off[3])]["sum"] == 2.5 * 100 * 100).all()
    sc.close()


def test_codes_near_2_27_in_f32(ctx):
    """20 fractional bits on values around 50: codes near 2^27, several codes decode to one float."""
    from dcdf_b200 import Superchunk
    rng = np.random.default_rng(34)
    T, R, Cc = 6, 64, 128
    data = (50.0 + rng.integers(0, 1 << 22, (T, R, Cc)) * 2.0 ** -18).astype(np.float32)
    sc = Superchunk.build(ctx, data, [1, 6], fractional_bits=20, compute_bits=False)
    ref = orc.superchunk_build(data, [1, 6], fractional_bits=20, compute_bits=False)
    assert sc.info(0).fractional_bits == 20
    _check(sc, lambda c: ref.window_f32(*c), [[0, T, 0, R, 0, Cc], [1, 5, 3, 61, 7, 120]])
    sc.close()


@pytest.mark.parametrize("dtype", [np.float64, np.int32, np.int64])
def test_f64_and_integer_encodings(ctx, dtype):
    from dcdf_b200 import Superchunk
    rng = np.random.default_rng(35)
    T, R, Cc = 7, 128, 128
    if dtype == np.float64:
        data = rng.integers(-1000, 1000, (T, R, Cc)) / 64.0
        data[:, :30, :30] = np.nan
        data[:, 64:, 64:] = np.nan                                        # an all-NaN subchunk
    elif dtype == np.int32:
        data = rng.integers(-5, 6, (T, R, Cc)).astype(dtype)
        data[:, 64:, 64:128] = 0                                          # code 0 is the value 0 for integers
    else:
        data = (rng.integers(-(1 << 20), 1 << 20, (T, R, Cc)) + (1 << 60)).astype(np.int64)   # far beyond 2^53
        data[:, 64:, :64] = (1 << 60) + 3                                 # constant: elided
    sc = Superchunk.build(ctx, data, [1, 6])
    cubes = [[0, T, 0, R, 0, Cc], [1, 6, 5, 120, 60, 125], [3, 4, 64, 128, 64, 128], [0, T, 70, 71, 0, 64]]
    recs, _ = _check(sc, lambda c: sc.window(*c), cubes)
    if dtype == np.int64:
        assert recs["max"].max() > (1 << 60) and recs["min"].dtype == np.int64
    sc.close()


def _random_cubes(rng, n, T, R, Cc):
    t0 = rng.integers(0, T, n)
    t1 = np.minimum(t0 + rng.integers(1, T + 1, n), T)
    r0, c0 = rng.integers(0, R, n), rng.integers(0, Cc, n)
    r1, c1 = np.minimum(r0 + rng.integers(0, 90, n), R), np.minimum(c0 + rng.integers(0, 90, n), Cc)
    return np.stack([t0, t1, r0, r1, c0, c1], axis=1)


def test_batch_equals_alone_and_repeats_bitwise(ctx):
    from dcdf_b200 import Superchunk
    data = _mixed_bits(T=20)
    T, R, Cc = data.shape
    sc = Superchunk.build(ctx, data, [2, 6], chunk_size=8)
    cubes = _random_cubes(np.random.default_rng(36), 2000, T, R, Cc)
    recs, off = sc.window_stats_batch(cubes)
    again, off2 = sc.window_stats_batch(cubes)
    assert recs.tobytes() == again.tobytes() and np.array_equal(off, off2)
    for i in range(0, 2000, 7):
        alone = sc.window_stats(*cubes[i])
        assert alone.tobytes() == recs[int(off[i]):int(off[i + 1])].tobytes(), i
    for i in range(0, 2000, 97):
        _truth_check(recs[int(off[i]):int(off[i + 1])], sc.window(*cubes[i]))
    sc.close()


def test_wide_expansion_and_reopened_superchunk_are_bitwise_equal(ctx):
    from dcdf_b200 import Superchunk, synth
    data = synth.raster_slice(0, 24, 150, 200, nan_ocean=True, scale=1.37).numpy()
    cubes = _random_cubes(np.random.default_rng(37), 300, 24, 150, 200)
    sc = Superchunk.build(ctx, data, [2, 6], chunk_size=8)
    recs, _ = sc.window_stats_batch(cubes)
    for opts in OPTIONS.values():                    # the same bytes queried with either expansion
        c2 = _context(opts)
        sc2 = Superchunk.build(c2, data, [2, 6], chunk_size=8)
        assert sc2.window_stats_batch(cubes)[0].tobytes() == recs.tobytes()
        sc2.close()
        c2.close()
    store, roots = {}, []
    for s in range(sc.n_slices):
        nodes, _ = sc.save(s)
        store.update({cid: b for cid, _, b in nodes})
        roots.append(nodes[-1][0])
    op = Superchunk.open(ctx, roots, store)
    assert op.window_stats_batch(cubes)[0].tobytes() == recs.tobytes()
    op.close()
    sc.close()


def test_device_outputs_equal_host_outputs(ctx):
    import torch
    from dcdf_b200 import Superchunk, _ffi
    data = _mixed_bits()
    sc = Superchunk.build(ctx, data, [2, 6])
    cubes = np.ascontiguousarray(_random_cubes(np.random.default_rng(38), 50, *data.shape), dtype=np.int64)
    recs, off = sc.window_stats_batch(cubes)
    n = int(off[-1])
    dev = torch.device("cuda", 0)
    count = torch.empty(n, dtype=torch.int64, device=dev)
    vmin, vmax = torch.empty(n, dtype=torch.float32, device=dev), torch.empty(n, dtype=torch.float32, device=dev)
    s, q = torch.empty(n, dtype=torch.float64, device=dev), torch.empty(n, dtype=torch.float64, device=dev)
    torch.cuda.synchronize()
    ptr = lambda t: C.c_void_p(t.data_ptr())
    ctx.check(ctx._lib.dcdf_superchunk_window_stats(ctx._h, sc._h, len(cubes), C.c_void_p(cubes.ctypes.data), C.c_void_p(off.ctypes.data),
                                                    ptr(count), ptr(vmin), ptr(vmax), ptr(s), ptr(q), _ffi.MEM_DEVICE))
    assert np.array_equal(count.cpu().numpy().view(np.uint64), recs["count"])
    for name, t in (("min", vmin), ("max", vmax), ("sum", s), ("sum_sq", q)):
        assert t.cpu().numpy().tobytes() == np.ascontiguousarray(recs[name]).tobytes(), name
    sc.close()


def test_bounds_and_errors(ctx):
    from dcdf_b200 import DcdfError, Superchunk
    data = _mixed_bits()
    T, R, Cc = data.shape
    sc = Superchunk.build(ctx, data, [2, 6])
    fwd = sc.window_stats(2, 8, 10, 100, 20, 150)
    assert sc.window_stats(8, 2, 100, 10, 150, 20).tobytes() == fwd.tobytes()            # reversed bounds are swapped
    z = sc.window_stats(1, 5, 30, 30, 0, 50)                                              # zero-area window
    assert len(z) == 4 and (z["count"] == 0).all() and (z["sum"] == 0).all()
    assert len(sc.window_stats(3, 3, 0, 10, 0, 10)) == 0                                  # start == end: no records
    recs, off = sc.window_stats_batch([[0, 2, 0, 5, 0, 5], [4, 4, 0, 5, 0, 5], [1, 3, 0, 5, 0, 5]])
    assert off.tolist() == [0, 2, 2, 4]
    for bad in ([0, T + 1, 0, 5, 0, 5], [0, 2, 0, R + 1, 0, 5], [0, 2, 0, 5, -1, 5]):
        with pytest.raises(DcdfError) as e:
            sc.window_stats(*bad)
        assert e.value.code == 5
    cubes = np.array([[0, 3, 0, 5, 0, 5]], np.int64)
    off = np.array([0, 2], np.uint64)                                                     # wrong out_off
    outs = [np.empty(3, np.uint64), np.empty(3, np.float32), np.empty(3, np.float32), np.empty(3), np.empty(3)]
    p = [C.c_void_p(a.ctypes.data) for a in outs]
    code = ctx._lib.dcdf_superchunk_window_stats(ctx._h, sc._h, 1, C.c_void_p(cubes.ctypes.data), C.c_void_p(off.ctypes.data), *p, 0)
    assert code == 8
    off = np.array([0, 3], np.uint64)
    code = ctx._lib.dcdf_superchunk_window_stats(ctx._h, sc._h, 1, C.c_void_p(cubes.ctypes.data), C.c_void_p(off.ctypes.data), p[0], None, p[2], p[3], p[4], 0)
    assert code == 8
    sc.close()


@pytest.mark.parametrize("cache_bytes", [1 << 30, 1])
def test_variable_window_stats_across_span_groups(ctx, cache_bytes):
    from dcdf_b200 import Variable
    rng = np.random.default_rng(39)
    T, R, Cc = 40, 256, 200
    data = (rng.integers(-800, 800, (T, R, Cc)) / 16.0).astype(np.float32)
    data[:, :64, 64:128] = np.round(data[:, :64, 64:128])
    data[:, 128:192, :64] = np.nan
    data[:, 64:128, 128:192] = 0.0
    v = Variable(ctx, {}, [1, 1, 6], chunk_size=8, span_size=3, cache_bytes=cache_bytes)
    v.append(data)
    for q in ((3, 37, 10, 250, 20, 190), (0, 40, 0, R, 0, Cc), (22, 26, 130, 140, 0, 10)):
        got = v.window_stats(*q)
        assert len(got) == q[1] - q[0]
        _truth_check(got, v.window(*q))
    assert len(v.window_stats(5, 5, 0, 10, 0, 10)) == 0
    v.close()


def test_two_launches_and_kernel_time(ctx):
    from dcdf_b200 import Superchunk, _ffi
    data = _mixed_bits()
    sc = Superchunk.build(ctx, data, [2, 6])
    cubes = _random_cubes(np.random.default_rng(40), 100, *data.shape)
    sc.window_stats_batch(cubes)                     # the superchunk's query directory is built on first use
    n0 = ctx.launch_count
    sc.window_stats_batch(cubes)
    assert ctx.launch_count - n0 <= 2
    assert ctx.last_kernel_ms(_ffi.KT_REDUCE) > 0
    sc.close()
