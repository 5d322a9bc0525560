"""Per-cell statistics over time reduced on the device (dcdf_superchunk_time_stats, Superchunk.time_stats_batch,
Variable.time_stats).  Truth is numpy over the decoded window: the oracle's window_f32 for f32, Superchunk.window
(parity-tested elsewhere) otherwise.  The order of the sums is part of the contract (one running double sum per time
slice, in time order, then the slices' sums in order), so every field is compared by equality: count and n_band
exactly, min / max by value and NaN-ness, sum and sum_sq bitwise.  Every case runs under the default 32-bit expansion
and with "window_wide"."""
import ctypes as C

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


def _truth(w, start, chunk_size, lower=-np.inf, upper=np.inf):
    """Records of a decoded [T, R, C] window whose first instant is `start`, in the order the header states."""
    T, R, Cc = w.shape
    flt = np.issubdtype(w.dtype, np.floating)
    count, n_band = np.zeros((R, Cc), np.uint64), np.zeros((R, Cc), np.uint64)
    total, total_sq = np.zeros((R, Cc)), np.zeros((R, Cc))
    lo, hi = min(lower, upper), max(lower, upper)
    t = 0
    while t < T:
        t_end = min(T, ((start + t) // chunk_size + 1) * chunk_size - start)     # the piece inside one slice
        acc, acc_sq = np.zeros((R, Cc)), np.zeros((R, Cc))
        for u in range(t, t_end):
            x = w[u].astype(np.float64)
            ok = ~np.isnan(x)
            x = np.where(ok, x, 0.0)
            acc = acc + x
            acc_sq = acc_sq + x * x
            count += ok
            n_band += ok & (x >= lo) & (x <= hi)
        total, total_sq = total + acc, total_sq + acc_sq
        t = t_end
    if T == 0:
        mn = mx = np.full((R, Cc), np.nan if flt else 0, w.dtype)
    elif flt:
        mn, mx = np.fmin.reduce(w, axis=0), np.fmax.reduce(w, axis=0)
    else:
        mn, mx = w.min(axis=0), w.max(axis=0)
    return {"count": count, "n_band": n_band, "min": mn, "max": mx, "sum": total, "sum_sq": total_sq}


def _same(rec, truth):
    rec = rec.reshape(truth["count"].shape)
    for f in ("count", "n_band"):
        assert np.array_equal(rec[f], truth[f]), f
    for f in ("min", "max"):
        assert np.array_equal(rec[f], truth[f].astype(rec.dtype[f]), equal_nan=np.issubdtype(rec.dtype[f], np.floating)), f
    for f in ("sum", "sum_sq"):
        bad = np.flatnonzero(rec[f].ravel().view(np.uint64) != np.ascontiguousarray(truth[f]).ravel().view(np.uint64))
        assert bad.size == 0, (f, bad[:5], rec[f].ravel()[bad[:5]], truth[f].ravel()[bad[:5]])


def _check(sc, values, cubes, chunk_size, lower=None, upper=None):
    recs, off = sc.time_stats_batch(cubes, lower, upper)
    lo = np.broadcast_to(-np.inf if lower is None else lower, len(cubes))
    hi = np.broadcast_to(np.inf if upper is None else upper, len(cubes))
    for i, c in enumerate(cubes):
        s, e = min(c[0], c[1]), max(c[0], c[1])
        _same(recs[int(off[i]):int(off[i + 1])], _truth(values(c), s, chunk_size, lo[i], hi[i]))
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
    recs, off = _check(sc, lambda c: ref.window_f32(*c), cubes, T, -2.0, 4.5)
    nan = recs[int(off[4]):int(off[5])]                                   # all NaN in time
    assert (nan["count"] == 0).all() and np.isnan(nan["min"]).all() and np.isnan(nan["max"]).all() and (nan["sum"] == 0).all()
    const = recs[int(off[5]):int(off[6])]                                 # the constant slot: T times 3.25
    assert (const["sum"] == 3.25 * T).all() and (const["count"] == T).all() and (const["n_band"] == T).all()
    sc.close()


def test_slices_and_windows_starting_inside_a_block(ctx):
    """chunk_size 8: windows crossing slice boundaries that start on Log instants (the snapshot is expanded first)."""
    from dcdf_b200 import Superchunk, synth
    data = synth.raster_slice(0, 40, 130, 200, nan_ocean=True).numpy()
    sc = Superchunk.build(ctx, data, [2, 6], chunk_size=8)
    assert sc.n_slices == 5
    cubes = [[3, 37, 0, 130, 0, 200], [5, 18, 17, 99, 33, 180], [9, 10, 0, 130, 0, 200], [15, 33, 64, 128, 0, 64],
             [1, 40, 129, 130, 199, 200]]
    _check(sc, lambda c: sc.window(*c), cubes, 8, 0.5, 12.0)
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
    _check(sc, lambda c: ref.window_f32(*c), cubes, T, 5.0, 7.5)
    sc.close()


def test_nested_2_4_6_with_an_elided_1024_node(ctx):
    """k2_levels [2, 4, 6] (the C5 layout): the second 1024-wide node of the root is constant, so the root elides it."""
    from dcdf_b200 import Superchunk, synth
    T, R, Cc = 3, 600, 2600
    data = synth.raster_slice(0, T, R, Cc, nan_ocean=True, scale=1.37).numpy()
    data[:, :, 1024:2048] = 2.5
    sc = Superchunk.build(ctx, data, [2, 4, 6])
    kinds, _, _, _ = sc.refs(0)
    assert 0 in set(int(k) for k in kinds)
    cubes = [[0, T, 0, R, 0, Cc], [1, 3, 17, 590, 1000, 2590], [0, T, 100, 200, 1100, 1200]]
    recs, off = _check(sc, lambda c: sc.window(*c), cubes, T)
    assert (recs[int(off[2]):int(off[3])]["sum"] == 2.5 * 3).all()
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
    _check(sc, lambda c: ref.window_f32(*c), [[0, T, 0, R, 0, Cc], [1, 5, 3, 61, 7, 120]], T, 51.0, 60.0)
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
        band = (-3.0, 5.5)
    elif dtype == np.int32:
        data = rng.integers(-5, 6, (T, R, Cc)).astype(dtype)
        data[:, 64:, 64:128] = 0                                          # code 0 is the value 0 for integers
        band = (-2.0, 0.0)
    else:
        data = (rng.integers(-(1 << 20), 1 << 20, (T, R, Cc)) + (1 << 60)).astype(np.int64)   # far beyond 2^53
        data[:, 64:, :64] = (1 << 60) + 3                                 # constant: elided
        band = (float(1 << 60), float((1 << 60) + (1 << 19)))
    sc = Superchunk.build(ctx, data, [1, 6], chunk_size=3)
    cubes = [[0, T, 0, R, 0, Cc], [1, 6, 5, 120, 60, 125], [3, 4, 64, 128, 64, 128], [0, T, 70, 71, 0, 64]]
    recs, _ = _check(sc, lambda c: sc.window(*c), cubes, 3, *band)
    if dtype == np.int64:
        assert recs["max"].max() > (1 << 60) and recs["min"].dtype == np.int64
        assert np.array_equal(recs[:R * Cc]["min"].reshape(R, Cc), data.min(axis=0))   # exact int64
    sc.close()


def _random_cubes(rng, n, T, R, Cc):
    t0 = rng.integers(0, T, n)
    t1 = np.minimum(t0 + rng.integers(1, T + 1, n), T)
    r0, c0 = rng.integers(0, R, n), rng.integers(0, Cc, n)
    r1, c1 = np.minimum(r0 + rng.integers(0, 90, n), R), np.minimum(c0 + rng.integers(0, 90, n), Cc)
    return np.stack([t0, t1, r0, r1, c0, c1], axis=1)


def test_band_counts_match_search_values(ctx):
    from dcdf_b200 import DcdfError, Superchunk
    data = _mixed_bits(T=16)
    T, R, Cc = data.shape
    sc = Superchunk.build(ctx, data, [2, 6], chunk_size=8)
    cubes = _random_cubes(np.random.default_rng(41), 60, T, R, Cc)
    lo, hi = np.linspace(-3.0, 1.0, 60), np.linspace(2.0, 8.0, 60)
    recs, off = sc.time_stats_batch(cubes, lo, hi)
    counts, _ = sc.search_values_batch(cubes, lo, hi, want_cells=False)
    got = np.array([int(recs[int(off[i]):int(off[i + 1])]["n_band"].sum()) for i in range(len(cubes))], np.uint64)
    assert np.array_equal(got, counts)
    rev, _ = sc.time_stats_batch(cubes, hi, lo)                                  # reversed bounds are swapped
    assert rev.tobytes() == recs.tobytes()
    every, _ = sc.time_stats_batch(cubes, -np.inf, np.inf)
    assert np.array_equal(every["n_band"], every["count"])
    plain, _ = sc.time_stats_batch(cubes)                                        # no band: n_band is count
    assert plain.tobytes() == every.tobytes()
    for f in ("count", "min", "max", "sum", "sum_sq"):
        assert np.ascontiguousarray(recs[f]).tobytes() == np.ascontiguousarray(every[f]).tobytes()
    for bad in ((np.nan, 1.0), (0.0, np.nan)):
        with pytest.raises(DcdfError) as e:
            sc.time_stats_batch(cubes[:3], *bad)
        assert e.value.code == 8
    sc.close()


def test_batch_equals_alone_and_repeats_bitwise(ctx):
    from dcdf_b200 import Superchunk
    data = _mixed_bits(T=20)
    T, R, Cc = data.shape
    sc = Superchunk.build(ctx, data, [2, 6], chunk_size=8)
    cubes = _random_cubes(np.random.default_rng(36), 2000, T, R, Cc)
    recs, off = sc.time_stats_batch(cubes, 0.0, 3.0)
    again, off2 = sc.time_stats_batch(cubes, 0.0, 3.0)
    assert recs.tobytes() == again.tobytes() and np.array_equal(off, off2)
    for i in range(0, 2000, 7):
        alone = sc.time_stats(*cubes[i], lower=0.0, upper=3.0)
        assert alone.tobytes() == recs[int(off[i]):int(off[i + 1])].tobytes(), i
    for i in range(0, 2000, 97):
        _same(recs[int(off[i]):int(off[i + 1])], _truth(sc.window(*cubes[i]), cubes[i][0], 8, 0.0, 3.0))
    sc.close()


def test_scratch_groups_do_not_change_results(ctx):
    from dcdf_b200 import Superchunk, synth
    data = synth.raster_slice(0, 48, 150, 200, nan_ocean=True, scale=1.37).numpy()
    sc = Superchunk.build(ctx, data, [2, 6], chunk_size=8)
    cubes = _random_cubes(np.random.default_rng(42), 200, 48, 150, 200)
    cubes[0] = [0, 48, 0, 150, 0, 200]
    recs, _ = sc.time_stats_batch(cubes, 1.0, 9.0)
    assert ctx.get_stat("time_stats_groups") == 1
    try:
        ctx.set_option("time_stats_scratch", 40 * 150 * 200 * 2)                  # about two slices of the full window
        small, _ = sc.time_stats_batch(cubes, 1.0, 9.0)
        assert ctx.get_stat("time_stats_groups") >= 3
        assert ctx.get_stat("time_stats_scratch_bytes") <= 40 * 150 * 200 * 2 + 40 * int(
            ((cubes[:, 3] - cubes[:, 2]) * (cubes[:, 5] - cubes[:, 4])).sum())
        ctx.set_option("time_stats_scratch", 1)                                   # one slice per group
        tiny, _ = sc.time_stats_batch(cubes, 1.0, 9.0)
        assert ctx.get_stat("time_stats_groups") == sc.n_slices
    finally:
        ctx.set_option("time_stats_scratch", 0)
    assert small.tobytes() == recs.tobytes() and tiny.tobytes() == recs.tobytes()
    sc.close()


def test_accumulate_continues_at_a_slice_boundary(ctx):
    from dcdf_b200 import Superchunk, synth
    from dcdf_b200.api import _TIME_FIELDS
    data = synth.raster_slice(0, 40, 130, 200, nan_ocean=True).numpy()
    sc = Superchunk.build(ctx, data, [2, 6], chunk_size=8)
    whole = sc.time_stats(3, 37, 10, 120, 5, 190, lower=2.0, upper=6.0)
    n = whole.size
    cols = {f: np.empty(n, whole.dtype[f]) for f in _TIME_FIELDS}
    off = np.array([0, n], np.uint64)
    for k, (a, b) in enumerate(((3, 16), (16, 37))):
        cube = np.array([[a, b, 10, 120, 5, 190]], np.int64)
        sc._time_stats_into(cube, 2.0, 6.0, cols, off, k > 0)
    for f in _TIME_FIELDS:
        assert cols[f].tobytes() == np.ascontiguousarray(whole[f]).ravel().tobytes(), f
    before = {f: cols[f].copy() for f in _TIME_FIELDS}                          # a zero-instant call leaves them as they are
    sc._time_stats_into(np.array([[20, 20, 10, 120, 5, 190]], np.int64), 2.0, 6.0, cols, off, True)
    for f in _TIME_FIELDS:
        assert cols[f].tobytes() == before[f].tobytes(), f
    sc.close()


def test_wide_expansion_and_reopened_superchunk_are_bitwise_equal(ctx):
    from dcdf_b200 import Superchunk, synth
    data = synth.raster_slice(0, 24, 150, 200, nan_ocean=True, scale=1.37).numpy()
    cubes = _random_cubes(np.random.default_rng(37), 300, 24, 150, 200)
    sc = Superchunk.build(ctx, data, [2, 6], chunk_size=8)
    recs, _ = sc.time_stats_batch(cubes, 2.0, 5.0)
    for opts in OPTIONS.values():                    # the same bytes queried with either expansion
        c2 = _context(opts)
        sc2 = Superchunk.build(c2, data, [2, 6], chunk_size=8)
        assert sc2.time_stats_batch(cubes, 2.0, 5.0)[0].tobytes() == recs.tobytes()
        sc2.close()
        c2.close()
    store, roots = {}, []
    for s in range(sc.n_slices):
        nodes, _ = sc.save(s)
        store.update({cid: b for cid, _, b in nodes})
        roots.append(nodes[-1][0])
    op = Superchunk.open(ctx, roots, store)
    assert op.time_stats_batch(cubes, 2.0, 5.0)[0].tobytes() == recs.tobytes()
    op.close()
    sc.close()


def test_device_outputs_equal_host_outputs(ctx):
    import torch
    from dcdf_b200 import Superchunk, _ffi
    data = _mixed_bits()
    sc = Superchunk.build(ctx, data, [2, 6])
    cubes = np.ascontiguousarray(_random_cubes(np.random.default_rng(38), 50, *data.shape), dtype=np.int64)
    lo, hi = np.full(50, -1.0), np.full(50, 2.5)
    recs, off = sc.time_stats_batch(cubes, lo, hi)
    n = int(off[-1])
    dev = torch.device("cuda", 0)
    count, n_band = torch.empty(n, dtype=torch.int64, device=dev), torch.empty(n, dtype=torch.int64, device=dev)
    vmin, vmax = torch.empty(n, dtype=torch.float32, device=dev), torch.empty(n, dtype=torch.float32, device=dev)
    s, q = torch.empty(n, dtype=torch.float64, device=dev), torch.empty(n, dtype=torch.float64, device=dev)
    torch.cuda.synchronize()
    ptr = lambda t: C.c_void_p(t.data_ptr())
    hp = lambda a: C.c_void_p(a.ctypes.data)
    ctx.check(ctx._lib.dcdf_superchunk_time_stats(ctx._h, sc._h, len(cubes), hp(cubes), hp(off), hp(lo), hp(hi), ptr(count), ptr(n_band),
                                                  ptr(vmin), ptr(vmax), ptr(s), ptr(q), 0, _ffi.MEM_DEVICE))
    for name, t in (("count", count), ("n_band", n_band), ("min", vmin), ("max", vmax), ("sum", s), ("sum_sq", q)):
        assert t.cpu().numpy().tobytes() == np.ascontiguousarray(recs[name]).tobytes(), name
    sc.close()


@pytest.mark.parametrize("cache_bytes", [1 << 30, 1])
def test_variable_time_stats_across_span_groups(ctx, cache_bytes):
    from dcdf_b200 import Superchunk, Variable
    rng = np.random.default_rng(39)
    T, R, Cc = 40, 256, 200
    data = (rng.integers(-800, 800, (T, R, Cc)) / 16.0).astype(np.float32)
    data[:, :64, 64:128] = np.round(data[:, :64, 64:128])
    data[:, 128:192, :64] = np.nan
    data[:, 64:128, 128:192] = 0.0
    v = Variable(ctx, {}, [1, 1, 6], chunk_size=8, span_size=3, cache_bytes=cache_bytes)
    v.append(data)
    sc = Superchunk.build(ctx, data, [1, 1, 6], chunk_size=8)
    for q in ((3, 37, 10, 250, 20, 190), (0, 40, 0, R, 0, Cc), (22, 26, 130, 140, 0, 10)):
        got = v.time_stats(*q, lower=-10.0, upper=10.0)
        assert got.shape == (q[3] - q[2], q[5] - q[4])
        assert got.tobytes() == sc.time_stats(*q, lower=-10.0, upper=10.0).tobytes()
        _same(got, _truth(v.window(*q), q[0], 8, -10.0, 10.0))
    empty = v.time_stats(5, 5, 0, 10, 0, 10)
    assert empty.shape == (10, 10) and (empty["count"] == 0).all() and np.isnan(empty["min"]).all()
    assert empty.tobytes() == sc.time_stats(5, 5, 0, 10, 0, 10).tobytes()
    sc.close()
    v.close()


def test_bounds_and_errors(ctx):
    from dcdf_b200 import DcdfError, Superchunk
    data = _mixed_bits()
    T, R, Cc = data.shape
    sc = Superchunk.build(ctx, data, [2, 6])
    fwd = sc.time_stats(2, 8, 10, 100, 20, 150)
    assert sc.time_stats(8, 2, 100, 10, 150, 20).tobytes() == fwd.tobytes()            # reversed bounds are swapped
    z = sc.time_stats(3, 3, 0, 10, 0, 10)                                             # zero instants: empty records
    assert z.shape == (10, 10) and (z["count"] == 0).all() and (z["n_band"] == 0).all() and np.isnan(z["max"]).all()
    assert (z["sum"] == 0).all() and (z["sum_sq"] == 0).all()
    assert sc.time_stats(1, 5, 30, 30, 0, 50).size == 0                                # zero area: no records
    recs, off = sc.time_stats_batch([[0, 2, 0, 5, 0, 5], [4, 6, 0, 0, 0, 5], [1, 3, 0, 2, 0, 3]])
    assert off.tolist() == [0, 25, 25, 31]
    for bad in ([0, T + 1, 0, 5, 0, 5], [0, 2, 0, R + 1, 0, 5], [0, 2, 0, 5, -1, 5]):
        with pytest.raises(DcdfError) as e:
            sc.time_stats(*bad)
        assert e.value.code == 5
    cubes = np.array([[0, 3, 0, 2, 0, 2]], np.int64)
    outs = [np.empty(4, np.uint64), np.empty(4, np.uint64), np.empty(4, np.float32), np.empty(4, np.float32), np.empty(4), np.empty(4)]
    p = [C.c_void_p(a.ctypes.data) for a in outs]
    hp = lambda a: C.c_void_p(a.ctypes.data)
    lo, hi, nan = np.zeros(1), np.ones(1), np.full(1, np.nan)
    call = lambda off, lo_, hi_, ps: ctx._lib.dcdf_superchunk_time_stats(ctx._h, sc._h, 1, hp(cubes), hp(off), lo_, hi_, *ps, 0, 0)
    good = np.array([0, 4], np.uint64)
    assert call(good, hp(lo), hp(hi), p) == 0
    assert call(np.array([0, 3], np.uint64), hp(lo), hp(hi), p) == 8                # out_off does not match the area
    assert call(good, hp(lo), hp(hi), [p[0], p[1], None, p[3], p[4], p[5]]) == 8    # NULL output
    assert call(good, hp(lo), hp(hi), [p[0], None] + p[2:]) == 8                     # a band needs n_band
    assert call(good, hp(nan), hp(hi), p) == 8                                       # NaN bound
    assert call(good, hp(lo), None, p) == 8                                          # one bound missing
    assert call(good, None, None, [p[0], None] + p[2:]) == 0                         # no band: n_band may be NULL
    sc.close()


def test_slice_longer_than_the_16_bit_counters(ctx):
    """One slice of 70,000 instants: the per-cell counters restart every 65,535 instants and add up in the partials."""
    from dcdf_b200 import Superchunk
    rng = np.random.default_rng(43)
    T, R, Cc = 70000, 6, 8
    data = (rng.integers(-40, 40, (T, R, Cc)) / 4.0).astype(np.float32)
    data[rng.random((T, R, Cc)) < 0.1] = np.nan
    data[:, 0, 0] = 1.5                                                             # never NaN: count T
    sc = Superchunk.build(ctx, data, [1, 2])                                        # 4x4 leaves
    assert sc.n_slices == 1
    got = sc.time_stats(0, T, 0, R, 0, Cc, lower=-1.0, upper=2.0)
    _same(got, _truth(data, 0, T, -1.0, 2.0))
    assert got["count"][0, 0] == T
    sc.close()


def test_two_launches_per_group_and_kernel_time(ctx):
    from dcdf_b200 import Superchunk, _ffi
    data = _mixed_bits(T=24)
    sc = Superchunk.build(ctx, data, [2, 6], chunk_size=8)
    cubes = _random_cubes(np.random.default_rng(40), 100, *data.shape)
    sc.time_stats_batch(cubes)                       # the superchunk's query directory is built on first use
    for budget in (0, 40 * 192 * 192):
        ctx.set_option("time_stats_scratch", budget)
        n0 = ctx.launch_count
        sc.time_stats_batch(cubes, 1.0, 2.0)
        groups = ctx.get_stat("time_stats_groups")
        assert groups >= 1 and ctx.launch_count - n0 == 2 * groups
        assert ctx.last_kernel_ms(_ffi.KT_TIME_STATS) > 0
    ctx.set_option("time_stats_scratch", 0)
    sc.close()
