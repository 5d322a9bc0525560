"""Value-range search with bounds in the array's own units (dcdf_superchunk_search_values, Superchunk.search_values_batch):
a cell is a hit iff lower <= (double)value <= upper for the value the window decoder writes, NaN never.  Truth is numpy
over the oracle's decoded window (f32) or the GPU window (f64 / integers, parity-tested elsewhere): counts per window
exactly, cells as sets (lexsorted arrays), under every search path the context options select."""
import os

import numpy as np
import pytest

import oracle_lib as orc

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OPTIONS = {"default": {}, "search_dfs": {"search_dfs": 1}, "search_share_min": {"search_share_min": 1},
           "search_no_cache": {"search_no_cache": 1}}


@pytest.fixture(scope="module", params=list(OPTIONS))
def ctx(request):
    from dcdf_b200 import Context
    c = Context(0)
    for k, v in OPTIONS[request.param].items():
        c.set_option(k, v)
    yield c
    c.close()


def _lex(cells):
    cells = np.asarray(cells, np.int64).reshape(-1, 3)
    return cells[np.lexsort((cells[:, 2], cells[:, 1], cells[:, 0]))]


def _bands(w, rng, n=5):
    """Full range, the NaN-adjacent bands [0, 0] and [-1, 1e-9], reversed bounds, +-inf, single decoded values, bands
    whose edges are decoded values, and bands strictly between two adjacent decoded values (empty)."""
    v = np.unique(w[np.isfinite(w)].astype(np.float64))
    out = [(-np.inf, np.inf), (0.0, 0.0), (-1.0, 1e-9), (v[-1], v[0]), (v[0], v[0]), (v[-1], np.inf), (-np.inf, v[len(v) // 2])]
    for _ in range(n):
        i, j = sorted(int(x) for x in rng.integers(0, len(v), 2))
        out.append((v[i], v[j]))
        out.append((np.nextafter(v[i], np.inf), np.nextafter(v[j], -np.inf)))
        k = int(rng.integers(0, len(v)))
        out.append((v[k], v[k]))
        if k + 1 < len(v):
            out.append((np.nextafter(v[k], np.inf), np.nextafter(v[k + 1], -np.inf)))   # between two neighbours: empty
    return out


def _check(sc, values, cubes, bands):
    """values(cube) -> decoded window (f64); every (cube, band) pair in one batch, counts-only call as well."""
    qc, lo, hi = [], [], []
    for c in cubes:
        for a, b in bands:
            qc.append(c); lo.append(a); hi.append(b)
    counts, cells = sc.search_values_batch(qc, lo, hi)
    only, none = sc.search_values_batch(qc, lo, hi, want_cells=False)
    assert none is None and only.tolist() == counts.tolist()
    assert len(cells) == int(counts.sum())
    pos, wins = 0, {}
    for c, a, b, n in zip(qc, lo, hi, counts.tolist()):
        key = tuple(c)
        if key not in wins:
            wins[key] = values(c).astype(np.float64)
        w = wins[key]
        x, y = min(a, b), max(a, b)
        want = np.argwhere((w >= x) & (w <= y)) + np.array([c[0], c[2], c[4]])
        mine = cells[pos:pos + n]
        pos += n
        assert n == len(want), (c, a, b, n, len(want))
        assert np.array_equal(_lex(mine), _lex(want)), (c, a, b)
    return int(counts.sum())


def _oracle_values(ref):
    return lambda c: ref.window_f32(*c)


def _cubes(T, R, C):
    return [[0, T, 0, R, 0, C], [1, T - 1, 5, R - 7, 3, C - 2], [T // 2, T // 2 + 1, R // 3, R, 0, C // 2 + 5]]


def test_mixed_bits_nan_ocean_and_elided_subchunks(ctx):
    """Subchunks with 0, 4 and 22 fractional bits in one slice, NaN ocean, an all-NaN and a constant (elided) subchunk."""
    from dcdf_b200 import Superchunk
    rng = np.random.default_rng(11)
    T, R, C = 10, 192, 192
    data = np.empty((T, R, C), np.float32)
    data[:, 0:64, 0:64] = rng.integers(-20, 40, (T, 64, 64))                               # 0 bits, integers incl. 0
    data[:, 0:64, 64:128] = rng.integers(-300, 300, (T, 64, 64)) / 16.0                   # 4 bits
    data[:, 0:64, 128:192] = 1.0 + rng.integers(0, 1 << 20, (T, 64, 64)) * 2.0 ** -22     # 22 bits
    data[:, 64:128, 0:64] = np.nan                                                        # elided, all NaN
    data[:, 64:128, 64:128] = 3.25                                                        # elided, constant
    ocean = rng.random((64, 64)) < 0.5
    tile = rng.integers(0, 40, (T, 64, 64)) / 4.0
    tile[:, ocean] = np.nan
    data[:, 64:128, 128:192] = tile
    data[:, 128:, :] = rng.integers(-50, 50, (T, 64, 192)) / 8.0
    sc, ref = Superchunk.build(ctx, data, [2, 6]), orc.superchunk_build(data, [2, 6])
    kinds, _, _, bits = sc.refs(0)
    assert {int(b) for k, b in zip(kinds, bits) if k == 2} >= {0, 4, 22}
    assert 0 in set(int(k) for k in kinds)
    _check(sc, _oracle_values(ref), _cubes(T, R, C), _bands(data, rng) + [(3.25, 3.25), (1.0, 1.0 + 2.0 ** -22)])
    sc.close()


def test_rounded_values_at_the_band_edges(ctx):
    """round=True at 8 bits on un-rounded input: bands whose edges sit within one unit of stored values, so the pruning by
    the node's tables has to keep its margin."""
    from dcdf_b200 import Superchunk
    rng = np.random.default_rng(12)
    T, R, C = 8, 128, 192
    data = (rng.random((T, R, C)) * 10 - 3).astype(np.float32)
    data[:, 64:, :64] = np.nan
    sc = Superchunk.build(ctx, data, [2, 6], fractional_bits=8, round=True)
    ref = orc.superchunk_build(data, [2, 6], fractional_bits=8, round_=True)
    w = ref.window_f32(0, T, 0, R, 0, C).astype(np.float64)
    v = np.unique(w[np.isfinite(w)])
    bands = []
    for x in v[:: max(1, len(v) // 12)]:
        for d in (0.0, 2.0 ** -9, 2.0 ** -8, 1e-7):
            bands += [(x - d, x + d), (x + d, x + 1), (x - 1, x - d)]
    _check(sc, _oracle_values(ref), _cubes(T, R, C), bands)
    sc.close()


@pytest.mark.parametrize("levels", [[1, 1, 6], [1, 1, 1, 5]])
def test_nested_superchunk_with_elided_inner_quadrants(ctx, levels):
    """Nested superchunks: a constant quadrant elided at an inner level, an all-NaN subchunk, mixed bits below."""
    from dcdf_b200 import Superchunk
    rng = np.random.default_rng(13)
    T, R, C = 9, 256, 224
    data = (rng.integers(-400, 400, (T, R, C)) / 16.0).astype(np.float32)
    data[:, 0:128, 128:224] = 7.5                                     # a whole inner node is constant
    data[:, 128:192, 0:64] = np.nan
    data[:, 192:256, 64:128] = rng.integers(-9, 9, (T, 64, 64))       # 0 bits
    data[:, 128:192, 128:192] = (5.0 + rng.integers(0, 1 << 18, (T, 64, 64)) * 2.0 ** -20).astype(np.float32)
    sc, ref = Superchunk.build(ctx, data, levels), orc.superchunk_build(data, levels)
    assert sc.node_count() > 1
    _check(sc, _oracle_values(ref), _cubes(T, R, C), _bands(data, rng) + [(7.5, 7.5), (7.0, 8.0)])
    sc.close()


def _cpc_stack(T=16):
    day = np.load(os.path.join(ROOT, "tests", "golden", "cpc_day_360x720.npz"))["day"]
    out = np.empty((T,) + day.shape, np.float32)
    rng = np.random.default_rng(14)
    for t in range(T):
        f = day * np.float32(1.0 + 0.1 * t)
        for i in range(0, 360, 64):
            for j in range(0, 720, 64):
                u = rng.random()
                if u < 0.25:
                    f[i:i + 64, j:j + 64] = 0.0                        # a dry tile at this instant
                elif u < 0.3:
                    f[i:i + 64, j:j + 64] = np.nan                     # ocean / missing at this instant
        out[t] = f
    return out


def test_cpc_day_with_dry_and_ocean_tiles(ctx):
    """Un-rounded real data (64-bit decode path) whose dry tiles make single-node Logs (SURVEY App. B #15)."""
    from dcdf_b200 import Superchunk
    data = _cpc_stack()
    T, R, C = data.shape
    sc, ref = Superchunk.build(ctx, data, [4, 6]), orc.superchunk_build(data, [4, 6])
    rng = np.random.default_rng(15)
    cubes = [[0, T, 0, R, 0, C], [3, 14, 40, 300, 100, 650]]
    sub = ref.window_f32(0, T, 0, R, 0, C)
    n = _check(sc, _oracle_values(ref), cubes, [(0.0, 0.0), (-1.0, 1e-9), (0.5, 5.0), (10.0, np.inf)] + _bands(sub, rng, 3))
    assert n > 0
    sc.close()


def test_nan_bound_is_rejected(ctx):
    from dcdf_b200 import DcdfError, Superchunk
    data = (np.arange(2 * 64 * 64).reshape(2, 64, 64) / 4.0).astype(np.float32)
    sc = Superchunk.build(ctx, data, [0, 6])
    for lo, hi in ((np.nan, 1.0), (0.0, np.nan)):
        with pytest.raises(DcdfError) as e:
            sc.search_values(0, 2, 0, 64, 0, 64, lo, hi)
        assert e.value.code == 8
    sc.close()


def test_codes_past_2_24_in_f32(ctx):
    """20 fractional bits on values around 50: codes near 2^27, where f32 maps several codes to one float."""
    from dcdf_b200 import Superchunk
    rng = np.random.default_rng(16)
    T, R, C = 6, 64, 128
    data = (50.0 + rng.integers(0, 1 << 22, (T, R, C)) * 2.0 ** -18).astype(np.float32)
    sc = Superchunk.build(ctx, data, [1, 6], fractional_bits=20, compute_bits=False)
    ref = orc.superchunk_build(data, [1, 6], fractional_bits=20, compute_bits=False)
    assert sc.info(0).fractional_bits == 20
    _check(sc, _oracle_values(ref), _cubes(T, R, C), _bands(data, rng, 8))
    sc.close()


@pytest.mark.parametrize("dtype", [np.float64, np.int32, np.int64])
def test_f64_and_integer_variables(ctx, dtype):
    from dcdf_b200 import Superchunk
    rng = np.random.default_rng(17)
    T, R, C = 7, 128, 128
    if dtype == np.float64:
        data = rng.integers(-1000, 1000, (T, R, C)) / 64.0
        data[:, :30, :30] = np.nan
    else:
        data = rng.integers(-5, 6, (T, R, C)).astype(dtype)
        data[:, 64:, 64:] = 0                                           # code 0 is the value 0 for integers
    sc = Superchunk.build(ctx, data, [1, 6])
    bands = _bands(data.astype(np.float64), rng) + [(-0.5, 0.5), (0.0, 0.0), (-2.5, 1.5)]
    _check(sc, lambda c: sc.window(*c), _cubes(T, R, C), bands)
    sc.close()


def test_order_equals_search_batch_on_uniform_bits(ctx):
    """A uniform-bit slice without single-node Logs and a band that excludes code 0: the strict search is array-equal to
    the fixed-bound search with the converted bounds."""
    from dcdf_b200 import Superchunk
    rng = np.random.default_rng(18)
    T, R, C = 9, 128, 192
    data = (rng.integers(1, 4000, (T, R, C)) / 16.0).astype(np.float32)
    data[:, :, :] += (rng.integers(0, 2, (T, R, C)) * 2 + 1) / 16.0          # every cell odd in 1/16: 4 bits everywhere
    sc = Superchunk.build(ctx, data, [2, 6])
    kinds, _, _, bits = sc.refs(0)
    assert {int(b) for k, b in zip(kinds, bits) if k == 2} == {4} and sc.info(0).fractional_bits == 4
    cubes = _cubes(T, R, C)
    for lo, hi in ((1.0, 100.0), (30.0, 30.0625), (0.01, 300.0), (200.0, 120.5)):
        a, b = min(lo, hi), max(lo, hi)
        fl, fh = 2 * int(np.ceil(a * 16)) + 1, 2 * int(np.floor(b * 16)) + 1
        c1, x1 = sc.search_values_batch(cubes, lo, hi)
        c2, x2 = sc.search_batch(cubes, fl, fh)
        assert c1.tolist() == c2.tolist() and np.array_equal(x1, x2), (lo, hi)
    sc.close()


def _single_node_log_frames():
    import fixtures as fx
    a = fx.array8_3()
    frames = [a[0], np.full((8, 8), 5, np.int64), a[0] + 3, a[0] - 2, np.full((8, 8), -4, np.int64), a[1], np.full((8, 8), 9, np.int64), a[1] + 1]
    data = np.stack([np.tile(f, (2, 2)) for f in frames])
    data[:, 8:, 8:] += 1
    return data, range(-8, 14, 2), (0, 1, 3, 20)


def _single_node_snapshot_frames():
    import fixtures as fx
    a = fx.array8_3()
    frames = [np.full((8, 8), -13, np.int64), a[0] - 40, a[0] - 41, a[1] - 40, np.full((8, 8), 7, np.int64), a[0] - 39, a[1] + 50, a[0] - 40]
    data = np.stack([np.tile(f, (2, 2)) for f in frames])
    data[:, 8:, :8] -= 3
    return data, range(-60, 70, 5), (0, 4, 12, 200)


@pytest.mark.parametrize("shape", ["single_node_logs", "logs_over_single_node_snapshot"])
@pytest.mark.parametrize("kind", ["int64", "f32"])
def test_strict_where_the_reference_traversal_is_wrong(ctx, shape, kind):
    """SURVEY App. B #15: on these shapes search_batch returns the reference's set, which is not the set of cells in the
    band for some bands; search_values returns the true set."""
    from dcdf_b200 import Superchunk
    data, los, widths = (_single_node_log_frames if shape == "single_node_logs" else _single_node_snapshot_frames)()
    T = len(data)
    if kind == "f32":
        data = (data / 8.0).astype(np.float32)
        scale = 8.0
    else:
        scale = 1.0
    sc = Superchunk.build(ctx, data, [1, 3])
    rng = np.random.default_rng(19)
    cubes, lo, hi = [], [], []
    for x in los:
        for wd in widths:
            t0 = int(rng.integers(0, T - 1))
            r0, c0 = int(rng.integers(0, 14)), int(rng.integers(0, 14))
            cubes.append([t0, int(rng.integers(t0 + 1, T + 1)), r0, int(rng.integers(r0 + 1, 17)), c0, int(rng.integers(c0 + 1, 17))])
            lo.append(x / scale); hi.append((x + wd) / scale)
    cubes.append([0, T, 0, 16, 0, 16]); lo.append(-np.inf); hi.append(np.inf)
    cubes.append([0, T, 0, 16, 0, 16]); lo.append(-30 / scale); hi.append(1000 / scale)
    cubes.append([0, T, 0, 16, 0, 16]); lo.append(-1000 / scale); hi.append(-36 / scale)    # everything below a bound
    counts, cells = sc.search_values_batch(cubes, lo, hi)
    pos, wrong = 0, 0
    bits = sc.info(0).fractional_bits
    for c, a, b, n in zip(cubes, lo, hi, counts.tolist()):
        w = data[c[0]:c[1], c[2]:c[3], c[4]:c[5]].astype(np.float64)
        want = np.argwhere((w >= a) & (w <= b)) + np.array([c[0], c[2], c[4]])
        assert np.array_equal(_lex(cells[pos:pos + n]), _lex(want)), (c, a, b)
        pos += n
        if kind == "int64":
            fl, fh = int(np.ceil(a)) if np.isfinite(a) else -(1 << 62), int(np.floor(b)) if np.isfinite(b) else 1 << 62
        else:
            fl = 2 * int(np.ceil(a * 2 ** bits)) + 1 if np.isfinite(a) else 1
            fh = 2 * int(np.floor(b * 2 ** bits)) + 1 if np.isfinite(b) else 1 << 62
        ref_cells = sc.search(*c, fl, fh)
        wrong += not np.array_equal(_lex(ref_cells), _lex(want))
    if not (kind == "int64" and shape == "logs_over_single_node_snapshot"):
        # (the int64 build of that shape: the fixed-bound search's sets happen to be the true ones for these bands)
        assert wrong > 0, "the fixed-bound search should reproduce the reference's wrong set on some band"
    sc.close()


def test_variable_search_runs_on_the_device(ctx, monkeypatch):
    """Variable.search over a nested, mixed-bit variable across two span groups equals numpy and never decodes a window."""
    from dcdf_b200 import Superchunk, Variable
    rng = np.random.default_rng(20)
    T, R, C = 40, 256, 200
    data = (rng.integers(-800, 800, (T, R, C)) / 16.0).astype(np.float32)
    data[:, :64, 64:128] = np.round(data[:, :64, 64:128])              # 0 bits
    data[:, 128:192, :64] = np.nan
    data[:, 64:128, 128:192] = 0.0
    v = Variable(ctx, {}, [1, 1, 6], chunk_size=8, span_size=3)
    v.append(data)

    def no_window(*a, **k):
        raise AssertionError("Variable.search decoded a window")
    monkeypatch.setattr(Superchunk, "window", no_window)
    for lo, hi in ((1.0, 2.5), (-1.0, 0.0), (0.0, 0.0), (5.0, -3.0), (-np.inf, np.inf), (0.3, 0.31)):
        got = v.search(3, 37, 10, 250, 20, 190, lo, hi)
        a, b = min(lo, hi), max(lo, hi)
        w = data[3:37, 10:250, 20:190].astype(np.float64)
        want = np.argwhere((w >= a) & (w <= b)) + np.array([3, 10, 20])
        assert np.array_equal(_lex(got), _lex(want)), (lo, hi)
    v.close()
