"""GPU parity tests for the fast-path encoder's Log / Snapshot decision (csrc/encode_v5.cuh): the fused pass sizes both
candidates exactly and picks the smaller one, ties going to the Snapshot (chunk.rs:62).  Exact size ties (found with the
CPU oracle), a Snapshot at every instant, Snapshots whose level-5/6 entries take two bytes, clipped tiles of both
fast-path lists, NaN cells, and the 254-log cap.  Every chunk and both superchunk DACs are compared with the CPU oracle,
bit for bit, with structures staged in shared memory and emitted straight into the arena."""
import numpy as np
import pytest

import oracle_lib as orc
from test_gpu_parity import _check_superchunk

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module", params=["staged", "direct"])
def ctx(request):
    """staged: default; direct: stage_limit = 0 sends every structure straight into the arena."""
    from dcdf_b200 import Context
    c = Context(0)
    if request.param == "direct":
        c.set_option("stage_limit", 0)
    yield c
    c.close()


def _fixed(n):
    """to_fixed of integer-valued cells at 0 fractional bits (what compute_bits picks for them): 2n + 1."""
    return 2 * np.asarray(n, np.int64) + 1


def _sizes(image, t):
    """Serialized sizes of the Snapshot of frame t and of its Log against the snapshot image."""
    return len(orc.snapshot_build(_fixed(t)).serialize()), len(orc.log_build(_fixed(image), _fixed(t)).serialize())


def _tie(rng, image, spread):
    """A 64x64 frame whose Snapshot and Log (against `image`) have the same size: the first m cells of a random order
    are set to one constant.  The Log grows with m until the frame is nearly uniform, where the Snapshot shrinks below
    it; m is bisected to where the Log stops being the smaller one, then searched downwards for an exact tie."""
    for _ in range(200):
        order = rng.permutation(4096)
        c = int(image.min()) + int(rng.integers(-spread // 4, spread + spread // 4))

        def frame(m):
            t = image.copy().ravel()
            t[order[:m]] = c
            return t.reshape(64, 64)

        def excess(m):
            s, lg = _sizes(image, frame(m))
            return lg - s

        hi = next((m for m in range(256, 4096, 256) if excess(m) > 0), None)
        if hi is None:
            continue
        lo = hi - 256
        while hi - lo > 1:
            mid = (lo + hi) // 2
            if excess(mid) <= 0:
                lo = mid
            else:
                hi = mid
        for m in range(lo, max(0, lo - 40), -1):
            if excess(m) == 0:
                return frame(m)
    raise AssertionError("no Log / Snapshot size tie found")


def _tiles(frames):
    """[T, 64, 64] frames -> [T, 128, 128] f32 raster of four full tiles holding the same frames."""
    f = np.asarray(frames, np.float32)
    return np.tile(f, (1, 2, 2))


@pytest.mark.parametrize("spread", [40, 400])
def test_exact_size_ties(ctx, spread):
    """Instants whose Log and Snapshot are exactly as large become Snapshots.  spread 400 (800 fixed units): most
    level-4 nodes span more than 127, so the Snapshot's leaf and quad entries take two bytes in places."""
    rng = np.random.default_rng(spread)
    image = rng.integers(4000, 4000 + spread, (64, 64))
    frames = [image]
    ties = []
    for _ in range(3):
        t = _tie(rng, image, spread)
        s, lg = _sizes(image, t)
        assert s == lg
        ties.append(len(frames))
        frames.append(t)
        image = t                                    # the tie is a Snapshot: the next Logs refer to it
        nxt = t.copy()
        nxt[rng.random((64, 64)) < 0.02] += 1        # a Log in between
        frames.append(nxt)
    data = _tiles(frames)
    sc = _check_superchunk(ctx, data, [1, 6])
    assert ctx.get_stat("encode_units_fast") == 4 and ctx.get_stat("encode_units_edge") == 0
    assert sc.info(0).stats.snapshots == 4 * (1 + len(ties))
    assert np.array_equal(sc.window(0, data.shape[0], 0, 128, 0, 128), data)
    sc.close()


def test_snapshot_every_instant(ctx):
    """Jumps far larger than the field's own variation: every instant is a Snapshot."""
    rng = np.random.default_rng(71)
    frames = [rng.integers(0, 40, (64, 64)) + 1000 * (i % 2) * (3 + i % 5) for i in range(12)]
    data = _tiles(frames)
    sc = _check_superchunk(ctx, data, [1, 6])
    assert ctx.get_stat("encode_units_fast") == 4
    assert sc.info(0).stats.snapshots == 4 * 12 and sc.info(0).stats.logs == 0
    sc.close()


def test_two_byte_snapshot_entries(ctx):
    """Snapshots whose level-6 / level-5 entries take two bytes (level-4 nodes with a range above 127 fixed units),
    next to nodes that stay within one byte, with Logs that come close to the Snapshot's size."""
    rng = np.random.default_rng(72)
    frames = []
    f = rng.integers(4000, 4030, (64, 64))
    for i in range(16):
        f = f.copy()
        j = i % 4
        if j == 0:                                   # wide nodes in one quadrant, a single wide cell elsewhere
            f = rng.integers(4000, 4030, (64, 64))
            f[:32, 32:] = rng.integers(4000, 4000 + 60 * (1 + i), (32, 32))
            f[40, 9] += 70 + 30 * i
        elif j == 1:                                 # a few cells move by more than a byte
            m = rng.random((64, 64)) < 0.04
            f[m] += rng.integers(-900, 900, m.sum())
        elif j == 2:                                 # half the cells jump: close to the Snapshot's size
            f[rng.random((64, 64)) < 0.5] += 90
        else:
            f = f + 1
        frames.append(f)
    data = _tiles(frames)
    sc = _check_superchunk(ctx, data, [1, 6])
    assert ctx.get_stat("encode_units_fast") == 4
    assert np.array_equal(sc.window(0, data.shape[0], 0, 128, 0, 128), data)
    sc.close()


def _series(rng, rows, cols, T=24):
    """Integer frames (|2n + 1| well below 32767, so an entry next to a cell outside the raster fits two bytes) with
    new fields, wide fields, close calls, sparse changes, constant blocks and offsets."""
    f = rng.integers(2000, 2030, (rows, cols))
    out = [f]
    for i in range(1, T):
        f = out[-1].copy()
        j = i % 6
        if j == 0:
            f = rng.integers(2000, 4500, (rows, cols))
        elif j == 1:
            f = rng.integers(2000, 2040, (rows, cols))
        elif j == 2:
            f[rng.random((rows, cols)) < 0.5] += 90
        elif j == 3:
            m = rng.random((rows, cols)) < 0.05
            f[m] += rng.integers(-300, 300, m.sum())
        elif j == 4:
            f[:rows // 2, :cols // 3] = 2100
        else:
            f = f + 2
        out.append(f)
    return np.stack(out)


# (81, 90): the 17 x 26 corner unit has a tree smaller than 64 x 64 and takes the general encoder
@pytest.mark.parametrize("rows,cols,n_fast,edge", [(104, 100, 4, False), (81, 90, 3, True), (128, 83, 4, True), (113, 117, 4, False)])
def test_clipped_tiles_and_nan(ctx, rows, cols, n_fast, edge):
    """Clipped fast-path tiles with more than 32 rows and columns in the raster (two warps, list 6) and with at most 32
    (one warp, list 7); row and column counts that cut level-4 nodes; then the same with NaN cells."""
    rng = np.random.default_rng(rows * 1000 + cols)
    data = _series(rng, rows, cols).astype(np.float32)
    sc = _check_superchunk(ctx, data, [1, 6])
    assert ctx.get_stat("encode_units_fast") == n_fast
    assert (ctx.get_stat("encode_units_edge") > 0) == edge
    assert np.array_equal(sc.window(0, data.shape[0], 0, rows, 0, cols), data)
    sc.close()
    nan = data.copy()
    nan[rng.random(nan.shape) < 0.03] = np.nan
    nan[3:6, 10:30, 20:60] = np.nan
    nan[9] = np.nan
    sc = _check_superchunk(ctx, nan, [1, 6])
    assert ctx.get_stat("encode_units_fast") == n_fast
    assert np.array_equal(sc.window(0, nan.shape[0], 0, rows, 0, cols), nan, equal_nan=True)
    sc.close()


def test_log_cap_with_decisions(ctx):
    """More than 255 instants of slowly changing 64x64 frames: Logs win, the 254-log cap forces Snapshots, and a jump
    starts a block of its own (the cap counts from there)."""
    rng = np.random.default_rng(73)
    f = rng.integers(3000, 3040, (64, 64))
    frames = []
    for i in range(300):
        f = f.copy()
        if i == 20:
            f = rng.integers(6000, 6300, (64, 64))
        else:
            m = rng.random((64, 64)) < 0.01
            f[m] += rng.integers(-2, 3, m.sum())
        frames.append(f)
    data = _tiles(frames)
    sc = _check_superchunk(ctx, data, [1, 6])
    assert ctx.get_stat("encode_units_fast") == 4
    info = sc.info(0)
    assert info.stats.snapshots == 3 * 4 and info.stats.logs == 297 * 4   # instants 0, 20 and 275
    sc.close()
