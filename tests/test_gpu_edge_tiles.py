"""GPU parity tests for the one-warp edge-tile encoder (k_encode_v5_edge, csrc/encode_v5.cuh): clipped fast-path tiles
with at most 32 rows or 32 columns inside the raster, where half of the 64-side tree holds no cell.  The last row or
column of units keeps 1 .. 63 cells; up to 32 they take the edge kernel, from 33 on the two-warp clipped kernel.  Every
chunk and both superchunk DACs are compared with the CPU oracle, bit for bit, with structures staged in shared memory
and emitted straight into the arena."""
import numpy as np
import pytest

from test_gpu_parity import _check_superchunk

pytestmark = pytest.mark.gpu

LEFT = [1, 4, 16, 17, 31, 32, 33, 48, 63]


@pytest.fixture(scope="module", params=["staged", "direct"])
def ctx(request):
    """staged: default; direct: stage_limit = 0 sends every structure straight into the arena."""
    from dcdf_b200 import Context
    c = Context(0)
    if request.param == "direct":
        c.set_option("stage_limit", 0)
    yield c
    c.close()


def _series(rng, rows, cols, T=26):
    """Integer frames (values 4000 .. 9000, so |fixed| stays below 32767 at 4 fractional bits) whose instants give
    Snapshots and Logs: new fields (two-byte entries), whole-field offsets (equal Logs), sparse changes, half the cells
    moved by 300 (the Log does not beat the Snapshot's lower bound: exact Snapshot size), constant blocks, jitter."""
    f = rng.integers(4000, 4300, (rows, cols))
    out = [f]
    for i in range(1, T):
        f = out[-1].copy()
        j = i % 7
        if j == 0:
            f = rng.integers(4000, 9000, (rows, cols))
        elif j == 1:
            f = f + 3
        elif j == 2:
            m = rng.random((rows, cols)) < 0.05
            f[m] += rng.integers(-200, 200, m.sum())
        elif j == 3:
            f[rng.random((rows, cols)) < 0.5] += 300
        elif j == 4:
            f[:rows // 2, :cols // 2] = 4100
        elif j == 5:
            f = f + rng.integers(-2, 3, (rows, cols))
        else:
            f = np.clip(f - 300, 4000, 9000)
        out.append(f)
    return np.stack(out)


def _shape(orient, n):
    return {"bottom": (64 + n, 128), "right": (128, 64 + n), "both": (64 + n, 64 + n)}[orient]


@pytest.mark.parametrize("orient", ["bottom", "right", "both"])
@pytest.mark.parametrize("n", LEFT)
def test_edge_tiles(ctx, orient, n):
    rows, cols = _shape(orient, n)
    rng = np.random.default_rng(1000 * n + len(orient))
    data = (_series(rng, rows, cols) / 16.0).astype(np.float32)
    sc = _check_superchunk(ctx, data, [1, 6])
    edge = ctx.get_stat("encode_units_edge")
    if n <= 32:
        # the two clipped units of the last row / column of units (a corner of n x n cells has a smaller tree)
        assert edge in ((2, 3) if orient == "both" else (2,)), edge
    else:
        assert edge == 0
    assert ctx.get_stat("encode_units_fast") >= 3      # the full tiles and the clipped ones share the fast path
    assert np.array_equal(sc.window(0, data.shape[0], 0, rows, 0, cols), data)
    sc.close()


@pytest.mark.parametrize("rows,cols", [(81, 128), (128, 96), (65, 65), (100, 200)])
def test_edge_tiles_nan_and_time_slices(ctx, rows, cols):
    """NaN cells (code 0), a NaN block, an all-NaN instant, and several time slices of one superchunk."""
    rng = np.random.default_rng(rows * 1000 + cols)
    data = (_series(rng, rows, cols, T=21) / 16.0).astype(np.float32)
    data[rng.random(data.shape) < 0.03] = np.nan
    data[2:5, 3:30, 5:40] = np.nan
    data[9] = np.nan
    levels = [max(1, int(np.ceil(np.log2(max(rows, cols)))) - 6), 6]
    sc = _check_superchunk(ctx, data, levels, chunk_size=8)
    assert ctx.get_stat("encode_units_edge") > 0
    assert np.array_equal(sc.window(0, data.shape[0], 0, rows, 0, cols), data, equal_nan=True)
    sc.close()
