"""The limits of the fast encoder's 16-bit cell codes (csrc/encode_v5.cuh: full tiles hold each cell as its fixed code
minus the unit's smallest one, two cells per 32-bit word).  Units built to sit exactly on those limits -- codes spanning
32767, a minimum near -2^22, Log differences of +-32767, NaN cells (code 0) next to cells outside the raster -- go
through the fast path and must match the CPU oracle byte for byte."""
import numpy as np
import pytest

from test_gpu_parity import _check_superchunk

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module", params=["staged", "direct"])
def ctx(request):
    """staged: default; direct: every structure straight into the arena."""
    from dcdf_b200 import Context
    c = Context(0)
    if request.param == "direct":
        c.set_option("stage_limit", 0)
    yield c
    c.close()


def _span_tile(rng, T):
    """Integer values 0..16383 (codes 1..32767) and NaN cells (code 0): the codes span exactly 32767.  Cells jump
    between NaN and 16383 (Log differences of +-32767) and between 0 and 16383 (+-32766)."""
    f = rng.integers(0, 16384, (T, 64, 64)).astype(np.float32)
    f[:, :8, :8] = rng.integers(8000, 8010, (T, 8, 8))               # mostly one-byte entries elsewhere ...
    f[:, 8:, :] = f[0, 8:, :]                                         # ... and an unchanged bottom part
    for t in range(T):
        f[t, 20 + t % 3, 5] = np.nan if t % 2 == 0 else 16383.0     # +-32767
        f[t, 30, 7 + t % 2] = 0.0 if t % 2 == 0 else 16383.0        # +-32766
        f[t, 40:44, 40:44] = np.nan if t % 3 == 0 else 16383.0      # a whole level-4 node jumping by 32767
    f[:, 60, 60] = 0.0
    f[:, 61, 61] = 16383.0
    return f


def _low_tile(rng, T):
    """The smallest fixed code the fast path takes, -2^22 + 3, with codes spanning 32766 above it."""
    lo = -2097151.0
    f = lo + rng.integers(0, 16384, (T, 64, 64)).astype(np.float64)
    f[:, 32:, :] = lo + 50 + rng.integers(-3, 4, (T, 32, 64))
    f[:, 0, 0] = lo
    f[:, 0, 1] = lo + 16383
    return f.astype(np.float32)


def test_packed_codes_at_their_limits(ctx):
    rng = np.random.default_rng(0x16)
    T = 9
    data = np.concatenate([_span_tile(rng, T), _low_tile(rng, T)], axis=2)     # [T, 64, 128]: two full tiles
    assert np.nanmin(data[:, :, 64:]) == -2097151.0
    sc = _check_superchunk(ctx, data, [1, 6])
    assert ctx.get_stat("encode_units_fast") == 2                               # both tiles took the fast path
    assert np.array_equal(sc.window(0, T, 0, 64, 0, 128), data, equal_nan=True)
    sc.close()


def test_packed_clipped_tiles_nan_next_to_none(ctx):
    """A 90x120 raster: one full tile, a clipped tile of 56 columns and two of 26 rows (one-warp tiles).  NaN cells
    (code 0) line the raster's last row and column, next to the cells outside it (None); each clipped unit's codes reach
    within a few units of -32767 or 32767, and one cell jumps between NaN and 16383 (Log differences of +-32767)."""
    rng = np.random.default_rng(0x17)
    T = 8
    data = np.empty((T, 90, 120), np.float32)
    data[:, :64, :64] = rng.integers(0, 2000, (T, 64, 64))
    data[:, :64, 64:] = rng.integers(-16383, -16383 + 2000, (T, 64, 56))        # codes -32765 .. -28767, and 0
    data[:, 64:, :] = rng.integers(16383 - 2000, 16384, (T, 26, 120))           # codes 28767 .. 32767, and 0
    data[:, 89, :] = np.nan
    data[:, :, 119] = np.nan
    data[0::2, 88, 118] = np.nan
    data[1::2, 88, 118] = 16383.0
    sc = _check_superchunk(ctx, data, [1, 6])
    assert ctx.get_stat("encode_units_fast") == 4
    assert np.array_equal(sc.window(0, T, 0, 90, 0, 120), data, equal_nan=True)
    sc.close()
