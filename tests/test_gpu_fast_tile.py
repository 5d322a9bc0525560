"""GPU parity tests aimed at the fast-path encoder (csrc/encode_v5.cuh): full 64x64 f32 tiles inside a Superchunk
whose to_fixed is exact, without NaN, fixed values within 32767 of each other.  Uniform / equal sub-trees at every
level, one- and two-byte entries on both candidates, the heuristic mix, the 254-log cap, both emission paths
(shared-memory image and straight into the arena), and tiles that must NOT take the fast path.  Every chunk and
both superchunk DACs are compared with the CPU oracle, bit for bit."""
import numpy as np
import pytest

import oracle_lib as orc
from test_gpu_parity import _check_superchunk

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module", params=["staged", "direct", "general"])
def ctx(request):
    """staged: default; direct: stage_limit = 0 sends every structure straight into the arena; general: the same
    inputs through the general encoder (no_fast_encode), which must give the same bytes."""
    from dcdf_b200 import Context
    c = Context(0)
    if request.param == "direct":
        c.set_option("stage_limit", 0)
    if request.param == "general":
        c.set_option("no_fast_encode", 1)
    c.general = request.param == "general"
    yield c
    c.close()


def test_removed_encoder_options_are_refused():
    """fast_variant, fast_sync_mask and encode_tiles256 select no encoder path: set_option refuses them like any unknown
    name."""
    from dcdf_b200 import Context, DcdfError
    c = Context(0)
    try:
        for name in ("fast_variant", "fast_sync_mask", "encode_tiles256"):
            with pytest.raises(DcdfError, match=f"BAD_ARG: unknown option {name}"):
                c.set_option(name, 1)
    finally:
        c.close()


def _tiles(frames, bits=4, offset=0.0):
    """[T, 64, 64] integer frames -> [T, 128, 128] f32 raster of four full tiles: the frames, a shifted copy, a
    transposed copy and a time-reversed copy, as multiples of 2^-bits."""
    f = np.asarray(frames, dtype=np.int64)
    T = f.shape[0]
    out = np.zeros((T, 128, 128), np.int64)
    out[:, :64, :64] = f
    out[:, :64, 64:] = f + 17
    out[:, 64:, :64] = f.transpose(0, 2, 1)
    out[:, 64:, 64:] = f[::-1]
    return (out.astype(np.float64) / float(1 << bits) + offset).astype(np.float32)


def _frames(rng, kind, T=12):
    base = rng.integers(0, 50, (64, 64)) + 4000
    out = [base]
    for i in range(1, T):
        f = out[-1].copy()
        if kind == "sparse":            # a few cells change: logs with mostly equal quads
            m = rng.random((64, 64)) < 0.03
            f[m] += rng.integers(-3, 4, m.sum())
        elif kind == "offset":          # whole-field offsets: single-node equal logs
            f = f + int(rng.integers(-5, 6))
        elif kind == "blocks":          # changes confined to one quadrant / 16x16 / 8x8 / 4x4 / 2x2 block
            s = [32, 16, 8, 4, 2][i % 5]
            r, c = rng.integers(0, 64 // s, 2) * s
            f[r:r + s, c:c + s] += rng.integers(-100, 100, (s, s))
        elif kind == "two":             # two-byte entries on leaves, quads and upper levels
            f = 4000 + rng.integers(0, 9000, (64, 64))
        elif kind == "two_sparse":      # a few two-byte entries among one-byte ones
            m = rng.random((64, 64)) < 0.02
            f[m] += rng.integers(-3000, 3000, m.sum())
            f = np.clip(f, 0, 12000)
        elif kind == "dense":           # every cell jitters
            f = f + rng.integers(-2, 3, (64, 64))
        elif kind == "mixed":
            j = i % 6
            if j == 0:
                f = 4000 + rng.integers(0, 3000, (64, 64))
            elif j == 1:
                f = f + 7
            elif j == 2:
                f[:32, :32] = 4005
            elif j == 3:
                f[rng.random((64, 64)) < 0.5] += 300
            elif j == 4:
                f[10:12, 20:22] -= 1000
            else:
                f = f * 0 + 4009
        out.append(f)
    return np.stack(out)


KINDS = ["sparse", "offset", "blocks", "two", "two_sparse", "dense", "mixed"]


@pytest.mark.parametrize("kind", KINDS)
def test_fast_tiles(ctx, kind):
    rng = np.random.default_rng(KINDS.index(kind) + 50)
    data = _tiles(_frames(rng, kind))
    sc = _check_superchunk(ctx, data, [1, 6])
    assert ctx.get_stat("encode_units_fast") == (0 if ctx.general else 4)      # the kernel under test really ran
    assert np.array_equal(sc.window(0, data.shape[0], 0, 128, 0, 128), data)
    sc.close()


def test_fast_tiles_uniform_levels(ctx):
    """Uniform and equal sub-trees at every level of the quadtree, including the root."""
    rng = np.random.default_rng(61)
    frames = []
    for s in [64, 32, 16, 8, 4, 2, 1]:
        f = np.repeat(np.repeat(rng.integers(0, 1000, (64 // s, 64 // s)), s, 0), s, 1)
        frames.append(f)
        frames.append(f + 3)                 # equal at the root
        g = f.copy()
        g[:s, :s] += 1                       # equal everywhere but one node
        frames.append(g)
    _check_superchunk(ctx, _tiles(frames), [1, 6]).close()


def test_fast_tiles_negative_values_and_time_slices(ctx):
    rng = np.random.default_rng(62)
    frames = _frames(rng, "sparse", T=23) - 9000              # fixed values around -10000 .. -8000
    data = _tiles(frames, bits=3)
    _check_superchunk(ctx, data, [1, 6], chunk_size=8).close()
    data = _tiles(_frames(rng, "mixed", T=9), bits=0, offset=-4100.0)     # integers, both signs
    _check_superchunk(ctx, data, [1, 6]).close()


def test_fast_tiles_log_cap(ctx):
    """254 Logs per Block (chunk.rs:62): 300 identical instants give blocks of 255 and 45."""
    rng = np.random.default_rng(63)
    f = rng.integers(0, 50, (64, 64)) + 100
    data = _tiles(np.stack([f] * 300))
    sc = _check_superchunk(ctx, data, [1, 6])
    info = sc.info(0)
    assert info.stats.snapshots == 2 * 4 and info.stats.logs == 298 * 4
    sc.close()


def test_tiles_that_must_not_take_the_fast_path(ctx):
    """A value range above 32767 fixed units, values above 2^22, data that needs rounding: each disqualifies only its
    own tile; the neighbours (one of them with NaN cells, which the fast path handles) still go through the fast path
    and everything must stay exact."""
    rng = np.random.default_rng(64)
    data = _tiles(_frames(rng, "dense", T=8))
    data[3, 5, 70] = np.nan                                    # tile (0, 1): NaN (code 0 stays within 32767 of the values)
    data[:, 64:, :64] += np.float32(3000.0)                    # tile (1, 0): range 3000 * 32 > 32767 against ...
    data[2, 64:, :64] -= np.float32(3000.0)                    # ... one instant back at the old level
    data[:, 64:, 64:] += np.float32(200000.0)                  # tile (1, 1): fixed values above 2^22
    _check_superchunk(ctx, data, [1, 6]).close()
    assert ctx.get_stat("encode_units_fast") == (0 if ctx.general else 2) and ctx.get_stat("encode_units_general") == (4 if ctx.general else 2)
    noisy = _tiles(_frames(rng, "sparse", T=6)) * np.float32(0.3)   # full mantissas: Round without rounding fails ...
    _check_superchunk(ctx, noisy, [1, 6], fractional_bits=5, round_=True).close()   # ... with it, to_fixed rounds (not exact)


def test_fast_path_strided_device_input(ctx):
    """Device-resident views: rows 16-byte aligned (128-bit loads) and not (32-bit loads)."""
    import torch
    from dcdf_b200 import Superchunk
    rng = np.random.default_rng(65)
    data = _tiles(_frames(rng, "blocks", T=7))
    big = torch.zeros((7, 136, 140), dtype=torch.float32, device="cuda")
    for r0, c0 in ((4, 8), (3, 5)):
        big[:, r0:r0 + 128, c0:c0 + 128] = torch.from_numpy(data).cuda()
        view = big[:, r0:r0 + 128, c0:c0 + 128]
        sc = Superchunk.build(ctx, view, [1, 6])
        ref = orc.superchunk_build(data, [1, 6])
        kinds, child = ref.node_refs(0)
        chunks = sc.chunk_bytes(0)
        for slot, c in enumerate(child):
            assert chunks[slot] == ref.node_bytes(int(c)), (r0, c0, slot)
        sc.close()


@pytest.mark.parametrize("rows,cols", [(150, 200), (129, 191), (190, 130), (64, 100), (100, 64)])
def test_fast_clipped_tiles_and_nan(ctx, rows, cols):
    """Clipped tiles that keep a 64-side tree (cells outside the raster are None) and NaN cells (code 0) through the fast
    path: temperature-like values (|fixed| <= 32767 so that an entry next to a None cell still fits two bytes), NaN
    sprinkled, NaN blocks, an all-NaN instant, whole-field offsets, sparse changes."""
    rng = np.random.default_rng(rows * 1000 + cols)
    base = rng.integers(4000, 4300, (rows, cols))
    frames = [base]
    for i in range(1, 11):
        f = frames[-1].copy()
        if i % 5 == 0:
            f = rng.integers(4000, 9000, (rows, cols))
        elif i % 5 == 1:
            f = f + 3
        else:
            m = rng.random((rows, cols)) < 0.05
            f[m] += rng.integers(-200, 200, m.sum())
        frames.append(f)
    data = (np.stack(frames) / 16.0).astype(np.float32)
    levels = [max(1, int(np.ceil(np.log2(max(rows, cols)))) - 6), 6]
    sc = _check_superchunk(ctx, data, levels)
    n_fast = ctx.get_stat("encode_units_fast")
    if not ctx.general:                                                    # 191 columns: rows not 16-byte aligned -> 32-bit loads
        assert n_fast >= ((rows + 63) // 64) * ((cols + 63) // 64) - 1       # all but (at most) a corner tile with a smaller tree
    assert np.array_equal(sc.window(0, 11, 0, rows, 0, cols), data)
    sc.close()
    nan = data.copy()
    nan[rng.random(nan.shape) < 0.03] = np.nan
    nan[2:5, 10:40, 20:90] = np.nan
    nan[7] = np.nan
    sc = _check_superchunk(ctx, nan, levels)
    if not ctx.general:
        assert ctx.get_stat("encode_units_fast") == n_fast
    assert np.array_equal(sc.window(0, 11, 0, rows, 0, cols), nan, equal_nan=True)
    sc.close()


def test_fast_nan_ocean_precipitation_like(ctx):
    """configs[2]'s shape of data: clamped at 0, 60 % NaN in 16x16 blocks -- fast path with NaN codes and many uniform /
    equal sub-trees."""
    from dcdf_b200 import synth
    data = synth.raster_slice(0, 20, 200, 260, hourly=False, nan_ocean=True).numpy()
    sc = _check_superchunk(ctx, data, [3, 6], chunk_size=8)
    assert ctx.general or ctx.get_stat("encode_units_fast") > 0
    sc.close()
