"""Host-side mirror of the reference's interface for the hot path, over the C-ABI.

Names and argument meaning follow the reference (paths relative to dcdf/src):
  Chunk.build / get / fill_cell / fill_window / iter_search / write_to / read_from   chunk.rs:42-278
  Superchunk.build / get / fill_cell / fill_window / search                          superchunk.rs:88-585
  Superchunk.search_values (float bounds; mmarray.rs:407-417 is todo!() upstream)
  Superchunk.window_stats (per-instant count / min / max / sum / sum_sq of windows; no reference counterpart)
  Superchunk.time_stats (per-cell count / n_band / min / max / sum / sum_sq over time; no reference counterpart)
  MMArray3.{shape,get,cell,window,search}                                            mmarray.rs:135-536,
                                                                py-dcdf/src/lib.rs:411-581 (PyMMArray3*)
  to_fixed / from_fixed / suggest_fraction                                           fixed.rs:31-159
Data errors that are panics in the reference raise DcdfError here (code = C-ABI status).
Inputs may be numpy arrays (host) or torch CUDA tensors (device, zero-copy).
"""
import ctypes as C

import numpy as np

from . import _ffi
from ._ffi import (ENC_F32, ENC_F64, ENC_I32, ENC_I64, MEM_DEVICE, MEM_HOST, Array3, BuildStats, Cube, SuperchunkInfo)

_ENC_OF_DTYPE = {"int32": ENC_I32, "int64": ENC_I64, "float32": ENC_F32, "float64": ENC_F64}
_DTYPE_OF_ENC = {ENC_I32: np.int32, ENC_I64: np.int64, ENC_F32: np.float32, ENC_F64: np.float64}


class DcdfError(Exception):
    def __init__(self, code, msg):
        super().__init__(f"{_ffi.ERR_NAMES.get(code, code)}: {msg}")
        self.code = code


def _is_torch(a):
    return hasattr(a, "data_ptr") and hasattr(a, "is_cuda")


def _order_after_torch(ctx, t):
    """A Context runs on its own stream: before the library touches a CUDA tensor, wait for the work torch has queued
    on that device's current stream (a producer kernel may still be writing it) -- unless the context was told to use
    that very stream (Context.set_stream).  Calls return after the context's stream has drained, so torch may consume
    outputs right away."""
    if not t.is_cuda:
        return
    import torch
    if ctx is not None and t.device.index != ctx.device:
        raise ValueError(f"tensor lives on cuda:{t.device.index}, the context on cuda:{ctx.device}")
    cur = torch.cuda.current_stream(t.device)
    if ctx is None or ctx._stream_ptr != cur.cuda_stream:
        cur.synchronize()


def _check_out(out, n, enc, raw):
    """`out` must be a contiguous buffer of exactly the element type and at least the size the C call writes."""
    want = np.dtype(np.int64 if raw else _DTYPE_OF_ENC[enc])
    if _is_torch(out):
        name = str(out.dtype).replace("torch.", "")
        if name != want.name or not out.is_contiguous() or out.numel() < n:
            raise ValueError(f"out must be a contiguous {want.name} tensor with at least {n} elements")
    else:
        if out.dtype != want or not out.flags["C_CONTIGUOUS"] or out.size < n:
            raise ValueError(f"out must be a C-contiguous {want.name} array with at least {n} elements")


def _describe(a, ctx=None):
    """-> (Array3, keepalive)"""
    d = Array3()
    if _is_torch(a):
        if a.dim() != 3:
            raise ValueError("expected a [instants, rows, cols] tensor")
        name = str(a.dtype).replace("torch.", "")
        if name not in _ENC_OF_DTYPE:
            raise TypeError(f"unsupported dtype {a.dtype}")
        _order_after_torch(ctx, a)
        d.base = a.data_ptr()
        d.shape = (C.c_int64 * 3)(*a.shape)
        d.strides = (C.c_int64 * 3)(*a.stride())
        d.encoding = _ENC_OF_DTYPE[name]
        d.mem = MEM_DEVICE if a.is_cuda else MEM_HOST
        return d, a
    a = np.asarray(a)
    if a.ndim != 3:
        raise ValueError("expected a [instants, rows, cols] array")
    if a.dtype.name not in _ENC_OF_DTYPE:
        raise TypeError(f"unsupported dtype {a.dtype}")
    d.base = a.ctypes.data
    d.shape = (C.c_int64 * 3)(*a.shape)
    d.strides = (C.c_int64 * 3)(*[s // a.itemsize for s in a.strides])
    d.encoding = _ENC_OF_DTYPE[a.dtype.name]
    d.mem = MEM_HOST
    return d, a


def _ptr(a):
    return C.c_void_p(a.ctypes.data)


class Context:
    """One device + one stream + scratch arenas (dcdf_ctx).  Not re-entrant; one per host thread / GPU."""

    def __init__(self, device=0):
        self._lib = _ffi.lib()
        h = C.c_void_p()
        code = self._lib.dcdf_ctx_create(int(device), C.byref(h))
        if code != 0:
            raise DcdfError(code, f"cannot create a CUDA context on device {device} (no CPU fallback exists)")
        self._h = h
        self.device = device
        self._stream_ptr = None   # a borrowed stream (set_stream), else the context's private one

    def close(self):
        if getattr(self, "_h", None):
            self._lib.dcdf_ctx_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def check(self, code):
        if code != 0:
            raise DcdfError(code, self._lib.dcdf_last_error(self._h).decode())

    def set_stream(self, cuda_stream_ptr):
        self.check(self._lib.dcdf_ctx_set_stream(self._h, C.c_void_p(cuda_stream_ptr or 0)))
        self._stream_ptr = cuda_stream_ptr or None

    def set_option(self, name, value):
        """dcdf_ctx_set_option: select between equivalent code paths (tests, A/B measurements)."""
        self.check(self._lib.dcdf_ctx_set_option(self._h, name.encode(), int(value)))

    def get_stat(self, name):
        """dcdf_ctx_get_stat: counters of the last build (e.g. "encode_units_fast")."""
        v = C.c_int64()
        self.check(self._lib.dcdf_ctx_get_stat(self._h, name.encode(), C.byref(v)))
        return v.value

    def synchronize(self):
        self.check(self._lib.dcdf_ctx_synchronize(self._h))

    @property
    def launch_count(self):
        return int(self._lib.dcdf_ctx_launch_count(self._h))

    def last_kernel_ms(self, which):
        ms = C.c_float()
        self.check(self._lib.dcdf_ctx_last_kernel_ms(self._h, which, C.byref(ms)))
        return ms.value

    # ---- fixed.rs
    def suggest_fraction(self, a):
        d, keep = _describe(a, self)
        kind, bits = C.c_int32(), C.c_int32()
        self.check(self._lib.dcdf_suggest_fraction(self._h, C.byref(d), C.byref(kind), C.byref(bits)))
        return ("Round" if kind.value else "Precise", bits.value)

    def min_max(self, a, fractional_bits=0, round=False):
        d, keep = _describe(a, self)
        mn = np.empty(d.shape[0], np.int64)
        mx = np.empty(d.shape[0], np.int64)
        self.check(self._lib.dcdf_min_max(self._h, C.byref(d), fractional_bits, int(round), _ptr(mn), _ptr(mx)))
        return mn, mx

    def to_fixed(self, values, fractional_bits, round=False):
        v = np.ascontiguousarray(values)
        out = np.empty(v.shape, np.int64)
        self.check(self._lib.dcdf_to_fixed(self._h, _ptr(v), _ENC_OF_DTYPE[v.dtype.name], v.size, fractional_bits, int(round), _ptr(out), MEM_HOST))
        return out

    def from_fixed(self, fixed, fractional_bits, dtype=np.float32):
        f = np.ascontiguousarray(fixed, dtype=np.int64)
        out = np.empty(f.shape, dtype)
        self.check(self._lib.dcdf_from_fixed(self._h, _ptr(f), f.size, fractional_bits, _ptr(out), _ENC_OF_DTYPE[np.dtype(dtype).name], MEM_HOST))
        return out


def stats_dtype(dtype):
    """Record of Superchunk.window_stats_batch / Variable.window_stats for an array of `dtype`."""
    return np.dtype([("count", np.uint64), ("min", dtype), ("max", dtype), ("sum", np.float64), ("sum_sq", np.float64)])


def time_stats_dtype(dtype):
    """Record of Superchunk.time_stats_batch / Variable.time_stats for an array of `dtype`."""
    return np.dtype([("count", np.uint64), ("n_band", np.uint64), ("min", dtype), ("max", dtype), ("sum", np.float64),
                     ("sum_sq", np.float64)])


_TIME_FIELDS = ("count", "n_band", "min", "max", "sum", "sum_sq")


def _out_array(shape, enc, raw):
    return np.empty(shape, np.int64 if raw else _DTYPE_OF_ENC[enc])


class _Queryable:
    """Shared query surface of Chunk and Superchunk (prefix selects the C entry points)."""
    _prefix = None

    def _fn(self, name):
        return getattr(self.ctx._lib, f"dcdf_{self._prefix}_{name}")

    def get_batch(self, irc, raw=False):
        irc = np.ascontiguousarray(irc, dtype=np.int64).reshape(-1, 3)
        out = _out_array(len(irc), self.encoding, raw)
        self.ctx.check(self._fn("get_batch")(self.ctx._h, self._h, len(irc), _ptr(irc), _ptr(out),
                                             ENC_I64 if raw else self.encoding, MEM_HOST))
        return out

    def get(self, instant, row, col, raw=False):
        return self.get_batch([[instant, row, col]], raw)[0]

    def cell_batch(self, queries, raw=False, out=None, flat=False):
        """Chunk / Superchunk::fill_cell for n x (start, end, row, col).  `out`: optional destination (a numpy array or
        a torch tensor, e.g. pinned host memory or device memory) for all series back to back; flat=True returns
        (out, offsets) instead of one view per series."""
        q = np.ascontiguousarray(queries, dtype=np.int64).reshape(-1, 4)
        lens = np.abs(q[:, 1] - q[:, 0]).astype(np.uint64)
        off = np.zeros(len(q) + 1, np.uint64)
        np.cumsum(lens, out=off[1:])
        mem = MEM_HOST
        if out is None:
            out = _out_array(int(off[-1]), self.encoding, raw)
            ptr = _ptr(out)
        elif _is_torch(out):
            _check_out(out, int(off[-1]), self.encoding, raw)
            _order_after_torch(self.ctx, out)
            ptr, mem = C.c_void_p(out.data_ptr()), (MEM_DEVICE if out.is_cuda else MEM_HOST)
        else:
            _check_out(out, int(off[-1]), self.encoding, raw)
            ptr = _ptr(out)
        self.ctx.check(self._fn("cell_batch")(self.ctx._h, self._h, len(q), _ptr(q), _ptr(off), ptr,
                                              ENC_I64 if raw else self.encoding, mem))
        if flat:
            return out, off
        return [out[int(off[i]):int(off[i + 1])] for i in range(len(q))]

    def cell(self, start, end, row, col, raw=False):
        return self.cell_batch([[start, end, row, col]], raw)[0]

    def window(self, start, end, top, bottom, left, right, raw=False, out=None):
        cube = Cube(start, end, top, bottom, left, right)
        shape = (abs(end - start), abs(bottom - top), abs(right - left))
        mem = MEM_HOST
        if out is None:
            out = _out_array(shape, self.encoding, raw)
            ptr = _ptr(out)
        elif _is_torch(out):
            _check_out(out, shape[0] * shape[1] * shape[2], self.encoding, raw)
            _order_after_torch(self.ctx, out)
            ptr, mem = C.c_void_p(out.data_ptr()), (MEM_DEVICE if out.is_cuda else MEM_HOST)
        else:
            _check_out(out, shape[0] * shape[1] * shape[2], self.encoding, raw)
            ptr = _ptr(out)
        self.ctx.check(self._fn("window")(self.ctx._h, self._h, C.byref(cube), ptr, ENC_I64 if raw else self.encoding, mem))
        return out


class Chunk(_Queryable):
    """chunk.rs: a series of time instants as Blocks of one Snapshot + <=254 Logs, resident on the GPU."""
    _prefix = "chunk"

    def __init__(self, ctx, handle, stats=None):
        self.ctx, self._h, self.stats = ctx, handle, stats
        shape = (C.c_int64 * 3)()
        enc, fb, nb = C.c_int32(), C.c_int32(), C.c_uint32()
        ctx.check(ctx._lib.dcdf_chunk_info(handle, C.byref(shape), C.byref(enc), C.byref(fb), C.byref(nb)))
        self.shape = tuple(shape)
        self.encoding, self.fractional_bits, self.n_blocks = enc.value, fb.value, nb.value

    @classmethod
    def build(cls, ctx, array, k=2, fractional_bits=0, round=False):
        """Chunk::build chunk.rs:42-96 (fractional_bits / round are the MMBuffer3 fields)."""
        d, keep = _describe(array, ctx)
        h = C.c_void_p()
        st = BuildStats()
        ctx.check(ctx._lib.dcdf_chunk_build(ctx._h, C.byref(d), k, fractional_bits, int(round), C.byref(h), C.byref(st)))
        return cls(ctx, h, dict(size=st.size, snapshots=st.snapshots, logs=st.logs))

    @classmethod
    def read_from(cls, ctx, data):
        """Chunk::read_from chunk.rs:247-266."""
        b = np.frombuffer(bytes(data), dtype=np.uint8)
        h = C.c_void_p()
        ctx.check(ctx._lib.dcdf_chunk_open(ctx._h, _ptr(b), len(b), MEM_HOST, C.byref(h)))
        return cls(ctx, h)

    def size(self):
        n = C.c_uint64()
        self.ctx.check(self.ctx._lib.dcdf_chunk_size(self._h, C.byref(n)))
        return n.value

    def write_to(self):
        """Chunk::write_to chunk.rs:235-243 -> bytes."""
        n = self.size()
        buf = np.empty(n, np.uint8)
        self.ctx.check(self.ctx._lib.dcdf_chunk_bytes(self.ctx._h, self._h, _ptr(buf), n, MEM_HOST))
        return buf.tobytes()

    def block_instants(self):
        out = np.zeros(self.n_blocks, np.uint32)
        self.ctx.check(self.ctx._lib.dcdf_chunk_block_instants(self.ctx._h, self._h, _ptr(out)))
        return out.tolist()

    def search(self, start, end, top, bottom, left, right, lower, upper):
        """Chunk::iter_search chunk.rs:213-228 -> [n,3] (instant,row,col) in the reference's order."""
        cube = Cube(start, end, top, bottom, left, right)
        n = C.c_uint64()
        self.ctx.check(self.ctx._lib.dcdf_chunk_search(self.ctx._h, self._h, C.byref(cube), lower, upper, None, 0, C.byref(n), MEM_HOST))
        out = np.zeros((n.value, 3), np.int64)
        if n.value:
            self.ctx.check(self.ctx._lib.dcdf_chunk_search(self.ctx._h, self._h, C.byref(cube), lower, upper, _ptr(out), n.value, C.byref(n), MEM_HOST))
        return out

    def close(self):
        if getattr(self, "_h", None):
            self.ctx._lib.dcdf_chunk_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Superchunk(_Queryable):
    """superchunk.rs: a raster time series cut into k^levels x k^levels subchunks, per `chunk_size` slice."""
    _prefix = "superchunk"

    def __init__(self, ctx, handle, encoding, shape):
        self.ctx, self._h, self.encoding, self.shape = ctx, handle, encoding, tuple(shape)
        n = C.c_uint32()
        ctx.check(ctx._lib.dcdf_superchunk_count(handle, C.byref(n)))
        self.n_slices = n.value

    @classmethod
    def build(cls, ctx, array, levels, k=2, fractional_bits=0, round=False, compute_bits=True, chunk_size=0):
        """Superchunk::build superchunk.rs:88-270 for every chunk_size slice (dataset.rs:834-851)."""
        d, keep = _describe(array, ctx)
        lv = (C.c_uint32 * len(levels))(*levels)
        h = C.c_void_p()
        ctx.check(ctx._lib.dcdf_superchunk_build(ctx._h, C.byref(d), lv, len(levels), k, fractional_bits, int(round),
                                                 int(compute_bits), int(chunk_size or 0), C.byref(h)))
        return cls(ctx, h, d.encoding, tuple(d.shape))

    def node_count(self):
        n = C.c_uint32()
        self.ctx.check(self.ctx._lib.dcdf_superchunk_node_count(self._h, C.byref(n)))
        return n.value

    def info(self, slice_=0, node=0):
        info = SuperchunkInfo()
        self.ctx.check(self.ctx._lib.dcdf_superchunk_node_info(self._h, slice_, node, C.byref(info)))
        return info

    def refs(self, slice_=0, node=0, with_children=False):
        """Reference kinds of a node's subchunk slots (row-major), offsets / sizes / bits of stored Chunks and,
        with_children, the node index of nested superchunk references (-1 otherwise)."""
        n = self.info(slice_, node).n_refs
        kinds = np.zeros(n, np.int32)
        child = np.zeros(n, np.int32)
        off = np.zeros(n, np.uint64)
        size = np.zeros(n, np.uint64)
        bits = np.zeros(n, np.int32)
        self.ctx.check(self.ctx._lib.dcdf_superchunk_node_refs(self.ctx._h, self._h, slice_, node, _ptr(kinds), _ptr(child),
                                                               _ptr(off), _ptr(size), _ptr(bits)))
        return (kinds, off, size, bits, child) if with_children else (kinds, off, size, bits)

    def bytes(self, slice_=0, which=0, node=0):
        """which 0: every stored Chunk of the slice back to back; 1 / 2: max / min Dac of `node`."""
        if which == 0:
            n = self.info(slice_, 0).chunk_bytes
            buf = np.empty(max(n, 1), np.uint8)
            self.ctx.check(self.ctx._lib.dcdf_superchunk_bytes(self.ctx._h, self._h, slice_, 0, _ptr(buf), n, MEM_HOST))
            return buf[:n].tobytes()
        info = self.info(slice_, node)
        n = info.max_dac_bytes if which == 1 else info.min_dac_bytes
        buf = np.empty(max(n, 1), np.uint8)
        self.ctx.check(self.ctx._lib.dcdf_superchunk_node_bytes(self.ctx._h, self._h, slice_, node, which, _ptr(buf), n, MEM_HOST))
        return buf[:n].tobytes()

    def chunk_bytes(self, slice_=0, node=0, blob=None):
        """-> list (one per subchunk slot of `node`, row-major) of Chunk bytes, or None for Elided / nested slots."""
        kinds, off, size, _ = self.refs(slice_, node)
        blob = self.bytes(slice_, 0) if blob is None else blob
        return [blob[int(o):int(o + s)] if (k == _ffi.REF_EXTERNAL and s > 0) else None for k, o, s in zip(kinds, off, size)]

    def total_bytes(self):
        n = C.c_uint64()
        self.ctx.check(self.ctx._lib.dcdf_superchunk_total_bytes(self._h, C.byref(n)))
        return n.value

    def save(self, slice_=0):
        """The tail of Superchunk::build + Resolver::save (superchunk.rs:199-270, resolver.rs:126-138): the stored
        objects of one time slice in first-save order as (cid, node_type, bytes) -- the last one is the superchunk node
        -- and the reference's MMStruct3Build counters (External references de-duplicated by CID)."""
        lib = self.ctx._lib
        h = C.c_void_p()
        self.ctx.check(lib.dcdf_superchunk_save(self.ctx._h, self._h, slice_, C.byref(h)))
        try:
            n = C.c_uint32()
            self.ctx.check(lib.dcdf_saved_count(h, C.byref(n)))
            offs = np.zeros(n.value + 1, np.uint64)
            self.ctx.check(lib.dcdf_saved_all_bytes(self.ctx._h, h, None, 0, _ptr(offs)))
            buf = np.empty(max(int(offs[-1]), 1), np.uint8)
            self.ctx.check(lib.dcdf_saved_all_bytes(self.ctx._h, h, _ptr(buf), int(offs[-1]), _ptr(offs)))  # one transfer
            view = memoryview(buf)
            nodes = []
            cid = np.zeros(_ffi.CID_BYTES, np.uint8)
            t, size = C.c_int32(), C.c_uint64()
            for i in range(n.value):
                self.ctx.check(lib.dcdf_saved_node(h, i, _ptr(cid), C.byref(t), C.byref(size)))
                nodes.append((cid.tobytes(), t.value, bytes(view[int(offs[i]):int(offs[i + 1])])))
            st = BuildStats()
            self.ctx.check(lib.dcdf_saved_stats(h, C.byref(st)))
            stats = dict(size=st.size, elided=st.elided, local=st.local, external=st.external, snapshots=st.snapshots, logs=st.logs)
        finally:
            lib.dcdf_saved_free(h)
        return nodes, stats

    @classmethod
    def open(cls, ctx, root_cids, store):
        """Superchunk::load_from (superchunk.rs:713-768) for the superchunk nodes of consecutive time slices: `store`
        maps a CID (bytes) to the stored bytes of a node -- the Mapper::load of mapper.rs:10-38."""
        keep = {}

        def fetch(user, cid_p, bytes_pp, len_p):
            try:
                cid = C.string_at(cid_p, _ffi.CID_BYTES)
                data = store.get(cid) if hasattr(store, "get") else store[cid]
                if data is None:
                    return 1
                arr = keep.get(cid)
                if arr is None:
                    arr = np.frombuffer(bytes(data), dtype=np.uint8)
                    keep[cid] = arr
                bytes_pp[0] = C.cast(arr.ctypes.data, C.POINTER(C.c_uint8))
                len_p[0] = len(arr)
                return 0
            except Exception:
                return 1

        cb = _ffi.FETCH_FN(fetch)
        roots = np.frombuffer(b"".join(bytes(c) for c in root_cids), dtype=np.uint8)
        h = C.c_void_p()
        ctx.check(ctx._lib.dcdf_superchunk_open(ctx._h, len(root_cids), _ptr(roots), cb, None, C.byref(h)))
        info = SuperchunkInfo()
        ctx.check(ctx._lib.dcdf_superchunk_get_info(h, 0, C.byref(info)))
        n = C.c_uint32()
        ctx.check(ctx._lib.dcdf_superchunk_count(h, C.byref(n)))
        total = 0
        for s in range(n.value):
            si = SuperchunkInfo()
            ctx.check(ctx._lib.dcdf_superchunk_get_info(h, s, C.byref(si)))
            total += si.shape[0]
        return cls(ctx, h, info.encoding, (total, info.shape[1], info.shape[2]))

    def window_batch(self, cubes, raw=False, out=None):
        cubes = np.ascontiguousarray(cubes, dtype=np.int64).reshape(-1, 6)
        sizes = (np.abs(cubes[:, 1] - cubes[:, 0]) * np.abs(cubes[:, 3] - cubes[:, 2]) * np.abs(cubes[:, 5] - cubes[:, 4])).astype(np.uint64)
        off = np.zeros(len(cubes) + 1, np.uint64)
        np.cumsum(sizes, out=off[1:])
        mem = MEM_HOST
        if out is None:
            out = _out_array(int(off[-1]), self.encoding, raw)
            ptr = _ptr(out)
        elif _is_torch(out):
            _check_out(out, int(off[-1]), self.encoding, raw)
            _order_after_torch(self.ctx, out)
            ptr, mem = C.c_void_p(out.data_ptr()), (MEM_DEVICE if out.is_cuda else MEM_HOST)
        else:
            _check_out(out, int(off[-1]), self.encoding, raw)
            ptr = _ptr(out)
        self.ctx.check(self.ctx._lib.dcdf_superchunk_window_batch(self.ctx._h, self._h, len(cubes), _ptr(cubes), _ptr(off), ptr,
                                                                  ENC_I64 if raw else self.encoding, mem))
        return out, off

    def window_stats_batch(self, cubes):
        """Per-instant statistics of n windows reduced on the device (dcdf_superchunk_window_stats) -> (records, off):
        window i's records are records[off[i]:off[i + 1]], one per instant, ascending.  Fields: count (non-NaN cells),
        min / max (the superchunk's dtype; NaN / 0 when count is 0), sum and sum_sq (float64) of the values the window
        decoder writes."""
        cubes = np.ascontiguousarray(cubes, dtype=np.int64).reshape(-1, 6)
        off = np.zeros(len(cubes) + 1, np.uint64)
        np.cumsum(np.abs(cubes[:, 1] - cubes[:, 0]).astype(np.uint64), out=off[1:])
        dt = _DTYPE_OF_ENC[self.encoding]
        n = int(off[-1])
        count, vmin, vmax = np.empty(n, np.uint64), np.empty(n, dt), np.empty(n, dt)
        total, total_sq = np.empty(n, np.float64), np.empty(n, np.float64)
        self.ctx.check(self.ctx._lib.dcdf_superchunk_window_stats(self.ctx._h, self._h, len(cubes), _ptr(cubes), _ptr(off), _ptr(count),
                                                                  _ptr(vmin), _ptr(vmax), _ptr(total), _ptr(total_sq), MEM_HOST))
        records = np.empty(n, stats_dtype(dt))
        records["count"], records["min"], records["max"], records["sum"], records["sum_sq"] = count, vmin, vmax, total, total_sq
        return records, off

    def window_stats(self, start, end, top, bottom, left, right):
        return self.window_stats_batch([[start, end, top, bottom, left, right]])[0]

    def _time_stats_into(self, cubes, lower, upper, cols, off, accumulate):
        """dcdf_superchunk_time_stats into the column arrays `cols` (one per field of time_stats_dtype)."""
        band = lower is not None or upper is not None
        lo = hi = None
        if band:
            lo = np.ascontiguousarray(np.broadcast_to(np.asarray(-np.inf if lower is None else lower, np.float64), len(cubes)))
            hi = np.ascontiguousarray(np.broadcast_to(np.asarray(np.inf if upper is None else upper, np.float64), len(cubes)))
        p = lambda a: None if a is None else _ptr(a)
        self.ctx.check(self.ctx._lib.dcdf_superchunk_time_stats(self.ctx._h, self._h, len(cubes), _ptr(cubes), _ptr(off), p(lo), p(hi),
                                                                *[p(cols[f]) for f in _TIME_FIELDS], int(accumulate), MEM_HOST))

    def time_stats_batch(self, cubes, lower=None, upper=None):
        """Per-cell statistics over time of n windows reduced on the device (dcdf_superchunk_time_stats) -> (records, off):
        window i's records are records[off[i]:off[i + 1]], one per cell, row-major.  Fields: count (non-NaN instants),
        n_band (instants with lower <= value <= upper; bounds are scalars or one per window, a missing one is infinite;
        without bounds n_band equals count), min / max (the superchunk's dtype; NaN / 0 when count is 0), sum and sum_sq
        (float64, summed per time slice in time order, then over the slices)."""
        cubes = np.ascontiguousarray(cubes, dtype=np.int64).reshape(-1, 6)
        off = np.zeros(len(cubes) + 1, np.uint64)
        np.cumsum((np.abs(cubes[:, 3] - cubes[:, 2]) * np.abs(cubes[:, 5] - cubes[:, 4])).astype(np.uint64), out=off[1:])
        records = np.empty(int(off[-1]), time_stats_dtype(_DTYPE_OF_ENC[self.encoding]))
        cols = {f: np.empty(len(records), records.dtype[f]) for f in _TIME_FIELDS}
        self._time_stats_into(cubes, lower, upper, cols, off, False)
        for f in _TIME_FIELDS:
            records[f] = cols[f]
        return records, off

    def time_stats(self, start, end, top, bottom, left, right, lower=None, upper=None):
        """Single-window time_stats_batch: records shaped (rows, cols)."""
        rec, _ = self.time_stats_batch([[start, end, top, bottom, left, right]], lower, upper)
        return rec.reshape(abs(bottom - top), abs(right - left))

    def search_batch(self, cubes, lower, upper, want_cells=True):
        return self._search(self.ctx._lib.dcdf_superchunk_search_batch, np.int64, cubes, lower, upper, want_cells)

    def search(self, start, end, top, bottom, left, right, lower, upper):
        return self.search_batch([[start, end, top, bottom, left, right]], lower, upper)[1]

    def search_values_batch(self, cubes, lower, upper, want_cells=True):
        """Value-range search with bounds in the array's own units (dcdf_superchunk_search_values): the cells whose decoded
        value v has lower <= v <= upper, NaN never; exact where search_batch follows the reference's traversal.  Per window
        counts and the (instant, row, col) cells, window after window."""
        return self._search(self.ctx._lib.dcdf_superchunk_search_values, np.float64, cubes, lower, upper, want_cells)

    def search_values(self, start, end, top, bottom, left, right, lower, upper):
        return self.search_values_batch([[start, end, top, bottom, left, right]], lower, upper)[1]

    def _search(self, fn, bound_type, cubes, lower, upper, want_cells):
        cubes = np.ascontiguousarray(cubes, dtype=np.int64).reshape(-1, 6)
        n = len(cubes)
        lo = np.ascontiguousarray(np.broadcast_to(np.asarray(lower, bound_type), (n,)))
        hi = np.ascontiguousarray(np.broadcast_to(np.asarray(upper, bound_type), (n,)))
        counts = np.zeros(n, np.uint64)
        found = C.c_uint64()
        self.ctx.check(fn(self.ctx._h, self._h, n, _ptr(cubes), _ptr(lo), _ptr(hi), _ptr(counts), None, 0, C.byref(found), MEM_HOST))
        if not want_cells:
            return counts, None
        out = np.zeros((found.value, 3), np.int64)
        if found.value:
            self.ctx.check(fn(self.ctx._h, self._h, n, _ptr(cubes), _ptr(lo), _ptr(hi), _ptr(counts), _ptr(out), found.value, C.byref(found), MEM_HOST))
        return counts, out

    def close(self):
        if getattr(self, "_h", None):
            self.ctx._lib.dcdf_superchunk_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
