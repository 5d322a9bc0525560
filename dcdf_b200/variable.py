"""Host-side mirror of how the product drives the hot path (SURVEY 8f2-8f4), over the C-ABI.

  Variable.append        dataset.rs:268-325 (tail re-encode) + :834-878 (one Superchunk::build per chunk_size slice,
                         every node saved to the store)
  span routing           span.rs:139-279: a query is split by time slice; here by groups of `span_size` slices
  ChunkCache             the Resolver's LRU of loaded nodes (cache.rs:37-232, resolver.rs:118-122), but DEVICE resident:
                         a group of consecutive time-slice superchunks opened from the store stays in HBM, keyed by
                         the CIDs of its superchunk nodes, evicted least-recently-used by encoded bytes
  Variable.__getitem__   py-dcdf/dcdf/__init__.py:281-336 (lazy _Slice, scalar / cell / window dispatch)
  MMArray3.shape/get/cell/window   py-dcdf/src/lib.rs:497-538 (PyMMArray3F32), mmarray.rs:357-400
  search with float bounds         mmarray.rs:407-417 is todo!() upstream; dcdf_superchunk_search_values on the device
  window_stats                     per-instant count / min / max / sum / sum_sq of a window, dcdf_superchunk_window_stats
  time_stats                       per-cell count / n_band / min / max / sum / sum_sq over time, dcdf_superchunk_time_stats

The store is any mapping CID (bytes) -> stored node bytes.  The slices' superchunk CIDs are kept in the reference's span
tree (dcdf_b200/span.py: stored Span nodes, `Variable.cid` = the root span, dataset.rs:880-987), so a variable written here
can be re-opened from its serialized form (`write_to` / `Variable.load`, dataset.rs:1012-1075); the flat lists below are
what that tree resolves to, kept for routing.  Datasets and coordinates stay with the host application (DESIGN.md 7).
"""
import collections
import functools
import threading

import numpy as np

from . import span as _span
from .api import DcdfError, Superchunk


class ChunkCache:
    """LRU of opened superchunk groups resident on the device (cache.rs:37-232 semantics: size-bounded, least recently
    used out first, one load per key even under concurrent requests)."""

    def __init__(self, ctx, store, cache_bytes=1 << 30):
        self.ctx, self.store, self.cache_bytes = ctx, store, int(cache_bytes)
        self._items = collections.OrderedDict()   # key -> (handle, bytes)
        self._lock = threading.Lock()
        self.hits = self.misses = self.evictions = 0

    def get(self, root_cids):
        key = tuple(bytes(c) for c in root_cids)
        with self._lock:                          # single flight: the load happens under the lock (cache.rs:120-180)
            it = self._items.get(key)
            if it is not None:
                self._items.move_to_end(key)
                self.hits += 1
                return it[0]
            self.misses += 1
            sc = Superchunk.open(self.ctx, list(key), self.store)
            size = sc.total_bytes()
            self._items[key] = (sc, size)
            self._evict(keep=key)
            return sc

    def _evict(self, keep=None):
        total = sum(b for _, b in self._items.values())
        while total > self.cache_bytes and len(self._items) > 1:
            key, (sc, size) = next(iter(self._items.items()))
            if key == keep:
                break
            del self._items[key]
            sc.close()
            total -= size
            self.evictions += 1

    def invalidate(self, root_cids=None):
        with self._lock:
            keys = [k for k in self._items if root_cids is None or any(c in k for c in root_cids)]
            for k in keys:
                self._items.pop(k)[0].close()

    @property
    def resident_bytes(self):
        return sum(b for _, b in self._items.values())

    def close(self):
        self.invalidate()


class _Slice:
    """py-dcdf/dcdf/__init__.py:353-363: the result of Variable[...] is realised on first use."""

    def __init__(self, realize):
        self.realize = realize

    @functools.cached_property
    def data(self):
        return self.realize()

    def __getitem__(self, arg):
        return self.data.__getitem__(arg)


def _is_int(n):
    return isinstance(n, (int, np.integer))


def _as_slice(n):
    return slice(n, n + 1) if _is_int(n) else n


class MMArray3:
    """shape / get / cell / window (PyMMArray3*, py-dcdf/src/lib.rs:411-581) plus __getitem__ exactly as
    Variable.__getitem__ does it (py-dcdf/dcdf/__init__.py:281-336).  Subclasses provide shape, get, cell, window."""

    def __getitem__(self, indices):
        indices = [indices] if not isinstance(indices, tuple) else list(indices)
        n_indices = len(indices)
        if n_indices > 3:
            raise IndexError(f"too many indices for array: array is 3-dimensional, but {len(indices)} were indexed")
        while len(indices) < 3:
            indices.append(slice(0, None))
        fixed = []
        for index, stop in zip(indices, self.shape):
            if _is_int(index):
                fixed.append(int(index))
                continue
            if index.start is None:
                index = slice(0, index.stop)
            if index.stop is None:
                index = slice(index.start, stop)
            fixed.append(index)
        instant, row, col = indices = fixed
        scalars = tuple(map(_is_int, indices))

        def realize(instant=instant, row=row, col=col, indices=indices):
            if all(scalars):
                return self.get(instant, row, col)
            if scalars == (False, True, True):
                return self.cell(instant.start, instant.stop, row, col)
            instant, row, col = map(_as_slice, indices)
            array = self.window(instant.start, instant.stop, row.start, row.stop, col.start, col.stop)
            mask = tuple(0 if scalar else slice(None, None) for scalar in scalars[:n_indices])
            if len(mask) == 1:
                mask = mask[0]
            return array.__getitem__(mask)

        return _Slice(realize)


class Variable(MMArray3):
    """One variable of a dataset: a time series of rasters stored as one superchunk per `chunk_size` instants."""

    def __init__(self, ctx, store, k2_levels, chunk_size=64, round=None, span_size=8, dtype=np.float32, cache_bytes=1 << 30,
                 name="data"):
        self.ctx, self.store, self.name = ctx, store, str(name)
        self.tree = None           # span tree (created with the first append, when the raster shape is known)
        self.k2_levels, self.chunk_size, self.round, self.span_size = tuple(k2_levels), int(chunk_size), round, int(span_size)
        self.dtype = np.dtype(dtype)
        self.roots = []            # CID of every time slice's superchunk node, in time order
        self.instants = []         # instants per slice
        self.slice_bits = []       # fractional bits of every slice's superchunk
        self.rows = self.cols = None
        self.stats = []            # MMStruct3Build of every slice (Variable::append drops it, dataset.rs:850-851; kept here)
        self.cache = ChunkCache(ctx, store, cache_bytes)

    # ------------------------------------------------------------------ ingest
    def append(self, data):
        """Dataset::append_* + Variable::append: an incomplete last slice is decoded, prepended and re-encoded
        (dataset.rs:283-297, `update` at :866-870); then one Superchunk::build per chunk_size slice, all of them in one
        call of the C-ABI, every node of every slice saved to the store."""
        import torch
        is_t = hasattr(data, "is_cuda")
        if tuple(data.shape[1:]) != (self.rows or data.shape[1], self.cols or data.shape[2]):
            raise ValueError("shape of the appended raster does not match the variable")
        self.rows, self.cols = int(data.shape[1]), int(data.shape[2])
        if self.tree is None:      # Dataset::add_variable saves one empty span (dataset.rs:127-129)
            self.tree = _span.SpanTree(self.store, self.rows, self.cols, self.chunk_size, self.span_size,
                                       _span.ENCODINGS[self.dtype.name])
        if int(data.shape[0]) == 0:
            return self            # the loop of Variable::append does not run (dataset.rs:838)
        update = bool(self.roots) and self.instants[-1] < self.chunk_size
        if update:
            T = self.shape[0]
            tail = self.window(T - self.instants[-1], T, 0, self.rows, 0, self.cols)
            if is_t:
                data = torch.cat([torch.from_numpy(tail).to(data.device), data], dim=0)
            else:
                data = np.concatenate([tail, np.asarray(data, dtype=self.dtype)], axis=0)
        bits = self.round if self.round is not None else 0
        sc = Superchunk.build(self.ctx, data, list(self.k2_levels), fractional_bits=bits, round=self.round is not None,
                              compute_bits=True, chunk_size=self.chunk_size)
        new = []                   # nothing of the variable changes until every slice is built and saved (a data error
        try:                       # -- NaN-only input, precision loss -- leaves it as it was)
            for s in range(sc.n_slices):
                nodes, stats = sc.save(s)
                for cid, _, b in nodes:
                    self.store[cid] = b
                info = sc.info(s)
                new.append((nodes[-1][0], int(info.shape[0]), int(info.fractional_bits), stats))
        finally:
            sc.close()
        if update:
            old = self.roots.pop()
            self.instants.pop(); self.slice_bits.pop(); self.stats.pop()
            self.cache.invalidate([old])
        for cid, n, fb, stats in new:
            self.tree.append(cid, n, update=update)   # Span::update for the re-encoded tail, Span::append after it
            update = False
            self.roots.append(cid); self.instants.append(n); self.slice_bits.append(fb); self.stats.append(stats)
        self.tree.commit()         # Variable::save_spans
        return self

    def fork(self):
        """A second handle on the same stored state (the reference clones a Variable before it appends to it,
        dataset.rs:269-276): appending to the fork leaves this one as it is.  The device cache is shared."""
        v = Variable(self.ctx, self.store, self.k2_levels, chunk_size=self.chunk_size, round=self.round, span_size=self.span_size,
                     dtype=self.dtype, cache_bytes=self.cache.cache_bytes, name=self.name)
        v.cache = self.cache
        v.roots, v.instants, v.slice_bits, v.stats = list(self.roots), list(self.instants), list(self.slice_bits), list(self.stats)
        v.rows, v.cols = self.rows, self.cols
        if self.tree is not None:
            v.tree = _span.SpanTree(self.store, self.rows, self.cols, self.chunk_size, self.span_size,
                                    _span.ENCODINGS[self.dtype.name], root=self.tree.commit())
        return v

    # ------------------------------------------------------------------ stored form
    @property
    def cid(self):
        """CID of the root span (Variable.cid, dataset.rs:58); None before the first append."""
        return self.tree.commit() if self.tree is not None else None

    def write_to(self):
        """The variable as it sits inside a Dataset node (dataset.rs:1018-1040): name, rounding, span_size, chunk_size,
        k2_levels, encoding, CID of the root span."""
        if self.tree is None:
            raise ValueError("nothing appended yet: the root span needs the raster shape")
        name = self.name.encode()
        if len(name) > 255:
            raise ValueError("name longer than 255 bytes")            # write_str: one length byte (extio.rs:260-265)
        b = bytes([len(name)]) + name
        b += bytes([1, self.round]) if self.round is not None else b"\x00"
        b += self.span_size.to_bytes(4, "big") + self.chunk_size.to_bytes(4, "big") + bytes([len(self.k2_levels)])
        for lv in self.k2_levels:
            b += int(lv).to_bytes(4, "big")
        return b + bytes([_span.ENCODINGS[self.dtype.name]]) + self.cid

    @classmethod
    def load(cls, ctx, store, stored, cache_bytes=1 << 30):
        """Variable::load_from (dataset.rs:1042-1075) + a walk of the span tree down to the slices' superchunk nodes."""
        stored = bytes(stored)
        try:
            n = stored[0]
            name, p = stored[1:1 + n].decode(), 1 + n
            rnd = None
            if stored[p] == 1:
                rnd, p = stored[p + 1], p + 1
            p += 1
            span_size, chunk_size = int.from_bytes(stored[p:p + 4], "big"), int.from_bytes(stored[p + 4:p + 8], "big")
            nk, p = stored[p + 8], p + 9
            k2 = [int.from_bytes(stored[p + 4 * i:p + 4 * i + 4], "big") for i in range(nk)]
            p += 4 * nk
            enc, root = stored[p], stored[p + 1:p + 1 + _span.CID_BYTES]
            if len(root) != _span.CID_BYTES or len(stored) != p + 1 + _span.CID_BYTES:
                raise IndexError
        except IndexError:
            raise DcdfError(6, "truncated or oversized Variable record") from None
        dtypes = {v: k for k, v in _span.ENCODINGS.items()}
        if enc not in dtypes:
            raise DcdfError(6, f"unknown encoding {enc}")
        v = cls(ctx, store, k2, chunk_size=chunk_size, round=rnd, span_size=span_size, dtype=np.dtype(dtypes[enc]),
                cache_bytes=cache_bytes, name=name)
        top = _span.Span.from_bytes(bytes(store[root]))
        v.rows, v.cols = top.rows, top.cols
        v.tree = _span.SpanTree(store, top.rows, top.cols, chunk_size, span_size, enc, root=root)
        for cid in v.tree.chunks():
            instants, rows, cols, bits, cenc = _span.superchunk_header(bytes(store[cid]))
            if (rows, cols, cenc) != (top.rows, top.cols, enc):
                raise DcdfError(6, "a time slice does not match its variable")
            v.roots.append(cid)
            v.instants.append(instants)
            v.slice_bits.append(bits)
            v.stats.append(None)
        if sum(v.instants) != top.instants:
            raise DcdfError(6, "span tree and time slices disagree on the number of instants")
        return v

    # ------------------------------------------------------------------ geometry / routing
    @property
    def shape(self):
        return [sum(self.instants), self.rows, self.cols]

    @property
    def fractional_bits(self):
        return max(self.slice_bits) if self.slice_bits else 0

    def _groups(self, start, end):
        """(handle, first instant of the group, group-local [a, b)) for every group of span_size slices that [start, end)
        touches (span.rs:183-224 splits a window by its stride the same way)."""
        per = self.chunk_size * self.span_size
        for g in range(start // per, (end - 1) // per + 1):
            s0, s1 = g * self.span_size, min((g + 1) * self.span_size, len(self.roots))
            sc = self.cache.get(self.roots[s0:s1])
            t0 = g * per
            yield sc, t0, max(start, t0) - t0, min(end, t0 + sum(self.instants[s0:s1])) - t0

    def _check(self, start, end, top, bottom, left, right):
        T, R, Cc = self.shape
        if not (0 <= start <= end <= T and 0 <= top <= bottom <= R and 0 <= left <= right <= Cc):
            raise DcdfError(5, f"[{start}:{end}, {top}:{bottom}, {left}:{right}] out of bounds for shape {self.shape}")  # mmarray.rs:218-229

    # ------------------------------------------------------------------ queries
    def get(self, instant, row, col):
        self._check(instant, instant + 1, row, row + 1, col, col + 1)
        sc, t0, a, _ = next(self._groups(instant, instant + 1))
        return sc.get(a, row, col)

    def cell(self, start, stop, row, col):
        self._check(start, stop, row, row + 1, col, col + 1)
        parts = [sc.cell(a, b, row, col) for sc, _, a, b in self._groups(start, stop)] if stop > start else []
        return np.concatenate(parts) if parts else np.empty(0, self.dtype)

    def window(self, start, stop, top, bottom, left, right):
        self._check(start, stop, top, bottom, left, right)
        out = np.empty((stop - start, bottom - top, right - left), self.dtype)
        if out.size:
            for sc, t0, a, b in self._groups(start, stop):
                out[t0 + a - start:t0 + b - start] = sc.window(a, b, top, bottom, left, right)
        return out

    def search(self, start, stop, top, bottom, left, right, lower, upper):
        """Cells (instant, row, col) with lower <= value <= upper, bounds in the variable's own units; NaN cells never
        match.  One value-range search on the device per span group (Superchunk.search_values_batch), which converts the
        bounds with every subchunk's own fractional bits (the reference leaves float search as todo!(),
        mmarray.rs:407-417)."""
        self._check(start, stop, top, bottom, left, right)
        hits = []
        if stop > start:
            for sc, t0, a, b in self._groups(start, stop):
                cells = sc.search_values(a, b, top, bottom, left, right, lower, upper)
                cells[:, 0] += t0
                hits.append(cells)
        return np.concatenate(hits) if hits else np.zeros((0, 3), np.int64)

    def window_stats(self, start, stop, top, bottom, left, right):
        """Per-instant statistics of a window, reduced on the device from the encoded bytes (one
        Superchunk.window_stats_batch call per span group): stop - start records in time order with fields count (non-NaN
        cells), min, max (the variable's dtype; NaN for floats / 0 for integers when count is 0), sum and sum_sq (float64).
        For example

            r = v.window_stats(0, 365, 100, 200, 300, 400)
            mean = r["sum"] / r["count"]
            var = r["sum_sq"] / r["count"] - mean ** 2     # population variance
        """
        from .api import stats_dtype
        self._check(start, stop, top, bottom, left, right)
        parts = [sc.window_stats(a, b, top, bottom, left, right) for sc, _, a, b in self._groups(start, stop)] if stop > start else []
        return np.concatenate(parts) if parts else np.empty(0, stats_dtype(self.dtype))

    def time_stats(self, start, stop, top, bottom, left, right, lower=None, upper=None):
        """Per-cell statistics over instants [start, stop) of a window, reduced on the device from the encoded bytes (one
        dcdf_superchunk_time_stats call per span group, each continuing the records of the one before): records shaped
        (rows, cols) with fields count (non-NaN instants), n_band (instants with lower <= value <= upper; equals count
        without bounds), min, max (the variable's dtype; NaN for floats / 0 for integers when count is 0), sum and sum_sq
        (float64).  For example, a climatology and the days above a threshold:

            r = v.time_stats(0, 365, 100, 200, 300, 400, lower=30.0)
            mean = r["sum"] / r["count"]
            var = r["sum_sq"] / r["count"] - mean ** 2     # population variance
            hot_days = r["n_band"]
        """
        from .api import _TIME_FIELDS, time_stats_dtype
        self._check(start, stop, top, bottom, left, right)
        rows, cols_ = bottom - top, right - left
        rec = np.empty((rows, cols_), time_stats_dtype(self.dtype))
        cols = {f: np.empty(rows * cols_, rec.dtype[f]) for f in _TIME_FIELDS}
        cube = np.array([[start, start, top, bottom, left, right]], np.int64)
        off = np.array([0, rows * cols_], np.uint64)
        if stop > start and rec.size:
            for k, (sc, _, a, b) in enumerate(self._groups(start, stop)):    # a group's handle may not outlive the next load
                cube[0, 0], cube[0, 1] = a, b
                sc._time_stats_into(cube, lower, upper, cols, off, k > 0)
        else:                                        # zero instants: empty records
            cols["count"][:] = cols["n_band"][:] = 0
            cols["min"][:] = cols["max"][:] = np.nan if np.issubdtype(self.dtype, np.floating) else 0
            cols["sum"][:] = cols["sum_sq"][:] = 0.0
        for f in _TIME_FIELDS:
            rec[f] = cols[f].reshape(rows, cols_)
        return rec

    def close(self):
        self.cache.close()
