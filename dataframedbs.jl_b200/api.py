"""Host-side mirror of the reference's API for the scan path (names and argument meaning kept).

  open_table                      /root/reference/src/tables/creators.jl:7-16
  DFTable                         /root/reference/src/tables/table.jl:9-61
  DFView, selection, projection,
  selproj, getindex, nrow, ncol   /root/reference/src/tables/view.jl:26-232
  DFColumn + broadcasting         /root/reference/src/tables/column.jl:30-174, columnbroadcast.jl:1-72
  materialize, head               /root/reference/src/tables/materialization.jl:27-66
  sum/minimum/maximum/mean/count  Base folds over iterate(::DFColumn) column.jl:102-126

Julia syntax -> this mirror:
  t[t.a .> 50, [:b]]              t[t.a > 50, ["b"]]
  t[5:300:1000, :]                t[R(5, 300, 1000), :]            (1-based inclusive, Julia semantics)
  t[[1, 200, 20], :]              t[[1, 200, 20], :]
  10 .< t.a .< 40                 (t.a > 10) & (t.a < 40)
  startswith.(t.b, "1")           startswith(t.b, "1")
  coalesce.(t.a .> 50, false)     coalesce(t.a > 50, False)
  in.(t.a, Ref([1, 11]))          isin(t.a, [1, 11])
Every scan runs on the GPU through the C ABI (dfdb_b200.h); there is no CPU path here.
"""
from __future__ import annotations

import ctypes as C
import os
import math

import numpy as np

from . import _capi
from ._capi import DfdbError
from .plan import (ArgumentError, BlockBroadcasting, ColRef, InSet, JRange, JType, Projection, SelectionQueue, add, encode_plan,
                   required_columns)

_NP = {"Int8": np.int8, "Int16": np.int16, "Int32": np.int32, "Int64": np.int64, "UInt8": np.uint8, "UInt16": np.uint16,
       "UInt32": np.uint32, "UInt64": np.uint64, "Float16": np.float16, "Float32": np.float32, "Float64": np.float64,
       "Bool": np.bool_, "Char": np.uint32, "Date": np.int64, "DateTime": np.int64, "Time": np.int64}

_COLON = slice(None)


def _raise(e: DfdbError):
    """Map C status codes to the exception class the reference throws."""
    if e.code in (_capi.ERR_ARGUMENT, _capi.ERR_UNSUPPORTED):
        raise ArgumentError(str(e)) from None
    if e.code == _capi.ERR_KEY:
        raise KeyError(str(e)) from None
    if e.code == _capi.ERR_DIVIDE:
        raise ZeroDivisionError(str(e)) from None
    if e.code == _capi.ERR_CORRUPT:
        raise AssertionError(str(e)) from None
    raise e


# -----------------------------------------------------------------------------------------------
# result containers


class FlatStringsVector:
    """FlatStringsVector layout (src/FlatStringsVectors.jl:5-9): Int32 sizes (-1 = missing), Int64 offsets
    (exclusive scan of max(size, 0)) and the flat char buffer."""

    def __init__(self, sizes: np.ndarray, data):
        self.sizes = np.asarray(sizes, dtype=np.int32)
        self.data = data if isinstance(data, bytes) else memoryview(data).cast("B")   # bytes, or a zero-copy view of the result buffer
        self._offsets = None

    @property
    def offsets(self):
        """exclusive scan of max(size, 0) (unsafe_remake_offsets!, FlatStringsVectors.jl:61-70); built on first use"""
        if self._offsets is None:
            off = np.zeros(len(self.sizes), dtype=np.int64)
            if len(self.sizes) > 1:
                np.cumsum(np.maximum(self.sizes[:-1], 0), out=off[1:])
            self._offsets = off
        return self._offsets

    def __len__(self):
        return len(self.sizes)

    def __getitem__(self, i):
        if isinstance(i, (int, np.integer)):
            s = int(self.sizes[i])
            if s < 0:
                return None
            o = int(self.offsets[i])
            return bytes(self.data[o:o + s]).decode("utf-8")
        return [self[int(k)] for k in np.arange(len(self))[i]]

    def tolist(self):
        return [self[i] for i in range(len(self))]

    def __iter__(self):
        return iter(self.tolist())

    def __eq__(self, other):
        if isinstance(other, FlatStringsVector):
            return np.array_equal(self.sizes, other.sizes) and self.data == other.data
        return self.tolist() == list(other)

    def __repr__(self):
        return f"FlatStringsVector({self.tolist()[:8]!r}{'...' if len(self) > 8 else ''}, n={len(self)})"


class Frame:
    """Minimal stand-in for the DataFrame that `materialize(::DFView)` returns (materialization.jl:39)."""

    def __init__(self, names, columns):
        self.names = list(names)
        self.columns = list(columns)

    def __getitem__(self, k):
        return self.columns[self.names.index(k)] if isinstance(k, str) else self.columns[k]

    def __len__(self):
        return len(self.names)

    def nrow(self):
        return len(self.columns[0]) if self.columns else 0

    def to_dict(self):
        out = {}
        for n, c in zip(self.names, self.columns):
            if isinstance(c, FlatStringsVector):
                out[n] = c.tolist()
            elif isinstance(c, np.ma.MaskedArray):
                out[n] = [None if m else v for v, m in zip(c.data.tolist(), np.ma.getmaskarray(c).tolist())]
            else:
                out[n] = c.tolist()
        return out

    def to_pandas(self):
        import pandas as pd
        return pd.DataFrame(self.to_dict())

    def __repr__(self):
        return f"Frame({self.nrow()}x{len(self)}: {', '.join(self.names)})"


# -----------------------------------------------------------------------------------------------


class _ColumnMeta:
    def __init__(self, cid, name, typestring):
        self.id, self.name, self.typestring = cid, name, typestring
        self.type = JType.parse(typestring)


class DFTable:
    """table.jl:9-15.  Do not instantiate directly; use open_table."""

    def __init__(self, path: str, mode: int = _capi.LOAD_HBM, rank: int = 0, world: int = 1, device: int | None = None):
        # opening only parses headers on the host; the CUDA runtime is initialised by the first scan
        self.__dict__["path"] = path
        self.__dict__["_device"] = device
        h = C.c_void_p()
        try:
            _capi.check(_capi.lib().dfdb_table_open(path.encode(), C.byref(h)))
        except DfdbError as e:
            if e.code in (_capi.ERR_IO, _capi.ERR_FORMAT):
                raise RuntimeError(str(e)) from None
            _raise(e)
        L = _capi.lib()
        d = self.__dict__
        d["_h"] = h
        d["is_opened"] = True
        d["mode"] = mode
        d["_loaded"] = set()
        d["_scans"] = {}
        cols = []
        for i in range(L.dfdb_table_ncols(h)):
            cid = C.c_int64()
            name = C.create_string_buffer(512)
            ts = C.create_string_buffer(512)
            _capi.check(L.dfdb_table_column(h, i, C.byref(cid), name, 512, ts, 512, None, None, None))
            cols.append(_ColumnMeta(cid.value, name.value.decode(), ts.value.decode()))
        d["meta"] = cols
        d["block_size"] = L.dfdb_table_block_size(h)
        d["rank"], d["world"] = 0, 1
        if world > 1:
            self.set_shard(rank, world)

    # -- residency --
    def set_shard(self, rank: int, world: int):
        self._drop_scans()
        _capi.check(_capi.lib().dfdb_table_set_shard(self._h, rank, world))
        self._loaded.clear()
        self.__dict__["rank"], self.__dict__["world"] = rank, world

    def load(self, columns=None, mode: int | None = None):
        """Read the shard's compressed blocks of `columns` (default: all) into pinned host / HBM."""
        if mode is not None and mode != self.mode:
            self.__dict__["mode"] = mode
            self._loaded.clear()
        _capi.init(self._device)
        names = [m.name for m in self.meta] if columns is None else list(columns)
        ids = [self.getmeta(n).id for n in names if n not in self._loaded]
        if ids:
            arr = (C.c_int64 * len(ids))(*ids)
            try:
                _capi.check(_capi.lib().dfdb_table_load(self._h, arr, len(ids), self.mode))
            except DfdbError as e:
                _raise(e)
            self._loaded.update(names)

    def drop_decoded(self):
        _capi.check(_capi.lib().dfdb_table_drop_decoded(self._h))

    # ---- add_column! (table.jl:96-124): the new column file is written by the device write path ----
    def add_column(self, name: str, data, typestring: str | None = None):
        """`data`: array / masked array / strings (see create_table) or a DFColumn / computed column of THIS table
        (`t.add_column("c", t.a * t.b)`), which is materialized on the device first."""
        if name in [m.name for m in self.meta]:
            raise ArgumentError(f"Column :{name} already exists")
        if isinstance(data, DFColumn):
            fr = materialize(data.view)
            data = fr.columns[0]
        ts, nrows, vals, miss, sizes, chars = _column_buffers(data, typestring)
        total = self.total_rows()
        if total != 0 and total != nrows:
            raise ArgumentError("Column and table have different sizes")
        new_id = 1 + max([m.id for m in self.meta], default=0)
        cols = [(m.id, m.name, m.typestring) for m in self.meta] + [(new_id, name, ts)]
        write_column_file(self.path, new_id, ts, self.block_size, nrows, vals, miss, sizes, chars, self._device)
        _write_meta(self.path, self.block_size, cols)
        # the handle describes the old meta: reopen
        mode, rank, world, dev = self.mode, self.rank, self.world, self._device
        self.close()
        self.__init__(self.path, mode=mode, rank=rank, world=world, device=dev)
        return self

    # ---- block index + zone maps (optional sidecar <id>.zmap; no reference counterpart, SURVEY.md 8f) ----
    def build_zonemaps(self, columns=None):
        """Per-block (min, max, null count) of the given fixed-width numeric columns (default: all of them), computed on the
        device and written beside the column files; used from then on (also by later open_table calls) to skip blocks a
        predicate's constants rule out."""
        L = _capi.lib()
        self._drop_scans()
        try:
            if columns is None:
                _capi.check(L.dfdb_table_build_zonemaps(self._h, None, 0))
            else:
                ids = [self.getmeta(n).id for n in columns]
                _capi.check(L.dfdb_table_build_zonemaps(self._h, (C.c_int64 * len(ids))(*ids), len(ids)))
        except DfdbError as e:
            _raise(e)

    def zonemap(self, column: str, block: int):
        """dfdb_zone of one table block, or None when the column has no zone map."""
        z = _capi.Zone()
        rc = _capi.lib().dfdb_table_zonemap(self._h, self.getmeta(column).id, block, C.byref(z))
        if rc == _capi.ERR_STATE:
            return None
        _capi.check(rc)
        return z

    def _drop_scans(self):
        for s in self._scans.values():
            _capi.lib().dfdb_scan_free(s)
        self._scans.clear()

    def close(self):
        if self.__dict__.get("is_opened"):
            self._drop_scans()
            _capi.lib().dfdb_table_close(self._h)
            self.__dict__["is_opened"] = False

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- reference API --
    def getmeta(self, name: str) -> _ColumnMeta:
        for m in self.meta:
            if m.name == name:
                return m
        raise KeyError(name)

    def names(self):
        return [m.name for m in self.meta]

    def shard_rows(self):
        lo, hi = C.c_int64(), C.c_int64()
        _capi.check(_capi.lib().dfdb_table_shard_range(self._h, None, None, C.byref(lo), C.byref(hi)))
        return lo.value, hi.value

    def nblocks(self):
        return _capi.lib().dfdb_table_nblocks(self._h)

    def total_rows(self):
        return _capi.lib().dfdb_table_nrows(self._h)

    def __getitem__(self, key):
        return DFView(self)[key]

    def __getattr__(self, name):
        if name.startswith("_"):
            raise AttributeError(name)
        return DFView(self)[:, name]

    def __eq__(self, other):
        return isinstance(other, DFTable) and self.path == other.path and \
            [(m.id, m.name, m.typestring) for m in self.meta] == [(m.id, m.name, m.typestring) for m in other.meta]

    def __hash__(self):
        return hash(self.path)

    def __repr__(self):
        return f"DFTable path: {self.path}" if self.is_opened else "closed table"


def open_table(path: str, mode: int = _capi.LOAD_HBM, rank: int = 0, world: int = 1, device: int | None = None) -> DFTable:
    """creators.jl:7-16"""
    return DFTable(path, mode=mode, rank=rank, world=world, device=device)


# ---- write path: create_table / add_column! on the device (creators.jl:81-89, table.jl:96-124, columns.jl:65-84) --------------------
_TYPESTR_OF = {np.dtype(v): k for k, v in _NP.items() if k not in ("Char", "Date", "DateTime", "Time")}


def _column_buffers(data, typestring=None):
    """(typestring, nrows, values, missing, sizes, chars) of a column given as a numpy array (fixed width), a numpy masked array
    (Union{T,Missing}), a (values, missing) pair, a FlatStringsVector, or a sequence of str / None."""
    if isinstance(data, FlatStringsVector):
        sizes = np.ascontiguousarray(data.sizes, dtype=np.int32)
        chars = np.frombuffer(bytes(data.data), dtype=np.uint8) if not isinstance(data.data, np.ndarray) else np.ascontiguousarray(data.data, dtype=np.uint8)
        ts = typestring or ("Missing(String)" if (sizes < 0).any() else "String")
        return ts, len(sizes), None, None, sizes, chars
    if isinstance(data, np.ma.MaskedArray):
        data = (np.ma.getdata(data), np.ma.getmaskarray(data))
    if isinstance(data, tuple) and len(data) == 2 and isinstance(data[0], np.ndarray):
        vals, miss = np.ascontiguousarray(data[0]), np.ascontiguousarray(data[1], dtype=np.uint8)
        base = _TYPESTR_OF.get(vals.dtype)
        if base is None:
            raise ArgumentError(f"{vals.dtype} is not available as stored column type")
        vals = np.where(miss.astype(bool), np.zeros((), dtype=vals.dtype), vals)       # bytes under a missing flag are unspecified: write zeros
        return typestring or f"Missing({base})", len(vals), np.ascontiguousarray(vals), miss, None, None
    if isinstance(data, np.ndarray) and data.dtype.kind != "O" and data.dtype.kind not in "US":
        base = _TYPESTR_OF.get(data.dtype)
        if base is None:
            raise ArgumentError(f"{data.dtype} is not available as stored column type")
        return typestring or base, len(data), np.ascontiguousarray(data), None, None, None
    items = list(data)
    if all(x is None or isinstance(x, str) for x in items):
        enc = [None if x is None else x.encode("utf-8") for x in items]
        sizes = np.array([-1 if b is None else len(b) for b in enc], dtype=np.int32)
        chars = np.frombuffer(b"".join(b for b in enc if b), dtype=np.uint8)
        ts = typestring or ("Missing(String)" if any(b is None for b in enc) else "String")
        return ts, len(items), None, None, sizes, chars
    if any(x is None for x in items):
        miss = np.array([x is None for x in items], dtype=np.uint8)
        vals = np.array([0 if x is None else x for x in items])
        return _column_buffers((vals, miss), typestring)
    return _column_buffers(np.array(items), typestring)


def write_column_file(path: str, col_id: int, typestring: str, block_size: int, nrows: int, vals, miss, sizes, chars, device=None):
    """dfdb_write_column_file: bodies assembled, LZ4-compressed and compacted on the device, framed on the host."""
    _capi.init(device)
    comp, unc = C.c_int64(), C.c_int64()
    ptr = lambda a: a.ctypes.data if a is not None and a.size else None      # noqa: E731
    try:
        _capi.check(_capi.lib().dfdb_write_column_file(path.encode(), col_id, typestring.encode(), block_size, nrows, ptr(vals), ptr(miss), ptr(sizes),
                                                       ptr(chars), 0 if chars is None else chars.size, C.byref(comp), C.byref(unc)))
    except DfdbError as e:
        if e.code == _capi.ERR_IO:
            raise RuntimeError(str(e)) from None
        _raise(e)
    return comp.value, unc.value


def _write_meta(path: str, block_size: int, cols):
    n = len(cols)
    ids = (C.c_int64 * max(n, 1))(*[c[0] for c in cols])
    names = (C.c_char_p * max(n, 1))(*[c[1].encode() for c in cols])
    types = (C.c_char_p * max(n, 1))(*[c[2].encode() for c in cols])
    try:
        _capi.check(_capi.lib().dfdb_write_table_meta(path.encode(), block_size, n, ids, names, types))
    except DfdbError as e:
        if e.code == _capi.ERR_IO:
            raise RuntimeError(str(e)) from None
        _raise(e)


def create_table(path: str, columns, block_size: int = 65536, mode: int = _capi.LOAD_HBM, device=None) -> DFTable:
    """create_table(path; from = df, block_size) (creators.jl:81-89): `columns` is a dict name -> data or a list of
    (name, data) / (name, typestring, data); all columns must have the same number of rows.  The column files are written by
    the device write path (same on-disk format: the reference opens the table)."""
    if os.path.isdir(path):
        raise RuntimeError(f"Table {path} already exists")                     # filesystem.jl:36
    items = [(k, None, v) for k, v in columns.items()] if isinstance(columns, dict) else [(c[0], None, c[1]) if len(c) == 2 else tuple(c) for c in columns]
    bufs = [(name,) + _column_buffers(data, ts) for name, ts, data in items]
    if len({b[2] for b in bufs}) > 1:
        raise ArgumentError("Column and table have different sizes")
    _write_meta(path, block_size, [(i + 1, b[0], b[1]) for i, b in enumerate(bufs)])
    for i, (name, ts, nrows, vals, miss, sizes, chars) in enumerate(bufs):
        write_column_file(path, i + 1, ts, block_size, nrows, vals, miss, sizes, chars, device)
    return DFTable(path, mode=mode, device=device)


def _full_table_projection(table: DFTable) -> Projection:
    return Projection([(m.name, ColRef(m.name, m.type, m.id)) for m in table.meta])


class DFView:
    """view.jl:26-31 -- lazy (table, projection, selection)."""

    def __init__(self, table: DFTable, proj: Projection | None = None, sel: SelectionQueue | None = None):
        d = self.__dict__
        d["table"] = table
        d["projection"] = proj if proj is not None else _full_table_projection(table)
        d["selection"] = sel if sel is not None else SelectionQueue()

    def __eq__(self, other):
        return isinstance(other, DFView) and self.table == other.table and self.projection == other.projection and \
            self.selection == other.selection

    def __hash__(self):
        return hash((self.table.path, self.projection, self.selection))

    def names(self):
        return self.projection.keys()

    def __getattr__(self, name):
        if name.startswith("_"):
            raise AttributeError(name)
        return self[:, name]

    def __setattr__(self, name, value):
        # Base.setproperty!(v::DFView, name, value::DFColumn) column.jl:77-81
        if isinstance(value, DFColumn):
            if not issameselection(self, value.view):
                raise ArgumentError("Can't add column with another selection")
            self.__dict__["projection"] = add(self.projection, [(name, value.view.projection.cols[0][1])])
        else:
            self.__dict__[name] = value

    def __getitem__(self, key):
        if not isinstance(key, tuple) or len(key) != 2:
            raise TypeError("DFView is indexed as v[selection, projection]")
        s, p = key
        # getindex overloads view.jl:120-135
        if isinstance(p, (str, int, np.integer)) and not isinstance(p, bool):
            col = DFColumn(selproj(self, s, [p]))
            if isinstance(s, (int, np.integer)) and not isinstance(s, bool):
                return col[1]
            return col
        if isinstance(s, (int, np.integer)) and not isinstance(s, bool):
            fr = materialize(selproj(self, [int(s)], p))
            if fr.nrow() == 0:
                raise IndexError("BoundsError")
            return {n: (c[0] if not isinstance(c, np.ndarray) else c[0].item()) for n, c in zip(fr.names, fr.columns)}
        return selproj(self, s, p)

    def __repr__(self):
        return f"View of table {self.table.path}\n{self.projection!r}\n{self.selection!r}"


def view_from_columns(**cols) -> DFView:
    """DFView(cols::NamedTuple{..., <:Tuple{Vararg{DFColumn}}}) / DFView(; kwargs...) column.jl:143-164"""
    ts = None
    for c in cols.values():
        cur = (c.view.table, c.view.selection)
        if ts is None:
            ts = cur
        elif cur != ts:
            raise ArgumentError("All columns must have same selection and table")
    return DFView(ts[0], Projection([(k, c.view.projection.cols[0][1]) for k, c in cols.items()]), ts[1])


def issametable(a: DFView, b: DFView) -> bool:
    return a.table == b.table


def issameselection(a: DFView, b: DFView) -> bool:
    return issametable(a, b) and a.selection == b.selection


def selection(v: DFView, el) -> DFView:
    """view.jl:60-72, column.jl:72-75"""
    if isinstance(el, slice) and el == _COLON:
        return v
    if isinstance(el, DFColumn):
        # An expression built on the bare table (empty selection) plays the reference's Pair form
        # `cols => f` (view.jl:64-70), which is evaluated against the view's own columns; any other
        # selection must match (column.jl:72-75).
        if not issametable(v, el.view) or (v.selection != el.view.selection and not el.view.selection.isempty()):
            raise ArgumentError("col must have same selection as view")
        el = el.view.projection.cols[0][1]
        if isinstance(el, ColRef):
            # a stored Bool column used as predicate: `col .== true`
            el = BlockBroadcasting("==", (el, True))
    elif isinstance(el, (np.ndarray, tuple, list)):
        el = tuple(int(x) for x in el)
    elif isinstance(el, np.integer):
        el = int(el)
    return DFView(v.table, v.projection, add(v.selection, el))


def _proj_elem(v: DFView, elem):
    if isinstance(elem, str):
        pc = v.projection[elem].cols
        if not pc:
            raise ArgumentError(f"view don't have column :{elem}")
        return pc[0][1]
    if isinstance(elem, DFColumn):
        # bare-table expressions stand for the Pair form `name = cols => f` (view.jl:81-97)
        if not issametable(v, elem.view) or (v.selection != elem.view.selection and not elem.view.selection.isempty()):
            raise ArgumentError("All columns must have same selection and table")
        return elem.view.projection.cols[0][1]
    raise TypeError(f"unsupported projection element {elem!r}")


def projection(v: DFView, p) -> DFView:
    """view.jl:91-109"""
    if isinstance(p, slice) and p == _COLON:
        return v
    if isinstance(p, dict):
        return DFView(v.table, Projection([(k, _proj_elem(v, e)) for k, e in p.items()]), v.selection)
    if isinstance(p, JRange):
        return DFView(v.table, v.projection[p], v.selection)
    p = list(p)
    if p and isinstance(p[0], str):
        return DFView(v.table, Projection([(k, _proj_elem(v, k)) for k in p]), v.selection)
    if any(int(i) < 1 or int(i) > len(v.projection) for i in p):
        raise IndexError("BoundsError")
    return DFView(v.table, v.projection[[int(i) for i in p]], v.selection)


def selproj(v: DFView, select, project) -> DFView:
    """view.jl:112-118"""
    return projection(selection(v, select), project)


# -----------------------------------------------------------------------------------------------
# scans through the C ABI


def _scan_handle(v: DFView):
    t = v.table
    key = (v.projection, v.selection)
    h = t._scans.get(key)
    if h is None:
        plan = encode_plan(v.selection, v.projection)
        h = C.c_void_p()
        try:
            _capi.check(_capi.lib().dfdb_scan_prepare(t._h, plan, len(plan), C.byref(h)))
        except DfdbError as e:
            _raise(e)
        if len(t._scans) > 256:
            t._drop_scans()
        t._scans[key] = h
    need = list(v.projection.required_columns())
    for e in v.selection.queue:
        if isinstance(e, BlockBroadcasting):
            need += [n for n in required_columns(e) if n not in need]
    _capi.init(t._device)
    t.load(need)
    return h


def plan_bytes(v) -> bytes:
    """Serialized plan of a view / column (what dfdb_scan_prepare receives)."""
    if isinstance(v, DFColumn):
        v = v.view
    if isinstance(v, DFTable):
        v = DFView(v)
    return encode_plan(v.selection, v.projection)


def nrow(v) -> int:
    """view.jl:192-206 (BlockRowsIterator count pass); shard-local when the table is sharded."""
    if isinstance(v, DFTable):
        v = DFView(v)
    if isinstance(v, DFColumn):
        v = v.view
    n = C.c_int64()
    try:
        _capi.check(_capi.lib().dfdb_scan_count(_scan_handle(v), C.byref(n)))
    except DfdbError as e:
        _raise(e)
    return n.value


def resolve_sharded_selection(views, allgather=None):
    """Range / index-vector stages behind a predicate rank rows among ALL survivors (selection.jl:94-111); on a
    sharded table every shard therefore needs the survivor counts of the lower-ranked shards before such a stage.
    `views`: the same view on every shard held by this process (one per rank in the multi-process case, all of
    them in a single-process test); `allgather(count) -> [count of every rank]` for the multi-process case."""
    views = [DFView(v) if isinstance(v, DFTable) else (v.view if isinstance(v, DFColumn) else v) for v in views]
    handles = [_scan_handle(v) for v in views]
    L = _capi.lib()
    while True:
        counts, pending = [], []
        for h in handles:
            n, p = C.c_int64(), C.c_int32()
            try:
                _capi.check(L.dfdb_scan_exchange_count(h, C.byref(n), C.byref(p)))
            except DfdbError as e:
                _raise(e)
            counts.append(n.value)
            pending.append(p.value)
        if not any(pending):
            return
        if allgather is not None:           # one view per process: `counts` of all ranks come from the collective
            allc = allgather(counts[0])
            _capi.check(L.dfdb_scan_exchange_offset(handles[0], sum(allc[:views[0].table.rank])))
        else:                               # every shard lives in this process, in rank order
            by_rank = sorted(range(len(views)), key=lambda i: views[i].table.rank)
            run = 0
            for i in by_rank:
                _capi.check(L.dfdb_scan_exchange_offset(handles[i], run))
                run += counts[i]


def ncol(v) -> int:
    return len(v.meta) if isinstance(v, DFTable) else len(v.projection)


def size(v, dim=None):
    if isinstance(v, DFTable):
        v = DFView(v)
    if dim is None:
        return (nrow(v), ncol(v))
    if dim not in (1, 2):
        raise ArgumentError("DFView have only 2 dimensions")
    return nrow(v) if dim == 1 else ncol(v)


def _np_dtype(kind_name: str, elsize: int):
    if kind_name in _NP:
        return np.dtype(_NP[kind_name])
    return np.dtype((np.void, elsize))


def materialize(v):
    """materialization.jl:27-52: DFView/DFTable -> Frame ; DFColumn -> vector."""
    if isinstance(v, DFColumn):
        return materialize(v.view).columns[0]
    if isinstance(v, DFTable):
        v = DFView(v)
    L = _capi.lib()
    h = _scan_handle(v)
    ncols = len(v.projection)
    n = C.c_int64()
    sb = (C.c_int64 * max(ncols, 1))()
    try:
        _capi.check(L.dfdb_scan_materialize_sizes(h, C.byref(n), sb))
    except DfdbError as e:
        _raise(e)
    nrows = n.value
    outs = (_capi.OutCol * max(ncols, 1))()
    keep = []
    for i in range(ncols):
        kind, nullable, elsize = C.c_int32(), C.c_int32(), C.c_int32()
        _capi.check(L.dfdb_scan_proj_type(h, i, C.byref(kind), C.byref(nullable), C.byref(elsize)))
        kname = _capi.KIND_NAMES[kind.value]
        if kname == "String":
            sizes = _capi.result_array(nrows, np.int32)
            chars = _capi.result_array(sb[i], np.uint8)
            outs[i].str_sizes = sizes.ctypes.data
            outs[i].str_chars = chars.ctypes.data
            keep.append(("str", sizes, chars, sb[i]))
        else:
            vals = _capi.result_array(nrows, _np_dtype(kname, elsize.value))
            outs[i].values = vals.ctypes.data
            miss = None
            if nullable.value:
                miss = _capi.result_array(nrows, np.uint8)
                outs[i].missing = miss.ctypes.data
            keep.append(("fix", vals, miss, 0))
    try:
        _capi.check(L.dfdb_scan_materialize(h, outs, ncols))
    except DfdbError as e:
        _raise(e)
    cols = []
    for tag, a, b, nb in keep:
        if tag == "str":
            cols.append(FlatStringsVector(a[:nrows], b[:nb]))
        elif b is not None:
            cols.append(np.ma.MaskedArray(a[:nrows], mask=b[:nrows].view(np.bool_)))
        else:
            cols.append(a[:nrows])
    return Frame(v.projection.keys(), cols)


def head(v, rows: int = 10):
    """materialization.jl:64-66"""
    if isinstance(v, DFTable):
        v = DFView(v)
    return materialize(v[JRange.make(1, rows), :])


def selection_mask(v: DFView) -> np.ndarray:
    """Parity hook (dfdb_scan_mask): Bool per table row, True where the view selects the row."""
    t = v.table
    total = t.total_rows()
    nwords = (total + 63) // 64
    words = np.zeros(max(nwords, 1), dtype=np.uint64)
    try:
        _capi.check(_capi.lib().dfdb_scan_mask(_scan_handle(v), words.ctypes.data, len(words)))
    except DfdbError as e:
        _raise(e)
    bits = np.unpackbits(words.view(np.uint8), bitorder="little")[:total]
    return bits.astype(bool)


def selection_indices(v: DFView) -> np.ndarray:
    """Parity hook (dfdb_scan_indices): 1-based table row numbers of the selected rows, ascending."""
    t = v.table
    cap = max(t.total_rows(), 1)
    idx = np.zeros(cap, dtype=np.int64)
    n = C.c_int64()
    try:
        _capi.check(_capi.lib().dfdb_scan_indices(_scan_handle(v), idx.ctypes.data, cap, C.byref(n)))
    except DfdbError as e:
        _raise(e)
    return idx[:n.value]


# -----------------------------------------------------------------------------------------------


def _check_same_selection(args):
    ts = None
    for a in args:
        if isinstance(a, DFColumn):
            cur = (a.view.table, a.view.selection)
            if ts is None:
                ts = cur
            elif cur != ts:
                raise ArgumentError("All columns in broadcast must have same selection and table")
    return ts


def _bc(f: str, *args):
    """Base.copy(::Broadcasted{DFColumnStyle}) columnbroadcast.jl:46-62"""
    for a in args:
        if isinstance(a, (np.ndarray, list, tuple)):
            # arrays take part in ordinary array broadcasting in Julia, never in a lazy column
            raise ArgumentError("Cannot do BlockBroadcasting with arrays")
    ts = _check_same_selection(args)
    conv = tuple(a.view.projection.cols[0][1] if isinstance(a, DFColumn) else (a.item() if isinstance(a, np.generic) else a) for a in args)
    bb = BlockBroadcasting(f, conv)
    return DFColumn(DFView(ts[0], Projection([("a", bb)]), ts[1]))


class DFColumn:
    """column.jl:30-37 -- lazy one-column view; Python operators play Julia's dot-broadcasting."""

    def __init__(self, view: DFView):
        if len(view.projection) != 1:
            raise ArgumentError("Column projection must contains singe element")
        self.view = view

    def eltype(self) -> JType | None:
        return self.view.projection.coltype(1)

    def same_as(self, other) -> bool:
        """Base.:(==)(a::DFColumn, b::DFColumn) column.jl:39 (Python's == is the broadcast comparison)."""
        return isinstance(other, DFColumn) and self.view == other.view

    __hash__ = object.__hash__

    # broadcasting
    def __eq__(self, o): return _bc("==", self, o)
    def __ne__(self, o): return _bc("!=", self, o)
    def __lt__(self, o): return _bc("<", self, o)
    def __le__(self, o): return _bc("<=", self, o)
    def __gt__(self, o): return _bc(">", self, o)
    def __ge__(self, o): return _bc(">=", self, o)
    def __and__(self, o): return _bc("&", self, o)
    def __rand__(self, o): return _bc("&", o, self)
    def __or__(self, o): return _bc("|", self, o)
    def __ror__(self, o): return _bc("|", o, self)
    def __xor__(self, o): return _bc("xor", self, o)
    def __invert__(self): return _bc("!", self)
    def __add__(self, o): return _bc("+", self, o)
    def __radd__(self, o): return _bc("+", o, self)
    def __sub__(self, o): return _bc("-", self, o)
    def __rsub__(self, o): return _bc("-", o, self)
    def __mul__(self, o): return _bc("*", self, o)
    def __rmul__(self, o): return _bc("*", o, self)
    def __truediv__(self, o): return _bc("/", self, o)
    def __rtruediv__(self, o): return _bc("/", o, self)
    def __mod__(self, o): return _bc("%", self, o)
    def __rmod__(self, o): return _bc("%", o, self)
    def __neg__(self): return _bc("neg", self)

    def __bool__(self):
        raise TypeError("a lazy DFColumn has no truth value; use & | ~ for element-wise logic")

    def __len__(self):
        return nrow(self.view)

    def __getitem__(self, i):
        # column.jl:60-67, 93-99
        if isinstance(i, DFColumn):
            if self.view.selection != i.view.selection:
                raise ArgumentError("cols must have same selections")
            return DFColumn(selection(self.view, i))
        if isinstance(i, (int, np.integer)) and not isinstance(i, bool):
            res = materialize(DFColumn(selection(self.view, int(i))))
            if len(res) == 0:
                raise IndexError("BoundsError")
            x = res[0]
            return x.item() if isinstance(x, np.generic) else x
        return DFColumn(selection(self.view, i))

    def __iter__(self):
        return iter(materialize(self).tolist())

    def __repr__(self):
        return f"DFColumn{{{self.eltype()}}}"


def startswith(col: DFColumn, prefix: str): return _bc("startswith", col, prefix)
def endswith(col: DFColumn, suffix: str): return _bc("endswith", col, suffix)
def ismissing(col: DFColumn): return _bc("ismissing", col)
def coalesce(col: DFColumn, default): return _bc("coalesce", col, default)


def isin(col: DFColumn, values):
    """`in.(col, Ref(values))`"""
    ts = _check_same_selection((col,))
    bb = BlockBroadcasting("in", (col.view.projection.cols[0][1], InSet(values)))
    return DFColumn(DFView(ts[0], Projection([("a", bb)]), ts[1]))


# -----------------------------------------------------------------------------------------------
# aggregates (Base folds over iterate(::DFColumn), column.jl:102-126)


def aggregate(col: DFColumn) -> _capi.Agg:
    """Raw dfdb_agg of the column's selected rows (shard-local when sharded)."""
    out = _capi.Agg()
    try:
        _capi.check(_capi.lib().dfdb_scan_aggregate(_scan_handle(col.view), 0, C.byref(out)))
    except DfdbError as e:
        _raise(e)
    return out


def aggregate_all(col: DFColumn) -> _capi.Agg:
    """dfdb_scan_aggregate_all: every rank aggregates its shard, the partials are all-gathered over the library's NCCL
    communicator (dist.comm_init_from_torch / dfdb_comm_init) and folded in rank order; every rank gets the same bits."""
    out = _capi.Agg()
    try:
        _capi.check(_capi.lib().dfdb_scan_aggregate_all(_scan_handle(col.view), 0, C.byref(out)))
    except DfdbError as e:
        _raise(e)
    return out


def nrow_all(v) -> int:
    """dfdb_scan_count_all: nrow(v) over all shards (survivor-count exchanges resolved over the communicator first)."""
    if isinstance(v, DFTable):
        v = DFView(v)
    if isinstance(v, DFColumn):
        v = v.view
    n = C.c_int64()
    try:
        _capi.check(_capi.lib().dfdb_scan_count_all(_scan_handle(v), C.byref(n)))
    except DfdbError as e:
        _raise(e)
    return n.value


def _group_call(view, by, cols, fn, *args):
    """Runs one of the group-by calls `fn` over the view's `by` + value columns (projections 0.. in that order); returns the
    scan handle and the number of groups."""
    if isinstance(view, DFTable):
        view = DFView(view)
    vals = list(cols.values())
    h = _scan_handle(view[:, by + vals])
    ng = C.c_int64()
    try:
        _capi.check(getattr(_capi.lib(), fn)(h, *args, C.byref(ng)))
    except DfdbError as e:
        _raise(e)
    return h, ng.value


def _group_projs(by, cols):
    nk, nv = len(by), len(cols)
    return (C.c_int32 * nk)(*range(nk)), nk, (C.c_int32 * max(nv, 1))(*range(nk, nk + nv)), nv


def _group_results(h, n, nvals):
    """first rows (1-based table rows) and the n x nvals dfdb_agg of the handle's group-by result"""
    first = np.zeros(max(n, 1), dtype=np.int64)
    aggs = (_capi.Agg * max(n * nvals, 1))()
    _capi.check(_capi.lib().dfdb_scan_group_results(h, first.ctypes.data, aggs))
    return first[:n], aggs


def _group_dict(view, cols, keys, first, aggs):
    """groupreduce's result: the key columns (dict of lists), first rows, and per value column the reductions of every group"""
    if isinstance(view, DFTable):
        view = DFView(view)
    n = len(first)
    out = dict(keys)
    out["first_row"] = first.tolist()
    for j, (name, src) in enumerate(cols.items()):
        rec = {"count": [], "nmissing": [], "sum": [], "min": [], "max": [], "mean": []}
        isf = view.table.getmeta(src).type.is_float if hasattr(view.table.getmeta(src).type, "is_float") else view.table.getmeta(src).typestring.replace("Missing(", "").startswith("Float")
        for g in range(n):
            a = aggs[g * len(cols) + j]
            nv = a.count - a.nmissing
            rec["count"].append(a.count)
            rec["nmissing"].append(a.nmissing)
            if a.value_class == 0:
                rec["sum"].append(0.0 if isf else 0); rec["min"].append(None); rec["max"].append(None); rec["mean"].append(None)
                continue
            # (sum_f64_lo is 0 in a local result; a merged one carries the compensated pair)
            sm = a.sum_f64 + a.sum_f64_lo if isf else (a.sum_i64 & ((1 << 64) - 1) if a.value_class == 2 else a.sum_i64)
            rec["sum"].append(sm)
            rec["min"].append(a.min_f64 if isf else (a.min_i64 & ((1 << 64) - 1) if a.value_class == 2 else a.min_i64))
            rec["max"].append(a.max_f64 if isf else (a.max_i64 & ((1 << 64) - 1) if a.value_class == 2 else a.max_i64))
            rec["mean"].append(sm / nv if nv else None)
        out[name] = rec
    if not cols:
        out["ngroups"] = n
    return out


def groupreduce(view, by, **cols):
    """groupreduce(view, by; cols...) -- finishes the reference's stub (src/tables/aggregate.jl:1-36): groups of the view's
    selected rows by the tuple of `by` columns, numbered in order of first appearance like the stub's RobinDict, and per group
    the reductions of the value columns.  `cols`: result name = source column name.  Returns a dict: every `by` column -> list
    of key values (None = missing), "count" -> rows per group, and per result name a dict of lists count / nmissing / sum /
    min / max / mean (None where the group has no non-missing value)."""
    if isinstance(view, DFTable):
        view = DFView(view)
    by = [by] if isinstance(by, str) else list(by)
    h, n = _group_call(view, by, cols, "dfdb_scan_groupreduce", *_group_projs(by, cols))
    first, aggs = _group_results(h, n, len(cols))
    # key values: the key columns at the rows where the groups first appear (an index-vector selection of the TABLE)
    if n:
        keys = materialize(DFView(view.table)[first.tolist(), by]).to_dict()
    else:
        keys = {k: [] for k in by}
    return _group_dict(view, cols, keys, first, aggs)


def _group_keys(h, n, nkeys):
    """the handle's group-by key columns (dfdb_scan_group_keys), as materialize returns columns"""
    L = _capi.lib()
    nb = (C.c_int64 * nkeys)()
    _capi.check(L.dfdb_scan_group_key_bytes(h, nb))
    outs = (_capi.OutCol * nkeys)()
    wraps = [_result_column(h, k, n, nb[k], outs[k]) for k in range(nkeys)]
    _capi.check(L.dfdb_scan_group_keys(h, outs, nkeys))
    return [w() for w in wraps]


def groupreduce_all(view, by, **cols):
    """dfdb_scan_groupreduce_all: groupreduce over ALL shards -- every rank's groups (keys, first rows, raw aggregates) are
    all-gathered over the library's NCCL communicator, merged on the device and folded in rank order; every rank gets the same
    result.  Unsharded without a communicator: the local pass.  Same dict as groupreduce, with the keys returned by the library
    and Float64 sums as sum_f64 + sum_f64_lo."""
    by = [by] if isinstance(by, str) else list(by)
    h, n = _group_call(view, by, cols, "dfdb_scan_groupreduce_all", *_group_projs(by, cols))
    first, aggs = _group_results(h, n, len(cols))
    return _group_dict(view, cols, Frame(by, _group_keys(h, n, len(by))).to_dict(), first, aggs)


def groupreduce_local(view, by, **cols):
    """The shard-local half of groupreduce_all: this shard's groups as a part for groupreduce_merge -- a dict of "keys" (one
    column per `by` column, as materialize returns it), "first_rows" (1-based table rows) and "aggs" (the raw dfdb_agg, n x
    len(cols), row-major)."""
    by = [by] if isinstance(by, str) else list(by)
    h, n = _group_call(view, by, cols, "dfdb_scan_groupreduce", *_group_projs(by, cols))
    first, aggs = _group_results(h, n, len(cols))
    return {"keys": _group_keys(h, n, len(by)), "first_rows": first, "aggs": list(aggs)[:n * len(cols)]}


def groupreduce_merge(view, by, parts, **cols):
    """dfdb_scan_groupreduce_merge: merges per-rank groupreduce_local parts carried by the host (`parts` in rank order) into the
    groups of the whole table, on the device; same dict as groupreduce_all."""
    by = [by] if isinstance(by, str) else list(by)
    nk, nv = len(by), len(cols)
    keep, outs = [], (_capi.OutCol * max(len(parts) * nk, 1))()
    pn = (C.c_int64 * max(len(parts), 1))()
    pb = (C.c_int64 * max(len(parts) * nk, 1))()
    for r, p in enumerate(parts):
        pn[r] = len(p["first_rows"])
        for k, col in enumerate(p["keys"]):
            pb[r * nk + k] = _part_outcol(col, outs[r * nk + k], keep)
    first = np.ascontiguousarray(np.concatenate([np.asarray(p["first_rows"], dtype=np.int64) for p in parts]) if parts else np.zeros(1, np.int64))
    allaggs = [a for p in parts for a in p["aggs"]]
    aggs = (_capi.Agg * max(len(allaggs), 1))(*allaggs)
    kp, _, _, _ = _group_projs(by, cols)
    h, n = _group_call(view, by, cols, "dfdb_scan_groupreduce_merge", kp, nk, nv, outs, first.ctypes.data_as(C.POINTER(C.c_int64)), aggs, pn, pb,
                       len(parts))
    first, aggs = _group_results(h, n, nv)
    return _group_dict(view, cols, Frame(by, _group_keys(h, n, nk)).to_dict(), first, aggs)


def _result_column(h, proj, n, nbytes, out):
    """Buffers for a result column of projection `proj`'s type (n values, nbytes chars), set in the OutCol `out`; returns a
    function that wraps them, once the library has filled them, as materialize returns a column: ndarray (fixed width),
    MaskedArray (nullable), FlatStringsVector (String, None = missing)."""
    kind, nullable, elsize = C.c_int32(), C.c_int32(), C.c_int32()
    _capi.check(_capi.lib().dfdb_scan_proj_type(h, proj, C.byref(kind), C.byref(nullable), C.byref(elsize)))
    kname = _capi.KIND_NAMES[kind.value]
    if kname == "String":
        sizes, chars = _capi.result_array(n, np.int32), _capi.result_array(nbytes, np.uint8)
        out.str_sizes, out.str_chars = sizes.ctypes.data, chars.ctypes.data
        return lambda: FlatStringsVector(sizes[:n], chars[:nbytes])
    vals = _capi.result_array(n, _np_dtype(kname, elsize.value))
    miss = _capi.result_array(n, np.uint8) if nullable.value else None
    out.values = vals.ctypes.data
    out.missing = miss.ctypes.data if miss is not None else None
    if miss is not None:
        return lambda: np.ma.MaskedArray(vals[:n], mask=miss[:n].view(np.bool_))
    return lambda: vals[:n]


def _part_outcol(p, out, keep):
    """points the OutCol `out` at a host column laid out as materialize returns it (buffers appended to `keep`); returns its
    char bytes (0 for fixed width)"""
    if isinstance(p, FlatStringsVector):
        sizes = np.ascontiguousarray(p.sizes, dtype=np.int32)
        chars = np.frombuffer(bytes(p.data), dtype=np.uint8) if len(p.data) else np.zeros(1, np.uint8)
        out.str_sizes, out.str_chars = sizes.ctypes.data, chars.ctypes.data
        keep += [sizes, chars]
        return len(p.data)
    vals = np.ascontiguousarray(np.ma.getdata(p))
    out.values = vals.ctypes.data
    keep.append(vals)
    if isinstance(p, np.ma.MaskedArray):
        miss = np.ascontiguousarray(np.ma.getmaskarray(p), dtype=np.uint8)
        out.missing = miss.ctypes.data
        keep.append(miss)
    return 0


def _unique_call(col: DFColumn, fn: str, *args):
    """Runs dfdb_scan_unique / _all / _merge on the column's scan and copies the handle's result out, in the layout materialize
    returns: ndarray (fixed width), MaskedArray (nullable), FlatStringsVector (String, None = missing)."""
    L = _capi.lib()
    h = _scan_handle(col.view)
    n, nb = C.c_int64(), C.c_int64()
    try:
        _capi.check(getattr(L, fn)(h, *args, C.byref(n), C.byref(nb)))
    except DfdbError as e:
        _raise(e)
    out = _capi.OutCol()
    wrap = _result_column(h, 0, n.value, nb.value, out)
    _capi.check(L.dfdb_scan_unique_values(h, C.byref(out)))
    return wrap()


def unique(col: DFColumn):
    """Base.unique(col): the distinct values of the column's selected rows in order of first appearance, equality isequal
    (missing once, one NaN, -0.0 != 0.0, strings by bytes).  Shard-local when the table is sharded."""
    return _unique_call(col, "dfdb_scan_unique", 0)


def unique_all(col: DFColumn):
    """dfdb_scan_unique_all: unique over ALL shards -- every rank's local result is all-gathered over the library's NCCL
    communicator and merged on the device; every rank gets the same values.  Unsharded without a communicator: unique(col)."""
    return _unique_call(col, "dfdb_scan_unique_all", 0)


def unique_merge(col: DFColumn, parts):
    """dfdb_scan_unique_merge: merges per-rank unique results carried by the host (`parts` in rank order, each as unique
    returns it) into the unique of the whole column: every value where it first appears in the rank-order concatenation."""
    bufs, outs = [], (_capi.OutCol * max(len(parts), 1))()
    pn = (C.c_int64 * max(len(parts), 1))()
    pb = (C.c_int64 * max(len(parts), 1))()
    for i, p in enumerate(parts):
        pn[i] = len(p)
        pb[i] = _part_outcol(p, outs[i], bufs)
    return _unique_call(col, "dfdb_scan_unique_merge", outs, pn, pb, len(parts))


def pruned_blocks(v):
    """(blocks the zone maps ruled out in the view's last scan, blocks of the shard)"""
    if isinstance(v, DFColumn):
        v = v.view
    p, n = C.c_int64(), C.c_int64()
    _capi.check(_capi.lib().dfdb_scan_pruned(_scan_handle(v), C.byref(p), C.byref(n)))
    return p.value, n.value


def fold(partials) -> _capi.Agg:
    """dfdb_agg_fold: fixed rank-order combination of per-shard partials."""
    arr = (_capi.Agg * len(partials))(*partials)
    out = _capi.Agg()
    _capi.check(_capi.lib().dfdb_agg_fold(arr, len(partials), C.byref(out)))
    return out


def _is_bool_expr(col: DFColumn) -> bool:
    e = col.view.projection.cols[0][1]
    return isinstance(e, BlockBroadcasting) and col.eltype() == JType("Bool")


def agg_sum(a: _capi.Agg, eltype: JType | None):
    if a.nmissing:
        return None                      # missing + x == missing
    if a.value_class == 3 or (eltype is not None and eltype.name.startswith("Float")):
        s = a.sum_f64 + a.sum_f64_lo
        return float(np.float32(s)) if eltype is not None and eltype.name == "Float32" else s
    if a.value_class == 2:
        return a.sum_i64 & 0xFFFFFFFFFFFFFFFF
    return a.sum_i64


def agg_min(a: _capi.Agg):
    if a.count == 0:
        raise ArgumentError("reducing over an empty collection is not allowed")
    if a.nmissing:
        return None
    if a.value_class == 3 or a.has_nan:
        return math.nan if a.has_nan else a.min_f64
    if a.value_class == 2:
        return a.min_i64 & 0xFFFFFFFFFFFFFFFF
    return bool(a.min_i64) if a.value_class == 4 else a.min_i64


def agg_max(a: _capi.Agg):
    if a.count == 0:
        raise ArgumentError("reducing over an empty collection is not allowed")
    if a.nmissing:
        return None
    if a.value_class == 3 or a.has_nan:
        return math.nan if a.has_nan else a.max_f64
    if a.value_class == 2:
        return a.max_i64 & 0xFFFFFFFFFFFFFFFF
    return bool(a.max_i64) if a.value_class == 4 else a.max_i64


def sum(col: DFColumn):  # noqa: A001  (mirrors Base.sum)
    if _is_bool_expr(col):
        # sum of a lazy Bool column == number of selected rows where it holds
        return nrow(selection(col.view, col))
    return agg_sum(aggregate(col), col.eltype())


def count(col: DFColumn) -> int:
    """count(col) for a Bool column; length for anything else."""
    if col.eltype() == JType("Bool"):
        return sum(col)
    return len(col)


def minimum(col: DFColumn):
    return agg_min(aggregate(col))


def maximum(col: DFColumn):
    return agg_max(aggregate(col))


def mean(col: DFColumn):
    a = aggregate(col)
    if a.nmissing:
        return None
    if a.count == 0:
        return math.nan
    if a.value_class == 3 or a.has_nan:
        return (a.sum_f64 + a.sum_f64_lo) / a.count
    s = a.sum_i64 & 0xFFFFFFFFFFFFFFFF if a.value_class == 2 else a.sum_i64
    return s / a.count
