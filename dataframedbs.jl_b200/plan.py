"""Lazy plan algebra of the scan path and its wire format.

Mirrors the reference's plan objects (names kept):
  ColRef, BlockBroadcasting      /root/reference/src/tables/broadcast.jl:2-17
  SelectionQueue, add, _new_queue /root/reference/src/tables/selection.jl:4-60
  Projection, add                 /root/reference/src/tables/projection.jl:1-30
and serialises them into the byte plan consumed by `dfdb_scan_prepare` (include/dfdb_b200.h).

Wire format (little endian):
  u32 magic 'DFP1' | u32 nstages | stage* | u32 nproj | proj*
  stage := u8 1 RANGE  i64 start, i64 step, i64 stop      (Julia 1-based inclusive range, `stop` = last(range))
         | u8 2 INDEXVEC u32 n, i64[n]                     (1-based row numbers)
         | u8 3 PRED  expr
  proj  := u8 1 COL i64 column_id | u8 2 EXPR expr
  expr  := u32 nops, postfix ops; op := u8 opcode [payload]

`in.(x, Ref(C))` is one of two ops after the ops of x:
  0x60 IN     u32 n, i64[n]                  C is all Int64, `==` semantics (what the encoders emit for that case)
  0x61 INSET  u8 semantics, u32 n, elem[n]   semantics 0 = `==` (Ref(vector or tuple)), 1 = isequal (Ref(Set))
  elem := u8 tag payload: 1 i64 | 2 u64 (values >= 2^63) | 3 f64 | 4 u32 length + bytes (String) | 5 u8 (Bool) | 6 (missing)
"""
from __future__ import annotations

import struct
from dataclasses import dataclass
from typing import Any, Sequence, Tuple, Union

MAGIC = 0x31504644

ST_RANGE, ST_INDEXVEC, ST_PRED = 1, 2, 3
PJ_COL, PJ_EXPR = 1, 2

OP_COL, OP_I64, OP_F64, OP_STR, OP_BOOL = 0x01, 0x02, 0x03, 0x04, 0x05
OP_EQ, OP_NE, OP_LT, OP_LE, OP_GT, OP_GE = 0x10, 0x11, 0x12, 0x13, 0x14, 0x15
OP_AND, OP_OR, OP_XOR, OP_NOT = 0x20, 0x21, 0x22, 0x23
OP_ADD, OP_SUB, OP_MUL, OP_DIV, OP_REM, OP_NEG = 0x30, 0x31, 0x32, 0x33, 0x34, 0x35
OP_ISMISSING, OP_COALESCE = 0x40, 0x41
OP_STARTSWITH, OP_ENDSWITH = 0x50, 0x51
OP_IN, OP_INSET = 0x60, 0x61
EL_I64, EL_U64, EL_F64, EL_STR, EL_BOOL, EL_MISSING = 1, 2, 3, 4, 5, 6

_BINARY = {
    "==": OP_EQ, "!=": OP_NE, "<": OP_LT, "<=": OP_LE, ">": OP_GT, ">=": OP_GE,
    "&": OP_AND, "|": OP_OR, "xor": OP_XOR,
    "+": OP_ADD, "-": OP_SUB, "*": OP_MUL, "/": OP_DIV, "%": OP_REM,
    "coalesce": OP_COALESCE, "startswith": OP_STARTSWITH, "endswith": OP_ENDSWITH,
}
_UNARY = {"!": OP_NOT, "neg": OP_NEG, "ismissing": OP_ISMISSING}

_INT_BITS = {"Int8": 8, "Int16": 16, "Int32": 32, "Int64": 64, "UInt8": 8, "UInt16": 16, "UInt32": 32, "UInt64": 64}
_FLOATS = {"Float32": 32, "Float64": 64}


class ArgumentError(ValueError):
    """Julia's ArgumentError (thrown by the reference's plan algebra)."""


@dataclass(frozen=True)
class JType:
    """Element type of a column or expression: a Julia type name plus `Union{T, Missing}`-ness."""
    name: str
    nullable: bool = False

    @staticmethod
    def parse(typestring: str) -> "JType":
        s = typestring.strip()
        if s.startswith("Missing(") and s.endswith(")"):
            return JType(s[8:-1].strip(), True)
        return JType(s, False)

    def typestring(self) -> str:
        return f"Missing({self.name})" if self.nullable else self.name

    def __str__(self) -> str:
        return f"Union{{Missing, {self.name}}}" if self.nullable else self.name


BOOL = JType("Bool")


@dataclass(frozen=True)
class ColRef:
    """broadcast.jl:2 -- reference to a stored column."""
    name: str
    type: JType
    col_id: int

    def eltype(self) -> JType:
        return self.type


# left operands of `in` whose values Julia would compare false against every number: refused in the INSET form
_IN_REFUSED = ("Date", "DateTime", "Time", "Char", "Float16", "Int128", "UInt128")


def _set_element(v):
    """One element of an `in` collection as a Python value: None (missing), bool, int, float or str.  NumPy floats widen
    exactly to float."""
    if v is None or isinstance(v, (bool, str)):
        return v
    if hasattr(v, "dtype") and hasattr(v, "item"):       # NumPy scalars
        v = v.item()
        if v is None or isinstance(v, (bool, str)):
            return v
    if isinstance(v, int):
        if not -(1 << 63) <= v < (1 << 64):
            raise ArgumentError(f"in() element {v} is outside the Int64 / UInt64 range")
        return v
    if isinstance(v, float):
        return v
    raise ArgumentError(f"in() element of type {type(v).__name__} is not available on the GPU path")


class InSet:
    """`Ref(C)` argument of `in.(x, Ref(C))` (test/broadcast.jl:63-71).  A list, tuple, ndarray, MaskedArray or
    FlatStringsVector is a vector: Julia's `in(x, ::Vector)`, `==` with three-valued logic.  A set or frozenset is a `Set`:
    `in(x, ::Set)`, isequal.  None is missing."""

    def __init__(self, values):
        self.isequal = isinstance(values, (set, frozenset))
        items = values.tolist() if hasattr(values, "tolist") else list(values)   # (a MaskedArray's masked entries are None)
        self.values = tuple(_set_element(v) for v in items)
        self.has_missing = any(v is None for v in self.values)
        # 0x60 for all-Int64 vectors, byte for byte what it always was; everything else 0x61
        self.legacy = not self.isequal and all(type(v) is int and v < (1 << 63) for v in self.values)
        self.wire = self._encode()

    def _encode(self) -> bytes:
        n = len(self.values)
        if self.legacy:
            return struct.pack("<BI", OP_IN, n) + struct.pack(f"<{n}q", *self.values)
        out = bytearray(struct.pack("<BBI", OP_INSET, int(self.isequal), n))
        for v in self.values:
            if v is None:
                out += struct.pack("<B", EL_MISSING)
            elif isinstance(v, bool):
                out += struct.pack("<BB", EL_BOOL, int(v))
            elif isinstance(v, int):
                out += struct.pack("<Bq", EL_I64, v) if v < (1 << 63) else struct.pack("<BQ", EL_U64, v)
            elif isinstance(v, float):
                out += struct.pack("<Bd", EL_F64, v)
            else:
                b = v.encode("utf-8")
                out += struct.pack("<BI", EL_STR, len(b)) + b
        return bytes(out)

    def __eq__(self, other):
        return isinstance(other, InSet) and self.wire == other.wire

    def __hash__(self):
        return hash(self.wire)

    def __repr__(self):
        return f"{'Set' if self.isequal else 'Ref'}({list(self.values)!r})"


Scalar = Union[int, float, str, bool, InSet]


def _scalar_type(v: Any) -> JType:
    if isinstance(v, bool):
        return BOOL
    if isinstance(v, int):
        return JType("Int64")
    if isinstance(v, float):
        return JType("Float64")
    if isinstance(v, str):
        return JType("String")
    if isinstance(v, InSet):
        return JType("Set{Int64}")
    # _check_sig_arg: arrays / iterables are rejected (broadcast.jl:23-29)
    raise ArgumentError("Cannot do BlockBroadcasting with arrays")


def _promote_arith(f: str, a: JType, b: JType | None) -> str | None:
    names = [a.name] + ([b.name] if b is not None else [])
    if any(n == "String" for n in names):
        return None
    if f == "/":
        if all(n in _FLOATS and _FLOATS[n] == 32 or n in _INT_BITS or n == "Bool" for n in names) and any(n == "Float32" for n in names):
            return "Float32"
        return "Float64"
    if any(n in _FLOATS for n in names):
        return "Float64" if any(n == "Float64" for n in names) else "Float32"
    ints = [n for n in names if n in _INT_BITS]
    if not ints:
        return "Int64" if all(n == "Bool" for n in names) else None
    if len(ints) == 1:
        return ints[0]
    ba, bb = _INT_BITS[ints[0]], _INT_BITS[ints[1]]
    if ba == bb:
        return ints[0] if ints[0] == ints[1] else "UInt%d" % ba
    return ints[0] if ba > bb else ints[1]


class BlockBroadcasting:
    """broadcast.jl:6-17 -- expression node `f.(args...)`; `eltype` plays Base._return_type."""

    def __init__(self, f: str, args: Tuple[Any, ...]):
        if f not in _BINARY and f not in _UNARY and f != "in":
            raise ArgumentError(f"function {f!r} is not in the supported operator set")
        self.f = f
        self.args = tuple(args)
        self._rt = self._infer()

    def eltype(self) -> JType | None:
        return self._rt

    def _infer(self) -> JType | None:
        ts = []
        for a in self.args:
            if isinstance(a, (ColRef, BlockBroadcasting)):
                t = a.eltype()
                if t is None:
                    return None
                ts.append(t)
            else:
                ts.append(_scalar_type(a))
        nullable = any(t.nullable for t in ts)
        f = self.f
        if f in ("==", "!=", "<", "<=", ">", ">="):
            a, b = ts
            if (a.name == "String") != (b.name == "String") and f not in ("==", "!="):
                return None
            return JType("Bool", nullable)
        if f in ("&", "|", "xor", "!"):
            if any(t.name != "Bool" for t in ts):
                return None
            return JType("Bool", nullable)
        if f in ("+", "-", "*", "/", "%", "neg"):
            r = _promote_arith(f, ts[0], ts[1] if len(ts) > 1 else None)
            return JType(r, nullable) if r else None
        if f == "ismissing":
            return BOOL
        if f == "coalesce":
            return JType(ts[0].name, False) if ts[0].name == ts[1].name else None
        if f in ("startswith", "endswith"):
            if ts[0].name != "String" or ts[1].name != "String":
                return None
            return JType("Bool", nullable)
        if f == "in":
            x, c = ts[0], self.args[1]
            if not c.legacy and (x.name in _IN_REFUSED or x.name.startswith("Tuple")):
                raise ArgumentError(f"in() with a collection over {x.name} values is not available on the GPU path")
            if c.isequal:
                return BOOL
            return JType("Bool", x.nullable or c.has_missing)
        return None

    def __eq__(self, other):
        return isinstance(other, BlockBroadcasting) and self.f == other.f and self.args == other.args

    def __hash__(self):
        return hash((self.f, self.args))

    def __repr__(self):
        return f"{self.f}({', '.join(map(repr, self.args))})::{self._rt}"


def required_columns(node) -> Tuple[str, ...]:
    """broadcast.jl:33-35 / projection.jl:83-97 -- column names in first-use order."""
    out: list[str] = []

    def walk(n):
        if isinstance(n, ColRef):
            if n.name not in out:
                out.append(n.name)
        elif isinstance(n, BlockBroadcasting):
            for a in n.args:
                walk(a)

    walk(node)
    return tuple(out)


# ---------------------------------------------------------------------------------------------
# ranges (Julia semantics: 1-based, inclusive, `last` normalised)


@dataclass(frozen=True)
class JRange:
    """`start:step:stop` with Julia semantics.  `R(5, 20)` == 5:20, `R(5, 300, 1000)` == 5:300:1000."""
    start: int
    step: int
    stop: int   # normalised last element (start - step when empty)

    @staticmethod
    def make(start: int, stop: int, step: int = 1) -> "JRange":
        if step == 0:
            raise ArgumentError("step cannot be zero")
        n = (stop - start) // step + 1
        if n <= 0:
            return JRange(start, step, start - step)
        return JRange(start, step, start + (n - 1) * step)

    def __len__(self):
        return max(0, (self.stop - self.start) // self.step + 1)

    def __getitem__(self, i):
        """Julia `r[i]` (1-based) and `r[other_range]` / `r[indexvector]` (reindex, selection.jl:40)."""
        if isinstance(i, JRange):
            if len(i) == 0:
                return JRange(self.start, self.step * i.step, self.start - self.step * i.step)
            lo, hi = min(i.start, i.stop), max(i.start, i.stop)
            if lo < 1 or hi > len(self):
                raise IndexError("BoundsError")
            return JRange.make(self[i.start], self[i.stop], self.step * i.step)
        if isinstance(i, (list, tuple)):
            return [self[int(k)] for k in i]
        i = int(i)
        if i < 1 or i > len(self):
            raise IndexError("BoundsError")
        return self.start + (i - 1) * self.step

    def minimum(self):
        if len(self) == 0:
            raise ArgumentError("range must be non-empty")
        return min(self.start, self.stop)

    def maximum(self):
        if len(self) == 0:
            raise ArgumentError("range must be non-empty")
        return max(self.start, self.stop)


def R(start: int, second: int, third: int | None = None) -> JRange:
    """Julia range literal: R(a, b) = a:b ; R(a, s, b) = a:s:b."""
    if third is None:
        return JRange.make(int(start), int(second), 1)
    return JRange.make(int(start), int(third), int(second))


# ---------------------------------------------------------------------------------------------


class SelectionQueue:
    """selection.jl:4-10 -- ordered tuple of range-ish elements and Bool predicates."""

    def __init__(self, queue: Tuple[Any, ...] = ()):
        self.queue = tuple(queue)

    def __len__(self):
        return len(self.queue)

    def isempty(self):
        return not self.queue

    def __eq__(self, other):
        return isinstance(other, SelectionQueue) and self.queue == other.queue

    def __hash__(self):
        return hash(self.queue)

    def __repr__(self):
        return "Selection: " + " |> ".join(map(repr, self.queue))


def _is_rangeish(e) -> bool:
    return isinstance(e, (JRange, int, tuple)) and not isinstance(e, bool)


def _reindex(old, elem):
    # old[1][elem]  (selection.jl:40)
    if isinstance(old, JRange):
        r = old[elem]
        return tuple(r) if isinstance(r, list) else r
    if isinstance(old, tuple):
        if isinstance(elem, JRange):
            return tuple(old[k - 1] for k in (elem[i] for i in range(1, len(elem) + 1)))
        if isinstance(elem, tuple):
            return tuple(old[k - 1] for k in elem)
        return old[elem - 1]
    # integer indexed by something: Julia numbers are iterable of length 1
    if elem == 1 or elem == (1,) or (isinstance(elem, JRange) and len(elem) == 1 and elem.start == 1):
        return old
    raise IndexError("BoundsError")


def add(q, r):
    """selection.jl:37,57-60 (SelectionQueue) and projection.jl:25-30 (Projection)."""
    if isinstance(q, Projection):
        return q.add(r)
    if isinstance(r, slice) and r == slice(None):
        return q
    if isinstance(r, (list, tuple)):
        r = tuple(int(x) for x in r)      # index vectors are kept as tuples (hashable plan objects)
    if isinstance(r, BlockBroadcasting):
        # _check_element selection.jl:52-55
        if r.eltype() != BOOL:
            raise ArgumentError("Function for selection must have Bool result type")
    elif not _is_rangeish(r):
        raise TypeError(f"unsupported selection element {r!r}")
    old = q.queue
    if not old:
        return SelectionQueue((r,))
    last = old[-1]
    if _is_rangeish(last) and _is_rangeish(r):
        return SelectionQueue(old[:-1] + (_reindex(last, r),))
    if isinstance(last, BlockBroadcasting) and isinstance(r, BlockBroadcasting):
        return SelectionQueue(old[:-1] + (BlockBroadcasting("&", (last, r)),))
    return SelectionQueue(old + (r,))


class Projection:
    """projection.jl:1-9 -- ordered name => ColRef | BlockBroadcasting."""

    def __init__(self, cols: Sequence[Tuple[str, Any]] = ()):
        self.cols = tuple((str(k), v) for k, v in cols)

    def keys(self):
        return tuple(k for k, _ in self.cols)

    def values(self):
        return tuple(v for _, v in self.cols)

    def __len__(self):
        return len(self.cols)

    def isempty(self):
        return not self.cols

    def add(self, el: Sequence[Tuple[str, Any]]):
        names = set(self.keys())
        for k, _ in el:
            if k in names:
                raise ArgumentError(f"Duplicated column {k}")
        return Projection(self.cols + tuple(el))

    def __getitem__(self, i):
        """projection.jl:43-75: integer, range / int vector (1-based), name, names."""
        if isinstance(i, str):
            return Projection([c for c in self.cols if c[0] == i])
        if isinstance(i, int):
            return Projection([self.cols[i - 1]])
        if isinstance(i, JRange):
            return Projection([self.cols[k - 1] for k in (i[j] for j in range(1, len(i) + 1))])
        i = list(i)
        if i and isinstance(i[0], str):
            return Projection([c for c in self.cols if c[0] in i])
        return Projection([self.cols[k - 1] for k in i])

    def coltype(self, i) -> JType | None:
        v = dict(self.cols)[i] if isinstance(i, str) else self.cols[i - 1][1]
        return v.eltype()

    def required_columns(self):
        out: list[str] = []
        for _, v in self.cols:
            for n in required_columns(v):
                if n not in out:
                    out.append(n)
        return tuple(out)

    def __eq__(self, other):
        return isinstance(other, Projection) and self.cols == other.cols

    def __hash__(self):
        return hash(self.cols)

    def __repr__(self):
        return "Projection: " + "; ".join(f"{k}=>{v!r}" for k, v in self.cols)


# ---------------------------------------------------------------------------------------------
# serialisation


def _emit_expr(node, out: bytearray) -> int:
    n = 0
    if isinstance(node, ColRef):
        out += struct.pack("<Bq", OP_COL, node.col_id)
        return 1
    if isinstance(node, BlockBroadcasting):
        if node.f == "in":
            n += _emit_expr(node.args[0], out)
            s = node.args[1]
            if not isinstance(s, InSet):
                raise ArgumentError("in.() needs Ref(collection) as second argument")
            out += s.wire
            return n + 1
        for a in node.args:
            n += _emit_expr(a, out)
        out += struct.pack("<B", _BINARY.get(node.f) or _UNARY[node.f])
        return n + 1
    if isinstance(node, bool):
        out += struct.pack("<BB", OP_BOOL, int(node))
    elif isinstance(node, int):
        if not -(1 << 63) <= node < (1 << 63):
            raise ArgumentError("integer constant out of Int64 range")
        out += struct.pack("<Bq", OP_I64, node)
    elif isinstance(node, float):
        out += struct.pack("<Bd", OP_F64, node)
    elif isinstance(node, str):
        b = node.encode("utf-8")
        out += struct.pack("<BI", OP_STR, len(b)) + b
    else:
        raise ArgumentError(f"cannot serialise {node!r}")
    return 1


def encode_expr(node) -> bytes:
    body = bytearray()
    nops = _emit_expr(node, body)
    return struct.pack("<I", nops) + bytes(body)


def encode_plan(selection: SelectionQueue, projection: Projection) -> bytes:
    out = bytearray(struct.pack("<II", MAGIC, len(selection.queue)))
    for e in selection.queue:
        if isinstance(e, BlockBroadcasting):
            out += struct.pack("<B", ST_PRED) + encode_expr(e)
        elif isinstance(e, JRange):
            out += struct.pack("<Bqqq", ST_RANGE, e.start, e.step, e.stop)
        elif isinstance(e, int):
            out += struct.pack("<Bqqq", ST_RANGE, e, 1, e)
        else:
            v = [int(x) for x in e]
            out += struct.pack("<BI", ST_INDEXVEC, len(v)) + struct.pack(f"<{len(v)}q", *v)
    out += struct.pack("<I", len(projection.cols))
    for _, v in projection.cols:
        if isinstance(v, ColRef):
            out += struct.pack("<Bq", PJ_COL, v.col_id)
        else:
            out += struct.pack("<B", PJ_EXPR) + encode_expr(v)
    return bytes(out)
