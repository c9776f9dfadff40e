"""Host-side mirror of the reference's function API for the hot path.

Same names, argument meaning and error behaviour as arrow::compute::CallFunction
(cpp/src/arrow/compute/exec.cc:1362-1390) / pyarrow.compute, but operands are
DeviceArray and every kernel is a C-ABI call into libarrow_b200.so.  The dispatch rules
reproduced here are the reference's:
  * arithmetic / compare: exact match, else promote all operands to CommonNumeric
    (kernels/codegen_internal.cc:166-218) with an implicit safe cast
    (ArithmeticFunction::DispatchBest kernels/scalar_arithmetic.cc:734-781,
     CompareFunction::DispatchBest kernels/scalar_compare.cc:340-366,
     FunctionExecutorImpl::Execute function.cc:242-250),
  * filter / take / sort_indices meta-functions unwrap to array_* kernels
    (kernels/vector_selection_filter_internal.cc:1043-1072, vector_selection_take_internal.cc:660-701,
     kernels/vector_sort.cc:856-924).
"""
from __future__ import annotations

import builtins
import ctypes as C
from typing import Optional, Sequence, Union

import numpy as np
import pyarrow as pa

from . import _cabi as cabi
from .device import _NUMERIC as _NUMERIC_TYPES
from .device import Context, DeviceArray, arrow_type, check, type_id

Operand = Union[DeviceArray, pa.Scalar, int, float, bool, None]

_NUMERIC_IDS = (cabi.UINT8, cabi.INT8, cabi.UINT16, cabi.INT16, cabi.UINT32, cabi.INT32, cabi.UINT64,
                cabi.INT64, cabi.FLOAT, cabi.DOUBLE)
_SIGNED = {cabi.INT8: 8, cabi.INT16: 16, cabi.INT32: 32, cabi.INT64: 64}
_UNSIGNED = {cabi.UINT8: 8, cabi.UINT16: 16, cabi.UINT32: 32, cabi.UINT64: 64}
_NP = {cabi.INT8: np.int8, cabi.UINT8: np.uint8, cabi.INT16: np.int16, cabi.UINT16: np.uint16,
       cabi.INT32: np.int32, cabi.UINT32: np.uint32, cabi.INT64: np.int64, cabi.UINT64: np.uint64,
       cabi.FLOAT: np.float32, cabi.DOUBLE: np.float64}


def _ctx(*args) -> Context:
    for a in args:
        if isinstance(a, DeviceArray):
            return a.ctx
    return Context.get()


def _out(ctx: Context, c: cabi.B2Array, type: pa.DataType, dictionary=None) -> DeviceArray:
    return DeviceArray._from_c(ctx, c, type, dictionary)


# ------------------------------------------------------------------------------------
# dispatch helpers
# ------------------------------------------------------------------------------------
def common_numeric(ids: Sequence[int]) -> int:
    """CommonNumeric (kernels/codegen_internal.cc:166-218)."""
    for i in ids:
        if i not in _NUMERIC_IDS:
            raise pa.ArrowNotImplementedError("Function has no kernel matching input types")
    if cabi.DOUBLE in ids:
        return cabi.DOUBLE
    if cabi.FLOAT in ids:
        return cabi.FLOAT
    ms = builtins.max([_SIGNED[i] for i in ids if i in _SIGNED], default=0)
    mu = builtins.max([_UNSIGNED[i] for i in ids if i in _UNSIGNED], default=0)
    if ms == 0:
        return {8: cabi.UINT8, 16: cabi.UINT16, 32: cabi.UINT32}.get(mu, cabi.UINT64)
    if ms <= mu:
        ms = 1 << (mu + 1 - 1).bit_length()  # NextPower2(mu + 1)
    return {8: cabi.INT8, 16: cabi.INT16, 32: cabi.INT32}.get(ms, cabi.INT64)


def _require_numeric(t: pa.DataType) -> None:
    """Only the ten genuinely numeric Arrow types reach the numeric kernels.  Temporal / dictionary /
    other logical types share an integer STORAGE with them but not their semantics (the reference
    rescales units in casts, kernels/scalar_cast_temporal.cc, and dispatches timestamp/duration
    arithmetic to dedicated kernels, kernels/scalar_arithmetic.cc:1480-1529): refuse rather than
    compute on raw storage."""
    if t not in _NUMERIC_TYPES:
        raise pa.ArrowNotImplementedError(f"Function has no kernel matching input types ({t}) on arrow_b200 device arrays")


_SORTABLE_STRING_TYPES = (pa.utf8(), pa.large_utf8(), pa.binary(), pa.large_binary())


def _require_sortable(t: pa.DataType) -> None:
    """Sort keys: the numeric types and utf8 / large_utf8 / binary / large_binary (ordered byte-wise, unsigned)."""
    if t not in _SORTABLE_STRING_TYPES:
        _require_numeric(t)


def _as_scalar(x) -> pa.Scalar:
    if isinstance(x, pa.Scalar):
        return x
    return pa.scalar(x)


def _scalar_to(s: pa.Scalar, tid: int) -> cabi.B2Scalar:
    """Implicit safe cast of a host scalar to the dispatched type (done on the host: it is
    argument preparation, one value)."""
    out = cabi.B2Scalar()
    out.type = tid
    out.is_valid = 1 if s.is_valid else 0
    out.bits = 0
    if s.is_valid:
        v = s.as_py()
        dt = _NP[tid]
        if np.issubdtype(dt, np.integer):
            if isinstance(v, float):
                if v != int(v):
                    raise pa.ArrowInvalid(f"Float value {v:f} was truncated converting to {arrow_type(tid)}")
                v = int(v)
            info = np.iinfo(dt)
            if not (info.min <= int(v) <= info.max):
                raise pa.ArrowInvalid(f"Integer value {v} not in range: {info.min} to {info.max}")
            arr = np.array([int(v)], dtype=dt)
        else:
            arr = np.array([v], dtype=dt)
        out.bits = int(np.frombuffer(arr.tobytes().ljust(8, b"\0"), dtype=np.uint64)[0])
    return out


def _prepare_binary(left: Operand, right: Operand):
    ctx = _ctx(left, right)
    ops = []
    ids = []
    for x in (left, right):
        if isinstance(x, DeviceArray):
            _require_numeric(x.type)
            ids.append(type_id(x.type))
            ops.append(x)
        else:
            s = _as_scalar(x)
            if pa.types.is_null(s.type):
                raise pa.ArrowNotImplementedError("null-typed scalar operands are not supported")
            _require_numeric(s.type)
            ids.append(type_id(s.type))
            ops.append(s)
    if not any(isinstance(o, DeviceArray) for o in ops):
        raise pa.ArrowNotImplementedError("arrow_b200: at least one operand must be a device array")
    tid = ids[0] if ids[0] == ids[1] and ids[0] in _NUMERIC_IDS else common_numeric(ids)
    keep = []  # keep ctypes structs alive for the call
    vals = []
    for o, i in zip(ops, ids):
        v = cabi.B2Value()
        if isinstance(o, DeviceArray):
            if i != tid:
                o = cast(o, arrow_type(tid))  # implicit safe cast
            c = o._c()
            keep.append((o, c))
            v.array = C.pointer(c)
            v.scalar = None
        else:
            sc = _scalar_to(o, tid)
            keep.append(sc)
            v.array = None
            v.scalar = C.pointer(sc)
        vals.append(v)
    return ctx, tid, vals, keep


# ------------------------------------------------------------------------------------
# scalar kernels
# ------------------------------------------------------------------------------------
def cast(arr: DeviceArray, target_type=None, safe: Optional[bool] = None, options=None) -> DeviceArray:
    """pyarrow.compute.cast / CastMetaFunction (compute/cast.cc:78-127)."""
    allow_int_overflow = allow_float_truncate = False
    if options is not None:
        target_type = options.target_type if target_type is None else target_type
        allow_int_overflow = bool(options.allow_int_overflow)
        allow_float_truncate = bool(options.allow_float_truncate)
    if safe is False:
        allow_int_overflow = allow_float_truncate = True
    target_type = pa.lib.ensure_type(target_type)
    if arr.type == target_type:
        return arr
    # logical types (timestamp/date/time/duration/dictionary) have numeric STORAGE ids but unit / index
    # semantics the numeric cast kernel does not implement: only exact numeric types pass
    if arr.type not in _NUMERIC_TYPES or target_type not in _NUMERIC_TYPES:
        raise pa.ArrowNotImplementedError(
            f"Unsupported cast from {arr.type} to {target_type} using function cast_{target_type}")
    src, dst = type_id(arr.type), type_id(target_type)
    if src not in _NUMERIC_IDS or dst not in _NUMERIC_IDS:
        raise pa.ArrowNotImplementedError(
            f"Unsupported cast from {arr.type} to {target_type} using function cast_{target_type}")
    ctx = arr.ctx
    opt = cabi.B2CastOptions(dst, int(allow_int_overflow), int(allow_float_truncate), 0)
    cin, cout = arr._c(), cabi.B2Array()
    check(ctx.lib.b2_cast_numeric(ctx.handle, C.byref(cin), C.byref(opt), C.byref(cout), ctx.stream))
    return _out(ctx, cout, target_type)


def _arith(name: str, left: Operand, right: Operand) -> DeviceArray:
    ctx, tid, vals, keep = _prepare_binary(left, right)
    cout = cabi.B2Array()
    check(ctx.lib.b2_binary_arith(ctx.handle, cabi.ARITH_OPS[name], C.byref(vals[0]), C.byref(vals[1]),
                                  C.byref(cout), ctx.stream))
    return _out(ctx, cout, arrow_type(tid))


def _compare(name: str, left: Operand, right: Operand) -> DeviceArray:
    ctx, tid, vals, keep = _prepare_binary(left, right)
    cout = cabi.B2Array()
    check(ctx.lib.b2_compare(ctx.handle, cabi.COMPARE_OPS[name], C.byref(vals[0]), C.byref(vals[1]),
                             C.byref(cout), ctx.stream))
    return _out(ctx, cout, pa.bool_())


def add(x, y): return _arith("add", x, y)
def subtract(x, y): return _arith("subtract", x, y)
def multiply(x, y): return _arith("multiply", x, y)
def divide(x, y): return _arith("divide", x, y)
def add_checked(x, y): return _arith("add_checked", x, y)
def subtract_checked(x, y): return _arith("subtract_checked", x, y)
def multiply_checked(x, y): return _arith("multiply_checked", x, y)
def divide_checked(x, y): return _arith("divide_checked", x, y)
def equal(x, y): return _compare("equal", x, y)
def not_equal(x, y): return _compare("not_equal", x, y)
def greater(x, y): return _compare("greater", x, y)
def greater_equal(x, y): return _compare("greater_equal", x, y)
def less(x, y): return _compare("less", x, y)
def less_equal(x, y): return _compare("less_equal", x, y)


# ------------------------------------------------------------------------------------
# boolean logic + validity predicates (kernels/scalar_boolean.cc, kernels/scalar_validity.cc)
# ------------------------------------------------------------------------------------
def _bool_value(x, keep):
    v = cabi.B2Value()
    if isinstance(x, DeviceArray):
        if not pa.types.is_boolean(x.type):
            raise pa.ArrowNotImplementedError(f"Function has no kernel matching input types ({x.type})")
        c = x._c()
        keep.append((x, c))
        v.array, v.scalar = C.pointer(c), None
    else:
        s = _as_scalar(x)
        if not (pa.types.is_boolean(s.type) or pa.types.is_null(s.type)):
            raise pa.ArrowNotImplementedError(f"Function has no kernel matching input types ({s.type})")
        sc = cabi.B2Scalar()
        sc.type, sc.is_valid = cabi.BOOL, 1 if s.is_valid else 0
        sc.bits = 1 if (s.is_valid and s.as_py()) else 0
        keep.append(sc)
        v.array, v.scalar = None, C.pointer(sc)
    return v


def _boolean(name: str, left, right=None) -> DeviceArray:
    ctx = _ctx(left, right)
    keep = []
    lv = _bool_value(left, keep)
    rv = _bool_value(right, keep) if name != "invert" else None
    cout = cabi.B2Array()
    check(ctx.lib.b2_boolean(ctx.handle, cabi.BOOLEAN_OPS[name], C.byref(lv), C.byref(rv) if rv is not None else None,
                             C.byref(cout), ctx.stream))
    return _out(ctx, cout, pa.bool_())


def and_(x, y): return _boolean("and", x, y)
def or_(x, y): return _boolean("or", x, y)
def xor(x, y): return _boolean("xor", x, y)
def and_not(x, y): return _boolean("and_not", x, y)
def and_kleene(x, y): return _boolean("and_kleene", x, y)
def or_kleene(x, y): return _boolean("or_kleene", x, y)
def and_not_kleene(x, y): return _boolean("and_not_kleene", x, y)
def invert(x): return _boolean("invert", x)


def _validity(name: str, arr: DeviceArray, nan_is_null: bool = False) -> DeviceArray:
    ctx = arr.ctx
    ca, cout = arr._c(), cabi.B2Array()
    check(ctx.lib.b2_validity(ctx.handle, cabi.VALIDITY_OPS[name], C.byref(ca), int(bool(nan_is_null)), C.byref(cout),
                              ctx.stream))
    return _out(ctx, cout, pa.bool_())


def is_valid(x): return _validity("is_valid", x)
def is_null(x, nan_is_null=False): return _validity("is_null", x, nan_is_null)
def true_unless_null(x): return _validity("true_unless_null", x)
def is_nan(x): return _validity("is_nan", x)


def if_else(cond, left, right) -> DeviceArray:
    """if_else (kernels/scalar_if_else.cc:62-520): cond ? left : right, null where cond or the chosen side is null.
    cond: boolean DeviceArray or scalar; left / right: DeviceArrays or scalars, numerics promoted to their common type
    like the reference's DispatchBest (scalar_if_else.cc:1227-1266), or both boolean."""
    ctx = _ctx(cond, left, right)
    keep = []
    cv = _bool_value(cond, keep)
    sides = [x if isinstance(x, DeviceArray) else _as_scalar(x) for x in (left, right)]
    types = [x.type for x in sides]
    if all(pa.types.is_boolean(t) or pa.types.is_null(t) for t in types):
        vals = [_bool_value(x, keep) for x in (left, right)]
        out_type = pa.bool_()
    else:
        for t in types:
            if pa.types.is_null(t):
                raise pa.ArrowNotImplementedError("null-typed scalar operands are not supported")
            _require_numeric(t)
        ids = [type_id(t) for t in types]
        tid = ids[0] if ids[0] == ids[1] else common_numeric(ids)
        out_type = arrow_type(tid)
        vals = []
        for x, i in zip(sides, ids):
            v = cabi.B2Value()
            if isinstance(x, DeviceArray):
                if i != tid:
                    x = cast(x, out_type)
                c = x._c()
                keep.append((x, c))
                v.array, v.scalar = C.pointer(c), None
            else:
                sc = _scalar_to(x, tid)
                keep.append(sc)
                v.array, v.scalar = None, C.pointer(sc)
            vals.append(v)
    cout = cabi.B2Array()
    check(ctx.lib.b2_if_else(ctx.handle, C.byref(cv), C.byref(vals[0]), C.byref(vals[1]), C.byref(cout), ctx.stream))
    return _out(ctx, cout, out_type)


# ------------------------------------------------------------------------------------
# selection
# ------------------------------------------------------------------------------------
def _null_selection(v) -> int:
    if v in ("drop", 0, None):
        return 0
    if v in ("emit_null", 1):
        return 1
    raise ValueError(f'"{v}" is not a valid null selection behavior')


def filter(values: DeviceArray, mask: DeviceArray, null_selection_behavior="drop") -> DeviceArray:
    """pyarrow.compute.filter / array_filter (kernels/vector_selection_filter_internal.cc:1043-1072)."""
    if not pa.types.is_boolean(mask.type):
        raise pa.ArrowNotImplementedError(
            f"Function 'array_filter' has no kernel matching input types ({values.type}, {mask.type})")
    if len(values) != len(mask):  # raised by the reference's VectorExecutor before the kernel runs
        raise pa.ArrowInvalid("Arguments for execution of vector kernel function 'array_filter' must all be the same length")
    ctx = values.ctx
    cv, cm, cout = values._c(), mask._c(), cabi.B2Array()
    check(ctx.lib.b2_filter(ctx.handle, C.byref(cv), C.byref(cm), _null_selection(null_selection_behavior),
                            C.byref(cout), ctx.stream))
    return _out(ctx, cout, values.type, values.dictionary)


def array_filter(values, mask, null_selection_behavior="drop"):
    return filter(values, mask, null_selection_behavior)


def filter_output_size(mask: DeviceArray, null_selection_behavior="drop") -> int:
    ctx = mask.ctx
    n = C.c_int64()
    cm = mask._c()
    check(ctx.lib.b2_filter_output_size(ctx.handle, C.byref(cm), _null_selection(null_selection_behavior),
                                        C.byref(n), ctx.stream))
    return n.value


def take_indices_from_filter(mask: DeviceArray, null_selection_behavior="drop") -> DeviceArray:
    """GetTakeIndices (kernels/vector_selection_take_internal.cc:298-305)."""
    ctx = mask.ctx
    cm, cout = mask._c(), cabi.B2Array()
    check(ctx.lib.b2_filter_indices(ctx.handle, C.byref(cm), _null_selection(null_selection_behavior),
                                    C.byref(cout), ctx.stream))
    return _out(ctx, cout, arrow_type(cout.type))


def take(values: DeviceArray, indices: DeviceArray, boundscheck: bool = True) -> DeviceArray:
    """pyarrow.compute.take / array_take (kernels/vector_selection_take_internal.cc:660-701)."""
    if not pa.types.is_integer(indices.type):
        raise pa.ArrowNotImplementedError(
            f"Function 'array_take' has no kernel matching input types ({values.type}, {indices.type})")
    ctx = values.ctx
    cv, ci, cout = values._c(), indices._c(), cabi.B2Array()
    check(ctx.lib.b2_take(ctx.handle, C.byref(cv), C.byref(ci), int(bool(boundscheck)), C.byref(cout),
                          ctx.stream))
    return _out(ctx, cout, values.type, values.dictionary)


def take_cast_arith(values: DeviceArray, indices: DeviceArray, target_type, op: str, other) -> DeviceArray:
    """Fused `op(cast(take(values, indices), target_type, safe=False), other)` -- one kernel instead of three
    (b2_take_cast_arith; the reference evaluates the same Expression kernel by kernel, compute/expression.cc:722-797).
    Falls back to the three calls for operand shapes the fused kernel does not cover."""
    target_type = pa.lib.ensure_type(target_type)
    fusable = (values.type in (pa.float64(), pa.float32(), pa.int64(), pa.int32()) and target_type in (pa.float32(), pa.float64())
               and indices.type in (pa.int32(), pa.uint32(), pa.int64(), pa.uint64()) and op in ("add", "subtract", "multiply")
               and isinstance(other, DeviceArray) and other.type == target_type and len(other) == len(indices))
    if not fusable:
        return _arith(op, cast(take(values, indices), target_type, safe=False), other)
    ctx = values.ctx
    keep = []
    ov = cabi.B2Value()
    co = other._c()
    keep.append(co)
    ov.array, ov.scalar = C.pointer(co), None
    cv, ci, cout = values._c(), indices._c(), cabi.B2Array()
    check(ctx.lib.b2_take_cast_arith(ctx.handle, C.byref(cv), C.byref(ci), type_id(target_type), cabi.ARITH_OPS[op], C.byref(ov),
                                     C.byref(cout), ctx.stream))
    return _out(ctx, cout, target_type)


def array_take(values, indices, boundscheck=True):
    return take(values, indices, boundscheck)


# ------------------------------------------------------------------------------------
# sort
# ------------------------------------------------------------------------------------
def _order(v) -> int:
    if v in ("ascending", 0):
        return 0
    if v in ("descending", 1):
        return 1
    raise ValueError(f'"{v}" is not a valid order')


def _placement(v) -> int:
    if v in ("at_start", 0):
        return 0
    if v in ("at_end", 1):
        return 1
    raise ValueError(f'"{v}" is not a valid null placement')


def array_sort_indices(arr: DeviceArray, order="ascending", null_placement="at_end") -> DeviceArray:
    """array_sort_indices (kernels/vector_array_sort.cc:524-540): stable argsort -> uint64."""
    ctx = arr.ctx
    ca, cout = arr._c(), cabi.B2Array()
    check(ctx.lib.b2_sort_indices(ctx.handle, C.byref(ca), _order(order), _placement(null_placement),
                                  C.byref(cout), ctx.stream))
    return _out(ctx, cout, pa.uint64())


def sort_payload(arr: DeviceArray, payload: DeviceArray, order="ascending", null_placement="at_end") -> DeviceArray:
    """stable sort of `arr` where row i carries payload[i] (uint32) instead of i: returns the payloads in sorted order
    (uint64) -- array_sort_indices followed by take(payload, indices), in the radix passes themselves"""
    ctx = arr.ctx
    ca, cp_, cout = arr._c(), payload._c(), cabi.B2Array()
    check(ctx.lib.b2_sort_payload(ctx.handle, C.byref(ca), C.byref(cp_), _order(order), _placement(null_placement),
                                  C.byref(cout), ctx.stream))
    return _out(ctx, cout, pa.uint64())


def sort_strings_path(arr: DeviceArray) -> str:
    """which path the sort of this utf8 / binary column takes: "dict" (sort the distinct values, then their ranks) or
    "refine" (7-byte prefix rounds) -- B2_SORT_STRINGS_PATH when set, else the sampled estimate (csrc/sort_strings.cu)"""
    ctx = arr.ctx
    ca, p = arr._c(), C.c_int32(0)
    check(ctx.lib.b2_sort_strings_path(ctx.handle, C.byref(ca), C.byref(p), ctx.stream))
    return "dict" if p.value else "refine"


def sort_indices(arr, sort_keys=None, null_placement="at_end", order=None) -> DeviceArray:
    """sort_indices meta function (kernels/vector_sort.cc:850-1027): on one array, or -- given a mapping
    {name: DeviceArray} (a record batch / table of device columns) and sort_keys = [(name, order), ...] -- the
    multi-key sort: ordered by the first key, ties by the next, stable (b2_sort_indices_multi)."""
    if isinstance(arr, dict):
        if not sort_keys:
            raise pa.ArrowInvalid("Must specify one or more sort keys")
        cols, orders = [], []
        for k in sort_keys:
            name, o = (k[0], k[1]) if isinstance(k, (tuple, list)) else (k, "ascending")
            if name not in arr:
                raise pa.ArrowInvalid(f"No match for FieldRef.Name({name})")
            _require_sortable(arr[name].type)
            cols.append(arr[name])
            orders.append(_order(o))
        ctx = cols[0].ctx
        cks = (cabi.B2Array * len(cols))(*[c._c() for c in cols])
        cor = (C.c_int32 * len(cols))(*orders)
        cout = cabi.B2Array()
        check(ctx.lib.b2_sort_indices_multi(ctx.handle, cks, len(cols), cor, _placement(null_placement), C.byref(cout), ctx.stream))
        return _out(ctx, cout, pa.uint64())
    o = "ascending"
    if sort_keys:
        o = sort_keys[0][1] if isinstance(sort_keys[0], (tuple, list)) else sort_keys[0]
    if order is not None:
        o = order
    return array_sort_indices(arr, o, null_placement)


def select_k_unstable(arr: DeviceArray, k: int, sort_keys=None, null_placement="at_end") -> DeviceArray:
    """select_k_unstable (kernels/vector_select_k.cc:157-232, SelectKOptions api_vector.h:178-214) on one array: the
    indices of the first k rows in sort order; sort_keys = [(ignored name, order)] as in the reference.  Ties come out in
    row order (= sort_indices(...)[:k]), one of the answers the reference's unstable selection may give."""
    if k < 0:
        raise pa.ArrowInvalid(f"select_k_unstable requires a nonnegative `k`, got {k}")
    o = "ascending"
    if sort_keys:
        if len(sort_keys) != 1:
            raise pa.ArrowNotImplementedError("arrow_b200 select_k_unstable: one sort key (use sort_indices for several)")
        o = sort_keys[0][1] if isinstance(sort_keys[0], (tuple, list)) else "ascending"
    _require_sortable(arr.type)
    ctx = arr.ctx
    ca, cout = arr._c(), cabi.B2Array()
    check(ctx.lib.b2_select_k(ctx.handle, C.byref(ca), int(k), _order(o), _placement(null_placement), C.byref(cout), ctx.stream))
    return _out(ctx, cout, pa.uint64())


# ------------------------------------------------------------------------------------
# ungrouped aggregates (kernels/aggregate_basic.cc, aggregate_basic.inc.cc)
# ------------------------------------------------------------------------------------
def _reduce(arr: DeviceArray) -> "cabi.B2ReduceResult":
    _require_numeric(arr.type)
    ctx = arr.ctx
    ca, r = arr._c(), cabi.B2ReduceResult()
    check(ctx.lib.b2_reduce(ctx.handle, C.byref(ca), C.byref(r), ctx.stream))
    return r


def _from_bits(bits: int, t: pa.DataType):
    raw = np.array([bits], dtype=np.uint64)
    if pa.types.is_floating(t):
        return raw.view(np.float64)[0]
    return raw.view(np.int64)[0] if pa.types.is_signed_integer(t) else raw[0]


def _acc_type(t: pa.DataType) -> pa.DataType:
    if pa.types.is_floating(t):
        return pa.float64()
    return pa.int64() if pa.types.is_signed_integer(t) else pa.uint64()


def sum(arr: DeviceArray, skip_nulls: bool = True, min_count: int = 1) -> pa.Scalar:  # noqa: A001
    """sum (SumImpl::Finalize, aggregate_basic.inc.cc:95-103): null if a null was seen and
    !skip_nulls, or fewer than min_count valid values; accumulator = int64 / uint64 / double."""
    r, out_t = _reduce(arr), _acc_type(arr.type)
    if (not skip_nulls and r.null_count > 0) or r.count < min_count:
        return pa.scalar(None, out_t)
    return pa.scalar(_from_bits(r.sum_bits, out_t).item(), out_t)


def mean(arr: DeviceArray, skip_nulls: bool = True, min_count: int = 1) -> pa.Scalar:
    """mean (MeanImpl, aggregate_basic.inc.cc:263-283): the sum is accumulated in double, then / count."""
    r = _reduce(arr)
    if (not skip_nulls and r.null_count > 0) or r.count < min_count:
        return pa.scalar(None, pa.float64())
    with np.errstate(invalid="ignore", divide="ignore"):  # no valid value and min_count == 0: 0/0 = NaN like the reference
        return pa.scalar(float(_from_bits(r.dsum_bits, pa.float64()) / np.float64(r.count)), pa.float64())


def min_max(arr: DeviceArray, skip_nulls: bool = True, min_count: int = 1) -> pa.Scalar:
    """min_max (MinMaxImpl::Finalize, aggregate_basic.inc.cc:834-853): struct<min, max> of the input
    type; min_count is at least 1 (:783)."""
    r, t = _reduce(arr), arr.type
    st = pa.struct([("min", t), ("max", t)])
    if (r.null_count > 0 and not skip_nulls) or r.count < builtins.max(1, min_count):
        return pa.scalar({"min": None, "max": None}, st)
    wide = _acc_type(t)
    lo, hi = _from_bits(r.min_bits, wide), _from_bits(r.max_bits, wide)
    nt = np.dtype(t.to_pandas_dtype()).type
    return pa.scalar({"min": nt(lo).item(), "max": nt(hi).item()}, st)


def min(arr: DeviceArray, skip_nulls: bool = True, min_count: int = 1) -> pa.Scalar:  # noqa: A001
    return min_max(arr, skip_nulls, min_count)["min"]


def max(arr: DeviceArray, skip_nulls: bool = True, min_count: int = 1) -> pa.Scalar:  # noqa: A001
    return min_max(arr, skip_nulls, min_count)["max"]


def count(arr: DeviceArray, mode: str = "only_valid") -> pa.Scalar:
    """count (CountImpl, aggregate_basic.cc:98-130; CountOptions api_aggregate.h:64-78)."""
    ctx = arr.ctx
    nulls = arr.null_count
    if nulls < 0:  # unknown after slicing: count the validity bits on the device
        out = C.c_int64()
        check(ctx.lib.b2_bitmap_count(ctx.handle, arr.buffers[0].ptr, arr.offset, arr.length, C.byref(out), ctx.stream))
        nulls = arr.length - out.value
    if mode == "only_valid":
        return pa.scalar(arr.length - nulls, pa.int64())
    if mode == "only_null":
        return pa.scalar(nulls, pa.int64())
    if mode == "all":
        return pa.scalar(arr.length, pa.int64())
    raise ValueError(f'"{mode}" is not a valid count mode')


# ------------------------------------------------------------------------------------
# unique / value_counts / dictionary_encode (kernels/vector_hash.cc:782-830)
# ------------------------------------------------------------------------------------
def _null_encoding(v) -> int:
    if v in ("mask", 0):
        return 0
    if v in ("encode", 1):
        return 1
    raise ValueError(f'"{v}" is not a valid null encoding behavior')


def _vector_hash(arr: DeviceArray, null_encoding: int, want_indices: bool, want_counts: bool):
    ctx = arr.ctx
    ca, ci, cd, cc = arr._c(), cabi.B2Array(), cabi.B2Array(), cabi.B2Array()
    check(ctx.lib.b2_vector_hash(ctx.handle, C.byref(ca), null_encoding, C.byref(ci) if want_indices else None,
                                 C.byref(cd), C.byref(cc) if want_counts else None, ctx.stream))
    dictionary = _out(ctx, cd, arr.type)
    indices = _out(ctx, ci, pa.dictionary(pa.int32(), arr.type), dictionary) if want_indices else None
    counts = _out(ctx, cc, pa.int64()) if want_counts else None
    return indices, dictionary, counts


def unique(arr: DeviceArray) -> DeviceArray:
    """unique: distinct values in first-occurrence order, null included (vector_hash.cc:65-97,791)."""
    return _vector_hash(arr, 1, False, False)[1]


def value_counts(arr: DeviceArray):
    """value_counts: (values, counts) = the two fields of the reference's struct result
    (vector_hash.cc:101-168,634,807); `to_struct` below assembles the StructArray on the host."""
    _, values, counts = _vector_hash(arr, 1, False, True)
    return values, counts


def value_counts_to_struct(values: DeviceArray, counts: DeviceArray) -> pa.StructArray:
    return pa.StructArray.from_arrays([values.to_arrow(), counts.to_arrow()], names=["values", "counts"])


def count_distinct(arr: DeviceArray, mode: str = "only_valid") -> pa.Scalar:
    """count_distinct (CountDistinctImpl, kernels/aggregate_basic.cc:141-230; CountOptions api_aggregate.h:64-78): the size of
    the memo table = the number of uniques, with the null entry counted under only_null / all."""
    u = unique(arr)
    has_null = 1 if u.null_count > 0 else 0
    if mode == "only_valid":
        return pa.scalar(len(u) - has_null, pa.int64())
    if mode == "only_null":
        return pa.scalar(has_null, pa.int64())
    if mode == "all":
        return pa.scalar(len(u), pa.int64())
    raise ValueError(f'"{mode}" is not a valid count mode')


def dictionary_encode(arr: DeviceArray, null_encoding="mask") -> DeviceArray:
    """dictionary_encode: int32 indices + dictionary (vector_hash.cc:173-232,826;
    DictionaryEncodeOptions api_vector.h:66-82)."""
    return _vector_hash(arr, _null_encoding(null_encoding), True, False)[0]


# ------------------------------------------------------------------------------------
# grouper + hash aggregates
# ------------------------------------------------------------------------------------
class Grouper:
    """arrow::compute::Grouper (compute/row/grouper.h:104-196) over fixed-width and utf8 / binary key columns."""

    def __init__(self, key_types: Sequence[pa.DataType], ctx: Optional[Context] = None):
        self.ctx = ctx or Context.get()
        self.key_types = [pa.lib.ensure_type(t) for t in key_types]
        ids = (C.c_int32 * len(self.key_types))(*[type_id(t) for t in self.key_types])
        h = C.c_void_p()
        check(self.ctx.lib.b2_grouper_create(self.ctx.handle, ids, len(self.key_types), C.byref(h)))
        self.handle = h

    def __del__(self):
        if getattr(self, "handle", None):
            self.ctx.lib.b2_grouper_destroy(self.handle)
            self.handle = None

    def _keys(self, keys):
        if isinstance(keys, DeviceArray):
            keys = [keys]
        if len(keys) != len(self.key_types):
            raise pa.ArrowInvalid(f"expected batch size {len(self.key_types)} but got {len(keys)}")
        for k, t in zip(keys, self.key_types):
            if k.type != t:
                raise pa.ArrowInvalid(f"expected batch value of type {t} but got {k.type}")
        carr = (cabi.B2Array * len(keys))(*[k._c() for k in keys])
        return carr

    def consume(self, keys) -> DeviceArray:
        carr, cout = self._keys(keys), cabi.B2Array()
        check(self.ctx.lib.b2_grouper_consume(self.handle, carr, C.byref(cout), self.ctx.stream))
        return _out(self.ctx, cout, pa.uint32())

    def lookup(self, keys) -> DeviceArray:
        carr, cout = self._keys(keys), cabi.B2Array()
        check(self.ctx.lib.b2_grouper_lookup(self.handle, carr, C.byref(cout), self.ctx.stream))
        return _out(self.ctx, cout, pa.uint32())

    @property
    def num_groups(self) -> int:
        n = C.c_uint32()
        check(self.ctx.lib.b2_grouper_num_groups(self.handle, C.byref(n)))
        return n.value

    def get_uniques(self):
        couts = (cabi.B2Array * len(self.key_types))()
        check(self.ctx.lib.b2_grouper_uniques(self.handle, couts, self.ctx.stream))
        return [_out(self.ctx, couts[i], t) for i, t in enumerate(self.key_types)]

    def reset(self):
        check(self.ctx.lib.b2_grouper_reset(self.handle))


JOIN_TYPES = {"inner": 0, "left outer": 1, "left semi": 2, "left anti": 3, "full outer": 4}


def hash_join_indices(left_keys: Sequence[DeviceArray], right_keys: Sequence[DeviceArray], join_type: str = "inner"):
    """The matching row pairs of an equi-join (the build / probe / match core of acero's HashJoinNode, hash_join_node.cc;
    join types as pyarrow.Table.join spells them).  Returns (left_indices, right_indices) as uint32 DeviceArrays -- for
    "left outer" right_indices is null where a left row found no match ("full outer" appends the unmatched right rows with a
    null left index), for "left semi" / "left anti" right_indices is None.
    A null key matches nothing.  Gather the payload columns with take()."""
    if isinstance(left_keys, DeviceArray):
        left_keys = [left_keys]
    if isinstance(right_keys, DeviceArray):
        right_keys = [right_keys]
    if join_type not in JOIN_TYPES:
        raise ValueError(f'"{join_type}" is not a supported join type ({", ".join(JOIN_TYPES)})')
    if len(left_keys) != len(right_keys) or not left_keys:
        raise pa.ArrowInvalid("join needs the same, non-zero number of key columns on both sides")
    for l, r in zip(left_keys, right_keys):
        if l.type != r.type:
            raise pa.ArrowInvalid(f"Incompatible data types for corresponding join field keys: {l.type} and {r.type}")
    ctx = left_keys[0].ctx
    cl = (cabi.B2Array * len(left_keys))(*[k._c() for k in left_keys])
    cr = (cabi.B2Array * len(right_keys))(*[k._c() for k in right_keys])
    ol, orr = cabi.B2Array(), cabi.B2Array()
    pairs = JOIN_TYPES[join_type] in (0, 1, 4)
    check(ctx.lib.b2_hash_join(ctx.handle, cl, cr, len(left_keys), JOIN_TYPES[join_type], C.byref(ol), C.byref(orr) if pairs else None,
                               ctx.stream))
    return _out(ctx, ol, pa.uint32()), (_out(ctx, orr, pa.uint32()) if pairs else None)


class HashAggregator:
    """One HashAggregateKernel state (compute/kernel.h:720-769): resize/consume/merge/finalize."""

    def __init__(self, function: str, value_type: Optional[pa.DataType], *, skip_nulls=True, min_count=1,
                 mode="only_valid", ctx: Optional[Context] = None):
        self.ctx = ctx or Context.get()
        self.function = function
        kind = cabi.HASH_AGG_KINDS[function]
        cm = {"only_valid": 0, "only_null": 1, "all": 2}[mode]
        opts = cabi.B2HashAggOptions(int(skip_nulls), int(min_count), cm, 0)
        vt = type_id(value_type) if value_type is not None else cabi.NA
        h = C.c_void_p()
        check(self.ctx.lib.b2_hashagg_create(self.ctx.handle, kind, vt, C.byref(opts), C.byref(h)))
        self.handle = h

    def __del__(self):
        if getattr(self, "handle", None):
            self.ctx.lib.b2_hashagg_destroy(self.handle)
            self.handle = None

    def resize(self, num_groups: int):
        check(self.ctx.lib.b2_hashagg_resize(self.handle, int(num_groups), self.ctx.stream))

    def consume(self, values: Optional[DeviceArray], ids: DeviceArray):
        cv = values._c() if values is not None else None
        ci = ids._c()
        check(self.ctx.lib.b2_hashagg_consume(self.handle, C.byref(cv) if cv is not None else None,
                                              C.byref(ci), self.ctx.stream))

    def merge(self, other: "HashAggregator", group_id_mapping: DeviceArray):
        cm = group_id_mapping._c()
        check(self.ctx.lib.b2_hashagg_merge(self.handle, other.handle, C.byref(cm), self.ctx.stream))

    def finalize(self) -> DeviceArray:
        cout = cabi.B2Array()
        check(self.ctx.lib.b2_hashagg_finalize(self.handle, C.byref(cout), self.ctx.stream))
        return _out(self.ctx, cout, arrow_type(cout.type))


def group_by(keys: Sequence[DeviceArray], aggregates: Sequence[tuple], fused: bool = True):
    """The Acero aggregate node's Consume/Finalize over one batch
    (acero/groupby_aggregate_node.cc:210-253,300-337): aggregates = [(function, values|None, opts)].
    Returns (unique key columns, [aggregate columns]); group order is unspecified (as under use_threads in the
    reference, whose tests sort by key)."""
    if isinstance(keys, DeviceArray):
        keys = [keys]
    # config 3's shape -- one fixed-width key, hash_sum / hash_count(only_valid) / hash_mean with default options over
    # one value column -- takes the fused path (b2_groupby_sumcount_*), exactly as the C++ b200_aggregate node does;
    # pass fused=False or any option to force the Grouper path.  hash_mean = sum / count of the same state; 64-bit
    # integer columns keep the unfused kernel (the reference's mean accumulates in double,
    # hash_aggregate_numeric.cc:353-356, which an exact int64 sum that wraps would not match).
    if fused and len(keys) == 1 and aggregates and all(
            fn in ("hash_sum", "hash_count", "hash_mean") and values is not None and not opts and values is aggregates[0][1]
            for fn, values, opts in aggregates) and keys[0].type in _NUMERIC_TYPES and aggregates[0][1].type in _NUMERIC_TYPES \
            and not pa.types.is_floating(keys[0].type) \
            and not (any(fn == "hash_mean" for fn, _, _ in aggregates) and aggregates[0][1].type in (pa.int64(), pa.uint64())):
        gb = GroupBySumCount(keys[0].type, aggregates[0][1].type, ctx=keys[0].ctx)
        gb.consume(keys[0], aggregates[0][1])
        k, s_, c_ = gb.finalize()
        m_ = None
        if any(fn == "hash_mean" for fn, _, _ in aggregates):
            m_ = divide(cast(s_, pa.float64(), safe=False), cast(c_, pa.float64(), safe=False))
        return [k], [{"hash_sum": s_, "hash_count": c_, "hash_mean": m_}[fn] for fn, _, _ in aggregates]
    g = Grouper([k.type for k in keys], keys[0].ctx)
    ids = g.consume(keys)
    outs = []
    for fn, values, opts in aggregates:
        agg = HashAggregator(fn, values.type if values is not None else None, ctx=keys[0].ctx, **(opts or {}))
        agg.resize(g.num_groups)
        agg.consume(values, ids)
        outs.append(agg.finalize())
    return g.get_uniques(), outs


class GroupBySumCount:
    """Fused consume of the aggregate node for `hash_sum` + `hash_count` over one value column
    (b2_groupby_sumcount_*): same results as Grouper + two HashAggregators."""

    def __init__(self, key_type, value_type, expected_groups=0, ctx: Optional[Context] = None):
        self.ctx = ctx or Context.get()
        self.key_type, self.value_type = pa.lib.ensure_type(key_type), pa.lib.ensure_type(value_type)
        h = C.c_void_p()
        check(self.ctx.lib.b2_groupby_sumcount_create(self.ctx.handle, type_id(self.key_type),
                                                      type_id(self.value_type), int(expected_groups), C.byref(h)))
        self.handle = h

    def __del__(self):
        if getattr(self, "handle", None):
            self.ctx.lib.b2_groupby_sumcount_destroy(self.handle)
            self.handle = None

    def consume(self, keys: DeviceArray, values: DeviceArray):
        ck, cv = keys._c(), values._c()
        check(self.ctx.lib.b2_groupby_sumcount_consume(self.handle, C.byref(ck), C.byref(cv), self.ctx.stream))

    def merge(self, keys: DeviceArray, sums: DeviceArray, counts: DeviceArray):
        """add partial (key, sum, count) states of another group-by (HashAggregateKernel::merge for the fused table)"""
        ck, cs, cc = keys._c(), sums._c(), counts._c()
        check(self.ctx.lib.b2_groupby_sumcount_merge(self.handle, C.byref(ck), C.byref(cs), C.byref(cc), self.ctx.stream))

    def path_counts(self):
        """{dense, compact, general, atomic}: chunks consumed so far by each internal path"""
        d, a, b, c = C.c_int64(), C.c_int64(), C.c_int64(), C.c_int64()
        check(self.ctx.lib.b2_groupby_sumcount_path_counts(self.handle, C.byref(d), C.byref(a), C.byref(b), C.byref(c)))
        return {"dense": d.value, "compact": a.value, "general": b.value, "atomic": c.value}

    def finalize(self):
        k, s, c = cabi.B2Array(), cabi.B2Array(), cabi.B2Array()
        check(self.ctx.lib.b2_groupby_sumcount_finalize(self.handle, C.byref(k), C.byref(s), C.byref(c),
                                                        self.ctx.stream))
        return (_out(self.ctx, k, self.key_type), _out(self.ctx, s, arrow_type(s.type)),
                _out(self.ctx, c, pa.int64()))


# ------------------------------------------------------------------------------------
# CallFunction-style registry (compute/registry.cc:87-96 lookup by name)
# ------------------------------------------------------------------------------------
_REGISTRY = {
    "cast": cast, "filter": filter, "array_filter": array_filter, "take": take, "array_take": array_take,
    "sort_indices": sort_indices, "array_sort_indices": array_sort_indices, "select_k_unstable": select_k_unstable,
    "if_else": if_else,
    "add": add, "subtract": subtract, "multiply": multiply, "divide": divide,
    "add_checked": add_checked, "subtract_checked": subtract_checked,
    "multiply_checked": multiply_checked, "divide_checked": divide_checked,
    "equal": equal, "not_equal": not_equal, "greater": greater, "greater_equal": greater_equal,
    "less": less, "less_equal": less_equal,
    "unique": unique, "value_counts": value_counts, "dictionary_encode": dictionary_encode, "count_distinct": count_distinct,
    "sum": sum, "mean": mean, "min_max": min_max, "min": min, "max": max, "count": count,
    "and": and_, "or": or_, "xor": xor, "and_not": and_not, "and_kleene": and_kleene, "or_kleene": or_kleene,
    "and_not_kleene": and_not_kleene, "invert": invert, "is_valid": is_valid, "is_null": is_null,
    "true_unless_null": true_unless_null, "is_nan": is_nan,
}


def list_functions():
    return sorted(_REGISTRY)


def call_function(name: str, args: Sequence, options=None):
    """CallFunction(name, args, options): KeyError text follows registry.cc:95."""
    fn = _REGISTRY.get(name)
    if fn is None:
        raise pa.ArrowKeyError(f"No function registered with name: {name}")
    if options is None:
        return fn(*args)
    if name == "cast":
        return cast(args[0], options=options)
    if name in ("filter", "array_filter"):
        return fn(*args, null_selection_behavior=getattr(options, "null_selection_behavior", options))
    if name in ("take", "array_take"):
        return fn(*args, boundscheck=getattr(options, "boundscheck", True))
    if name == "array_sort_indices":
        return fn(*args, order=options.order, null_placement=options.null_placement)
    if name == "select_k_unstable":
        if isinstance(options, dict):
            return fn(*args, k=options["k"], sort_keys=options.get("sort_keys"))
        # pyarrow's SelectKOptions exposes no attributes: read k and the order from its repr
        # ("SelectKOptions(k=3, sort_keys=[FieldRef.Name(x) DESC])")
        import re
        text = str(options)
        return fn(*args, k=int(re.search(r"k=(-?\d+)", text).group(1)),
                  sort_keys=[("x", "descending" if " DESC" in text else "ascending")])
    if name == "dictionary_encode":
        return fn(*args, null_encoding=getattr(options, "null_encoding", options))
    if name in ("sum", "mean", "min_max", "min", "max"):
        return fn(*args, skip_nulls=options.skip_nulls, min_count=options.min_count)
    if name in ("count", "count_distinct"):
        return fn(*args, mode=getattr(options, "mode", options))
    if name == "is_null":
        return fn(*args, nan_is_null=getattr(options, "nan_is_null", False))
    return fn(*args)
