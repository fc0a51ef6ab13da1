"""The lean kernel's range-specialised arithmetic at its thresholds.

The plan compiler's interval analysis (compiler.cpp: lower_fast) reads each column's min/max statistics and picks a
narrower instruction or accumulator wherever it can prove the values fit: the 32-bit form of the decimal rescale
(DIVR b=2), the SUM value classes (32-bit words below 2^16, 64-bit below 2^47, a per-row check above), the packed tuple
operand widths, mul.wide.s32, checked ops with a 128-bit rerun, leaf ranges clipped to the column range, Decimal MIN/MAX
held as one u64, and the sign/zero extension of every narrow column load.  Each case below puts its data exactly on one
side of such a threshold: the values sit at the first row, the last row and next to 4096-row tile boundaries.

Two layers share the case builders:
* CPU (no marker): each case lowers to the form it targets (`gpu.debug_plan`), so a compiler change cannot move a case
  off its threshold unnoticed;
* GPU: each case runs on the interpreting and the specialised lean kernel, on the general interpreter and, for grouped
  plans with a hint above 128, in the partitioned form; every result must equal the oracle and a plain Python `int`
  reference bit for bit, and an error must carry the oracle's error code.
"""
import functools
import re
from dataclasses import dataclass
from typing import Callable, List, Optional, Tuple

import numpy as np
import pytest

from llkv_b200 import ffi, gpu
from llkv_b200.expr import (AggregateKind, AggregateSpec, Bound, CompareOp, DataType, Expr, Literal, Operator, ScalarExpr,
                            pred)
from llkv_b200.table import HostColumn, HostTable, LlkvError, decimal_from_i64

I64_MIN, I64_MAX = -(1 << 63), (1 << 63) - 1
I32_MIN, I32_MAX = -(1 << 31), (1 << 31) - 1
TILE = 4096  # the zone / tile granularity of the resident image
OVERFLOW = "overflow"  # a reference result: the exact total leaves i64, the oracle's error is expected
K_RESCALE = (1, 2, 9, 10, 12, 18)
col = ScalarExpr.Column


@dataclass
class Case:
    table: HostTable
    specs: list
    expr: Optional[Expr] = None
    group_by: Tuple[int, ...] = ()
    hint: int = 0
    expr_mode: Optional[int] = None
    forms: Tuple[str, ...] = ()         # regular expressions the lean listing must match
    lean: bool = True                   # False: the plan must stay on the general interpreter
    packed_forms: Tuple[str, ...] = ()  # regular expressions the listing of the partitioned form must match
    sum_width: int = 0                  # per-thread width in bytes of the word the first SUM accumulates into
    error: bool = False                 # the reference rejects the plan (a literal outside the column's type)
    reruns: bool = False                # a checked op overflows: the lean run is repeated on the 128-bit interpreter
    ref: Optional[Callable[[], object]] = None  # {group key: [values]} or OVERFLOW, from Python ints


# ------------------------------------------------------------------------------------------------ data helpers
def edge_positions(n: int) -> List[int]:
    """Row 0, the last row, and both sides of every 4096-row boundary."""
    pos = [0, n - 1]
    for b in range(TILE, n - 1, TILE):
        pos += [b - 1, b]
    return sorted(set(pos))


def with_specials(base: List[int], specials: List[int]) -> List[int]:
    """`base` with the special values cycled over the edge positions; those that found no edge position are spread over
    the rest of the table."""
    vals = list(base)
    edges = edge_positions(len(vals))
    for i, p in enumerate(edges):
        vals[p] = specials[i % len(specials)]
    rest = specials[len(edges):]
    step = (len(vals) - 4) // (len(rest) + 1)
    for j, v in enumerate(rest):
        p = 2 + step * (j + 1)
        while p in edges:
            p += 2
        vals[p] = v
    return vals


def rdiv(x: int, k: int) -> int:
    """x / 10^k rounded half away from zero (arrow-cast's decimal rescale)."""
    d = 10 ** k
    q, r = divmod(abs(x), d)
    if 2 * r >= d:
        q += 1
    return q if x >= 0 else -q


def dec_col(field_id: int, p: int, s: int, vals: List[int]) -> HostColumn:
    return HostColumn(field_id, DataType.Decimal128(p, s), decimal_from_i64(np.array(vals, dtype=np.int64)))


def group_totals(keys, cols, fn):
    """{(key,): [fn(row values) summed per aggregate]} in first-appearance order, or OVERFLOW when a total leaves i64."""
    out = {}
    for i, k in enumerate(keys):
        acc = out.setdefault((k,) if k is not None else (), None)
        row = fn(*(c[i] for c in cols))
        out[(k,) if k is not None else ()] = row if acc is None else [a + b for a, b in zip(acc, row)]
    return out


def no_prefix_overflow(vals):
    """The oracle reports SumInt64 overflow at the first prefix that leaves i64, the kernels iff the exact total does: the
    cases only build data on which the two agree."""
    s = 0
    for v in vals:
        s += v
        if not I64_MIN <= s <= I64_MAX:
            return False
    return True


def sum_spec(e, dt=DataType.Int64, name="s"):
    return AggregateSpec(name, AggregateKind.Sum(e, dt))


# ------------------------------------------------------------------------------------------------ 1. decimal rescale
def divr_mode(data_mode: int, k: int) -> int:
    """The rescale form a correct compiler picks: the 32-bit division needs the value *and* the divisor 10^k below 2^32."""
    if data_mode == 2:
        return 2 if k <= 9 else 1
    return data_mode


def halves(k: int, limit: int, count: int = 3) -> List[int]:
    """Exact halves m*10^k + 10^k/2 below `limit`, and their neighbours."""
    d = 10 ** k
    out = []
    for m in range(count):
        h = m * d + d // 2
        if h + 1 < limit:
            out += [h - 1, h, h + 1]
    return out


def rescale_values(mode: int, n: int, seed: int) -> List[int]:
    """Scale-18 raw values: mode 2 in [0, 2^32) ending exactly at 2^32 - 1; mode 1 non-negative, crossing 2^32; mode 0
    signed.  Exact halves of every rescale of K_RESCALE, zero and the interval ends are among them."""
    rng = np.random.default_rng(seed)
    if mode == 2:
        top = (1 << 32) - 1
        base = rng.integers(0, top, n, dtype=np.int64).tolist()
        specials = [0, top, top - 1] + [h for k in K_RESCALE for h in halves(k, top)]
    else:
        top = 1 << 62
        base = rng.integers(0, top, n, dtype=np.int64).tolist()
        specials = [0, top, (1 << 32) - 1, 1 << 32, (1 << 32) + 1] + [h for k in K_RESCALE for h in halves(k, top)]
        if mode == 0:
            base = [v if i % 2 else -v for i, v in enumerate(base)]
            specials += [-v for v in specials if v] + [-top]
    return with_specials(base, specials)


def _rescale_cast_case(mode: int, grouped: bool) -> List[Case]:
    n = 70_000
    vals = rescale_values(mode, n, seed=10 + mode)
    keys = [i % 5 for i in range(n)]
    t = HostTable(1).add(dec_col(1, 38, 18, vals)).add(HostColumn(2, DataType.Int64, np.array(keys, np.int64)))
    specs = [sum_spec(ScalarExpr.Cast(col(1), DataType.Decimal128(38, 18 - k)), DataType.Decimal128(38, 18 - k), f"k{k}") for k in K_RESCALE]
    forms = tuple(rf"DIVR +a={k} b={divr_mode(mode, k)} " for k in K_RESCALE)

    def ref():
        return group_totals(keys if grouped else [None] * n, [vals], lambda x: [rdiv(x, k) for k in K_RESCALE])

    if grouped:
        return [Case(t, specs, group_by=(2,), hint=8, expr_mode=ffi.EXPR_ARROW, forms=forms, ref=ref)]
    return [Case(t, specs, forms=forms, ref=ref)]


def product_operands(mode: int, n: int, k: int, seed: int):
    """Two scale-k raw columns whose product interval is [0, 2^32 - 1] exactly (mode 2), [0, 2^62] (mode 1) or
    [-2^62, 2^62] (mode 0); rows with the exact halves of 10^k as products."""
    rng = np.random.default_rng(seed)
    if mode == 2:
        xmax, ymax = 65537, 65535  # 65537 * 65535 = 2^32 - 1
    else:
        xmax = ymax = 1 << 31
    x = rng.integers(0, xmax + 1, n, dtype=np.int64).tolist()
    y = rng.integers(0, ymax + 1, n, dtype=np.int64).tolist()
    pairs = [(xmax, ymax), (0, ymax), (xmax, 0), (1, 1)]
    lim = xmax * ymax
    for h in halves(k, lim + 1, 2):
        for j in range(0, 19):  # h = a * 10^j with both factors inside their column's range
            if h % (10 ** j) == 0 and h // 10 ** j <= xmax and 10 ** j <= ymax:
                pairs.append((h // 10 ** j, 10 ** j))
                break
    if mode == 0:
        x = [v if i % 3 else -v for i, v in enumerate(x)]
        y = [v if i % 2 else -v for i, v in enumerate(y)]
        pairs += [(-a, b) for a, b in pairs] + [(-xmax, -ymax), (-xmax, ymax)]
    for i, p in enumerate(edge_positions(n)):
        x[p], y[p] = pairs[i % len(pairs)]
    return x, y


def _rescale_product_case(mode: int, grouped: bool) -> List[Case]:
    """SUM(x_k * y_k) of two Decimal128(38, k) columns under the arrow contract: the product (scale 2k) is rescaled back
    to scale k with DIVR a=k."""
    n = 40_000
    t = HostTable(1)
    data = {}
    for k in K_RESCALE:
        x, y = product_operands(mode, n, k, seed=100 * mode + k)
        data[k] = (x, y)
        t.add(dec_col(100 + k, 38, k, x)).add(dec_col(200 + k, 38, k, y))
    keys = [(i // 7) % 3 for i in range(n)]
    t.add(HostColumn(2, DataType.Int64, np.array(keys, np.int64)))
    specs = [sum_spec(col(100 + k) * col(200 + k), DataType.Decimal128(38, k), f"k{k}") for k in K_RESCALE]
    forms = tuple(rf"DIVR +a={k} b={divr_mode(mode, k)} " for k in K_RESCALE)

    def ref():
        cols = [c for k in K_RESCALE for c in data[k]]
        return group_totals(keys if grouped else [None] * n, cols,
                            lambda *xy: [rdiv(xy[2 * i] * xy[2 * i + 1], k) for i, k in enumerate(K_RESCALE)])

    if grouped:
        return [Case(t, specs, group_by=(2,), hint=4, expr_mode=ffi.EXPR_ARROW, forms=forms, ref=ref)]
    return [Case(t, specs, forms=forms, ref=ref)]


def _rescale_compare_case(mode: int) -> List[Case]:
    """OP_CAST_D_DOWN inside an Expr::Compare leaf: CAST(v AS DECIMAL(38, 18 - k)) > 0, one plan per k."""
    n = 30_000
    vals = rescale_values(mode, n, seed=20 + mode)
    t = HostTable(1).add(dec_col(1, 38, 18, vals))
    specs = [AggregateSpec("n", AggregateKind.CountStar())]
    cases = []
    for k in K_RESCALE:
        f = Expr.Compare(ScalarExpr.Cast(col(1), DataType.Decimal128(38, 18 - k)), CompareOp.Gt, ScalarExpr.Literal(Literal.Decimal128(0, 18 - k)))
        cases.append(Case(t, specs, expr=f, forms=(rf"DIVR +a={k} b={divr_mode(mode, k)} ", r" CMP "),
                          ref=lambda k=k: {(): [sum(1 for v in vals if rdiv(v, k) > 0)]}))
    return cases


# ------------------------------------------------------------------------------------------------ 2. SUM value classes
GROUPINGS = {
    "ungrouped": ((), 0),
    "slots": ((2,), 4),     # four groups, four CTA-local slots
    "spill": ((3,), 4),     # 1000 groups behind a hint of 4: rows go to the global table
    "packed": ((3,), 1000),  # hint > 128: the partitioned form runs too
}


def sum_class_values(kind: str, n: int, keys: List[int]) -> List[int]:
    rng = np.random.default_rng(abs(hash(kind)) % (1 << 32))
    if kind == "u16_in":
        return with_specials(rng.integers(0, 1 << 16, n).tolist(), [0, (1 << 16) - 1])
    if kind == "u16_out":
        return with_specials(rng.integers(0, 1 << 16, n).tolist(), [0, (1 << 16) - 1, 1 << 16])
    if kind == "i47_in":
        m = (1 << 47) - 1
        return with_specials(rng.integers(-m, m + 1, n).tolist(), [m, -m, 0])
    if kind == "i47_out":
        m = 1 << 47
        return with_specials(rng.integers(-m + 1, m, n).tolist(), [m, -m, m - 1, 0])
    if kind == "i64_extremes":
        # INT64_MAX / INT64_MIN in alternating rows (no prefix of the row order leaves i64, while a thread of the kernel,
        # which owns every 128th row, sums only one of the two: its partial totals need the 128-bit carries), the other
        # rows small and non-positive
        vals = (-rng.integers(0, 1000, n)).tolist()
        for i in range(0, 3 * TILE):
            vals[i] = I64_MAX if i % 2 == 0 else I64_MIN
        for p in edge_positions(n)[4:]:  # (n is even)
            vals[p - p % 2], vals[p - p % 2 + 1] = I64_MAX, I64_MIN
        return vals
    # totals exactly on (or one beyond) INT64_MAX / INT64_MIN in every group: sign-uniform values, so a prefix of the row
    # order overflows iff the total does; each group's first and last rows carry the large values
    sign = 1 if kind.startswith("total_max") else -1
    target = I64_MAX if sign > 0 else I64_MIN
    if kind.endswith("_beyond"):
        target += sign
    vals = (sign * rng.integers(0, 1 << 40, n)).tolist()
    first, last = {}, {}
    for i, k in enumerate(keys):
        first.setdefault(k, i)
        last[k] = i
    for k in first:
        rows = [i for i, kk in enumerate(keys) if kk == k] if len(first) > 1 else range(n)
        rest = sum(vals[i] for i in rows if i not in (first[k], last[k]))
        remaining = target - rest
        vals[first[k]] = remaining // 2
        vals[last[k]] = remaining - remaining // 2
    return vals


SUM_KINDS = {  # value class the compiler must pick (SUM a & 3), and the word width of the per-thread accumulator
    "u16_in": (1, 4), "u16_out": (2, 8), "i47_in": (2, 8), "i47_out": (0, 8), "i64_extremes": (0, 8),
    "total_max": (0, 8), "total_max_beyond": (0, 8), "total_min": (0, 8), "total_min_beyond": (0, 8),
}


def _sum_class_case(kind: str, grouping: str) -> List[Case]:
    n = 3 * TILE + 1500 if kind != "i64_extremes" else 8 * TILE + 78
    group_by, hint = GROUPINGS[grouping]
    k4 = [(i // 3) % 4 for i in range(n)]
    k1000 = [(i * 7919) % 1000 for i in range(n)]
    keys = k4 if group_by == (2,) else k1000 if group_by == (3,) else [0] * n
    if kind == "i64_extremes" and group_by:
        keys = k4 = [(i // 2) % 4 for i in range(n)]  # a group holds whole (MAX, MIN) pairs
        k1000 = [(i // 2) % 1000 for i in range(n)]
        keys = k4 if group_by == (2,) else k1000
    vals = sum_class_values(kind, n, keys)
    for g in set(keys):
        gv = [v for v, kk in zip(vals, keys) if kk == g]
        assert no_prefix_overflow(gv) or kind.endswith("_beyond"), (kind, grouping, g)
    t = HostTable(1).add(HostColumn(1, DataType.Int64, np.array(vals, np.int64))).add(
        HostColumn(2, DataType.Int64, np.array(k4, np.int64))).add(HostColumn(3, DataType.Int64, np.array(k1000, np.int64)))
    cls, width = SUM_KINDS[kind]
    specs = [sum_spec(1), AggregateSpec("n", AggregateKind.CountStar())]

    def ref():
        out = group_totals(keys if group_by else [None] * n, [vals], lambda v: [v, 1])
        if any(not I64_MIN <= s[0] <= I64_MAX for s in out.values()):
            return OVERFLOW
        return out

    return [Case(t, specs, group_by=group_by, hint=hint, forms=(rf"SUM +a={cls} ",), sum_width=width, ref=ref)]


def _packed_width_case(bits: int, over: bool) -> List[Case]:
    """A partitioned GROUP BY packs each row's SUM operand in `bit length of max` bits: max 2^k - 1 needs k bits, 2^k
    needs k + 1; an operand of 2^32 is no longer proven below 2^32 and has no packed width."""
    n = 3 * TILE + 900
    rng = np.random.default_rng(bits)
    top = (1 << bits) if over else (1 << bits) - 1
    vals = with_specials(rng.integers(0, top, n).tolist(), [0, top])
    keys = [(i * 7919) % 1000 for i in range(n)]
    t = HostTable(1).add(HostColumn(1, DataType.UInt32 if top < (1 << 32) else DataType.Int64,
                                    np.array(vals, np.uint32 if top < (1 << 32) else np.int64))).add(
        HostColumn(3, DataType.Int64, np.array(keys, np.int64)))
    # (a product with an Int64 literal: the oracle's SUM takes Int64 operands only)
    specs = [sum_spec(col(1) * ScalarExpr.Literal(1)), AggregateSpec("n", AggregateKind.CountStar())]
    width = top.bit_length()
    packed = (rf"operands {width} ",) if width <= 32 else ()
    return [Case(t, specs, group_by=(3,), hint=1000, forms=(rf"SUM +a=\d+ b=\d+ c=\d+",), packed_forms=packed,
                 ref=lambda: group_totals(keys, [vals], lambda v: [v, 1]))]


# ------------------------------------------------------------------------------------------------ 3. mul.wide.s32
def _mul32_case(kind: str) -> List[Case]:
    """SUM / MIN / MAX of a * b with INT32_MIN and INT32_MAX in both operands (INT32_MIN^2 = 2^62).  Int32 * Int32 keeps its
    Int64 product only under the exact contract; an Int64 column whose statistics fit i32 multiplies in 32 bits too;
    one value of 2^31 takes it to the 64-bit product."""
    n = 2 * TILE + 333
    rng = np.random.default_rng(len(kind))
    a = rng.integers(-1000, 1000, n).tolist()
    b = rng.integers(-1000, 1000, n).tolist()
    amax = (1 << 31) if kind == "int64_2p31" else I32_MAX
    pairs = [(I32_MIN, I32_MIN), (I32_MIN, I32_MAX), (amax, I32_MAX), (amax, I32_MIN), (I32_MAX, -1), (I32_MIN, 1)]
    pos = edge_positions(n)
    for i, p in enumerate(pos):
        a[p], b[p] = pairs[i % len(pairs)] if i < len(pairs) else (0, 0)
    assert no_prefix_overflow([x * y for x, y in zip(a, b)])
    ta = DataType.Int32 if kind == "int32" else DataType.Int64
    t = HostTable(1).add(HostColumn(1, ta, np.array(a, np.int32 if kind == "int32" else np.int64))).add(
        HostColumn(2, DataType.Int32, np.array(b, np.int32)))
    e = col(1) * col(2)
    specs = [sum_spec(e), AggregateSpec("mn", AggregateKind.Min(e, DataType.Int64)), AggregateSpec("mx", AggregateKind.Max(e, DataType.Int64))]
    fb = 2 if kind == "int64_2p31" else 3  # FB_MUL / FB_MUL32 (plan.h FastBin)
    prods = [x * y for x, y in zip(a, b)]
    return [Case(t, specs, expr_mode=ffi.EXPR_EXACT if kind == "int32" else None, forms=(rf"OP_COL +a={fb} ",),
                 ref=lambda: {(): [sum(prods), min(prods), max(prods)]})]


# ------------------------------------------------------------------------------------------------ 4. leaves at the column extremes
NARROW = {  # type: (numpy type, min, max)
    "Int8": (DataType.Int8, np.int8, -128, 127),
    "UInt8": (DataType.UInt8, np.uint8, 0, 255),
    "Int16": (DataType.Int16, np.int16, -(1 << 15), (1 << 15) - 1),
    "UInt16": (DataType.UInt16, np.uint16, 0, (1 << 16) - 1),
    "UInt32": (DataType.UInt32, np.uint32, 0, (1 << 32) - 1),
    "Int32": (DataType.Int32, np.int32, I32_MIN, I32_MAX),
    "Date32": (DataType.Date32, np.int32, I32_MIN, I32_MAX),
    "UInt64": (DataType.UInt64, np.uint64, 0, (1 << 64) - 1),
    "D32": (DataType.Decimal128(10, 2), None, I32_MIN, I32_MAX),
    "D64": (DataType.Decimal128(19, 2), None, I64_MIN, I64_MAX),
}


def s64(v: int) -> int:
    """The listing prints a leaf bound as the signed 64-bit image of its bits."""
    v &= (1 << 64) - 1
    return v - (1 << 64) if v >> 63 else v


def leaf_filters(name: str, lo: int, hi: int, L):
    """(operator, the values it accepts as [a, b]) at and beyond the type's extremes; L(v) is the literal of value v."""
    inf = 1 << 70
    ops = [
        (Operator.Equals(L(lo)), (lo, lo)), (Operator.Equals(L(hi)), (hi, hi)),
        (Operator.GreaterThan(L(lo)), (lo + 1, inf)), (Operator.LessThan(L(hi)), (-inf, hi - 1)),
        (Operator.GreaterThanOrEquals(L(lo)), (lo, inf)), (Operator.LessThanOrEquals(L(hi)), (-inf, hi)),
        (Operator.GreaterThan(L(hi)), (hi + 1, inf)), (Operator.LessThan(L(lo)), (-inf, lo - 1)),
        (Operator.Range(Bound.Excluded(L(lo)), Bound.Excluded(L(hi))), (lo + 1, hi - 1)),
    ]
    if name not in ("UInt64", "D64"):  # literals beyond the type's range
        ops += [(Operator.Range(Bound.Included(L(lo - 1)), Bound.Included(L(hi + 1))), (lo - 1, hi + 1)),
                (Operator.Equals(L(hi + 1)), (hi + 1, hi + 1)), (Operator.GreaterThan(L(hi + 1)), (hi + 2, inf))]
        if lo < 0:
            ops.append((Operator.Equals(L(lo - 1)), (lo - 1, lo - 1)))
    if name in ("UInt32", "Int32", "Date32", "D32", "UInt16"):  # beyond i32
        ops += [(Operator.Equals(L(1 << 31)), (1 << 31, 1 << 31)), (Operator.LessThan(L(1 << 31)), (-inf, (1 << 31) - 1)),
                (Operator.GreaterThanOrEquals(L(-(1 << 31) - 1)), (-(1 << 31) - 1, inf))]
    if name == "UInt64":  # at and above 2^63
        ops += [(Operator.Equals(L(1 << 63)), (1 << 63, 1 << 63)), (Operator.GreaterThanOrEquals(L(1 << 63)), (1 << 63, inf)),
                (Operator.LessThan(L(1 << 63)), (-inf, (1 << 63) - 1)),
                (Operator.Range(Bound.Included(L((1 << 63) - 1)), Bound.Excluded(L((1 << 63) + 2))), ((1 << 63) - 1, (1 << 63) + 1))]
    return ops


def _leaf_literal(name: str):
    if name in ("D32", "D64"):
        return lambda v: Literal.Decimal128(v, 2)
    if name == "Date32":
        return Literal.Date32
    return Literal.Int128


def _leaf_case(name: str) -> List[Case]:
    dtype, npt, lo, hi = NARROW[name]
    n = 3 * TILE + 211
    rng = np.random.default_rng(len(name) * 31)
    if name == "D64":
        lo, hi = I64_MIN + 1, I64_MAX  # a Decimal128 image strictly inside i64 narrows to 8 bytes
    base = [int(v) for v in rng.integers(max(lo, -(1 << 62)), min(hi, 1 << 62), n, dtype=np.int64)] if hi < (1 << 63) else \
        [int(v) for v in rng.integers(0, 1 << 64, n, dtype=np.uint64)]
    specials = [lo, hi, lo + 1, hi - 1, 0] + ([(1 << 63) - 1, 1 << 63, (1 << 63) + 1] if name == "UInt64" else [])
    vals = with_specials(base, specials)
    w = [(-1, 1, 2, -2)[i % 4] for i in range(n)]
    t = HostTable(1)
    t.add(dec_col(1, dtype.precision, dtype.scale, vals) if name in ("D32", "D64") else HostColumn(1, dtype, np.array(vals, dtype=npt)))
    t.add(HostColumn(2, DataType.Int64, np.array(w, np.int64)))
    specs = [AggregateSpec("n", AggregateKind.CountStar())]
    if name in ("UInt64", "D64"):
        specs.append(sum_spec(2))
        prod = None
    else:  # the narrow load inside the arithmetic (exact contract: arrow-arith has no UInt8 * Int64), its sign / zero
        # extension reaches the aggregates
        e = col(1) * col(2)
        dt = DataType.Decimal128(38, 2) if name == "D32" else DataType.Int64
        specs += [sum_spec(e, dt), AggregateSpec("mn", AggregateKind.Min(e, dt)), AggregateSpec("mx", AggregateKind.Max(e, dt))]
        prod = [v * x for v, x in zip(vals, w)]
    cmin, cmax = min(vals), max(vals)
    cases = []
    for op, (a, b) in leaf_filters(name, lo, hi, _leaf_literal(name)):
        flo, fhi = max(a, cmin), min(b, cmax)
        form = rf"range \[{s64(flo)}, {s64(fhi)}\]" if flo <= fhi else r"range \[1, 0\]"
        sel = [i for i, v in enumerate(vals) if a <= v <= b]
        outside = name not in ("D32", "D64") and any(not lo <= l.value <= hi for l in op.literals)

        def ref(sel=sel):
            r = [len(sel)]
            if prod is None:
                r.append(sum(w[i] for i in sel) if sel else None)
            else:
                p = [prod[i] for i in sel]
                # (over no rows a Decimal128 SUM is 0, an Int64 SUM is NULL: the reference's accumulators)
                r += [sum(p), min(p), max(p)] if p else [0 if name == "D32" else None, None, None]
            return {(): r}

        cases.append(Case(t, specs, expr=pred(1, op), expr_mode=ffi.EXPR_EXACT, forms=(r" LEAF ", form), error=outside,
                          ref=None if outside else ref))
    return cases


# ------------------------------------------------------------------------------------------------ 5. Decimal MIN/MAX
def _dec_minmax_case(kind: str) -> List[Case]:
    """Values strictly inside i64 keep the thread state as one order-preserving u64 (MIN_I / MAX_I with a = 0x80);
    INT64_MIN itself would be the identity of that state, so the plan stays on the general interpreter."""
    n = 2 * TILE + 999
    rng = np.random.default_rng(7)
    lo = I64_MIN if kind == "general" else I64_MIN + 1
    vals = with_specials(rng.integers(-(1 << 62), 1 << 62, n).tolist(), [lo, I64_MAX - 1, 0, -1])
    keys = [(i // 5) % 3 for i in range(n)]
    t = HostTable(1).add(dec_col(1, 38, 2, vals)).add(HostColumn(2, DataType.Int64, np.array(keys, np.int64)))
    dt = DataType.Decimal128(38, 2)
    specs = [AggregateSpec("mn", AggregateKind.Min(1, dt)), AggregateSpec("mx", AggregateKind.Max(1, dt)), AggregateSpec("n", AggregateKind.CountStar())]
    lean = kind != "general"

    def ref(grouped):
        out = {}
        for v, k in zip(vals, keys if grouped else [None] * n):
            key = (k,) if grouped else ()
            m = out.get(key)
            out[key] = [v, v, 1] if m is None else [min(m[0], v), max(m[1], v), m[2] + 1]
        return out

    forms = (r"MIN_I +a=128 ", r"MAX_I +a=128 ") if lean else ()
    return [Case(t, specs, forms=forms, lean=lean, ref=lambda: ref(False)),
            Case(t, specs, group_by=(2,), hint=4, forms=forms, lean=lean, ref=lambda: ref(True))]


# ------------------------------------------------------------------------------------------------ 6. checked ops
def checked_table(n: int):
    """x * y of two Decimal128(38, 2) columns whose statistics allow products beyond i64: FB_MUL_CK.  Every product fits
    i64 except the one in the last tile."""
    rng = np.random.default_rng(3)
    x = rng.integers(-(1 << 20), 1 << 20, n).tolist()
    y = rng.integers(-(1 << 20), 1 << 20, n).tolist()
    x[0], y[0] = (1 << 40), 5           # the statistics reach 2^40 in both columns ...
    x[1], y[1] = -3, (1 << 40)
    x[n - 2], y[n - 2] = (1 << 40), (1 << 40)  # ... and only this product leaves i64 (2^80)
    keys = [(i // 11) % 4 for i in range(n)]
    t = HostTable(1).add(dec_col(1, 38, 2, x)).add(dec_col(2, 38, 2, y)).add(HostColumn(3, DataType.Int64, np.array(keys, np.int64)))
    return t, x, y, keys


def checked_specs():
    dt = DataType.Decimal128(38, 4)
    return [sum_spec(col(1) * col(2), dt), AggregateSpec("n", AggregateKind.CountStar())]


def _checked_case(grouped: bool) -> List[Case]:
    n = 5 * TILE + 17
    t, x, y, keys = checked_table(n)

    def ref():
        out = {}
        for i in range(n):
            key = (keys[i],) if grouped else ()
            p = x[i] * y[i]
            m = out.get(key)
            out[key] = [p, 1] if m is None else [m[0] + p, m[1] + 1]
        return out

    return [Case(t, checked_specs(), group_by=(3,) if grouped else (), hint=4 if grouped else 0, expr_mode=ffi.EXPR_EXACT,
                 forms=(r"OP_COL +a=6 ",), reruns=True, ref=ref)]


# ------------------------------------------------------------------------------------------------ registry
BUILDERS = {}
for _m in (2, 1, 0):
    BUILDERS[f"rescale_cast_b{_m}"] = functools.partial(_rescale_cast_case, _m, False)
    BUILDERS[f"rescale_product_b{_m}"] = functools.partial(_rescale_product_case, _m, False)
    BUILDERS[f"rescale_compare_b{_m}"] = functools.partial(_rescale_compare_case, _m)
# grouped plans under the arrow contract (each grouped shape costs a few seconds of NVRTC: the 32-bit mode only)
BUILDERS["rescale_cast_b2_grouped"] = functools.partial(_rescale_cast_case, 2, True)
BUILDERS["rescale_product_b2_grouped"] = functools.partial(_rescale_product_case, 2, True)
for _k in SUM_KINDS:
    for _g in GROUPINGS:
        BUILDERS[f"sum_{_k}_{_g}"] = functools.partial(_sum_class_case, _k, _g)
for _b in (8, 16, 31, 32):
    BUILDERS[f"packed_width_{_b}"] = functools.partial(_packed_width_case, _b, False)
    BUILDERS[f"packed_width_{_b}_plus1"] = functools.partial(_packed_width_case, _b, True)
for _k in ("int32", "int64_fits_i32", "int64_2p31"):
    BUILDERS[f"mul_{_k}"] = functools.partial(_mul32_case, _k)
for _t in NARROW:
    BUILDERS[f"leaf_{_t}"] = functools.partial(_leaf_case, _t)
BUILDERS["decimal_minmax_lean"] = functools.partial(_dec_minmax_case, "lean")
BUILDERS["decimal_minmax_general"] = functools.partial(_dec_minmax_case, "general")
BUILDERS["checked_mul"] = functools.partial(_checked_case, False)
BUILDERS["checked_mul_grouped"] = functools.partial(_checked_case, True)


@functools.lru_cache(maxsize=None)
def cases(name: str) -> List[Case]:
    return BUILDERS[name]()


def listing(case: Case, **kw) -> str:
    return gpu.debug_plan(case.table, case.expr, case.specs, group_by=case.group_by, expr_mode=case.expr_mode,
                          cardinality_hint=case.hint, **kw)


# ================================================================================================ CPU layer
@pytest.mark.parametrize("name", sorted(BUILDERS))
def test_case_lowers_to_its_target_form(name):
    from oracle import oracle
    for i, case in enumerate(cases(name)):
        if case.error:  # a literal the column's type cannot hold: the reference's error, raised by both
            with pytest.raises(LlkvError) as e:
                listing(case)
            with pytest.raises(LlkvError) as ei:
                oracle.aggregate(case.table, case.expr, case.specs, group_by=case.group_by, expr_mode=case.expr_mode)
            assert ei.value.code == e.value.code, (name, i, e.value, ei.value)
            continue
        text = listing(case)
        if not case.lean:
            assert text.startswith("general interpreter"), (name, i, text)
            continue
        assert text.startswith("lean plan"), (name, i, text)
        for f in case.forms:
            assert re.search(f, text), (name, i, f, text)
        if case.sum_width:
            word = re.search(r"SUM +a=\d+ b=(\d+) ", text).group(1)
            assert re.search(rf"word {word}: kind \d+ width {case.sum_width} ", text), (name, i, text)
        if case.packed_forms:
            packed = listing(case, packed=True)
            for f in case.packed_forms:
                assert re.search(f, packed), (name, i, f, packed)


@pytest.mark.parametrize("k, mode", [(9, 2), (10, 1), (12, 1), (18, 1)])
def test_decimal_rescale_takes_the_32_bit_division_only_with_a_32_bit_divisor(k, mode):
    """DIVR b=2 divides in 32 bits: the value (proven in [0, 2^32)) *and* the divisor 10^k must fit.  10^10 truncated to
    32 bits is 1 410 065 408."""
    t = HostTable(1).add(dec_col(1, 38, 12, [0, 59_999, 12_345]))
    text = gpu.debug_plan(t, None, [sum_spec(col(1) * col(1), DataType.Decimal128(38, 12))])
    assert re.search(r"DIVR +a=12 b=1 ", text), text
    t = HostTable(1).add(dec_col(1, 38, 18, [0, (1 << 32) - 1]))
    text = gpu.debug_plan(t, None, [sum_spec(ScalarExpr.Cast(col(1), DataType.Decimal128(38, 18 - k)), DataType.Decimal128(38, 18 - k))])
    assert re.search(rf"DIVR +a={k} b={mode} ", text), text


def test_reference_values_are_plain_integer_arithmetic():
    """The Python reference the GPU layer compares with: exact halves round away from zero in both signs."""
    assert [rdiv(v, 1) for v in (5, 4, -5, -4, 15, -15, 0)] == [1, 0, -1, 0, 2, -2, 0]
    assert rdiv(10 ** 18 // 2, 18) == 1 and rdiv(10 ** 18 // 2 - 1, 18) == 0 and rdiv(-(10 ** 18) // 2, 18) == -1
    assert rdiv((1 << 32) - 1, 10) == 0 and rdiv(5 * 10 ** 9, 10) == 1
    assert no_prefix_overflow([I64_MAX, I64_MIN, I64_MAX]) and not no_prefix_overflow([I64_MAX, 1])


# ================================================================================================ GPU layer
WAYS = ("interpreted", "specialised", "general", "partitioned")


def _values(rows):
    return {key: [v.value for v in vals] for key, vals in rows}


def _run(ctx, dt, case: Case, way: str):
    if way == "interpreted":
        ctx.set_jit(0)
    elif way == "specialised":
        ctx.set_jit(2)
    elif way == "general":
        ctx.set_tuning(force_wide=2)
    else:
        ctx.set_jit(2)
        ctx.set_partitioning(2)
    prog = gpu.Program(ctx, case.expr) if case.expr is not None else None
    agg = None
    try:
        agg = gpu.Aggregation(dt, case.specs, case.group_by, case.expr_mode, case.hint)
        agg.run(prog)
        return agg.finalize(), agg.run_info()
    finally:
        if agg:
            agg.destroy()
        if prog:
            prog.destroy()
        ctx.set_jit(1)
        ctx.set_tuning()
        ctx.set_partitioning(1)


def _check_case(ctx, dt, case: Case, label):
    import util
    from oracle import oracle
    try:
        want, want_err = oracle.aggregate(case.table, case.expr, case.specs, group_by=case.group_by, expr_mode=case.expr_mode), None
    except LlkvError as e:
        want, want_err = None, e
    expect = case.ref() if case.ref else None
    assert (want_err is not None) == (case.error or expect is OVERFLOW), (label, want_err)
    if expect is OVERFLOW:
        assert want_err is not None, (label, "the oracle accepted a total beyond i64")
    elif expect is not None:
        assert want_err is None, (label, want_err)
        assert _values(want) == expect, (label, "oracle != Python reference")
    ways = list(WAYS[:3])
    partitioned = False
    if case.group_by and case.hint > 128:
        ways.append("partitioned")
        partitioned = "partitioned" in listing(case, partition=True)
    for way in ways:
        if want_err is not None:
            with pytest.raises(LlkvError) as ei:
                _run(ctx, dt, case, way)
            assert ei.value.code == want_err.code, (label, way, ei.value, want_err)
            continue
        got, info = _run(ctx, dt, case, way)
        util.assert_same_result(got, want, ordered=False)
        if expect is not None:
            assert _values(got) == expect, (label, way)
        if case.reruns:
            if way != "general":  # (the run info then describes the rerun)
                assert info.used_wide_path == 1 and info.used_fast_kernel == 0, (label, way)
        elif case.lean:
            assert info.used_fast_kernel == (0 if way == "general" else 1), (label, way)
            if way in ("specialised", "partitioned") and info.kernel_launches:  # (no launch: every tile pruned)
                assert info.used_jit_kernel == 1, (label, way)
        if way == "partitioned":
            assert (info.partitions > 0) == partitioned, (label, info.partitions)
            if case.packed_forms:
                assert info.packed_tuples != 0, label


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(BUILDERS))
def test_case_matches_oracle_and_reference_on_every_kernel(gpu_ctx, name):
    group = cases(name)
    dt = gpu.DeviceTable.from_host(gpu_ctx, group[0].table)
    try:
        for i, case in enumerate(group):
            assert case.table is group[0].table
            _check_case(gpu_ctx, dt, case, (name, i))
    finally:
        dt.destroy()


@pytest.mark.gpu
@pytest.mark.parametrize("grouped", [False, True])
def test_checked_product_overflowing_in_the_last_range_reruns_from_the_saved_state(gpu_ctx, grouped):
    """Three runs over consecutive row ranges into one accumulator; only the third meets the product beyond i64.  The
    128-bit rerun of that range must start from the state the first two left (the group table's backup when grouped),
    so the result equals the oracle over the whole range."""
    import util
    from oracle import oracle
    n = 5 * TILE + 17
    t, x, y, keys = checked_table(n)
    group_by = (3,) if grouped else ()
    specs = checked_specs()
    want = oracle.aggregate(t, None, specs, group_by=group_by, expr_mode=ffi.EXPR_EXACT)
    dt = gpu.DeviceTable.from_host(gpu_ctx, t)
    cuts = [0, 2 * TILE + 5, 4 * TILE - 1, n]
    try:
        for jit in (0, 2):
            gpu_ctx.set_jit(jit)
            agg = gpu.Aggregation(dt, specs, group_by, ffi.EXPR_EXACT, 4 if grouped else 0)
            try:
                agg.reset()
                for r in range(3):
                    agg.run(None, False, cuts[r], cuts[r + 1])
                    if r < 2:
                        info = agg.run_info()
                        assert (info.used_fast_kernel, info.used_wide_path) == (1, 0), (jit, r)
                util.assert_same_result(agg.finalize(), want, ordered=False)
                # the third range overflowed and was run again on the 128-bit interpreter (settled by finalize)
                info = agg.run_info()
                assert (info.used_fast_kernel, info.used_wide_path) == (0, 1), jit
            finally:
                agg.destroy()
                gpu_ctx.set_jit(1)
    finally:
        dt.destroy()


@pytest.mark.gpu
def test_narrowed_decimal_column_rewidens_when_a_later_chunk_leaves_i32(gpu_ctx):
    """A Decimal128 column holding +-(2^31 - 1) and -2^31 is resident as 4-byte values (D32); a chunk appended after the
    seal with 2^31 widens it.  MIN / MAX / SUM / a leaf at the extremes agree with the oracle before and after."""
    import util
    from oracle import oracle
    n = 2 * TILE + 100
    rng = np.random.default_rng(11)
    vals = with_specials(rng.integers(-1000, 1000, n).tolist(), [I32_MAX, -I32_MAX, I32_MIN])
    more = with_specials(rng.integers(-1000, 1000, TILE + 3).tolist(), [1 << 31, I32_MIN])
    dtype = DataType.Decimal128(12, 2)
    dt_out = DataType.Decimal128(38, 2)
    specs = [AggregateSpec("mn", AggregateKind.Min(1, dt_out)), AggregateSpec("mx", AggregateKind.Max(1, dt_out)),
             sum_spec(1, dt_out), AggregateSpec("n", AggregateKind.CountStar())]
    flt = pred(1, Operator.Range(Bound.Included(Literal.Decimal128(I32_MIN, 2)), Bound.Excluded(Literal.Decimal128(I32_MAX, 2))))
    before = HostTable(1).add(dec_col(1, 12, 2, vals))
    after = HostTable(1).add(dec_col(1, 12, 2, vals + more))
    assert "col 0: 4 B/row" in gpu.debug_plan(before, flt, specs) and "col 0: 8 B/row" in gpu.debug_plan(after, flt, specs)
    dt = gpu.DeviceTable.from_host(gpu_ctx, before)
    try:
        for table in (before, after):
            if table is after:
                dt.columns[1].append(dec_col(1, 12, 2, more))
                dt.n_rows = len(vals) + len(more)
                dt.seal()
            for expr in (None, flt):
                want = oracle.aggregate(table, expr, specs)
                ref_rows = [v for v in decimal_values(table) if expr is None or I32_MIN <= v < I32_MAX]
                assert _values(want) == {(): [min(ref_rows), max(ref_rows), sum(ref_rows), len(ref_rows)]}
                for jit in (0, 2):
                    gpu_ctx.set_jit(jit)
                    try:
                        util.assert_same_result(dt.aggregate(expr, specs), want)
                    finally:
                        gpu_ctx.set_jit(1)
    finally:
        dt.destroy()


def decimal_values(table: HostTable) -> List[int]:
    v = table.columns[1].values
    return [int(x) for x in v[:, 0].view(np.int64)]
