"""Repeated steps on the one-kernel path (a lean scan that publishes its result to page-locked memory and re-arms the
state) for every accumulator class, and every way a step sequence leaves or re-enters that path.

The re-arm writes each accumulator word back to its class's starting value and every key back to empty.  A word of one
class re-armed with the wrong value makes only that class wrong, and only from the second step on, so each case here
runs a script of steps and checks every one of them:

* A: the whole table under a filter;  E: nothing selected (a filter no row meets, or an empty row range);  B: a row range
  holding the extreme rows, among them values equal to a class's starting value (INT64_MIN under MAX, INT64_MAX under
  MIN, NaN payloads whose order image is all ones or all zeros).
* Every result equals the oracle (bit-exact integers, decimals, counts and keys; 1e-12 relative for f64).
* `run_info().published_steps` grows by one for each step whose scan published the result: every step of a plan whose
  table fits the 64 KiB stage, except a step over an empty row range (no launch, the result is the armed state) and the
  aggregate's first step (its state is created after the reset that would have armed it).
* The stage boundary: the largest tables that fit publish, the smallest that do not keep the reset / scan / copy form,
  and a table that grows past the stage during a step stops publishing from then on.
* A seeded random walk over the step state machine on a mutable table: execute / run / reset / finalize / set_output,
  appends, deletes and updates, knob changes, bitmaps and column scans between execute and finalize, and 128-bit
  reruns.

The CPU tests (no marker) pin the plan listing of every case, so a lowering change cannot move a case off the path
it is meant to exercise."""
import re
from dataclasses import dataclass, field
from typing import List, Optional, Tuple

import numpy as np
import pytest

import util
from llkv_b200 import ffi, gpu
from llkv_b200.expr import AggregateKind, AggregateSpec, AggregateValue, Bound, DataType, Expr, Operator, ScalarExpr, pred
from llkv_b200.table import HostColumn, HostTable, LlkvError, Snapshot, decimal_from_i64, pack_validity
from oracle import oracle

ONE_KERNEL = "step: one kernel, the scan publishes the result to page-locked memory and re-arms the state"
THREE_PARTS = "step: reset, scan, result copy"
STAGE_BYTES = 64 << 10
I64_MIN, I64_MAX = -(1 << 63), (1 << 63) - 1
col = ScalarExpr.Column


def group_table_cap(hint: int) -> int:
    """Rows of a grouped aggregate's global table at its first run (llkv_gpu.cu: group_table_cap)."""
    if not hint:
        return 1024
    cap = 1
    while cap < max(32, 2 * hint):
        cap *= 2
    return cap


def result_bytes(gcap: int, n_gwords: int, n_keys: int) -> int:
    return (gcap + 2) * n_gwords * 8 + (gcap * 8 if n_keys else 0)


def listing_words(text: str) -> int:
    return int(re.match(r"lean plan: \d+ instr, \d+ cols, (\d+) words", text).group(1))


def step_line(text: str) -> str:
    lines = [ln for ln in text.splitlines() if ln.startswith("step: ")]
    assert len(lines) == 1, text
    return lines[0]


# ================================================================================================ 2a: the class matrix
N = 6 * 4096 + 777
B_LO, B_HI = 9_000, 13_500   # the extreme rows live here
SEL = 30                     # filter column: even values 0..98 in every zone, so a filter on it never prunes a tile
F_A = pred(SEL, Operator.Range(Bound.Included(0), Bound.Included(90)))
F_NONE = pred(SEL, Operator.Equals(51))
NAN_ONES = np.array([0x7FFFFFFFFFFFFFFF], np.uint64).view(np.float64)[0]   # order image all ones
NAN_ZEROS = np.array([0xFFFFFFFFFFFFFFFF], np.uint64).view(np.float64)[0]  # order image all zeros
NAN32_ONES = np.array([0x7FFFFFFF], np.uint32).view(np.float32)[0]
NAN32_ZEROS = np.array([0xFFFFFFFF], np.uint32).view(np.float32)[0]


def _nullable(rng, vals, share=0.15):
    valid = rng.random(vals.shape[0]) > share
    return valid, pack_validity(valid)


def matrix_table() -> HostTable:
    rng = np.random.default_rng(2024)
    t = HostTable(61)
    b = slice(B_LO, B_HI)

    def ints(npt, lo, hi, specials):
        v = rng.integers(lo, hi, N, endpoint=True).astype(npt)
        pos = rng.choice(np.arange(B_LO, B_HI), size=len(specials), replace=False)
        v[pos] = np.array(specials).astype(npt)
        return v

    i8, i16, i32 = np.iinfo(np.int8), np.iinfo(np.int16), np.iinfo(np.int32)
    t.add(HostColumn(1, DataType.Int8, ints(np.int8, -100, 100, [i8.min, i8.max])))
    t.add(HostColumn(2, DataType.Int16, ints(np.int16, -30_000, 30_000, [i16.min, i16.max])))
    t.add(HostColumn(3, DataType.Int32, ints(np.int32, -(1 << 30), 1 << 30, [i32.min, i32.max])))
    t.add(HostColumn(4, DataType.Int64, ints(np.int64, -(1 << 40), 1 << 40, [-(1 << 47), 1 << 47])))
    t.add(HostColumn(5, DataType.UInt8, ints(np.uint8, 1, 200, [0, 255])))
    t.add(HostColumn(6, DataType.UInt16, ints(np.uint16, 1, 60_000, [0, 65_535])))
    t.add(HostColumn(7, DataType.UInt32, ints(np.uint32, 1, 1 << 31, [0, (1 << 32) - 1])))
    t.add(HostColumn(9, DataType.Date32, ints(np.int32, 8_000, 12_000, [i32.min, i32.max])))
    f32 = (rng.integers(-4000, 4000, N) / 8).astype(np.float32)
    f32[B_LO:B_LO + 8] = [np.nan, -np.nan, 0.0, -0.0, np.inf, -np.inf, NAN32_ONES, NAN32_ZEROS]
    t.add(HostColumn(10, DataType.Float32, f32))
    f64 = rng.integers(-4000, 4000, N) / 8
    f64[B_LO + 10:B_LO + 18] = [np.nan, -np.nan, 0.0, -0.0, np.inf, -np.inf, NAN_ONES, NAN_ZEROS]
    t.add(HostColumn(11, DataType.Float64, f64))
    t.add(HostColumn(12, DataType.Decimal128(9, 2), decimal_from_i64(ints(np.int64, -(1 << 28), 1 << 28, [i32.min, i32.max]))))
    t.add(HostColumn(13, DataType.Decimal128(18, 2), decimal_from_i64(ints(np.int64, -(1 << 50), 1 << 50, [I64_MIN + 1, I64_MAX - 1]))))
    # nullable copies
    _, v14 = _nullable(rng, t.columns[4].values)
    t.add(HostColumn(14, DataType.Int64, t.columns[4].values.copy(), v14))
    _, v15 = _nullable(rng, f64)
    t.add(HostColumn(15, DataType.Float64, (rng.integers(-4000, 4000, N) / 8).astype(np.float64), v15))
    _, v16 = _nullable(rng, f64)
    t.add(HostColumn(16, DataType.Decimal128(18, 2), decimal_from_i64(rng.integers(-(1 << 40), 1 << 40, N)), v16))
    valid17, v17 = _nullable(rng, f64, 0.5)
    valid17[b] = False  # a column with no valid row in B: COUNT 0, MIN / MAX / SUM NULL there
    t.add(HostColumn(17, DataType.Int32, rng.integers(-1000, 1000, N).astype(np.int32), pack_validity(valid17)))
    # the starting values of the MIN / MAX words: every row of B holds INT64_MAX (under MIN) / INT64_MIN (under MAX)
    mx = rng.integers(-(1 << 40), 1 << 40, N)
    mx[b] = I64_MIN
    t.add(HostColumn(18, DataType.Int64, mx))
    mn = rng.integers(-(1 << 40), 1 << 40, N)
    mn[b] = I64_MAX
    t.add(HostColumn(19, DataType.Int64, mn))
    t.add(HostColumn(SEL, DataType.Int64, 2 * rng.integers(0, 50, N)))
    # keys
    t.add(HostColumn(40, DataType.Int64, rng.integers(0, 4, N)))
    k41 = rng.integers(0, 10, N).astype(np.int32)
    _, v41 = _nullable(rng, f64, 0.1)
    t.add(HostColumn(41, DataType.Int32, k41, v41))
    short = ["A", "N", "R", "xy", "zzzzzzz"]
    t.add(HostColumn.utf8(42, [short[i] for i in rng.integers(0, len(short), N)]))
    long_ = ["DELIVER IN PERSON", "COLLECT COD", "TAKE BACK RETURN", "NONE-AT-ALL", "a somewhat longer string"]
    t.add(HostColumn.utf8(43, [long_[i] for i in rng.integers(0, len(long_), N)]))
    t.add(HostColumn(44, DataType.Int64, rng.integers(0, 300, N) * 7 - 1000))
    dv = rng.integers(0, 1500, N)
    _, v45 = _nullable(rng, f64, 0.05)
    t.add(HostColumn(45, DataType.Int64, dv, v45))
    return t


def _s(name, kind):
    return AggregateSpec(name, kind)


I64, F64 = DataType.Int64, DataType.Float64
DEC38 = DataType.Decimal128(38, 2)


def int_specs():
    return [_s("n", AggregateKind.CountStar()), _s("c14", AggregateKind.Count(14)), _s("nn14", AggregateKind.CountNulls(14)),
            _s("c17", AggregateKind.Count(17)), _s("nn17", AggregateKind.CountNulls(17)),
            _s("s4", AggregateKind.Sum(4, I64)), _s("s14", AggregateKind.Sum(14, I64)), _s("a4", AggregateKind.Avg(4, F64)),
            _s("t14", AggregateKind.Total(14, I64)), _s("s17", AggregateKind.Sum(ScalarExpr.Cast(col(17), I64), I64)),
            _s("mn4", AggregateKind.Min(4, I64)), _s("mx4", AggregateKind.Max(4, I64)), _s("mn14", AggregateKind.Min(14, I64)),
            _s("mx18", AggregateKind.Max(18, I64)), _s("mn19", AggregateKind.Min(19, I64))]


def narrow_specs():
    """MIN / MAX of the narrow integer, date and unsigned columns (the reference aggregates Int64 and Float64 arguments:
    through a cast)."""
    c64 = lambda f: ScalarExpr.Cast(col(f), I64)
    cf = lambda f: ScalarExpr.Cast(col(f), F64)
    return [_s("n", AggregateKind.CountStar()),
            _s("mn1", AggregateKind.Min(c64(1), I64)), _s("mx1", AggregateKind.Max(c64(1), I64)),
            _s("mn2", AggregateKind.Min(c64(2), I64)), _s("mx2", AggregateKind.Max(c64(2), I64)),
            _s("mn3", AggregateKind.Min(c64(3), I64)), _s("mx3", AggregateKind.Max(c64(3), I64)),
            _s("mn9", AggregateKind.Min(c64(9), I64)), _s("mx9", AggregateKind.Max(c64(9), I64)), _s("mx17", AggregateKind.Max(c64(17), I64)),
            _s("mn5", AggregateKind.Min(cf(5), F64)), _s("mx6", AggregateKind.Max(cf(6), F64)),
            _s("mx7", AggregateKind.Max(cf(7), F64)), _s("s7", AggregateKind.Sum(cf(7), F64))]


def float_specs():
    cf = lambda f: ScalarExpr.Cast(col(f), F64)
    return [_s("n", AggregateKind.CountStar()), _s("c15", AggregateKind.Count(15)), _s("nn15", AggregateKind.CountNulls(15)),
            _s("s11", AggregateKind.Sum(11, F64)), _s("t11", AggregateKind.Total(11, F64)), _s("a11", AggregateKind.Avg(11, F64)),
            _s("mn11", AggregateKind.Min(11, F64)), _s("mx11", AggregateKind.Max(11, F64)),
            _s("s15", AggregateKind.Sum(15, F64)), _s("a15", AggregateKind.Avg(15, F64)),
            _s("mn15", AggregateKind.Min(15, F64)), _s("mx15", AggregateKind.Max(15, F64)),
            _s("s10", AggregateKind.Sum(cf(10), F64)), _s("mn10", AggregateKind.Min(cf(10), F64)), _s("mx10", AggregateKind.Max(cf(10), F64)),
            _s("t4", AggregateKind.Total(4, F64))]


def dec_specs():
    return [_s("n", AggregateKind.CountStar()), _s("c16", AggregateKind.Count(16)), _s("nn16", AggregateKind.CountNulls(16)),
            _s("s12", AggregateKind.Sum(12, DEC38)), _s("a12", AggregateKind.Avg(12, DEC38)),
            _s("mn12", AggregateKind.Min(12, DEC38)), _s("mx12", AggregateKind.Max(12, DEC38)),
            _s("s13", AggregateKind.Sum(13, DEC38)), _s("mn13", AggregateKind.Min(13, DEC38)), _s("mx13", AggregateKind.Max(13, DEC38)),
            _s("s16", AggregateKind.Sum(16, DEC38)), _s("a16", AggregateKind.Avg(16, DEC38)),
            _s("mn16", AggregateKind.Min(16, DEC38)), _s("mx16", AggregateKind.Max(16, DEC38)),
            _s("p", AggregateKind.Sum(col(12) * col(12), DataType.Decimal128(38, 4)))]


def distinct_specs():
    return [_s("cd", AggregateKind.Count(45, distinct=True)), _s("sd", AggregateKind.Sum(45, I64, distinct=True)),
            _s("ad", AggregateKind.Avg(45, I64, distinct=True)), _s("td", AggregateKind.Total(45, I64, distinct=True))]


# (the arrow contract keeps the casts on the lean kernel in grouped plans too; the decimal product needs the exact one)
SPEC_SETS = {"int": (int_specs, ffi.EXPR_ARROW), "narrow": (narrow_specs, ffi.EXPR_ARROW), "float": (float_specs, ffi.EXPR_ARROW),
             "dec": (dec_specs, ffi.EXPR_EXACT)}
GROUPINGS = {  # (keys, hint)
    "ungrouped": ((), 0),
    "int64_four_slots": ((40,), 4),
    "nullable_int32_cta": ((41,), 64),
    "short_utf8_cta": ((42,), 64),
    "dict_utf8_four_slots": ((43,), 4),
    "pair_cta": ((40, 42), 64),
    "spill_growth": ((44,), 2),
}


@dataclass
class MatrixCase:
    name: str
    specs: list
    keys: Tuple[int, ...]
    hint: int
    expr_mode: Optional[int]
    distinct: bool = False


def matrix_cases() -> List[MatrixCase]:
    out = []
    for sname, (mk, mode) in SPEC_SETS.items():
        for gname, (keys, hint) in GROUPINGS.items():
            out.append(MatrixCase(f"{sname}-{gname}", mk(), keys, hint, mode))
    out.append(MatrixCase("distinct-ungrouped", distinct_specs(), (), 0, None, distinct=True))
    return out


CASE_IDS = [c.name for c in matrix_cases()]
_TABLE = []


def the_table() -> HostTable:
    if not _TABLE:
        _TABLE.append(matrix_table())
    return _TABLE[0]


def case_listing(t: HostTable, case: MatrixCase) -> str:
    """The plan listing of the scan that runs: for DISTINCT aggregates, the inner GROUP BY <column> of
    llkv_gpu_agg_create (COUNT(*) per distinct value, hint 1024 when none is given)."""
    if case.distinct:
        return gpu.debug_plan(t, F_A, [_s("n", AggregateKind.CountStar())], group_by=(45,), cardinality_hint=case.hint or 1024)
    return gpu.debug_plan(t, F_A, case.specs, group_by=case.keys, expr_mode=case.expr_mode, cardinality_hint=case.hint)


# ------------------------------------------------------------------------------------------------ CPU layer
@pytest.mark.parametrize("name", CASE_IDS)
def test_matrix_case_is_a_one_kernel_step(name):
    t = the_table()
    case = next(c for c in matrix_cases() if c.name == name)
    text = case_listing(t, case)
    assert text.startswith("lean plan"), (name, text)
    # (the listing sees column statistics, not dictionaries: a long-string key reads as a hashed wide key there, while the
    # runtime packs its dictionary ranks, and the GPU test checks that those steps publish)
    assert step_line(text) == (THREE_PARTS if 43 in case.keys else ONE_KERNEL), (name, text)
    assert "OP_COL      a=6" not in text, (name, "a checked product would rerun on the 128-bit interpreter")
    # the reference accepts every aggregate of the case over every step's rows
    for kind in set(SCRIPT):
        flt, lo, hi = step_args(kind)
        matrix_want(t, case, flt, lo, hi)


def test_matrix_covers_every_accumulator_class():
    """Word classes in the listings of the matrix: MIN, MAX, FSUM, Decimal MIN / MAX (MIN_I / MAX_I a=128: one u64 thread
    state over a 128-bit word pair, WC_MIN128 / WC_MAX128 and their low halves), a FIRSTROW word (grouped)."""
    t = the_table()
    kinds = set()
    for case in matrix_cases():
        kinds.update(re.findall(r"^ +\d+ ([A-Z_0-9]+) ", case_listing(t, case), re.M))
    for op in ("COUNT_STAR", "COUNT", "SUM", "MIN_I", "MAX_I", "FSUM", "MIN_F", "MAX_F", "GROUP", "FIRSTROW"):
        assert op in kinds, (op, sorted(kinds))
    dec = case_listing(t, next(c for c in matrix_cases() if c.name == "dec-ungrouped"))
    assert re.search(r" MIN_I +a=128 ", dec) and re.search(r" MAX_I +a=128 ", dec), dec


# ------------------------------------------------------------------------------------------------ GPU layer
SCRIPT = ["A"] * 4 + ["E_filter", "E_empty", "E_filter"] + ["B"] * 4 + ["A"] * 3


def step_args(kind: str):
    """(filter, row_begin, row_end) of a step of the script."""
    return {"A": (F_A, 0, N), "E_filter": (F_NONE, 0, N), "E_empty": (F_A, B_LO, B_LO), "B": (None, B_LO, B_HI)}[kind]


def matrix_want(t: HostTable, case: MatrixCase, flt, lo: int, hi: int):
    """The oracle's result; DISTINCT aggregates (which the oracle does not take) from numpy over the selected rows."""
    if not case.distinct:
        return oracle.aggregate(t, flt, case.specs, None, case.keys, case.expr_mode, lo, hi, group_capacity=1 << 12)
    c = t.columns[45]
    sel = np.zeros(t.n_rows, bool)
    if hi > lo:
        words, _ = oracle.filter_bitmap(t, flt, None, lo, hi)
        sel[lo + util.selected_positions(words, hi - lo)] = True
    sel &= np.unpackbits(c.validity, bitorder="little")[:t.n_rows].astype(bool)
    u = np.unique(c.values[sel])
    return [((), [AggregateValue(ffi.PT_INT64, u.size), AggregateValue(ffi.PT_INT64, int(u.sum()) if u.size else None),
                  AggregateValue(ffi.PT_FLOAT64, float(u.sum()) / u.size if u.size else None),
                  AggregateValue(ffi.PT_FLOAT64, float(u.sum()))])]


def slot_groups(rows) -> int:
    """Groups that occupy a slot of the global table (a single NULL key has a row of its own)."""
    return sum(1 for key, _ in rows if not (len(key) == 1 and key[0] is None))


@pytest.fixture(scope="module")
def matrix_device(gpu_ctx):
    t = the_table()
    dt = gpu.DeviceTable.from_host(gpu_ctx, t)
    yield t, dt
    dt.destroy()


# every case on the interpreting lean build; the specialised build (an NVRTC compile of several seconds per shape) for
# the ungrouped, four-slot and growing-table cases of each set and one case of each other key kind
SPECIALISED = [c for c in CASE_IDS if c.endswith(("-ungrouped", "-int64_four_slots", "-spill_growth"))] + [
    "int-pair_cta", "dec-nullable_int32_cta", "float-short_utf8_cta", "narrow-dict_utf8_four_slots"]
MATRIX_RUNS = [(c, 0) for c in CASE_IDS] + [(c, 2) for c in SPECIALISED]


@pytest.mark.gpu
@pytest.mark.parametrize("name, jit", MATRIX_RUNS, ids=[f"{c}-{'specialised' if j else 'interpreted'}" for c, j in MATRIX_RUNS])
def test_matrix_case_every_step(gpu_ctx, matrix_device, name, jit):
    t, dt = matrix_device
    case = next(c for c in matrix_cases() if c.name == name)
    n_words = listing_words(case_listing(t, case))
    n_keys = 1 if case.distinct else len(case.keys)
    cap = group_table_cap(case.hint or 1024) if n_keys else 1
    wants = {}
    for kind in set(SCRIPT):
        flt, lo, hi = step_args(kind)
        wants[kind] = matrix_want(t, case, flt, lo, hi)
    progs = {"A": gpu.Program(gpu_ctx, F_A), "E": gpu.Program(gpu_ctx, F_NONE)}
    gpu_ctx.set_jit(jit)
    dt.set_snapshot(None)
    agg = gpu.Aggregation(dt, case.specs, case.keys, case.expr_mode, case.hint)
    try:
        for i, kind in enumerate(SCRIPT):
            label = f"{name} jit={jit} step {i} ({kind})"
            flt, lo, hi = step_args(kind)
            before = agg.run_info()
            agg.execute(progs["E" if flt is F_NONE else "A"] if flt is not None else None, False, lo, hi)
            got = agg.finalize(1 << 12)
            info = agg.run_info()
            try:
                if case.distinct:  # (values only: the reference's result types are not restated here)
                    gv, wv = [v.value for v in got[0][1]], [v.value for v in wants[kind][0][1]]
                    assert len(got) == 1 and all(a == b or (isinstance(b, float) and a is not None and abs(a - b) <= 1e-12 * abs(b))
                                                 for a, b in zip(gv, wv)), (gv, wv)
                else:
                    util.assert_same_result(got, wants[kind])
            except AssertionError as e:
                raise AssertionError(f"{label}: {e}") from e
            assert info.used_fast_kernel == 1 or hi == lo, label
            # (the first step allocates and initialises the state after the reset that would have armed it, so it never
            # publishes)
            publishes = i > 0 and hi > lo and result_bytes(cap, n_words, n_keys) <= STAGE_BYTES
            if case.distinct:
                # the inner GROUP BY's table; the distinct values of the step decide its growth
                g = len(np.unique(t.columns[45].values[lo:hi])) if hi > lo else 0
            else:
                g = slot_groups(wants[kind]) if n_keys else 0
            while n_keys and g > cap:
                cap *= 4
            assert info.published_steps - before.published_steps == int(publishes), \
                (label, "published_steps", before.published_steps, info.published_steps)
            # a step repeated unchanged is captured as a CUDA graph once the plan and the table's statistics have
            # settled (the third unchanged run at the earliest) and replayed after that
            block_pos = next(k for k in range(i + 1) if i - k == 0 or SCRIPT[i - k - 1] != kind)
            if block_pos < 3:
                assert info.graph_replays == before.graph_replays, (label, "graph_replays", before.graph_replays, info.graph_replays)
            if kind == "B" and block_pos == 3:  # (by the B block the plan and the statistics have settled)
                assert info.graph_replays == before.graph_replays + 1, (label, "graph_replays", before.graph_replays, info.graph_replays)
    finally:
        agg.destroy()
        for p in progs.values():
            p.destroy()
        gpu_ctx.set_jit(1)


# ================================================================================================ 2b: the stage boundary
def boundary_table() -> HostTable:
    rng = np.random.default_rng(77)
    n = 40_000
    t = HostTable(62).add(HostColumn(1, DataType.Int64, rng.integers(0, 300, n) * 3 + 5))
    t.add(HostColumn(2, DataType.Int64, rng.integers(-(1 << 30), 1 << 30, n)))
    return t


def boundary_specs(n_max: int):
    """COUNT(*) and `n_max` MAX aggregates over distinct expressions: 2 + n_max words per group (COUNT(*), the group's first
    row, one word per MAX)."""
    return [_s("n", AggregateKind.CountStar())] + [_s(f"m{j}", AggregateKind.Max(col(2) + j, I64)) for j in range(n_max)]


# (name, hint, MAX aggregates, words, one kernel): at 2048 rows 2 words fit and 3 do not (49 184 / 65 632 B); at 512 rows
# 14 fit and 15 do not (61 664 / 65 776 B)
BOUNDARY = [("cap2048_fits", 1024, 0, 2, True), ("cap2048_over", 1024, 1, 3, False),
            ("cap512_fits", 256, 12, 14, True), ("cap512_over", 256, 13, 15, False)]


@pytest.mark.parametrize("name, hint, n_max, words, one", BOUNDARY, ids=[b[0] for b in BOUNDARY])
def test_stage_boundary_forms(name, hint, n_max, words, one):
    t = boundary_table()
    text = gpu.debug_plan(t, None, boundary_specs(n_max), group_by=(1,), cardinality_hint=hint)
    assert listing_words(text) == words, text
    size = result_bytes(group_table_cap(hint), words, 1)
    assert (size <= STAGE_BYTES) == one, (name, size)
    assert step_line(text) == (ONE_KERNEL if one else THREE_PARTS), (name, text)


def test_low_hint_starts_inside_the_stage():
    """Hint 2: a 32-row table, so the step's listing says one kernel although the table later grows past the stage."""
    t = boundary_table()
    text = gpu.debug_plan(t, None, boundary_specs(13), group_by=(1,), cardinality_hint=2)
    assert step_line(text) == ONE_KERNEL and result_bytes(32, 15, 1) <= STAGE_BYTES < result_bytes(512, 15, 1)


@pytest.mark.gpu
@pytest.mark.parametrize("jit", [0, 2], ids=["interpreted", "specialised"])
def test_stage_boundary_on_the_device(gpu_ctx, jit):
    t = boundary_table()
    dt = gpu.DeviceTable.from_host(gpu_ctx, t)
    gpu_ctx.set_jit(jit)
    try:
        for name, hint, n_max, words, one in BOUNDARY + [("grows_past_the_stage", 2, 13, 15, None)]:
            specs = boundary_specs(n_max)
            wants = {end: oracle.aggregate(t, None, specs, None, (1,), row_end=end, group_capacity=1024) for end in (20, 5000, t.n_rows)}
            agg = gpu.Aggregation(dt, specs, (1,), cardinality_hint=hint)
            try:
                for i in range(6):
                    label = f"{name} jit={jit} step {i}"
                    end = {0: 20, 4: 5000}.get(i, t.n_rows)  # (step 0, which creates the state, never publishes; its 20 rows fill no table)
                    before = agg.run_info().published_steps
                    agg.execute(None, False, 0, end)
                    try:
                        util.assert_same_result(agg.finalize(1024), wants[end])
                    except AssertionError as e:
                        raise AssertionError(f"{label}: {e}") from e
                    # growing past the stage: step 1 publishes from the 32-row table, fills it and runs again in a
                    # larger one without publishing; every later step is reset, scan and copy
                    expect = (i == 1) if one is None else (one and i > 0)
                    assert agg.run_info().published_steps - before == int(expect), label
            finally:
                agg.destroy()
    finally:
        gpu_ctx.set_jit(1)
        dt.destroy()


# ================================================================================================ reruns and graph replays
@pytest.mark.gpu
def test_rerunning_step_then_run_then_execute(gpu_ctx):
    """A step that asks for a 128-bit rerun every time is never captured (it ends on the general interpreter), so a replay
    can never follow a continuing run with that run's bookkeeping: re-running step x4, run, execute; no graph replays."""
    rng = np.random.default_rng(5)
    n = 30_000
    a = rng.integers(-10_000, 10_000, n)
    b = rng.integers(-10_000, 10_000, n)
    a[-1] = b[-1] = 4_000_000_000_000
    dec = DataType.Decimal128(15, 2)
    t = HostTable(63).add(HostColumn(1, dec, decimal_from_i64(a))).add(HostColumn(2, dec, decimal_from_i64(b))).add(
        HostColumn(3, DataType.Int64, rng.integers(0, 5, n)))
    specs = [_s("s", AggregateKind.Sum(col(1) * col(2), DataType.Decimal128(38, 4))), _s("n", AggregateKind.CountStar())]
    dt = gpu.DeviceTable.from_host(gpu_ctx, t)
    try:
        for keys in ((), (3,)):
            once = oracle.aggregate(t, None, specs, None, keys, ffi.EXPR_EXACT)
            doubled = oracle.aggregate(concat(t, t), None, specs, None, keys, ffi.EXPR_EXACT)
            agg = gpu.Aggregation(dt, specs, keys, ffi.EXPR_EXACT, 4 if keys else 0)
            try:
                for i in range(4):
                    agg.execute()
                    util.assert_same_result(agg.finalize(64), once, ordered=False)
                    assert agg.run_info().used_wide_path == 1, (keys, i)
                agg.execute()
                agg.run()
                util.assert_same_result(agg.finalize(64), doubled, ordered=False)
                agg.execute()
                util.assert_same_result(agg.finalize(64), once, ordered=False)
                info = agg.run_info()
                # every execute but the first publishes before its rerun; the continuing run does not
                assert info.graph_replays == 0 and info.published_steps == 5, (keys, info.graph_replays, info.published_steps)
            finally:
                agg.destroy()
    finally:
        dt.destroy()


@pytest.mark.gpu
@pytest.mark.parametrize("grouped", [False, True], ids=["ungrouped", "grouped"])
def test_aggregate_goes_on_after_deletes_and_appends(gpu_ctx, grouped):
    """A prepared aggregate over a table that changes under it.  Deleted rows make the columns nullable, so a COUNT that
    was the row count needs a word of its own: the next step (which starts afresh) takes the new accumulator layout, a
    run continuing a state of the old one is refused with a clear error until the aggregate is reset, and a run after a
    sparse append continues the step before it."""
    rng = np.random.default_rng(12)
    n = 20_000
    keys = rng.integers(0, 5, n)
    vals = rng.integers(-1000, 1000, n)
    live = np.ones(n + 400, bool)
    live[n:] = False
    all_keys = np.concatenate([keys, rng.integers(0, 7, 400)])
    all_vals = np.concatenate([vals, rng.integers(-1000, 1000, 400)])
    specs = [_s("n", AggregateKind.CountStar()), _s("c", AggregateKind.Count(2)), _s("s", AggregateKind.Sum(2, I64)),
             _s("mn", AggregateKind.Min(2, I64)), _s("mx", AggregateKind.Max(2, I64))]
    group_by = (1,) if grouped else ()

    def compact():
        ids = np.nonzero(live)[0]
        return HostTable(65).add(HostColumn(1, I64, all_keys[ids])).add(HostColumn(2, I64, all_vals[ids]))

    def want(*tables):
        return oracle.aggregate(concat(*tables), None, specs, None, group_by, group_capacity=64)

    dt = gpu.DeviceTable.from_host(gpu_ctx, compact())
    agg = gpu.Aggregation(dt, specs, group_by, cardinality_hint=8 if grouped else 0)
    fresh = gpu.Aggregation(dt, specs, group_by, cardinality_hint=8 if grouped else 0)
    try:
        for i in range(3):
            agg.execute()
            util.assert_same_result(agg.finalize(64), want(compact()), ordered=False)
        fresh.execute()
        before = compact()
        util.assert_same_result(fresh.finalize(64), want(before), ordered=False)
        gone = np.arange(3, n, 7)
        for c in dt.columns.values():
            c.delete_rows(gone.astype(np.uint64))
            c.seal()
        live[gone] = False
        for i in range(3):
            published = agg.run_info().published_steps
            agg.execute()
            util.assert_same_result(agg.finalize(64), want(compact()), ordered=False)
            assert agg.run_info().published_steps == published + 1, i
        with pytest.raises(LlkvError) as e:  # continuing a state started before the columns had NULLs
            fresh.run()
        assert e.value.code == ffi.ERR_INVALID_ARGUMENT, e.value
        fresh.reset()
        fresh.run()
        util.assert_same_result(fresh.finalize(64), want(compact()), ordered=False)
        # rows appended at every other row id past the end, then a run that continues the last step
        first = compact()
        ids = np.arange(n, n + 400, 2)
        dt.columns[1].append_rows(all_keys[ids], ids.astype(np.uint64))
        dt.columns[2].append_rows(all_vals[ids], ids.astype(np.uint64))
        for c in dt.columns.values():
            c.seal()
        dt.n_rows = max(c.rows() for c in dt.columns.values())
        live[ids] = True
        agg.run()
        util.assert_same_result(agg.finalize(64), want(first, compact()), ordered=False)
        agg.execute()
        util.assert_same_result(agg.finalize(64), want(compact()), ordered=False)
    finally:
        agg.destroy()
        fresh.destroy()
        dt.destroy()


def concat(*tables: HostTable) -> HostTable:
    out = HostTable(tables[0].table_id)
    for f, c in tables[0].columns.items():
        parts = [t.columns[f] for t in tables]
        validity = None
        if any(p.validity is not None for p in parts):
            bits = np.concatenate([np.unpackbits(p.validity, bitorder="little")[:p.n_rows] if p.validity is not None
                                   else np.ones(p.n_rows, np.uint8) for p in parts])
            validity = pack_validity(bits.astype(bool))
        if c.dtype.type == ffi.PT_UTF8:
            offs, data, base = [np.zeros(1, np.int32)], [], 0
            for p in parts:
                offs.append(p.values[1:] + base)
                data.append(p.aux)
                base += int(p.values[-1])
            out.add(HostColumn(f, c.dtype, np.concatenate(offs), validity, np.concatenate(data) if data else None))
        else:
            out.add(HostColumn(f, c.dtype, np.concatenate([p.values for p in parts]), validity))
    if all(t.created_by is not None for t in tables):
        out.add_mvcc(np.concatenate([t.created_by.values for t in tables]), np.concatenate([t.deleted_by.values for t in tables]))
    return out


# ================================================================================================ 2c: a random walk
WALK_DENSE = 20_000
WALK_TABLE = 64
W_KEY, W_V, W_F, W_D, W_X, W_P, W_Q = 1, 2, 3, 4, 5, 6, 7
W_DEC = DataType.Decimal128(18, 2)
W_CUT = 1_234     # a range boundary
W_WIDE = 17_000   # W_D * W_Q leaves i64 in this row only


def walk_specs():
    return {
        # ungrouped, arrow contract
        "plain": ([_s("n", AggregateKind.CountStar()), _s("mn", AggregateKind.Min(W_V, I64)), _s("mx", AggregateKind.Max(W_V, I64)),
                   _s("f", AggregateKind.Sum(W_F, F64)), _s("fmn", AggregateKind.Min(W_F, F64)), _s("fmx", AggregateKind.Max(W_F, F64)),
                   _s("d", AggregateKind.Sum(W_D, DEC38)), _s("dmn", AggregateKind.Min(W_D, DEC38)), _s("dmx", AggregateKind.Max(W_D, DEC38))], (), ffi.EXPR_ARROW, 0),
        # grouped on a nullable key, exact contract: the checked product W_D * W_Q needs 128 bits on one row
        "grouped": ([_s("n", AggregateKind.CountStar()), _s("s", AggregateKind.Sum(W_V, I64)), _s("c", AggregateKind.Count(W_V)),
                     _s("mn", AggregateKind.Min(W_V, I64)), _s("fmx", AggregateKind.Max(W_F, F64)),
                     _s("dq", AggregateKind.Sum(col(W_D) * col(W_Q), DataType.Decimal128(38, 4)))], (W_KEY,), ffi.EXPR_EXACT, 16),
        "distinct": ([_s("cd", AggregateKind.Count(W_X, distinct=True)), _s("sd", AggregateKind.Sum(W_X, I64, distinct=True))], (), None, 0),
    }


class WalkModel:
    """The walk's table by row id: values and validity per field, MVCC ids, and which row ids exist."""

    FIELDS = {W_KEY: DataType.Int64, W_V: DataType.Int64, W_F: DataType.Float64, W_D: W_DEC, W_X: DataType.Int64,
              W_P: DataType.Int64, W_Q: W_DEC}
    CAP = 1 << 16

    def __init__(self, rng):
        self.rng = rng
        self.vals = {f: np.zeros(self.CAP, np.float64 if f == W_F else np.int64) for f in self.FIELDS}
        self.valid = {f: np.zeros(self.CAP, bool) for f in self.FIELDS}
        self.mvcc = {"c": np.zeros(self.CAP, np.uint64), "d": np.zeros(self.CAP, np.uint64)}
        self.live = np.zeros(self.CAP, bool)
        self.write(np.arange(WALK_DENSE))
        self.write(np.arange(WALK_DENSE, WALK_DENSE + 600, 2))  # the row-id-sparse part: every other id
        self.next_id = WALK_DENSE + 600

    def write(self, ids):
        """New values for the rows `ids` (appended or rewritten)."""
        r, n = self.rng, len(ids)
        self.vals[W_KEY][ids] = r.integers(0, 9, n)
        self.vals[W_V][ids] = r.integers(-1000, 1000, n)
        self.vals[W_F][ids] = r.integers(-800, 800, n) / 8
        self.vals[W_D][ids] = r.integers(-10**6, 10**6, n)
        self.vals[W_X][ids] = r.integers(0, 400, n)
        self.vals[W_P][ids] = r.integers(-1000, 1000, n)
        self.vals[W_Q][ids] = r.integers(-1000, 1000, n)
        for f in self.FIELDS:
            self.valid[f][ids] = True
        self.valid[W_KEY][ids] = r.random(n) > 0.1
        self.valid[W_V][ids] = r.random(n) > 0.05
        self.mvcc["c"][ids] = r.integers(1, 4, n)
        self.mvcc["d"][ids] = np.where(r.random(n) > 0.1, 0, r.integers(2, 6, n))
        self.live[ids] = True
        for i in ids:
            if i == W_WIDE:
                self.vals[W_D][i] = self.vals[W_Q][i] = 4_000_000_000_000

    def table(self, lo, hi) -> HostTable:
        """The rows with row ids in [lo, hi), in row-id order (the oracle's view of a step over that range)."""
        ids = lo + np.nonzero(self.live[lo:hi])[0]
        t = HostTable(WALK_TABLE)
        for f, dtype in self.FIELDS.items():
            raw = self.vals[f][ids]
            valid = self.valid[f][ids]
            arr = decimal_from_i64(raw) if dtype.type == ffi.PT_DECIMAL128 else raw
            t.add(HostColumn(f, dtype, arr, None if valid.all() else pack_validity(valid)))
        t.add_mvcc(self.mvcc["c"][ids], self.mvcc["d"][ids])
        return t


def device_walk_table(ctx, model: WalkModel) -> gpu.DeviceTable:
    """The dense part as sealed chunks, then the row-id-sparse part through append_rows."""
    dt = gpu.DeviceTable.from_host(ctx, model.table(0, WALK_DENSE))
    push_rows(dt, model, np.nonzero(model.live[WALK_DENSE:])[0] + WALK_DENSE)
    return dt


def device_columns(dt):
    return [(f, dt.columns[f]) for f in WalkModel.FIELDS] + [("c", dt.created_by), ("d", dt.deleted_by)]


def push_rows(dt, model: WalkModel, ids):
    """append_rows of the rows `ids` (new or rewritten: last writer wins) to every column.  A NULL is an absent cell: a
    rewritten row whose new value is NULL loses its old one."""
    ids = np.sort(np.asarray(ids, np.int64))
    for f, dc in device_columns(dt):
        if f in WalkModel.FIELDS:
            has = model.valid[f][ids]
            vals = model.vals[f][ids[has]]
            arr = decimal_from_i64(vals).reshape(-1) if WalkModel.FIELDS[f].type == ffi.PT_DECIMAL128 else vals
        else:
            has = np.ones(ids.size, bool)
            arr = model.mvcc[f][ids]
        if has.any():
            dc.append_rows(arr, ids[has].astype(np.uint64), first_row_id=0)
        if not has.all():
            dc.delete_rows(ids[~has].astype(np.uint64))
    for _, dc in device_columns(dt):
        dc.seal()
    dt.n_rows = max(dc.rows() for _, dc in device_columns(dt))


WALK_SNAPSHOTS = [None, Snapshot(4, 4, ()), Snapshot(3, 3, (2,))]
WALK_FILTERS = [None, pred(W_V, Operator.Range(Bound.Included(-500), Bound.Excluded(600))),
                Expr.Or([pred(W_KEY, Operator.Equals(3)), pred(W_F, Operator.LessThan(-20.0))])]


@dataclass
class AggState:
    agg: gpu.Aggregation
    specs: list
    keys: tuple
    mode: Optional[int]
    runs: list = field(default_factory=list)  # per run since the last reset: the rows it selected, or the error it raises
    pending_reset: bool = False                      # reset called: finalize must be empty until the next run
    failed: bool = False                             # the last step raised: a run cannot continue from it
    output: Optional[tuple] = None                   # (limit, count threshold) of set_output on the grouped aggregation


def apply_output(rows, output):
    if output is None:
        return rows
    limit, above = output
    keep = [r for r in rows if r[1][0].value > above]
    keep.sort(key=lambda r: (-r[1][0].value, r[0][0] is not None, r[0][0] if r[0][0] is not None else 0))
    return keep[:limit]


def run_part(model: WalkModel, st: AggState, run):
    """What one run contributes, taken from the table as it is when the run is queued: the rows it selects, or the
    reference's error."""
    lo, hi, fi, si = run
    part = model.table(lo, hi)
    try:
        oracle.aggregate(part, WALK_FILTERS[fi], [_s("n", AggregateKind.CountStar())] if st.specs[0].kind.distinct else st.specs,
                         WALK_SNAPSHOTS[si], st.keys, st.mode, group_capacity=1 << 12)
    except LlkvError as e:
        return e
    return filtered(part, WALK_FILTERS[fi], WALK_SNAPSHOTS[si])


def expected(model: WalkModel, st: AggState):
    """The oracle over the runs since the last reset: each run's rows in row-id order, concatenated in run order."""
    errors = [p for p in st.runs if isinstance(p, LlkvError)]
    if errors:
        return errors[0]
    tables = list(st.runs)
    if st.specs[0].kind.distinct:  # (the oracle takes no DISTINCT aggregates: COUNT / SUM of the distinct values)
        x = [c.values[np.unpackbits(c.validity, bitorder="little")[:c.n_rows].astype(bool)] if c.validity is not None else c.values
             for c in (tb.columns[W_X] for tb in tables)]
        u = np.unique(np.concatenate(x)) if x else np.zeros(0, np.int64)
        return [((), [AggregateValue(ffi.PT_INT64, int(u.size)), AggregateValue(ffi.PT_INT64, int(u.sum()) if u.size else None)])]
    if not tables:
        return oracle.aggregate(model.table(0, 0), None, st.specs, None, st.keys, st.mode, group_capacity=1 << 12)
    return oracle.aggregate(concat(*tables), None, st.specs, None, st.keys, st.mode, group_capacity=1 << 12)


def filtered(t: HostTable, flt, snap) -> HostTable:
    """The rows of `t` a run selects (the oracle's selection bitmap), as a table of their own."""
    words, _ = oracle.filter_bitmap(t, flt, snap)
    pos = util.selected_positions(words, t.n_rows)
    out = HostTable(t.table_id)
    for f, c in t.columns.items():
        validity = None
        if c.validity is not None:
            bits = np.unpackbits(c.validity, bitorder="little")[:t.n_rows][pos]
            validity = pack_validity(bits.astype(bool))
        out.add(HostColumn(f, c.dtype, c.values[pos], validity))
    out.add_mvcc(t.created_by.values[pos], t.deleted_by.values[pos])
    return out


def run_walk(ctx, seed: int, n_ops: int = 60):
    rng = np.random.default_rng(9000 + seed)
    model = WalkModel(rng)
    dt = device_walk_table(ctx, model)
    progs = [None] + [gpu.Program(ctx, f) for f in WALK_FILTERS[1:]]
    states = {name: AggState(gpu.Aggregation(dt, specs, keys, mode, hint), specs, keys, mode)
              for name, (specs, keys, mode, hint) in walk_specs().items()}
    log = []
    ranges = [(0, None), (0, W_CUT), (W_CUT + 1, None), (5_000, W_WIDE), (W_WIDE, None)]

    def pick_run():
        lo, hi = ranges[int(rng.integers(0, len(ranges)))]
        return lo, dt.n_rows if hi is None else hi, int(rng.integers(0, len(WALK_FILTERS))), int(rng.integers(0, len(WALK_SNAPSHOTS)))

    def launch(st, how, run):
        lo, hi, fi, si = run
        dt.set_snapshot(WALK_SNAPSHOTS[si])
        if how == "execute":
            st.agg.execute(progs[fi], WALK_SNAPSHOTS[si] is not None, lo, hi)
            st.runs, st.failed = [run_part(model, st, run)], False
        else:
            st.agg.run(progs[fi], WALK_SNAPSHOTS[si] is not None, lo, hi)
            st.runs = ([] if st.pending_reset else st.runs) + [run_part(model, st, run)]
        st.pending_reset = False

    def check(name, st):
        want = expected(model, st)
        if isinstance(want, LlkvError):
            with pytest.raises(LlkvError) as got:
                st.agg.finalize(1 << 12)
            assert got.value.code == want.code, (got.value, want)
            st.runs, st.failed = [], True  # (a failed step leaves nothing to continue from)
            st.pending_reset = True
            return
        got = st.agg.finalize(1 << 12)
        if st.specs[0].kind.distinct:
            assert [v.value for v in got[0][1]] == [v.value for v in want[0][1]], (got, want)
        else:
            # (first-appearance order of groups follows the kernel's row order across runs: compared as a set, unless
            # ORDER BY fixes it)
            util.assert_same_result(got, apply_output(want, st.output), ordered=st.output is not None)

    try:
        for op_i in range(n_ops):
            name = ["plain", "grouped", "distinct"][int(rng.integers(0, 3))]
            st = states[name]
            op = ["execute", "execute", "execute", "repeat", "twice", "run", "reset", "finalize2", "output", "mutate", "knob",
                  "bitmap"][int(rng.integers(0, 12))]
            log.append(f"{op_i}: {op} {name}")
            try:
                if op in ("execute", "repeat"):
                    run = pick_run()
                    log[-1] += f" {run}"
                    for _ in range(1 if op == "execute" else 4):  # repeated unchanged: captured and replayed
                        launch(st, "execute", run)
                        check(name, st)
                elif op == "twice":
                    first, run = pick_run(), pick_run()
                    log[-1] += f" {first} {run}"
                    launch(st, "execute", first)
                    launch(st, "execute", run)
                    check(name, st)
                elif op == "run" and not st.failed and not isinstance(expected(model, st), LlkvError):  # (a failed step must be reset first)
                    run = pick_run()
                    log[-1] += f" {run}"
                    launch(st, "run", run)
                    check(name, st)
                elif op == "reset":
                    st.agg.reset()
                    st.runs, st.pending_reset, st.failed = [], True, False
                    check(name, st)
                elif op == "finalize2":
                    check(name, st)
                    check(name, st)
                    if st.keys and not isinstance(expected(model, st), LlkvError):
                        assert st.agg.group_count() == len(expected(model, st))
                elif op == "output" and name == "grouped":
                    st.output = None if st.output is not None else (int(rng.integers(1, 6)), int(rng.integers(0, 300)))
                    log[-1] += f" {st.output}"
                    if st.output is None:
                        st.agg.set_output()
                    else:
                        st.agg.set_output(having=[("agg", 0, ffi.CMP_GT, st.output[1])],
                                          order_by=[("agg", 0, True, False), ("key", 0, False, True)], limit=st.output[0])
                    check(name, st)
                elif op == "mutate":
                    for nm, s_ in states.items():  # (settles what is queued: its results describe the rows before the change)
                        check(nm, s_)
                    kind = int(rng.integers(0, 3))
                    live = np.nonzero(model.live)[0]
                    if kind == 0:  # append rows at the end (the row-id-sparse part: every other id)
                        ids = np.arange(model.next_id, model.next_id + 2 * int(rng.integers(10, 300)), 2)
                        model.next_id = int(ids[-1]) + 1
                        model.write(ids)
                    elif kind == 1:  # rewrite live rows in place
                        ids = rng.choice(live, size=int(rng.integers(1, 40)), replace=False)
                        model.write(ids)
                    else:
                        gone = rng.choice(live, size=int(rng.integers(1, 40)), replace=False)
                        gone = gone[gone != W_WIDE].astype(np.uint64)
                        for _, dc in device_columns(dt):
                            dc.delete_rows(gone)
                            dc.seal()
                        model.live[gone.astype(np.int64)] = False
                        ids = []
                    log[-1] += f" kind {kind} rows {len(ids)}"
                    if len(ids):
                        push_rows(dt, model, ids)
                    # the aggregations go on over the changed table: the next execute starts afresh (its captured graph no
                    # longer applies), a run continues what the earlier runs left
                elif op == "knob":
                    k = int(rng.integers(0, 3))
                    v = int(rng.integers(0, 3)) if k < 2 else int(rng.integers(0, 2))
                    (ctx.set_jit, ctx.set_pruning, ctx.set_graphs)[k](v)
                    log[-1] += f" {('jit', 'pruning', 'graphs')[k]}={v}"
                elif op == "bitmap":
                    # a selection bitmap and a column scan on the same context between execute and finalize
                    run = pick_run()
                    launch(st, "execute", run)
                    lo, hi, fi, si = run
                    _, count = dt.filter_bitmap(WALK_FILTERS[fi], WALK_SNAPSHOTS[si], lo, hi)
                    _, want_count = oracle.filter_bitmap(model.table(lo, hi), WALK_FILTERS[fi], WALK_SNAPSHOTS[si])
                    assert count == want_count
                    acc = [0]
                    dt.columns[W_V].scan(lambda vals, ids: acc.__setitem__(0, acc[0] + (0 if vals is None else int(vals.sum()))))
                    assert acc[0] == int(model.vals[W_V][model.live & model.valid[W_V]].sum())
                    check(name, st)
            except (AssertionError, LlkvError, pytest.fail.Exception) as e:
                raise AssertionError(f"seed {seed}: {e!r}\noperations:\n  " + "\n  ".join(log)) from e
        return sum(s.agg.run_info().graph_replays for s in states.values()), sum(s.agg.run_info().published_steps for s in states.values())
    finally:
        for s in states.values():
            s.agg.destroy()
        for p in progs:
            if p is not None:
                p.destroy()
        dt.destroy()
        ctx.set_jit(1)
        ctx.set_pruning(1)
        ctx.set_graphs(1)


@pytest.mark.gpu
@pytest.mark.parametrize("seed", range(8))
def test_random_step_walk(gpu_ctx, seed):
    replays, published = run_walk(gpu_ctx, seed)
    assert published > 0, seed
