"""GPU: steps whose scan publishes the result itself (the lean kernel copies the status word and the table to page-locked
memory and re-arms the state, so a replayed step is one kernel).  Every step of every case is checked against the oracle:
repeated steps on the benchmark shapes, aggregations interleaved on one table, a run that continues a published result,
unfinished steps, zone-map tile lists, reruns (a checked product that needs 128 bits, a group table that fills up) and a
device error followed by a clean step."""
import numpy as np
import pytest

import util
from llkv_b200 import ffi, gpu, tpch
from llkv_b200.expr import AggregateKind, AggregateSpec, DataType, ScalarExpr
from llkv_b200.table import HostColumn, HostTable, LlkvError, decimal_from_i64
from oracle import oracle

pytestmark = pytest.mark.gpu
STEPS = 10


def rows_of(t: HostTable, lo: int, hi: int, tid=None) -> HostTable:
    out = HostTable(t.table_id if tid is None else tid)
    for c in t.columns.values():
        out.add(HostColumn(c.field_id, c.dtype, c.values[lo:hi]))
    return out


def twice(t: HostTable) -> HostTable:
    out = HostTable(t.table_id)
    for c in t.columns.values():
        out.add(HostColumn(c.field_id, c.dtype, np.concatenate([c.values, c.values])))
    return out


def keyed_table(n, groups, seed, tid):
    rng = np.random.default_rng(seed)
    return HostTable(tid).add(HostColumn(1, DataType.Int64, rng.integers(0, groups, n, dtype=np.int64))).add(
        HostColumn(2, DataType.Int64, rng.integers(-1000, 1000, n, dtype=np.int64)))


KEYED_SPECS = [AggregateSpec("n", AggregateKind.CountStar()), AggregateSpec("s", AggregateKind.Sum(2, DataType.Int64)),
               AggregateSpec("mx", AggregateKind.Max(2, DataType.Int64))]


def steps(agg, prog, want, n_steps=STEPS, mvcc=False, cap=64, **kw):
    for i in range(n_steps):
        agg.execute(prog, mvcc, **kw)
        util.assert_same_result(agg.finalize(cap), want)


@pytest.fixture(scope="module")
def lineitem(gpu_ctx):
    t, snap = tpch.lineitem_table(300_000, seed=6, with_q1=True, with_mvcc=True)
    dt = gpu.DeviceTable.from_host(gpu_ctx, t)
    yield t, snap, dt
    dt.destroy()


def test_benchmark_shapes_every_step(gpu_ctx, lineitem):
    t, snap, dt = lineitem
    for flt, specs, keys, sn, hint in ((tpch.q6_filter(), tpch.q6_aggregates(), (), None, 0),
                                       (tpch.q1_filter(), tpch.q1_aggregates(), tpch.Q1_GROUP_BY, snap, 4)):
        want = oracle.aggregate(t, flt, specs, sn, keys, group_capacity=64)
        prog = gpu.Program(gpu_ctx, flt)
        dt.set_snapshot(sn)
        agg = gpu.Aggregation(dt, specs, keys, cardinality_hint=hint)
        try:
            steps(agg, prog, want, mvcc=sn is not None)
            assert agg.run_info().graph_replays >= 3
        finally:
            agg.destroy()
            prog.destroy()
    dt.set_snapshot(None)
    # configs[0]
    c0, _ = tpch.int64_table(200_000, seed=1, table_id=3)
    x = c0.columns[tpch.X_FIELD].values
    lo, hi = (int(v) for v in np.percentile(x, [25, 75]).astype(np.int64))
    flt = tpch.between_filter(tpch.X_FIELD, lo, hi)
    d0 = gpu.DeviceTable.from_host(gpu_ctx, c0)
    prog = gpu.Program(gpu_ctx, flt)
    agg = gpu.Aggregation(d0, tpch.sum_int64(tpch.X_FIELD))
    try:
        steps(agg, prog, oracle.aggregate(c0, flt, tpch.sum_int64(tpch.X_FIELD)))
        assert agg.run_info().graph_replays >= 3
    finally:
        agg.destroy()
        prog.destroy()
        d0.destroy()


def test_two_aggregations_interleaved_on_one_table(gpu_ctx, lineitem):
    t, _, dt = lineitem
    dt.set_snapshot(None)
    p6, p1 = gpu.Program(gpu_ctx, tpch.q6_filter()), gpu.Program(gpu_ctx, tpch.q1_filter())
    a6 = gpu.Aggregation(dt, tpch.q6_aggregates())
    a1 = gpu.Aggregation(dt, tpch.q1_aggregates(), tpch.Q1_GROUP_BY, cardinality_hint=4)
    w6 = oracle.aggregate(t, tpch.q6_filter(), tpch.q6_aggregates())
    w1 = oracle.aggregate(t, tpch.q1_filter(), tpch.q1_aggregates(), None, tpch.Q1_GROUP_BY, group_capacity=64)
    try:
        for i in range(STEPS):
            a6.execute(p6)
            a1.execute(p1)
            util.assert_same_result(a1.finalize(64), w1)
            util.assert_same_result(a6.finalize(1), w6)
        assert a6.run_info().graph_replays >= 3 and a1.run_info().graph_replays >= 3
    finally:
        for o in (a6, a1, p6, p1):
            o.destroy()


@pytest.mark.parametrize("grouped", [False, True], ids=["ungrouped", "grouped"])
def test_run_after_execute_accumulates(gpu_ctx, grouped):
    t = keyed_table(150_000, 40, seed=3, tid=41)
    dt = gpu.DeviceTable.from_host(gpu_ctx, t)
    keys = (1,) if grouped else ()
    once = oracle.aggregate(t, None, KEYED_SPECS, None, keys, group_capacity=64)
    doubled = oracle.aggregate(twice(t), None, KEYED_SPECS, None, keys, group_capacity=64)
    agg = gpu.Aggregation(dt, KEYED_SPECS, keys, cardinality_hint=64 if grouped else 0)
    try:
        for i in range(STEPS):
            agg.execute()
            if i % 3 == 2:
                agg.run()  # continues from the step's result: the published table goes back onto the device first
                util.assert_same_result(agg.finalize(64), doubled)
            else:
                util.assert_same_result(agg.finalize(64), once)
    finally:
        agg.destroy()
        dt.destroy()


def test_execute_twice_without_finalize(gpu_ctx, lineitem):
    t, _, dt = lineitem
    dt.set_snapshot(None)
    prog = gpu.Program(gpu_ctx, tpch.q6_filter())
    agg = gpu.Aggregation(dt, tpch.q6_aggregates())
    want = oracle.aggregate(t, tpch.q6_filter(), tpch.q6_aggregates())
    try:
        for i in range(STEPS):
            agg.execute(prog)
            if i % 2:
                agg.execute(prog)
            util.assert_same_result(agg.finalize(1), want)
    finally:
        agg.destroy()
        prog.destroy()


def test_tile_list_runs(gpu_ctx):
    """A range on a clustered key: the scan walks the zone-map tile list of the surviving tiles."""
    n = 400_000
    keys = np.arange(n, dtype=np.int64)
    t = HostTable(42).add(HostColumn(tpch.K_FIELD, DataType.Int64, keys)).add(
        HostColumn(tpch.V_FIELD, DataType.Int64, np.random.default_rng(5).integers(0, 1001, n, dtype=np.int64)))
    dt = gpu.DeviceTable.from_host(gpu_ctx, t)
    flt = tpch.between_filter(tpch.K_FIELD, 50_000, 90_000)
    specs = [AggregateSpec("s", AggregateKind.Sum(tpch.V_FIELD, DataType.Int64)), AggregateSpec("n", AggregateKind.CountStar())]
    prog = gpu.Program(gpu_ctx, flt)
    agg = gpu.Aggregation(dt, specs)
    gpu_ctx.set_pruning(2)
    try:
        steps(agg, prog, oracle.aggregate(t, flt, specs))
        assert agg.run_info().tiles_pruned > 0
    finally:
        gpu_ctx.set_pruning(1)
        agg.destroy()
        prog.destroy()
        dt.destroy()


def test_checked_product_reruns_on_one_step_and_not_the_next(gpu_ctx):
    """SUM(a * b) over Decimal128 columns whose product may leave 64 bits: the last row's product does.  A step over all
    rows reruns with 128-bit arithmetic; a step that stops before that row does not."""
    n = 120_000
    rng = np.random.default_rng(7)
    a = rng.integers(-10_000, 10_000, n, dtype=np.int64)
    b = rng.integers(-10_000, 10_000, n, dtype=np.int64)
    a[-1] = b[-1] = 4_000_000_000_000
    dec = DataType.Decimal128(15, 2)
    t = HostTable(43).add(HostColumn(1, dec, decimal_from_i64(a))).add(HostColumn(2, dec, decimal_from_i64(b)))
    dt = gpu.DeviceTable.from_host(gpu_ctx, t)
    specs = [AggregateSpec("s", AggregateKind.Sum(ScalarExpr.Column(1) * ScalarExpr.Column(2), DataType.Decimal128(38, 4))),
             AggregateSpec("n", AggregateKind.CountStar())]
    mode = ffi.EXPR_EXACT  # the lean program multiplies in 64 bits, checked (the listing's OP_COL a=6)
    assert gpu.debug_plan(t, None, specs, expr_mode=mode).startswith("lean plan")
    w_all = oracle.aggregate(t, None, specs, expr_mode=mode)
    w_head = oracle.aggregate(rows_of(t, 0, n - 1), None, specs, expr_mode=mode)
    agg = gpu.Aggregation(dt, specs, expr_mode=mode)
    try:
        for i in range(STEPS):
            end = n if i % 2 else n - 1
            agg.execute(row_end=end)
            util.assert_same_result(agg.finalize(1), w_all if end == n else w_head)
    finally:
        agg.destroy()
        dt.destroy()


def test_low_hint_fills_the_group_table(gpu_ctx):
    """A cardinality hint far below the groups: the first step fills the table, grows it and runs again."""
    t = keyed_table(100_000, 300, seed=9, tid=44)
    dt = gpu.DeviceTable.from_host(gpu_ctx, t)
    agg = gpu.Aggregation(dt, KEYED_SPECS, (1,), cardinality_hint=2)
    try:
        steps(agg, None, oracle.aggregate(t, None, KEYED_SPECS, None, (1,), group_capacity=512), cap=512)
    finally:
        agg.destroy()
        dt.destroy()


def test_device_error_then_a_clean_step(gpu_ctx):
    """An arrow-arith overflow raised on the device, then a step over rows that do not overflow, alternately."""
    t = HostTable(45).add(HostColumn(1, DataType.Int64, np.array([5, 2**62, 2**62, 7], dtype=np.int64)))
    dt = gpu.DeviceTable.from_host(gpu_ctx, t)
    specs = [AggregateSpec("s", AggregateKind.Sum(ScalarExpr.Column(1) * ScalarExpr.Column(1), DataType.Int64))]
    with pytest.raises(LlkvError) as want_err:
        oracle.aggregate(t, None, specs)
    clean = oracle.aggregate(rows_of(t, 0, 1), None, specs)
    agg = gpu.Aggregation(dt, specs)
    try:
        for i in range(STEPS):
            if i % 2 == 0:
                agg.execute(row_end=4)
                with pytest.raises(LlkvError) as got:
                    agg.finalize(1)
                assert got.value.code == want_err.value.code
            else:
                agg.execute(row_end=1)
                util.assert_same_result(agg.finalize(1), clean)
    finally:
        agg.destroy()
        dt.destroy()
