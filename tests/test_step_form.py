"""CPU: the step form the plan listing reports (llkv_gpu_debug_plan asks the runtime's policy, step_publishes).  A repeated
step is one kernel — the scan publishes its result to page-locked memory and re-arms the state — only for a lean plan in
its per-row form whose result fits the page-locked stage, without hashed wide keys, on one rank, and for a run that
starts from the initial state.  Every other run is reset, scan and result copy, as before."""
import numpy as np

from llkv_b200 import gpu, tpch
from llkv_b200.expr import AggregateKind, AggregateSpec, DataType
from llkv_b200.table import HostColumn, HostTable

ONE_KERNEL = "step: one kernel, the scan publishes the result to page-locked memory and re-arms the state"
THREE_PARTS = "step: reset, scan, result copy"


def step_line(text):
    lines = [ln for ln in text.splitlines() if ln.startswith("step: ")]
    assert len(lines) == 1, text
    return lines[0]


def test_benchmark_plans_publish_from_the_scan():
    t, snap = tpch.lineitem_table(20_000, seed=6, with_q1=True, with_mvcc=True)
    assert step_line(gpu.debug_plan(t, tpch.q6_filter(), tpch.q6_aggregates())) == ONE_KERNEL
    q1 = gpu.debug_plan(t, tpch.q1_filter(), tpch.q1_aggregates(), snap, group_by=tpch.Q1_GROUP_BY, cardinality_hint=4)
    assert step_line(q1) == ONE_KERNEL
    # a run that continues the previous one without a reset keeps the reset-free sequence of today: no publishing
    assert step_line(gpu.debug_plan(t, tpch.q6_filter(), tpch.q6_aggregates(), continues=True)) == THREE_PARTS
    q1c = gpu.debug_plan(t, tpch.q1_filter(), tpch.q1_aggregates(), snap, group_by=tpch.Q1_GROUP_BY, cardinality_hint=4, continues=True)
    assert step_line(q1c) == THREE_PARTS


def test_partitioned_and_large_tables_keep_the_result_copy():
    t = tpch.highcard_table(50_000, 20_000, seed=4)
    for kw in (dict(partition=True), dict(packed=True)):
        text = gpu.debug_plan(t, None, tpch.highcard_aggregates(), group_by=(tpch.K_FIELD,), cardinality_hint=20_000, **kw)
        assert "partitioned" in text and step_line(text) == THREE_PARTS, (kw, text)
    # the same plan per row: its table is far beyond the 64 KB stage
    text = gpu.debug_plan(t, None, tpch.highcard_aggregates(), group_by=(tpch.K_FIELD,), cardinality_hint=20_000)
    assert "partitioned" not in text and step_line(text) == THREE_PARTS
    # a small grouped table per row fits
    text = gpu.debug_plan(t, None, tpch.highcard_aggregates(), group_by=(tpch.K_FIELD,), cardinality_hint=64)
    assert step_line(text) == ONE_KERNEL


def test_hashed_wide_keys_keep_the_table_on_the_device():
    """Keys wider than 64 bits group by a hash; finalize proves on the device that no two keys share one, so the table
    stays there."""
    rng = np.random.default_rng(1)
    n = 2000
    t = HostTable(71).add(HostColumn(1, DataType.Int64, rng.integers(-(1 << 62), 1 << 62, n, dtype=np.int64))).add(
        HostColumn(2, DataType.UInt64, rng.integers(0, (1 << 64) - 1, n, dtype=np.uint64))).add(
        HostColumn(5, DataType.Int64, rng.integers(-1000, 1000, n, dtype=np.int64)))
    specs = [AggregateSpec("c", AggregateKind.CountStar()), AggregateSpec("s", AggregateKind.Sum(5, DataType.Int64))]
    text = gpu.debug_plan(t, None, specs, group_by=(1, 2), cardinality_hint=16)
    assert text.startswith("lean plan") and "2 keys" in text and step_line(text) == THREE_PARTS
    # one of the two keys alone packs into 64 bits
    assert step_line(gpu.debug_plan(t, None, specs, group_by=(2,), cardinality_hint=16)) == ONE_KERNEL

