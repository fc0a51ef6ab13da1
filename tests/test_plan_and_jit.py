"""CPU: the plan compiler's lean lowering and the run-time specialisation of the lean kernel, through the diagnostics
entry of the C ABI (llkv_gpu_debug_plan).  NVRTC compiles for sm_100a without a GPU, so the specialised build of the
benchmark plans is checked here: it must compile, keep its registers in bounds and contain the Blackwell path
(cp.async.bulk = UBLKCP, mbarrier = SYNCS) and no shared-memory CAS loop in the ungrouped kernel."""
import os
import shutil
import subprocess

import pytest

from llkv_b200 import gpu, tpch
import numpy as np

from llkv_b200.expr import AggregateKind, AggregateSpec, DataType, Expr, Literal, Operator, pred
from llkv_b200.table import HostColumn, HostTable


@pytest.fixture(scope="module")
def lineitem():
    return tpch.lineitem_table(20_000, seed=6, with_q1=True, with_mvcc=True)


def test_q6_lowers_to_the_lean_program(lineitem):
    t, _ = lineitem
    text = gpu.debug_plan(t, tpch.q6_filter(), tpch.q6_aggregates())
    assert text.startswith("lean plan:")
    ops = [ln.split()[1] for ln in text.splitlines() if ln.startswith("  ") and ln.split()[0].isdigit()]
    # three typed range leaves, early exit, revenue = round(price * discount / 100) summed exactly
    assert ops[:4] == ["LEAF", "LEAF", "LEAF", "SELECT_DONE"] and ops[-1] == "END"
    assert "OP_COL" in ops and "DIVR" in ops and "SUM" in ops
    # the date range and the decimal bounds were folded against the columns' own min/max statistics
    assert "range [8766, 9130]" in text and "range [5, 7]" in text


def test_q1_lowers_to_the_lean_program_with_narrow_accumulators(lineitem):
    t, snap = lineitem
    text = gpu.debug_plan(t, tpch.q1_filter(), tpch.q1_aggregates(), snap, group_by=tpch.Q1_GROUP_BY, cardinality_hint=6)
    assert text.startswith("lean plan:")
    ops = [ln.split()[1] for ln in text.splitlines() if ln.startswith("  ") and ln.split()[0].isdigit()]
    assert ops[:4] == ["LEAF", "MVCC", "SELECT_DONE", "GROUP"]
    assert ops.count("SUM") == 5  # qty, price, disc_price, charge, disc: the AVGs share the SUM words, COUNT(*) the count
    words = [ln for ln in text.splitlines() if ln.startswith("  word")]
    assert sum("width 4" in w for w in words) == 4 and sum("width 8" in w for w in words) == 3
    assert "fg=8" in text  # six expected groups -> eight CTA-local slots


def test_or_and_not_trees_lower_to_the_mask_stack_of_the_lean_kernel(lineitem):
    """OR / NOT trees run on the lean kernel since round 2: leaves push (rows, not-in-domain) masks, MASK_* combine them."""
    t, _ = lineitem
    text = gpu.debug_plan(t, Expr.Or([tpch.q1_filter(), Expr.Not(tpch.q6_filter())]), tpch.q6_aggregates())
    assert text.startswith("lean plan")
    ops = [ln.split()[1] for ln in text.splitlines() if ln.strip()[:1].isdigit()]
    assert ops.count("LEAF") == 4 and "MASK_AND" in ops and "MASK_OR" in ops and "MASK_NOT" in ops and ops.count("MASK_FILTER") == 1
    # IN lists too (decimal entries compare as the 64-bit images the narrowed column holds)
    from llkv_b200.expr import Operator, pred
    text = gpu.debug_plan(t, Expr.Or([tpch.q1_filter(), pred(tpch.L_QUANTITY, Operator.In([100, 200]))]), tpch.q6_aggregates())
    assert text.startswith("lean plan") and "IN list of 2 literals (pushed)" in text


def test_expression_comparisons_lower_to_the_lean_kernel(lineitem):
    """Expr::Compare over two scalar expressions (compute_compare, llkv-compute/src/kernels.rs:269-297) is a lean
    instruction: one side in the accumulator, the other a column / literal / temporary, the result on the mask stack."""
    from llkv_b200.expr import CompareOp, ScalarExpr
    t, _ = lineitem
    c = ScalarExpr.Column
    price, disc, qty = tpch.L_EXTENDEDPRICE, tpch.L_DISCOUNT, tpch.L_QUANTITY
    big = Expr.Compare(c(price) * c(disc), CompareOp.Gt, ScalarExpr.Literal(Literal.Decimal128(50_000_0000, 4)))
    text = gpu.debug_plan(t, big, tpch.q6_aggregates())
    ops = [ln.split()[1] for ln in text.splitlines() if ln.strip()[:1].isdigit()]
    assert text.startswith("lean plan") and ops.count("CMP") == 1 and ops.count("MASK_FILTER") == 1
    # inside a tree, next to typed leaves; operand order mirrored when the right side ends up in the accumulator
    tree = Expr.Or([Expr.Not(big), Expr.And([tpch.q6_filter(), Expr.Compare(c(qty), CompareOp.LtEq, c(disc) * c(disc))])])
    text = gpu.debug_plan(t, tree, tpch.q6_aggregates())
    ops = [ln.split()[1] for ln in text.splitlines() if ln.strip()[:1].isdigit()]
    assert text.startswith("lean plan") and ops.count("CMP") == 2 and "MASK_NOT" in ops and "MASK_OR" in ops
    if _nvrtc_available():
        assert "specialised cubin:" in gpu.debug_plan(t, tree, tpch.q6_aggregates(), jit=True)


def test_every_reference_held_filter_lowers_to_the_lean_kernel():
    """The reference's own filter tests (tests/golden: ranges, IN lists over integers and floats, AND / OR / NOT, the
    two-column comparison) as the selection of COUNT(*): each is a lean program, and the oracle counts what the reference's
    test expects."""
    import util
    from oracle import oracle
    G = util.golden()
    t = util.table_from_json(G["table_t4"])
    for case in G["filter_cases"]:
        f = util.expr_from_json(case["filter"])
        specs = [AggregateSpec("n", AggregateKind.CountStar())]
        assert gpu.debug_plan(t, f, specs).startswith("lean plan"), case["name"]
        (_, vals), = oracle.aggregate(t, f, specs)
        assert vals[0].value == len(case["expect"]), case["name"]


def test_nullable_group_keys_lower_to_the_lean_kernel():
    """A nullable key column adds a null bit to its field of the packed key (NULL is its own group): GROUP BY over columns
    with NULLs no longer leaves the lean kernel."""
    rng = np.random.default_rng(3)
    n = 4000
    t = HostTable(1)
    k = HostColumn(1, DataType.Int32, rng.integers(0, 40, n).astype(np.int32))
    k.validity = np.packbits(rng.random(n) > 0.2, bitorder="little")
    t.add(k)
    t.add(HostColumn(2, DataType.Int64, rng.integers(-1000, 1000, n, dtype=np.int64)))
    specs = [AggregateSpec("n", AggregateKind.CountStar()), AggregateSpec("s", AggregateKind.Sum(2, DataType.Int64))]
    text = gpu.debug_plan(t, None, specs, group_by=(1,), cardinality_hint=64)
    assert text.startswith("lean plan") and " GROUP " in text


def test_geometry_respects_tuning_and_shared_memory(lineitem):
    t, snap = lineitem
    text = gpu.debug_plan(t, tpch.q1_filter(), tpch.q1_aggregates(), snap, group_by=tpch.Q1_GROUP_BY, cardinality_hint=6,
                          block_threads=64, rows_per_thread=4, stages=2, ctas_per_sm=4)
    head = text.splitlines()[0]
    assert "NC=64 R=4 tile=256 stages=2" in head and "ctas/SM=4" in head
    smem = int(head.split("smem=")[1].split()[0])
    assert 4 * (smem + 1024) <= 227 * 1024


def _nvrtc_available():
    return any(os.path.exists(p) for p in ("/usr/local/cuda/lib64/libnvrtc.so.12", "/usr/local/cuda/lib64/libnvrtc.so"))


@pytest.mark.skipif(not _nvrtc_available(), reason="NVRTC is not installed")
@pytest.mark.parametrize("query", ["q6", "q1"])
def test_specialised_kernel_compiles_for_sm_100a(lineitem, tmp_path, query):
    t, snap = lineitem
    cubin = str(tmp_path / f"{query}.cubin")
    if query == "q6":
        text = gpu.debug_plan(t, tpch.q6_filter(), tpch.q6_aggregates(), jit=True, cubin_path=cubin)
    else:
        text = gpu.debug_plan(t, tpch.q1_filter(), tpch.q1_aggregates(), snap, group_by=tpch.Q1_GROUP_BY, cardinality_hint=6, jit=True,
                              cubin_path=cubin)
    assert "specialised cubin:" in text and os.path.getsize(cubin) > 10_000
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        return
    sass = subprocess.run([cuobjdump, "-sass", cubin], capture_output=True, text=True, check=True).stdout
    assert "sm_100a" in sass and "llkv_lean_jit" in sass
    assert "UBLKCP" in sass and "SYNCS.ARRIVE" in sass and "SYNCS.PHASECHK" in sass
    usage = subprocess.run([cuobjdump, "-res-usage", cubin], capture_output=True, text=True, check=True).stdout
    regs = int(usage.split("REG:")[1].split()[0])
    assert regs <= (80 if query == "q6" else 128)
    # the per-row state (accumulator, slot offsets, masks) must stay in registers: any stack frame means some helper took
    # the address of the tile state or indexed a register array dynamically
    assert int(usage.split("STACK:")[1].split()[0]) == 0
    if query == "q6":
        assert "ATOMS" not in sass  # ungrouped: thread-private accumulators, no shared-memory atomics at all


@pytest.mark.skipif(not _nvrtc_available(), reason="NVRTC is not installed")
def test_partitioned_scan_compiles_for_sm_100a(tmp_path):
    """The partitioned form of a high-cardinality GROUP BY: the specialised scan stages tuples in shared memory (consumer
    barrier 1), reserves partition space with one global atomic per partition and tile, and writes streaming stores."""
    t = tpch.highcard_table(50_000, 20_000, seed=4)
    cubin = str(tmp_path / "part.cubin")
    text = gpu.debug_plan(t, None, tpch.highcard_aggregates(), group_by=(tpch.K_FIELD,), cardinality_hint=20_000, jit=True, partition=True,
                          cubin_path=cubin)
    assert "partitioned: 3 fields per tuple" in text and "specialised cubin:" in text
    plain = gpu.debug_plan(t, None, tpch.highcard_aggregates(), group_by=(tpch.K_FIELD,), cardinality_hint=20_000)
    assert "partitioned" not in plain
    # a plan whose aggregate masks depend on the values (f64 MIN ignores NaN) keeps the per-row path
    tf = HostTable(1).add(HostColumn(tpch.K_FIELD, DataType.Int64, np.arange(100, dtype=np.int64))).add(
        HostColumn(tpch.V_FIELD, DataType.Float64, np.arange(100, dtype=np.float64)))
    nan_dependent = gpu.debug_plan(tf, None, [AggregateSpec("m", AggregateKind.Min(tpch.V_FIELD, DataType.Float64))], group_by=(tpch.K_FIELD,),
                                   cardinality_hint=20_000, partition=True)
    assert "partitioned" not in nan_dependent
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        return
    sass = subprocess.run([cuobjdump, "-sass", cubin], capture_output=True, text=True, check=True).stdout
    assert "UBLKCP" in sass and "BAR.SYNC" in sass and "ATOMS.ADD" in sass and "ATOMG.E.ADD" in sass and "STG.E.EF.64" in sass
    usage = subprocess.run([cuobjdump, "-res-usage", cubin], capture_output=True, text=True, check=True).stdout
    assert int(usage.split("STACK:")[1].split()[0]) == 0


def test_listing_partitions_only_where_the_runtime_does():
    """The listing asks the runtime's form policy: a GROUP BY with a cardinality hint of 128 or less (or none) keeps its
    CTA-local group slots and runs per row in every partitioning mode, so its listing shows no partitioned form."""
    t = tpch.highcard_table(50_000, 20_000, seed=4)
    for hint in (0, 1, 100, 128):
        for kw in (dict(partition=True), dict(packed=True)):
            text = gpu.debug_plan(t, None, tpch.highcard_aggregates(), group_by=(tpch.K_FIELD,), cardinality_hint=hint, **kw)
            assert text.startswith("lean plan") and "partitioned" not in text, (hint, kw, text)
    text = gpu.debug_plan(t, None, tpch.highcard_aggregates(), group_by=(tpch.K_FIELD,), cardinality_hint=129, partition=True)
    assert "partitioned: 3 fields per tuple" in text, text


def test_pinned_geometry_that_does_not_fit_keeps_the_group_slots(lineitem):
    """llkv_gpu_ctx_set_tuning may pin a geometry that does not fit in shared memory.  The fallback gives up consumer
    threads (whole warps) before CTA-local group slots: Q1's four groups keep their four slots."""
    t, snap = lineitem
    for tune in ((96, 2, 2, 6), (128, 1, 4, 5), (128, 2, 2, 4)):
        text = gpu.debug_plan(t, tpch.q1_filter(), tpch.q1_aggregates(), snap, group_by=tpch.Q1_GROUP_BY, cardinality_hint=4,
                              block_threads=tune[0], rows_per_thread=tune[1], stages=tune[2], ctas_per_sm=tune[3])
        head = text.splitlines()[0]
        nc = int(head.split("NC=")[1].split()[0])
        assert " fg=4 " in head and nc % 32 == 0 and f"stages={tune[2]}" in head and f"ctas/SM={tune[3]}" in head, head


@pytest.mark.skipif(not _nvrtc_available(), reason="NVRTC is not installed")
def test_specialising_a_long_program_stays_fast(tmp_path):
    """A specialised build instantiates only the switch case of the instruction at each program position
    (LeanTile::live<PC>): twenty aggregates used to take NVRTC 11 s, and take about 2 s now.  Guard with a wide margin."""
    import time
    from test_gpu_parity import PREDICATES, all_aggs, mixed_table
    t = mixed_table(5000, seed=5)
    t0 = time.time()
    gpu.debug_plan(t, PREDICATES[0], all_aggs()[:1], jit=True, cubin_path=str(tmp_path / "one.cubin"))
    small = time.time() - t0  # the yardstick: the same machine, the same load, one aggregate
    t0 = time.time()
    text = gpu.debug_plan(t, PREDICATES[0], all_aggs(), jit=True, cubin_path=str(tmp_path / "many.cubin"))
    took = time.time() - t0
    assert "specialised cubin:" in text
    # measured: 0.6 s / 1.8 s (ratio 3); before the change 0.9 s / 11.3 s (ratio 12)
    assert took < 6.0 * small + 2.0, f"NVRTC took {took:.1f} s ({small:.1f} s for one aggregate) for {text.splitlines()[0]}"


@pytest.mark.skipif(not _nvrtc_available(), reason="NVRTC is not installed")
def test_every_kernel_variant_specialises_without_a_stack_frame(lineitem, tmp_path):
    """Dense / tile-list scans of Q6 and Q1, the per-row and the partitioned high-cardinality GROUP BY: each shape compiles
    for sm_100a and keeps its per-row state in registers."""
    t, snap = lineitem
    hc = tpch.highcard_table(50_000, 20_000, seed=4)
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    variants = [
        ("q6_list", dict(table=t, expr=tpch.q6_filter(), specs=tpch.q6_aggregates(), tile_list=True)),
        ("q1_list", dict(table=t, expr=tpch.q1_filter(), specs=tpch.q1_aggregates(), snapshot=snap, group_by=tpch.Q1_GROUP_BY, cardinality_hint=4,
                         tile_list=True)),
        ("per_row", dict(table=hc, expr=None, specs=tpch.highcard_aggregates(), group_by=(tpch.K_FIELD,), cardinality_hint=20_000)),
        ("partitioned_list", dict(table=hc, expr=tpch.between_filter(tpch.K_FIELD, 10, 5000), specs=tpch.highcard_aggregates(),
                                  group_by=(tpch.K_FIELD,), cardinality_hint=20_000, partition=True, tile_list=True)),
    ]
    for name, kw in variants:
        cubin = str(tmp_path / f"{name}.cubin")
        text = gpu.debug_plan(jit=True, cubin_path=cubin, **kw)
        assert "specialised cubin:" in text, name
        if os.path.exists(cuobjdump):
            usage = subprocess.run([cuobjdump, "-res-usage", cubin], capture_output=True, text=True, check=True).stdout
            assert int(usage.split("STACK:")[1].split()[0]) == 0, (name, usage)


def test_float_in_list_and_prefix_leaves_lower_to_the_lean_kernel():
    """Float ranges (as integer ranges over the ordered image of the bits), IN lists and string prefixes (a range of packed
    keys) are lean-kernel leaves, also inside OR / NOT trees over nullable columns; the specialised kernel compiles."""
    from test_gpu_parity import mixed_table
    t = mixed_table(1000, 1, nulls=True, long_strings=False)
    specs = [AggregateSpec("n", AggregateKind.CountStar()), AggregateSpec("s1", AggregateKind.Sum(1, DataType.Int64))]
    f = Expr.And([pred(3, Operator.GreaterThan(-0.0)), pred(7, Operator.Equals(0.25)), pred(1, Operator.In([1, 2, -3])),
                  Expr.Or([pred(10, Operator.StartsWith("a")), pred(5, Operator.In([Literal.Decimal128(100, 2), Literal.Int128(7)])),
                           Expr.Not(pred(3, Operator.LessThan(float("nan"))))])])
    listing = gpu.debug_plan(t, f, specs, jit=True)
    assert listing.startswith("lean plan") and "specialised cubin" in listing
    assert "range [1, 9218868437227405312] over the ordered image of the float bits" in listing  # (0, +inf]: -0 == +0
    assert "range [1048576000, 1048576000] over the ordered image" in listing                    # f32 0.25
    assert "IN list of 3 literals" in listing and "IN list of 2 literals (pushed)" in listing
    assert "range [1, 0] over the ordered image of the float bits (pushed)" in listing           # NaN literal: empty
    # suffix / substring patterns are interpreter ops
    g = gpu.debug_plan(t, pred(10, Operator.Contains("a")), specs)
    assert g.startswith("general interpreter")
