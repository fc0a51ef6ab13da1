"""GPU: row-id-sparse Utf8 columns.

Utf8 chunks that arrive with their row-id shadow columns: last-writer-wins updates of strings, NULL by absence (a chunk row
marked NULL is not written) and deletes, on packed short-string columns (scatter_utf8_kernel), one-byte flag columns and
dictionary-coded columns.  Statistics of a sparse packed column are recomputed over the rows that exist at seal
(str_stats_kernel), so a flag column stays at one byte per row and GROUP BY keys keep their full length.  Every query is
checked against the oracle over the compacted table: only the rows that exist, in row-id order."""
import numpy as np
import pytest

import util
from llkv_b200 import ffi, tpch
from llkv_b200.expr import AggregateKind, AggregateSpec, Bound, DataType, Expr, Filter, Operator, pred
from llkv_b200.table import HostColumn, HostTable, LlkvError, decimal_from_i64
from oracle import oracle

pytestmark = pytest.mark.gpu

COUNT = [AggregateSpec("n", AggregateKind.CountStar()), AggregateSpec("s", AggregateKind.Sum(2, DataType.Int64))]


def utf8_chunk(strings):
    """(offsets, data, validity or None) of one Utf8 chunk; None marks a NULL row."""
    c = HostColumn.utf8(0, strings)
    return c.values, c.aux, c.validity


def append_strings(dc, ids, strings):
    offs, data, valid = utf8_chunk(strings)
    dc.append_rows(offs, np.asarray(ids, dtype=np.uint64), first_row_id=0, validity=valid, aux=data)


def new_column(gpu_ctx, table_id, field, dtype):
    from llkv_b200 import gpu
    if dtype.type == ffi.PT_UTF8:
        host = HostColumn.utf8(field, [])
    elif dtype.type == ffi.PT_DECIMAL128:
        host = HostColumn(field, dtype, np.zeros((0, 2), np.uint64))
    else:
        host = HostColumn(field, dtype, np.zeros(0, np.int64))
    return gpu.DeviceColumn(gpu_ctx, gpu.logical_field_id(table_id, field), host)


# ------------------------------------------------------------------------------------------------ Q1 on a mutated lineitem
def mutated_lineitem(n_ids: int, seed: int):
    """The life of a lineitem table, as a list of phases, plus the compacted HostTable of what is left at the end.

    Phase 1 appends the rows that exist below 90 % of the id range (15 % of ids never exist); l_returnflag is absent on
    about 10 % of rows and on the last 1 000 ids.  The table is sealed.  Phase 2 deletes 3 % of those rows from every
    column.  Phase 3 appends the remaining rows, then rewrites 5 % of the surviving rows (quantity, both flags: last writer
    wins); a few rewritten flags are NULL in their chunk, so the earlier value stays.  The table is sealed again."""
    rng = np.random.default_rng(seed)
    a = tpch.lineitem_arrays(n_ids, seed, with_q1=True)
    ids = np.arange(n_ids, dtype=np.uint64)
    exists = rng.random(n_ids) > 0.15
    exists[0] = False
    has_rf = exists & (rng.random(n_ids) > 0.1)
    has_rf[-1000:] = False
    late = ids >= np.uint64(int(n_ids * 0.9))
    deleted = exists & ~late & (rng.random(n_ids) < 0.03)
    alive = exists & ~deleted
    upd = alive & (rng.random(n_ids) < 0.05)
    qty, rf, ls = a["quantity"].copy(), a["returnflag"].copy(), a["linestatus"].copy()
    new_qty = 100 * rng.integers(1, 51, n_ids)
    new_rf = np.array([ord(ch) for ch in "ANR"], np.uint8)[rng.integers(0, 3, n_ids)]
    new_ls = np.array([ord(ch) for ch in "FO"], np.uint8)[rng.integers(0, 2, n_ids)]
    rf_null_in_update = rng.random(n_ids) < 0.1  # the update chunk marks these NULL: not written

    def pieces(mask, piece=7_000):
        sel = np.nonzero(mask)[0]
        return [sel[i:i + piece] for i in range(0, sel.size, piece)]

    def flags(codes):
        return [chr(c) for c in codes]

    def rows(mask):
        out = []
        for p in pieces(mask):
            rfp = p[has_rf[p]]
            out.append({
                tpch.L_QUANTITY: (p, decimal_from_i64(qty[p])),
                tpch.L_EXTENDEDPRICE: (p, decimal_from_i64(a["extendedprice"][p])),
                tpch.L_DISCOUNT: (p, decimal_from_i64(a["discount"][p])),
                tpch.L_TAX: (p, decimal_from_i64(a["tax"][p])),
                tpch.L_SHIPDATE: (p, a["shipdate"][p]),
                tpch.L_RETURNFLAG: (rfp, flags(rf[rfp])),
                tpch.L_LINESTATUS: (p, flags(ls[p])),
                "created": (p, created[p]),
                "deleted": (p, deleted_by[p]),
            })
        return out

    created, deleted_by, snap = tpch.mvcc_arrays(n_ids, seed)
    phase1 = rows(exists & ~late)
    phase3 = rows(exists & late)
    # the rewrite: quantity and linestatus of every updated row, returnflag where the row has one
    upd_chunks = []
    for p in pieces(upd, 3_000):
        rfp = p[has_rf[p]]
        upd_chunks.append({tpch.L_QUANTITY: (p, decimal_from_i64(new_qty[p])),
                           tpch.L_RETURNFLAG: (rfp, [None if rf_null_in_update[i] else chr(new_rf[i]) for i in rfp]),
                           tpch.L_LINESTATUS: (p, flags(new_ls[p]))})
    qty[upd] = new_qty[upd]
    w = upd & has_rf & ~rf_null_in_update
    rf[w] = new_rf[w]
    ls[upd] = new_ls[upd]
    e = np.nonzero(alive)[0]
    t = HostTable(41)
    t.add(HostColumn(tpch.L_QUANTITY, tpch.DEC_15_2, decimal_from_i64(qty[e])))
    t.add(HostColumn(tpch.L_EXTENDEDPRICE, tpch.DEC_15_2, decimal_from_i64(a["extendedprice"][e])))
    t.add(HostColumn(tpch.L_DISCOUNT, tpch.DEC_15_2, decimal_from_i64(a["discount"][e])))
    t.add(HostColumn(tpch.L_TAX, tpch.DEC_15_2, decimal_from_i64(a["tax"][e])))
    t.add(HostColumn(tpch.L_SHIPDATE, DataType.Date32, a["shipdate"][e]))
    t.add(HostColumn.utf8(tpch.L_RETURNFLAG, [chr(rf[i]) if has_rf[i] else None for i in e]))
    t.add(HostColumn.utf8(tpch.L_LINESTATUS, [chr(ls[i]) for i in e]))
    t.add_mvcc(created[e], deleted_by[e])
    return phase1, ids[deleted], phase3 + upd_chunks, t, snap


Q1_TYPES = {tpch.L_QUANTITY: tpch.DEC_15_2, tpch.L_EXTENDEDPRICE: tpch.DEC_15_2, tpch.L_DISCOUNT: tpch.DEC_15_2, tpch.L_TAX: tpch.DEC_15_2,
            tpch.L_SHIPDATE: DataType.Date32, tpch.L_RETURNFLAG: DataType.Utf8, tpch.L_LINESTATUS: DataType.Utf8}


def apply_chunks(dt, chunks):
    for ch in chunks:
        for key, (rid, vals) in ch.items():
            dc = dt.created_by if key == "created" else dt.deleted_by if key == "deleted" else dt.columns[key]
            if key in (tpch.L_RETURNFLAG, tpch.L_LINESTATUS):
                if len(rid):
                    append_strings(dc, rid, vals)
            else:
                dc.append_rows(vals, np.asarray(rid, dtype=np.uint64), first_row_id=0)


def upload_mutated(gpu_ctx, phase1, gone, later, table_id=41):
    from llkv_b200 import gpu
    dt = gpu.DeviceTable(gpu_ctx, table_id)
    for fid, dtype in Q1_TYPES.items():
        dt.columns[fid] = new_column(gpu_ctx, table_id, fid, dtype)
    u64 = HostColumn(0, DataType.UInt64, np.zeros(0, np.uint64))
    dt.created_by = gpu.DeviceColumn(gpu_ctx, gpu.logical_field_id(table_id, 0xFFFFFFFF, gpu.NS_TXN_CREATED_BY), u64)
    dt.deleted_by = gpu.DeviceColumn(gpu_ctx, gpu.logical_field_id(table_id, 0xFFFFFFFE, gpu.NS_TXN_DELETED_BY), u64)
    apply_chunks(dt, phase1)
    dt.seal()
    for dc in dt._all():
        dc.delete_rows(gone)
    apply_chunks(dt, later)
    dt.seal()
    dt.n_rows = max(c.rows() for c in dt._all())
    return dt


def test_q1_on_a_mutated_lineitem_matches_the_oracle(gpu_ctx):
    from llkv_b200 import gpu
    phase1, gone, later, compact, snap = mutated_lineitem(200_000, seed=23)
    dt = upload_mutated(gpu_ctx, phase1, gone, later)
    try:
        assert dt.columns[tpch.L_RETURNFLAG].rows() < dt.n_rows  # (the flag column's last ids are absent: it is grown to the span)
        specs = tpch.q1_aggregates()
        for sn in (None, snap):
            want = oracle.aggregate(compact, tpch.q1_filter(), specs, sn, group_by=tpch.Q1_GROUP_BY, group_capacity=16)
            assert any(k[0] is None for k, _ in want)  # the NULL returnflag group
            for jit in (1, 2):
                gpu_ctx.set_jit(jit)
                for _ in range(2):  # (mode 1 specialises a shape from its second run on)
                    prog = gpu.Program(gpu_ctx, tpch.q1_filter())
                    dt.set_snapshot(sn)
                    agg = gpu.Aggregation(dt, specs, tpch.Q1_GROUP_BY, cardinality_hint=8)
                    try:
                        agg.run(prog, sn is not None)
                        got = agg.finalize(16)
                        info = agg.run_info()
                    finally:
                        agg.destroy()
                        prog.destroy()
                    util.assert_same_result(got, want)
                    assert info.used_fast_kernel == 1
                assert jit == 1 or info.used_jit_kernel == 1
                if sn is not None:  # 4 date + 4 x 4 narrowed decimals + 1 + 1 flags + 8 + 8 MVCC: the flags stayed one byte per row
                    assert info.physical_bytes_per_row == 38
    finally:
        gpu_ctx.set_jit(1)
        dt.destroy()


# ------------------------------------------------------------------------------------------------ last writer wins
SHORT = ["A", "N", "R", "xy", "abc", "TRUCK", "1234567", "é", "Zü", "ab", "zzzzzz"]


def lww_column(rng, n_ids, words, n_chunks, null_share=0.1):
    """Chunks of distinct existing ids with strings from `words`, some marked NULL in their chunk; returns the exists mask,
    the chunks and the last value written per id (None: nothing written)."""
    exists = rng.random(n_ids) > 0.1
    exists[0] = False
    pool = np.nonzero(exists)[0]
    final = [None] * n_ids
    chunks = []
    for _ in range(n_chunks):
        ids = rng.choice(pool, size=int(pool.size * rng.uniform(0.2, 0.6)), replace=False)
        strs = [None if rng.random() < null_share else words[int(rng.integers(0, len(words)))] for _ in ids]
        for i, s in zip(ids, strs):
            if s is not None:
                final[i] = s
        chunks.append((ids, strs))
    return exists, chunks, final


def string_table(gpu_ctx, table_id, exists, x):
    """A sparse table of a Utf8 column (field 1, appended by the caller) and an Int64 column (field 2) holding every row."""
    from llkv_b200 import gpu
    dt = gpu.DeviceTable(gpu_ctx, table_id)
    dt.columns[1] = new_column(gpu_ctx, table_id, 1, DataType.Utf8)
    dt.columns[2] = new_column(gpu_ctx, table_id, 2, DataType.Int64)
    e = np.nonzero(exists)[0].astype(np.uint64)
    for lo in range(0, e.size, 10_000):
        dt.columns[2].append_rows(x[e[lo:lo + 10_000]], e[lo:lo + 10_000], first_row_id=0)
    return dt


def compacted(exists, final, x):
    e = np.nonzero(exists)[0]
    return e, HostTable(1).add(HostColumn.utf8(1, [final[i] for i in e])).add(HostColumn(2, DataType.Int64, x[e]))


def test_last_writer_wins_per_row(gpu_ctx):
    rng = np.random.default_rng(5)
    n_ids = 60_000
    exists, chunks, final = lww_column(rng, n_ids, SHORT, n_chunks=6)
    x = rng.integers(-100, 100, n_ids, dtype=np.int64)
    dt = string_table(gpu_ctx, 42, exists, x)
    try:
        for k, (ids, strs) in enumerate(chunks):
            append_strings(dt.columns[1], ids, strs)
            if k == 2:
                dt.columns[1].seal()  # later chunks land on a sealed column
        dt.seal()
        dt.n_rows = max(c.rows() for c in dt._all())
        assert dt.columns[1].dict_size() == 0  # short strings only: packed keys
        e, t = compacted(exists, final, x)
        for s in SHORT:
            words, count = dt.filter_bitmap(Expr.Pred(Filter(1, Operator.Equals(s))))
            want = np.array([i for i in e if final[i] == s])
            assert count == want.size and np.array_equal(util.selected_positions(words, dt.n_rows), want), s
        words, count = dt.filter_bitmap(pred(1, Operator.IsNull))
        want = np.array([i for i in e if final[i] is None])
        assert count == want.size and np.array_equal(util.selected_positions(words, dt.n_rows), want)
        util.assert_same_result(dt.aggregate(None, COUNT, None, (1,), cardinality_hint=16), oracle.aggregate(t, None, COUNT, None, (1,)))
    finally:
        dt.destroy()


def test_one_byte_strings_written_sparsely_seal_to_one_byte_per_row(gpu_ctx):
    """A sparse flag column, NULL by absence and rewritten: one byte per row at seal, again after more chunks and a delete."""
    from llkv_b200 import gpu
    rng = np.random.default_rng(9)
    n_ids = 30_000
    exists, chunks, final = lww_column(rng, n_ids, ["A", "N", "R"], n_chunks=4)
    x = rng.integers(-100, 100, n_ids, dtype=np.int64)
    dt = string_table(gpu_ctx, 43, exists, x)
    try:
        for k, (ids, strs) in enumerate(chunks):
            append_strings(dt.columns[1], ids, strs)
            if k == 1:
                dt.columns[1].seal()
        gone = np.nonzero(exists)[0][::17].astype(np.uint64)
        for dc in dt._all():
            dc.delete_rows(gone)
        dt.seal()
        dt.n_rows = max(c.rows() for c in dt._all())
        alive = exists.copy()
        alive[gone.astype(np.int64)] = False
        e, t = compacted(alive, final, x)
        for jit in (1, 2):
            gpu_ctx.set_jit(jit)
            agg = gpu.Aggregation(dt, COUNT, (1,), cardinality_hint=4)
            try:
                agg.run(None)
                got = agg.finalize(16)
                info = agg.run_info()
            finally:
                agg.destroy()
            util.assert_same_result(got, oracle.aggregate(t, None, COUNT, None, (1,)))
            assert info.used_fast_kernel == 1 and info.physical_bytes_per_row == 1 + 8  # the flag column: one byte per row
    finally:
        gpu_ctx.set_jit(1)
        dt.destroy()


# ------------------------------------------------------------------------------------------------ dictionary form
LONG = ["DELIVER IN PERSON", "TAKE BACK RETURN", "COLLECT COD", "Zürich Hauptbahnhof", "NONE", "AIR", "REG AIR", "DELIVER", "MAIL"]


def dict_leaves():
    return [Operator.Equals("NONE"), Operator.Equals("DELIVER IN PERSON"), Operator.Equals("nope"),
            Operator.In(["AIR", "TAKE BACK RETURN", "xy", "missing"]),
            Operator.Range(Bound.Included("B"), Bound.Excluded("N")), Operator.GreaterThan("MAIL"), Operator.LessThanOrEquals("AIR"),
            Operator.StartsWith("DELIVER"), Operator.StartsWith("R"), Operator.EndsWith("AIR"), Operator.EndsWith("N"),
            Operator.Contains("IN"), Operator.Contains("ü")]


def check_dict_column(gpu_ctx, dt, t, written):
    from llkv_b200 import gpu
    assert dt.columns[1].dict_size() == len(written)
    for jit in (1, 2):
        gpu_ctx.set_jit(jit)
        for op in dict_leaves():
            flt = Expr.Pred(Filter(1, op))
            prog = gpu.Program(gpu_ctx, flt)
            agg = gpu.Aggregation(dt, COUNT)
            try:
                agg.run(prog)
                got = agg.finalize(1)
                assert agg.run_info().used_fast_kernel == 1, op
            finally:
                agg.destroy()
                prog.destroy()
            util.assert_same_result(got, oracle.aggregate(t, flt, COUNT), ordered=True)
        for flt in (None, pred(2, Operator.LessThan(30))):
            want = oracle.aggregate(t, flt, COUNT, None, (1,))
            assert any(k[0] is None for k, _ in want)
            util.assert_same_result(dt.aggregate(flt, COUNT, None, (1,), cardinality_hint=32), want)


def test_sparse_packed_column_meets_a_long_string(gpu_ctx):
    """Short strings with gaps, NULL rows and rewrites, then a sparse chunk with long strings: the column is re-coded, and only
    the strings of rows that exist enter the dictionary (a gap's zero key is not "")."""
    rng = np.random.default_rng(11)
    n_ids = 40_000
    exists, chunks, final = lww_column(rng, n_ids, SHORT, n_chunks=3)
    _, more, _ = lww_column(np.random.default_rng(12), n_ids, LONG + SHORT[:3], n_chunks=2)
    x = rng.integers(-100, 100, n_ids, dtype=np.int64)
    pool = np.nonzero(exists)[0]
    more = [(ids[np.isin(ids, pool)], [s for i, s in zip(ids, strs) if exists[i]]) for ids, strs in more]
    dt = string_table(gpu_ctx, 44, exists, x)
    try:
        for k, (ids, strs) in enumerate(chunks):
            append_strings(dt.columns[1], ids, strs)
            if k == 1:
                dt.columns[1].seal()  # the short form is sealed before the long strings arrive
        # what the dictionary starts from: the strings the packed column holds (rewritten ones are gone with their keys)
        written = {s for s in final if s is not None}
        for ids, strs in more:
            append_strings(dt.columns[1], ids, strs)
            written |= {s for s in strs if s is not None}
            for i, s in zip(ids, strs):
                if s is not None:
                    final[i] = s
        dt.seal()
        dt.n_rows = max(c.rows() for c in dt._all())
        _, t = compacted(exists, final, x)
        check_dict_column(gpu_ctx, dt, t, written)
    finally:
        gpu_ctx.set_jit(1)
        dt.destroy()


def test_dictionary_column_with_rewrites_and_deletes(gpu_ctx):
    """A column that is dictionary-coded from its first chunk: rewrites keep replaced strings in the dictionary, deletes
    leave gaps, then more chunks arrive after the seal."""
    rng = np.random.default_rng(13)
    n_ids = 40_000
    exists, chunks, final = lww_column(rng, n_ids, LONG, n_chunks=5)
    x = rng.integers(-100, 100, n_ids, dtype=np.int64)
    dt = string_table(gpu_ctx, 45, exists, x)
    alive = exists.copy()
    try:
        written = set()
        for k, (ids, strs) in enumerate(chunks):
            append_strings(dt.columns[1], ids, strs)
            written |= {s for s in strs if s is not None}
            if k == 2:
                dt.seal()
                gone = np.nonzero(alive)[0][::13].astype(np.uint64)
                for dc in dt._all():
                    dc.delete_rows(gone)
                alive[gone.astype(np.int64)] = False
                for i in gone:
                    final[int(i)] = None
        # the last chunks may write deleted ids again: such a row exists once more only if the Int64 column has it too
        for ids, strs in chunks[3:]:
            for i, s in zip(ids, strs):
                if s is not None:
                    final[i] = s
        back = np.array(sorted({int(i) for ids, strs in chunks[3:] for i, s in zip(ids, strs) if s is not None and not alive[i]}), dtype=np.uint64)
        if back.size:
            dt.columns[2].append_rows(x[back.astype(np.int64)], back, first_row_id=0)
            alive[back.astype(np.int64)] = True
        dt.seal()
        dt.n_rows = max(c.rows() for c in dt._all())
        _, t = compacted(alive, final, x)
        check_dict_column(gpu_ctx, dt, t, written)
    finally:
        gpu_ctx.set_jit(1)
        dt.destroy()


# ------------------------------------------------------------------------------------------------ deletes on a dense column
@pytest.mark.parametrize("words", [["A", "N", "R"], ["A", "N", "R", "xy", "abc", "é", "Zürich", "TRUCK"]], ids=["flags", "mixed"])
@pytest.mark.parametrize("when", ["before_seal", "after_seal"])
def test_deletes_on_a_dense_packed_column(gpu_ctx, words, when):
    """GROUP BY over a dense packed Utf8 column after deletes: every key keeps its full length, and a case-insensitive pattern
    over non-ASCII strings is still refused."""
    from llkv_b200 import gpu
    rng = np.random.default_rng(17)
    n = 50_000
    vals = [words[i] for i in rng.integers(0, len(words), n)]
    x = rng.integers(-100, 100, n, dtype=np.int64)
    t_full = HostTable(46).add(HostColumn.utf8(1, vals)).add(HostColumn(2, DataType.Int64, x))
    dt = gpu.DeviceTable(gpu_ctx, 46)
    for col in t_full.columns.values():
        dt.add_column(col, chunk_rows=8192)
    try:
        if when == "after_seal":
            dt.seal()
        gone = np.sort(rng.choice(n, size=n // 7, replace=False)).astype(np.uint64)
        for dc in dt._all():
            dc.delete_rows(gone)
        dt.seal()
        keep = np.ones(n, bool)
        keep[gone.astype(np.int64)] = False
        e = np.nonzero(keep)[0]
        t = HostTable(46).add(HostColumn.utf8(1, [vals[i] for i in e])).add(HostColumn(2, DataType.Int64, x[e]))
        for jit in (1, 2):
            gpu_ctx.set_jit(jit)
            util.assert_same_result(dt.aggregate(None, COUNT, None, (1,), cardinality_hint=16), oracle.aggregate(t, None, COUNT, None, (1,)))
        if any(ord(ch) >= 128 for w in words for ch in w):
            with pytest.raises(LlkvError) as ei:
                dt.aggregate(Expr.Pred(Filter(1, Operator.Contains("a", False))), COUNT)
            assert ei.value.code == ffi.ERR_PREDICATE_BUILD
        else:
            flt = Expr.Pred(Filter(1, Operator.StartsWith("a", False)))
            util.assert_same_result(dt.aggregate(flt, COUNT), oracle.aggregate(t, flt, COUNT))
    finally:
        gpu_ctx.set_jit(1)
        dt.destroy()


def test_utf8_chunk_errors_leave_the_column_unchanged(gpu_ctx):
    """Offsets that run backwards, and a missing data buffer, are refused before anything is uploaded."""
    dc = new_column(gpu_ctx, 47, 1, DataType.Utf8)
    try:
        append_strings(dc, [3, 5], ["ab", "c"])
        with pytest.raises(LlkvError) as ei:
            dc.append_rows(np.array([0, 2, 1], np.int32), np.array([7, 9], np.uint64), aux=np.frombuffer(b"abc", np.uint8))
        assert ei.value.code == ffi.ERR_INVALID_ARGUMENT
        with pytest.raises(LlkvError) as ei:
            dc.append_rows(np.array([0, 2, 3], np.int32), np.array([7, 9], np.uint64))
        assert ei.value.code == ffi.ERR_INVALID_ARGUMENT
        assert dc.rows() == 6 and dc.present_rows() == 2
    finally:
        dc.destroy()
