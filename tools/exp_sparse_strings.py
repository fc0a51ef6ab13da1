"""Q1+MVCC on a lineitem uploaded dense and uploaded row-id-sparse with the same rows, and the append rate of Utf8 flag
columns through scatter_utf8_kernel next to the dense pack path.

The sparse table holds the n rows at row ids with gaps (15 % of an id range of n / 0.85 never exist), every column appended
chunk by chunk with its row ids.  The flags have no NULLs, so both tables are 38 B/row resident and the comparison isolates
the sparse form: positions are row ids and every column carries a validity bitmap.  A third upload, dense with an
all-valid bitmap on every column, separates the cost of the validity bits from that of the gaps.  Q1 kernel times
(`set_timing`) are taken alternating the uploads; the results must be equal.  Append rates are host time of append + seal of one flag
column (copies included), and, when torch.profiler can see the kernels, the device time of pack_utf8_kernel and
scatter_utf8_kernel in a separate run.
Usage: python tools/exp_sparse_strings.py [rows] [reps]"""
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [os.path.join(ROOT, "rust-llkv_b200"), ROOT]
import numpy as np

from llkv_b200 import ffi, gpu, tpch
from llkv_b200.table import HostColumn

n = int(sys.argv[1]) if len(sys.argv) > 1 else tpch.lineitem_rows(10.0)
reps = int(sys.argv[2]) if len(sys.argv) > 2 else 10
CHUNK = 1 << 20
try:
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
except OSError:
    card = "unknown"
print(f"card: {card}; rows {n}", flush=True)

ctx = gpu.Context(0)
ctx.set_timing(True)
ctx.set_jit(2)
t, snap = tpch.lineitem_table(n, seed=6, with_q1=True, with_mvcc=True)
rng = np.random.default_rng(7)
ids = np.nonzero(rng.random(int(n / 0.85) + 100_000) > 0.15)[0][:n].astype(np.uint64)  # row id of each row
n_ids = int(ids[-1]) + 1


def flag_chunk(col, lo, hi):
    return np.arange(hi - lo + 1, dtype=np.int32), col.aux[lo:hi]


def append_sparse_column(dc, col):
    for lo in range(0, n, CHUNK):
        hi = min(n, lo + CHUNK)
        if col.dtype.type == ffi.PT_UTF8:
            offs, data = flag_chunk(col, lo, hi)
            dc.append_rows(offs, ids[lo:hi], first_row_id=0, aux=data)
        else:
            dc.append_rows(col.values[lo:hi], ids[lo:hi], first_row_id=0)


def sparse_table():
    dt = gpu.DeviceTable(ctx, 2)
    for fid, col in t.columns.items():
        dc = gpu.DeviceColumn(ctx, gpu.logical_field_id(2, fid), col)
        append_sparse_column(dc, col)
        dt.columns[fid] = dc
    dt.created_by = gpu.DeviceColumn(ctx, gpu.logical_field_id(2, 0xFFFFFFFF, gpu.NS_TXN_CREATED_BY), t.created_by)
    dt.deleted_by = gpu.DeviceColumn(ctx, gpu.logical_field_id(2, 0xFFFFFFFE, gpu.NS_TXN_DELETED_BY), t.deleted_by)
    append_sparse_column(dt.created_by, t.created_by)
    append_sparse_column(dt.deleted_by, t.deleted_by)
    dt.seal()
    dt.n_rows = max(c.rows() for c in dt._all())
    return dt


def dense_nullable_table():
    """The dense upload with an all-valid bitmap on every column: per-column validity without gaps or an exists bitmap."""
    from llkv_b200.table import HostTable
    ones = np.full((n + 7) // 8, 0xFF, np.uint8)
    tn = HostTable(3)
    for col in t.columns.values():
        tn.add(HostColumn(col.field_id, col.dtype, col.values, ones, col.aux))
    tn.created_by = HostColumn(t.created_by.field_id, t.created_by.dtype, t.created_by.values, ones)
    tn.deleted_by = HostColumn(t.deleted_by.field_id, t.deleted_by.dtype, t.deleted_by.values, ones)
    return gpu.DeviceTable.from_host(ctx, tn, chunk_rows=CHUNK)


tables = {"dense": gpu.DeviceTable.from_host(ctx, t, chunk_rows=CHUNK), "dense, every column with a validity bitmap": dense_nullable_table(),
          "sparse": sparse_table()}
aggs, results, ms = {}, {}, {k: [] for k in tables}
prog = gpu.Program(ctx, tpch.q1_filter())
for k, dt in tables.items():
    dt.set_snapshot(snap)
    aggs[k] = gpu.Aggregation(dt, tpch.q1_aggregates(), tpch.Q1_GROUP_BY, cardinality_hint=8)
    for _ in range(3):  # warm-up: specialisation, first launches
        aggs[k].execute(prog, True)
        aggs[k].finalize(16)
for _ in range(reps):
    for k in tables:
        tables[k].set_snapshot(snap)
        aggs[k].execute(prog, True)
        results[k] = aggs[k].finalize(16)
        ms[k].append(aggs[k].run_info().last_kernel_ms)
for k in tables:
    info = aggs[k].run_info()
    v = sorted(ms[k])
    print(f"Q1+MVCC {k}: kernel ms median {v[len(v) // 2]:.4f} min {v[0]:.4f} max {v[-1]:.4f} lean={info.used_fast_kernel} "
          f"jit={info.used_jit_kernel} bytes/row={info.physical_bytes_per_row}", flush=True)
same = all([(a[0], [x.value for x in a[1]]) for a in results["dense"]] == [(a[0], [x.value for x in a[1]]) for a in r] for r in results.values())
print(f"Q1 results equal: {same}", flush=True)
for a in aggs.values():
    a.destroy()
prog.destroy()
for dt in tables.values():
    dt.destroy()

# append rate of one flag column: dense pack path against the sparse scatter, same rows
flag = t.columns[tpch.L_RETURNFLAG]


def append_dense(dc):
    dc.append(flag, chunk_rows=CHUNK)


def append_scattered(dc):
    append_sparse_column(dc, flag)


def timed(fn, tid):
    dc = gpu.DeviceColumn(ctx, gpu.logical_field_id(tid, 1), flag)
    dc.reserve(n_ids)
    t0 = time.perf_counter()
    fn(dc)
    dc.seal()  # ends in a device synchronise
    dt = time.perf_counter() - t0
    dc.destroy()
    return dt


for label, fn in (("dense pack", append_dense), ("sparse scatter", append_scattered)):
    secs = sorted(timed(fn, 10 + i) for i in range(5))
    print(f"append {label}: {n / secs[2] / 1e6:.1f} M rows/s host time (median of 5, {secs[2] * 1e3:.1f} ms)", flush=True)

try:
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.init()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for fn in (append_dense, append_scattered):
            timed(fn, 20)
    dev = {}
    for ev in prof.events():
        if "utf8_kernel" in ev.name:
            name = ev.name.split("(")[0]
            dev[name] = dev.get(name, 0.0) + ev.device_time_total / 1e3
    for name, total in sorted(dev.items()):
        print(f"kernel {name}: {total:.3f} ms for {n} rows = {n / total / 1e6:.2f} G rows/s", flush=True)
    if not dev:
        print("kernel times: not measured (the profiler saw no Utf8 kernels)", flush=True)
except Exception as exc:  # the host-time rates above stand on their own
    print(f"kernel times: not measured ({exc})", flush=True)
ctx.close()
