#!/usr/bin/env python
"""bench.py — rows/s and HBM GB/s (fraction of the measured roofline) for TPC-H Q6 / Q1 over synthetic lineitem, plus the
other BASELINE.json configurations, every result checked against a numpy restatement of the query (`"verified": true`, or
a non-zero exit).

  python bench.py --gpus N --steps K --warmup W            our arm: the CUDA path through the C ABI
  python bench.py --impl reference --gpus N ...            the reference's CPU path (oracle port), host threads
  python bench.py ... --dump-outputs DIR                   also write what each timed leg returned in its last step

A step = one pass of scan -> predicate -> MVCC -> aggregate over the batch, through llkv_gpu_agg_execute (fresh accumulators,
one fused scan, merge of the ranks' partial states) and llkv_gpu_agg_finalize (result in host memory).
N = 1: BASELINE.json configs[1], TPC-H Q6 on synthetic lineitem SF10 (59 986 052 rows) resident in HBM; configs[2] (Q1 + MVCC),
       configs[0] (10 M-row Int64 BETWEEN + SUM, without / with MVCC columns) and configs[3] (1 B rows, 10 M keys) ride along.
N > 1: BASELINE.json configs[4]: every rank holds one chunk-aligned row-range shard of SF100 lineitem cut in eight
       (600 037 902 rows / 8 = 75.0 M rows per GPU; weak scaling: N of the eight shards are resident), partial states merge
       over NVLink peer mailboxes every step.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

# the benchmark writes nothing into the source tree, which may be read-only
sys.dont_write_bytecode = True
# stdout carries exactly one JSON line: NCCL's own banner ("NCCL version ...") goes to stderr
os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (os.path.join(ROOT, "rust-llkv_b200"), ROOT):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402

from llkv_b200 import ffi, tpch  # noqa: E402
from llkv_b200.expr import DataType  # noqa: E402
from llkv_b200.table import HostColumn, HostTable  # noqa: E402

METRIC = "tpch_q6_lineitem_rows_per_sec"
UNIT = "rows/s"
SF100_ROWS = tpch.LINEITEM_ROWS[100]
# how SUM(l_extendedprice * l_discount) is typed and rounded: arrow-arith product, cast back to Decimal128(15,2) per row
# (SURVEY.md section 8a note D1, "as written")
DECIMAL_CONTRACT = "arrow-as-written"


def measured_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for name, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm)}


def kernel_name(info) -> str:
    if info.used_jit_kernel:
        return "llkv_lean_jit (lean_kernel.cuh specialised on the plan shape by jit.cpp)"
    if info.used_fast_kernel:
        return "llkv::lean_scan_kernel<R> (lean_kernel.cuh, interpreted)"
    return "llkv::scan_kernel<WIDE,R> (general interpreter)"


def pinned_column(gpu, field_id, dtype, values: np.ndarray):
    """Copies `values` into page-locked host memory and returns (HostColumn view, raw ptr, nbytes)."""
    raw = np.ascontiguousarray(values)
    buf, ptr = gpu.pinned_empty(raw.nbytes)
    buf[:] = raw.view(np.uint8).reshape(-1)
    view = buf.view(raw.dtype).reshape(raw.shape)
    return HostColumn(field_id, dtype, view), ptr, raw.nbytes


def build_lineitem_pinned(gpu, a, with_q1):
    from llkv_b200.table import decimal_from_i64
    cols, ptrs = {}, []

    def add(fid, dtype, vals):
        c, p, _ = pinned_column(gpu, fid, dtype, vals)
        cols[fid] = c
        ptrs.append(p)

    add(tpch.L_QUANTITY, tpch.DEC_15_2, decimal_from_i64(a["quantity"]))
    add(tpch.L_EXTENDEDPRICE, tpch.DEC_15_2, decimal_from_i64(a["extendedprice"]))
    add(tpch.L_DISCOUNT, tpch.DEC_15_2, decimal_from_i64(a["discount"]))
    add(tpch.L_SHIPDATE, DataType.Date32, a["shipdate"])
    if with_q1:
        add(tpch.L_TAX, tpch.DEC_15_2, decimal_from_i64(a["tax"]))
    return cols, ptrs


def upload_column(dc, col: HostColumn, chunk_bytes: int, row_id_base: int):
    """ColumnStore::append shape: one append per chunk of ~chunk_bytes straight from the pinned buffer."""
    n = col.n_rows
    width = col.values.dtype.itemsize * (2 if col.dtype.type == ffi.PT_DECIMAL128 else 1)
    rows = max(1, chunk_bytes // width)
    base = col.values.ctypes.data
    for lo in range(0, n, rows):
        m = min(rows, n - lo)
        dc.append_raw(base + lo * width, m, row_id_base + lo)


class Failed(Exception):
    pass


def check(cond, what):
    if not cond:
        raise Failed(what)


def run_ours(args):
    import torch
    from llkv_b200 import gpu

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    # ---- the rows this rank holds
    if args.rows:
        n, row_base, workload_rows = args.rows, rank * args.rows, f"{args.rows} rows per GPU (--rows)"
    elif world > 1:
        lo, hi = gpu.shard_rows(SF100_ROWS, 8, rank % 8)
        n, row_base = hi - lo, lo
        workload_rows = f"SF100 (600 037 902 rows) cut into 8 chunk-aligned row-range shards of ~75.0 M rows, {world} of them resident, one per GPU"
    else:
        n, row_base = tpch.lineitem_rows(args.sf), 0
        workload_rows = f"SF{args.sf:g}, {n} rows"
    cores = os.cpu_count() or 1
    ctx = gpu.Context(local, n_streams=4, pinned_bytes=64 << 20)
    # host workers that narrow Decimal128 chunks before the DMA: this rank's share of the host threads
    upload_threads = args.upload_threads if args.upload_threads >= 0 else max(0, min(32, cores // world - 1))
    if args.upload_threads < 0 and world > 1:
        # several ranks share the host's memory system: narrowing on the host loses against plain DMA there
        # (12 threads per rank at N = 2: 113 ms against 72 ms per step)
        upload_threads = 0
    # N = 1: a hybrid upload — the workers narrow their share of the Decimal128 bytes (about 4.5 GB/s of Arrow bytes each,
    # bound by the host's memory system), the copy engine takes the rest as it lies and a kernel narrows it on the device;
    # the split follows the worker count (llkv_gpu_ctx_set_dma_share, -1)
    ctx.set_dma_share(args.dma_share)
    ctx.set_upload_threads(upload_threads)
    if world > 1:
        ids = [ctx.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(ids, src=0)
        ctx.comm_init(ids[0], world, rank)
    ctx.set_timing(True)

    with_q1 = not args.no_q1
    seed = 6 + rank
    a = tpch.lineitem_arrays(n, seed, with_q1)
    cols, ptrs = build_lineitem_pinned(gpu, a, with_q1)
    table = gpu.DeviceTable(ctx, 1)
    chunk_bytes = 1 << 20
    dcs = {}
    for fid, c in cols.items():
        dc = gpu.DeviceColumn(ctx, gpu.logical_field_id(1, fid), c)
        dc.reserve(n)
        upload_column(dc, c, chunk_bytes, row_base)
        dcs[fid] = dc
        table.columns[fid] = dc
    table.n_rows = n
    snap = created = deleted = None
    if with_q1:
        from llkv_b200.tpch import _utf8_single_char
        for fid, key in ((tpch.L_RETURNFLAG, "returnflag"), (tpch.L_LINESTATUS, "linestatus")):
            dc = gpu.DeviceColumn(ctx, gpu.logical_field_id(1, fid), _utf8_single_char(fid, a[key]))
            dc.reserve(n)
            dc.append(_utf8_single_char(fid, a[key]), chunk_rows=1 << 20, row_id_base=row_base)
            table.columns[fid] = dc
        created, deleted, snap = tpch.mvcc_arrays(n, seed=seed)
        table.created_by = gpu.DeviceColumn(ctx, gpu.logical_field_id(1, 0xFFFFFFFF, gpu.NS_TXN_CREATED_BY), HostColumn(0xFFFFFFFF, DataType.UInt64, created))
        table.deleted_by = gpu.DeviceColumn(ctx, gpu.logical_field_id(1, 0xFFFFFFFE, gpu.NS_TXN_DELETED_BY), HostColumn(0xFFFFFFFE, DataType.UInt64, deleted))
        for dc, arr in ((table.created_by, created), (table.deleted_by, deleted)):
            dc.reserve(n)
            dc.append(HostColumn(0, DataType.UInt64, arr), chunk_rows=1 << 17, row_id_base=row_base)
    table.seal()
    ctx.synchronize()

    # ---- expected answers: numpy over this rank's arrays, exact integers; the union over ranks through the host
    exp_q6_local = tpch.expected_q6(a)
    exp_q1_local = tpch.expected_q1_partials(a, created, deleted, snap) if with_q1 else None

    def gather(obj):
        if dist is None:
            return [obj]
        out = [None] * world
        dist.all_gather_object(out, obj)
        return out

    exp_q6_all = sum(gather(exp_q6_local))
    exp_q1_all = tpch.q1_rows_from_partials(tpch.add_partials(gather((row_base, exp_q1_local)))) if with_q1 else None
    exp_q1_own = tpch.q1_rows_from_partials(tpch.add_partials([(row_base, exp_q1_local)])) if with_q1 else None

    def barrier():
        torch.cuda.synchronize()
        ctx.synchronize()
        if dist is not None:
            dist.barrier()
            torch.cuda.synchronize()

    def max_over_ranks(x: float) -> float:
        if dist is None:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def plain_rows(rows):
        return [(k, [v.value for v in vals]) for k, vals in rows]

    def bench_query(name, filter_expr, specs, group_by=(), snapshot=None, hint=0, want_own=None, want_all=None, steps=args.steps, warmup=args.warmup):
        prog = gpu.Program(ctx, filter_expr)
        table.set_snapshot(snapshot)
        agg = gpu.Aggregation(table, specs, group_by, cardinality_hint=hint)
        cap = 64 if group_by else 1
        # this rank's shard on its own, before any merge
        agg.execute(prog, snapshot is not None, 0, n, merge=False)
        own = plain_rows(agg.finalize(cap))
        check(own == want_own, f"{name}: rank {rank}'s own shard gives {own}, numpy says {want_own}")
        kernel_ms, merge_ms, launches = [], [], 0
        raw = None

        def step(record):
            nonlocal launches, raw
            agg.execute(prog, snapshot is not None, 0, n, merge=True)
            raw = agg.finalize_raw(cap)  # the result is in host memory here; it is decoded and checked after the timed region
            if record:
                info = agg.run_info()
                kernel_ms.append(info.last_kernel_ms)
                merge_ms.append(info.last_merge_ms)
                launches += info.kernel_launches + 1 + (1 if world > 1 else 0)  # scan launches + accumulator init + merge kernel

        for _ in range(warmup):
            step(False)
        barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            step(True)
        barrier()
        dt = max_over_ranks(time.perf_counter() - t0)
        rows = agg.decode(*raw)
        merged = plain_rows(rows)
        check(merged == want_all, f"{name}: merged result {merged} != numpy over all shards {want_all}")
        info = agg.run_info()
        agg.destroy()
        prog.destroy()
        # the merge kernel's device time on every rank (it includes waiting for the slowest peer's scan)
        merge_all = gather(statistics.mean(merge_ms)) if merge_ms and world > 1 else None
        return {"seconds": dt, "kernel_ms": kernel_ms, "merge_ms": merge_all, "launches": launches, "info": info, "result": merged, "rows": rows}

    failed = None
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    line = {}
    try:
        q6 = bench_query("Q6", tpch.q6_filter(), tpch.q6_aggregates(), want_own=[((), [exp_q6_local])], want_all=[((), [exp_q6_all])])
        q1 = None
        if with_q1:
            q1 = bench_query("Q1", tpch.q1_filter(), tpch.q1_aggregates(), tpch.Q1_GROUP_BY, snap, hint=4,  # BASELINE.json: "4-group GROUP BY"
                             want_own=exp_q1_own, want_all=exp_q1_all)

        # ---- end to end: host (pinned) buffers -> chunk appends -> fused scan -> result on the host, every step
        e2e_cols = [tpch.L_QUANTITY, tpch.L_EXTENDEDPRICE, tpch.L_DISCOUNT, tpch.L_SHIPDATE]
        host_bytes = sum(cols[f].values.nbytes for f in e2e_cols)
        prog = gpu.Program(ctx, tpch.q6_filter())
        table.set_snapshot(None)
        agg = gpu.Aggregation(table, tpch.q6_aggregates())

        def e2e_step():
            for f in e2e_cols:
                dcs[f].clear()
                upload_column(dcs[f], cols[f], chunk_bytes, row_base)
            for f in e2e_cols:
                dcs[f].seal()
            agg.execute(prog, False, 0, n, merge=True)
            return agg.finalize(1)

        for _ in range(max(1, min(args.warmup, 2))):
            e2e_step()
        barrier()
        e2e_steps = args.steps
        moved0 = sum(dcs[f].h2d_bytes() for f in e2e_cols)
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            e2e_result = e2e_step()
        barrier()
        e2e_dt = max_over_ranks(time.perf_counter() - t0)
        h2d = (sum(dcs[f].h2d_bytes() for f in e2e_cols) - moved0) // e2e_steps
        check(plain_rows(e2e_result) == [((), [exp_q6_all])], f"end to end: {plain_rows(e2e_result)} != numpy {exp_q6_all}")
        d2h = 4 + 3 * 6 * 8  # status word + the ungrouped state row (6 words) and its two spare rows, read back by finalize
        agg.destroy()
        prog.destroy()

        # --dump-outputs: the merged results are the same on every rank, rank 0 writes them
        dump = {} if args.dump_outputs and rank == 0 else None
        if dump is not None:
            add_result(dump, "q6", q6["rows"])
            if q1 is not None:
                add_result(dump, "q1", q1["rows"])
            add_result(dump, "e2e_q6", e2e_result)
        extra = {}
        if world == 1 and not args.no_configs:
            extra["config0"] = bench_config0(ctx, gpu, args, dump)
        if world == 1 and not args.no_highcard:
            extra["highcard"] = bench_highcard(ctx, gpu, torch, args, big=n >= 20_000_000, dump=dump)
        if dump is not None:
            write_outputs(args.dump_outputs, dump)
        clocks = sampler.stop() if rank == 0 else None  # sampled across the timed regions

        total_rows = sum(gather_rows(dist, n, world))
        if rank == 0:
            peak, peak_src = measured_peak()
            kms = statistics.mean(q6["kernel_ms"]) if q6["kernel_ms"] else float("nan")
            # bytes per row: `arrow` = Arrow-layout value buffers (Decimal128 = 16 B), `resident` = what the kernel reads from HBM
            # (Decimal128 columns whose values fit i32 / i64 are kept as 4 / 8 B per row, DESIGN.md "data layout").  The roofline
            # uses the resident bytes, so the fraction can never exceed what the memory system delivered.
            arrow_bpr = q6["info"].algorithmic_bytes_per_row
            alg_bpr = q6["info"].physical_bytes_per_row
            achieved = alg_bpr * n / (kms * 1e-3) / 1e9 if kms == kms and kms > 0 else None
            achieved_arrow = arrow_bpr * n / (kms * 1e-3) / 1e9 if kms == kms and kms > 0 else None
            traffic, traffic_source = None, None  # dram__bytes_read + dram__bytes_write of the Q6 kernel from the committed ncu capture
            prof = os.path.join(ROOT, "profiles", "r02_q6_traffic.json")
            if os.path.exists(prof):
                try:
                    t = json.load(open(prof))
                    if t.get("resident_bytes_per_row") == alg_bpr:
                        traffic = (t["dram_bytes_read"] + t["dram_bytes_write"]) / t["rows"] * n
                        traffic_source = (f"replayed, not measured in this run: profiles/r02_q6_traffic.json (ncu --set full, {t['rows']} rows, "
                                          f"build {t.get('build', '?')}), scaled by rows")
                except Exception:
                    pass
            line = {
                "metric": METRIC, "value": total_rows * args.steps / q6["seconds"], "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": q6["seconds"] / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "i128/i64 (Decimal128, Date32)", "data": "synthetic", "verified": True,
                "decimal_contract": DECIMAL_CONTRACT,
                "config": {"workload": f"TPC-H Q6 (filter + SUM(l_extendedprice*l_discount)) on synthetic lineitem {workload_rows}, resident in HBM"
                                       + (" (BASELINE.json configs[4])" if world > 1 and not args.rows else " (BASELINE.json configs[1])"),
                           "rows_per_gpu": n, "total_rows": total_rows, "sharding": "row-range per rank" if world > 1 else "none",
                           "l2_policy": "inputs larger than L2 (%.2f GB resident per pass vs 126 MB)" % (alg_bpr * n / 1e9), "chunk_bytes": chunk_bytes,
                           "step": "llkv_gpu_agg_execute (reset + scan + merge, one CUDA graph launch once the step repeats) + llkv_gpu_agg_finalize",
                           "graph_replays": q6["info"].graph_replays, "merge": ("NVLink peer mailboxes" if q6["info"].merged_p2p else "NCCL") if world > 1 else "none",
                           "merge_kernel_ms": q6["merge_ms"],
                           "kernel": {"grid": q6["info"].grid, "block": q6["info"].block, "rows_per_tile": q6["info"].rows_per_tile,
                                      "stages": q6["info"].stages, "smem_bytes": q6["info"].smem_bytes, "wide": q6["info"].used_wide_path,
                                      "specialised": q6["info"].used_jit_kernel}},
                "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak if achieved else None,
                             "traffic": traffic, "traffic_source": traffic_source, "peak_source": peak_src, "kernel": kernel_name(q6["info"]), "kernel_ms": kms,
                             "basis": "resident bytes: what the kernel reads from HBM (Decimal128(15,2) columns whose values fit are kept as i32 / i64 "
                                      "after seal, DESIGN.md section 2); SURVEY.md section 8(d) counts Arrow-layout bytes, given beside it",
                             "resident_bytes_per_row": alg_bpr, "algorithmic_bytes_per_row": arrow_bpr,
                             "algorithmic_gbs": achieved_arrow},
                "e2e": {"value": total_rows * e2e_steps / e2e_dt, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                        "host_bytes_per_step": host_bytes, "upload_threads": upload_threads, "dma_share_percent": args.dma_share,
                        "narrow_isa": host_narrow_isa(),
                        "note": "host buffers hold the Arrow layout (Decimal128 = 16 B/value); host workers narrow the chunks that fit before the DMA, "
                                "h2d_bytes_per_step is what crossed the link (llkv_gpu_column_h2d_bytes)",
                        "ms_per_step": e2e_dt / e2e_steps * 1e3, "steps": e2e_steps},
                "gpu_launches": q6["launches"],
                "clocks": clocks,
                "result": {"q6_revenue_raw": q6["result"][0][1][0], "q6_expected_numpy": exp_q6_all, "e2e_revenue_raw": e2e_result[0][1][0].value},
            }
            if q1 is not None:
                k1 = statistics.mean(q1["kernel_ms"])
                b1 = q1["info"].physical_bytes_per_row
                a1 = b1 * n / (k1 * 1e-3) / 1e9
                line["q1"] = {"workload": f"TPC-H Q1 (4-group GROUP BY, Decimal SUM/AVG/COUNT) with MVCC on the same lineitem, {n} rows per GPU"
                                          + (" (BASELINE.json configs[4])" if world > 1 and not args.rows else " (BASELINE.json configs[2])"),
                              "value": total_rows * args.steps / q1["seconds"], "unit": UNIT, "ms_per_step": q1["seconds"] / args.steps * 1e3, "verified": True,
                              "roofline": {"bound": "hbm", "achieved": a1, "peak": peak, "unit": "GB/s", "frac": a1 / peak, "kernel_ms": k1,
                                           "resident_bytes_per_row": b1, "algorithmic_bytes_per_row": q1["info"].algorithmic_bytes_per_row,
                                           "algorithmic_gbs": q1["info"].algorithmic_bytes_per_row * n / (k1 * 1e-3) / 1e9},
                              "groups": [[list(k), v] for k, v in q1["result"]], "graph_replays": q1["info"].graph_replays,
                              "merge": ("NVLink peer mailboxes" if q1["info"].merged_p2p else "NCCL") if world > 1 else "none",
                              "merge_kernel_ms": q1["merge_ms"],
                              "kernel_name": kernel_name(q1["info"]), "kernel": {"grid": q1["info"].grid, "block": q1["info"].block,
                                                                                  "rows_per_tile": q1["info"].rows_per_tile, "stages": q1["info"].stages,
                                                                                  "smem_bytes": q1["info"].smem_bytes, "fast_groups": q1["info"].fast_groups,
                                                                                  "wide": q1["info"].used_wide_path}}
            line.update(extra)
            if world == 1 and not args.no_cpu_baseline:
                line["cpu_baseline"] = cpu_baseline_subprocess()
    except Failed as e:
        failed = str(e)
    except Exception as e:  # a rank that raises must not leave the others in a collective
        import traceback
        traceback.print_exc()
        failed = repr(e)

    if dist is not None:
        flags = [None] * world
        dist.all_gather_object(flags, failed)
        failed = next((f for f in flags if f), None)
    if rank == 0:
        if failed:
            emit({"metric": METRIC, "unit": UNIT, "n_gpus": world, "verified": False, "error": failed})
        else:
            emit(line)
    for p in ptrs:
        gpu.pinned_free(p)
    if dist is not None:
        dist.barrier()
        ctx.comm_destroy()
        dist.destroy_process_group()
    ctx.close()
    if failed:
        sys.exit(1)


DUMP_LIMIT_BYTES = 64 << 20
DUMP_GROUPS = 1 << 18  # groups of a high-cardinality result that --dump-outputs keeps


def add_result(dump, name, rows):
    """Decoded result rows as float64 arrays `<name>_values` [groups, aggregates] and, when grouped, `<name>_keys`
    [groups, keys]: a Decimal128 as its value (unscaled / 10^scale), a one-character Utf8 key as its code point, NULL as NaN."""
    def num(x, scale=0):
        if x is None:
            return float("nan")
        return float(ord(x)) if isinstance(x, str) else x / 10 ** scale
    dump[name + "_values"] = np.array([[num(v.value, v.scale) for v in vals] for _, vals in rows], dtype=np.float64)
    if rows and rows[0][0]:
        dump[name + "_keys"] = np.array([[num(k) for k in key] for key, _ in rows], dtype=np.float64)


def write_outputs(directory, dump):
    total = sum(a.nbytes for a in dump.values())
    check(total <= DUMP_LIMIT_BYTES, f"--dump-outputs: {total} bytes, more than {DUMP_LIMIT_BYTES}")
    os.makedirs(directory, exist_ok=True)
    for name, a in dump.items():
        np.save(os.path.join(directory, name + ".npy"), a)


def gather_rows(dist, n, world):
    if dist is None:
        return [n]
    out = [None] * world
    dist.all_gather_object(out, n)
    return out


def bench_config0(ctx, gpu, args, dump):
    """BASELINE.json configs[0]: SELECT SUM(x) FROM t WHERE x BETWEEN a AND b over one Int64 column of 10 M rows (a, b = 25th / 75th
    percentile), without and with the MVCC columns every SQL table carries.  Launch-latency bound at this size: the 1 B-row figure is
    the Q6 / Q1 legs' business.  Results against numpy; with `dump` (a dict), the last step's results are added to it."""
    n = 10_000_000
    t, snap = tpch.int64_table(n, seed=1, table_id=3)
    x = t.columns[tpch.X_FIELD].values
    lo, hi = (int(v) for v in np.percentile(x[:1_000_000], [25, 75]).astype(np.int64))
    want = int(x[(x >= lo) & (x <= hi)].sum())
    dt = gpu.DeviceTable.from_host(ctx, t, chunk_rows=1 << 20)
    out = {"workload": "SELECT SUM(x) WHERE x BETWEEN a AND b, single Int64 column, 10 M rows, ~50 % selectivity (BASELINE.json configs[0])",
           "rows": n, "unit": UNIT, "verified": True}
    try:
        for name, sn in (("no_mvcc", None), ("mvcc", snap)):
            prog = gpu.Program(ctx, tpch.between_filter(tpch.X_FIELD, lo, hi))
            dt.set_snapshot(sn)
            agg = gpu.Aggregation(dt, tpch.sum_int64(tpch.X_FIELD))
            ms = []
            for _ in range(max(3, args.warmup)):
                agg.execute(prog, sn is not None)
                got = agg.finalize(1)
            torch_sync(ctx)
            steps = args.steps
            t0 = time.perf_counter()
            for _ in range(steps):
                agg.execute(prog, sn is not None)
                raw = agg.finalize_raw(1)
                ms.append(agg.run_info().last_kernel_ms)
            torch_sync(ctx)
            dtm = time.perf_counter() - t0
            got = agg.decode(*raw)
            check(got[0][1][0].value == want, f"configs[0] {name}: {got[0][1][0].value} != numpy {want}")
            if dump is not None:
                add_result(dump, f"config0_{name}", got)
            info = agg.run_info()
            kms = statistics.mean(ms)
            out[name] = {"value": n * steps / dtm, "ms_per_step": dtm / steps * 1e3, "kernel_ms": kms, "bytes_per_row": info.physical_bytes_per_row,
                         "kernel_gbs": info.physical_bytes_per_row * n / (kms * 1e-3) / 1e9, "graph_replays": info.graph_replays,
                         "specialised": info.used_jit_kernel, "result": got[0][1][0].value}
            agg.destroy()
            prog.destroy()
    finally:
        dt.destroy()
    return out


def torch_sync(ctx):
    ctx.synchronize()


def bench_highcard(ctx, gpu, torch, args, big, dump):
    """BASELINE.json configs[3]: GROUP BY over 10 M distinct Int64 keys, SUM + COUNT, 1 B rows (key = SplitMix64(i) mod 10^7,
    value = SplitMix64(i + 2^40) mod 1001).  The two columns are generated on the device in pieces (16 GB of input) and appended from
    device memory; kernel time only (CUDA events around the scan + apply launches).  Every group's SUM and COUNT is compared
    with an integer scatter-add of the same arrays (torch, exact int64).  With `dump` (a dict), a fixed sample of the last run's
    groups is added to it."""
    rows, n_keys = (args.highcard_rows or 1_000_000_000, 10_000_000) if big else (1 << 22, 2_000_000)
    dev = torch.device("cuda", ctx.device)
    piece = 1 << 26
    dt = gpu.DeviceTable(ctx, 2)
    cols = {}
    want_sum = torch.zeros(n_keys, dtype=torch.int64, device=dev)
    want_cnt = torch.zeros(n_keys, dtype=torch.int64, device=dev)
    first = torch.full((n_keys,), rows, dtype=torch.int64, device=dev)

    def splitmix(i):  # int64 arithmetic wraps like uint64; shifts are made logical by masking
        def shr(z, k):
            return (z >> k) & ((1 << (64 - k)) - 1)
        z = i + (-7046029254386353131)            # 0x9E3779B97F4A7C15
        z = (z ^ shr(z, 30)) * (-4658895280553007687)   # 0xBF58476D1CE4E5B9
        z = (z ^ shr(z, 27)) * (-7723592293110705685)   # 0x94D049BB133111EB
        z = z ^ shr(z, 31)
        return z

    def umod(z, m):  # unsigned 64-bit z mod m from the signed image
        r = (shr1(z) % m) * 2 + (z & 1)
        return r % m

    def shr1(z):
        return (z >> 1) & 0x7FFFFFFFFFFFFFFF

    for lo in range(0, rows, piece):
        m = min(piece, rows - lo)
        i = torch.arange(lo, lo + m, dtype=torch.int64, device=dev)
        k = umod(splitmix(i), n_keys)
        v = umod(splitmix(i + (1 << 40)), 1001)
        want_sum.scatter_add_(0, k, v)
        want_cnt.scatter_add_(0, k, torch.ones_like(k))
        first.scatter_reduce_(0, k, i, reduce="amin")
        torch.cuda.synchronize()
        for fid, arr in ((tpch.K_FIELD, k), (tpch.V_FIELD, v)):
            if fid not in cols:
                cols[fid] = gpu.DeviceColumn(ctx, gpu.logical_field_id(2, fid), HostColumn(fid, DataType.Int64, np.zeros(0, np.int64)))
                cols[fid].reserve(rows)
                dt.columns[fid] = cols[fid]
            cols[fid].append_raw(arr.data_ptr(), m, lo)
            cols[fid].flush()
        del i, k, v
    dt.n_rows = rows
    dt.seal()
    # the generator against its numpy statement (first rows)
    probe = np.arange(0, 4096, dtype=np.uint64)
    k_np = (tpch.splitmix64(probe) % np.uint64(n_keys)).astype(np.int64)
    check(np.array_equal(cols[tpch.K_FIELD].read(0, 4096), k_np), "configs[3]: the device key generator disagrees with numpy SplitMix64")
    out = {"workload": f"GROUP BY over {n_keys} distinct Int64 keys (key = SplitMix64(i) mod {n_keys}), SUM + COUNT, {rows} rows (BASELINE.json configs[3])",
           "rows": rows, "keys": n_keys, "unit": UNIT, "verified": True}
    try:
        modes = (("partitioned", 1),) if rows > (1 << 28) else (("partitioned", 2), ("per_row", 0))
        for name, mode in modes:
            ctx.set_partitioning(mode)
            hagg = gpu.Aggregation(dt, tpch.highcard_aggregates(), (tpch.K_FIELD,), cardinality_hint=n_keys)
            ms = []
            for i in range(1 + args.steps):
                hagg.reset()
                hagg.run(None, False, 0, rows)
                groups = hagg.group_count()
                if i:
                    ms.append(hagg.run_info().last_kernel_ms)
            hinfo = hagg.run_info()
            vals, keys, n_groups = hagg.finalize_numpy(groups)
            kk = torch.from_numpy(keys["bits"][:, 0].astype(np.int64)).to(dev)
            got_sum = torch.from_numpy(vals["lo"][:, 0].astype(np.int64)).to(dev)
            got_cnt = torch.from_numpy(vals["lo"][:, 1].astype(np.int64)).to(dev)
            check(n_groups == int((want_cnt > 0).sum().item()), f"configs[3] {name}: {n_groups} groups, expected {int((want_cnt > 0).sum().item())}")
            check(bool((vals["valid"] == 1).all()) and bool((keys["valid"] == 1).all()), f"configs[3] {name}: NULL cells in the result")
            check(bool(torch.equal(want_sum[kk], got_sum)) and bool(torch.equal(want_cnt[kk], got_cnt)), f"configs[3] {name}: per-key SUM / COUNT differ from the scatter-add")
            check(int(torch.unique(kk).numel()) == n_groups, f"configs[3] {name}: duplicate keys in the result")
            order = first[kk]
            check(bool((order[1:] > order[:-1]).all().item()), f"configs[3] {name}: groups are not in first-appearance order")
            if dump is not None:
                # the same groups from run to run: a seeded choice of positions in key order
                by_key = np.argsort(keys["bits"][:, 0].astype(np.int64), kind="stable")
                pick = by_key[np.sort(np.random.default_rng(0).choice(n_groups, min(n_groups, DUMP_GROUPS), replace=False))]
                dump[f"highcard_{name}_keys"] = keys["bits"][pick, :1].astype(np.int64).astype(np.float64)
                dump[f"highcard_{name}_values"] = vals["lo"][pick].astype(np.int64).astype(np.float64)
            hagg.destroy()
            del kk, got_sum, got_cnt, order
            kms_hc = statistics.mean(ms)
            out[name] = {"kernel_ms": kms_hc, "value": rows / (kms_hc * 1e-3), "groups": n_groups, "partitions": hinfo.partitions,
                         "launches_per_run": hinfo.kernel_launches, "algorithmic_bytes_per_row": 16,
                         "algorithmic_gbs": 16 * rows / (kms_hc * 1e-3) / 1e9}
    finally:
        ctx.set_partitioning(1)
        dt.destroy()
    return out


def cpu_baseline_subprocess():
    """The CPU leg runs in its own process (the product process never maps the oracle library)."""
    try:
        out = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "cpu-baseline"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL,
                             text=True, timeout=600)
        return json.loads(out.stdout.strip().splitlines()[-1])
    except Exception as e:
        return {"value": None, "unit": UNIT, "cores": os.cpu_count() or 1, "kind": "port", "sample": f"CPU baseline leg failed: {e!r}"}


def cpu_baseline(seed: int = 6, target_seconds: float = 6.0):
    """The reference-shaped CPU path (oracle port of the Rust code: one scan per predicate leaf -> bitmaps -> gather in
    64 K windows -> arrow-style temporaries -> scalar accumulators) on a bounded sample, two ways (BASELINE.md section 3):
    (i) one thread, as the reference runs this path; (ii) the leaf scans on all host threads (the Rayon-equivalent)."""
    from oracle import oracle
    cores = os.cpu_count() or 1
    probe = 1_000_000
    t, _ = tpch.lineitem_table(probe, seed=seed, with_q1=False)
    t0 = time.perf_counter()
    oracle.aggregate(t, tpch.q6_filter(), tpch.q6_aggregates(), n_threads=cores)
    rate = probe / (time.perf_counter() - t0)
    n = int(min(max(rate * target_seconds, probe), 24_000_000))
    t, _ = tpch.lineitem_table(n, seed=seed, with_q1=False)

    def best_of(threads, reps):
        best = None
        for _ in range(reps):
            t0 = time.perf_counter()
            oracle.aggregate(t, tpch.q6_filter(), tpch.q6_aggregates(), n_threads=threads)
            dt = time.perf_counter() - t0
            best = dt if best is None else min(best, dt)
        return best

    multi = best_of(cores, 2)
    n1 = min(n, 4_000_000)
    t1 = t if n1 == n else tpch.lineitem_table(n1, seed=seed, with_q1=False)[0]
    t_save, t = t, t1
    single = best_of(1, 1)
    t = t_save
    return {"value": n / multi, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"TPC-H Q6 over the first {n} rows of the same synthetic lineitem (seed {seed}); best of 2; oracle/llkv_oracle.c, "
                      f"leaf scans on {cores} threads, the rest single-threaded like the reference",
            "single_thread": {"value": n1 / single, "unit": UNIT, "cores": 1, "kind": "port",
                              "sample": f"the same path on one thread (how the reference runs it), first {n1} rows"}}


def run_reference(args):
    """--impl reference: the reference's own CPU path cannot be built here (pure Rust, no cargo/rustc in the image), so
    this arm times the oracle port of it on the host cores."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import oracle
    cores = os.cpu_count() or 1
    n = args.rows or 4_000_000
    t, _ = tpch.lineitem_table(n, seed=6, with_q1=False)
    want = tpch.expected_q6(tpch.lineitem_arrays(n, 6, False))
    for _ in range(args.warmup):
        oracle.aggregate(t, tpch.q6_filter(), tpch.q6_aggregates(), n_threads=cores)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        got = oracle.aggregate(t, tpch.q6_filter(), tpch.q6_aggregates(), n_threads=cores)
    dt = time.perf_counter() - t0
    v = n * args.steps / dt
    sample = f"each step = TPC-H Q6 over a {n}-row sample of the synthetic lineitem (seed 6)"
    emit({
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": int(os.environ.get("WORLD_SIZE", "1")), "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "i128/i64 (Decimal128, Date32)", "data": "synthetic", "verified": bool(got[0][1][0].value == want),
        "decimal_contract": DECIMAL_CONTRACT,
        "config": {"workload": f"TPC-H Q6 on synthetic lineitem SF{args.sf:g} — bounded CPU sample: {sample}"},
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    })


# stdout carries exactly one JSON line.  Native libraries print there too (NCCL's "NCCL version ..." banner is a plain
# printf when NCCL_DEBUG=VERSION), so file descriptor 1 points at stderr while the benchmark runs and the JSON line goes to
# the real stdout.
_REAL_STDOUT = None


def emit(obj):
    data = (json.dumps(obj) + "\n").encode()
    sys.stdout.flush()
    if _REAL_STDOUT is None:
        os.write(1, data)
    else:
        os.write(_REAL_STDOUT, data)


def host_narrow_isa():
    """Widest form of the host narrowing loops this CPU runs (upload.cpp dispatches to it), through the library's test hook."""
    try:
        import ctypes
        from llkv_b200 import gpu
        fn = ctypes.CDLL(gpu.LIB_PATH).llkv_internal_narrow_d128
        fn.restype = ctypes.c_int
        fn.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint64]
        return {1: "sse2", 2: "avx2", 3: "avx512"}[max(i for i in (1, 2, 3) if fn(4, i, None, None, 0) >= 0)]
    except Exception as e:  # (a label only: never fail the bench over it)
        return f"unknown ({e!r})"


def main():
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "cpu-baseline"])
    ap.add_argument("--sf", type=float, default=10.0)
    ap.add_argument("--rows", type=int, default=0, help="override the row count per GPU (smoke runs)")
    ap.add_argument("--highcard-rows", type=int, default=0, help="override the row count of the configs[3] leg")
    ap.add_argument("--upload-threads", type=int, default=-1, help="host workers narrowing Decimal128 chunks before the DMA (0 = off)")
    ap.add_argument("--dma-share", type=int, default=-1, help="percent of the Decimal128 bytes of the end-to-end upload that take the copy engine unnarrowed (-1 = from the worker count)")
    ap.add_argument("--no-q1", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-highcard", action="store_true")
    ap.add_argument("--no-configs", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="after the timed steps, write what each timed leg returned in its last step as DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    elif args.impl == "cpu-baseline":
        emit(cpu_baseline())
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
