# Where the fixed cost of one query step goes (execute + finalize, replayed as a CUDA graph), on the shapes bench.py times:
# Q6 and Q1+MVCC (hint 4) on lineitem SF10, and configs[0] (Int64 BETWEEN + SUM over 10 M rows, no MVCC).
#
#   python tools/exp_step.py [steps] [--trace DIR]
#
# Without --trace: host time per step over `steps` replayed steps (default 400), split into execute and finalize, against
# the scan's own time (CUDA events, run_info().last_kernel_ms).  With --trace: a torch.profiler run with CUDA activities
# over 20 replayed steps of each leg; prints every device node of a step (kernels, copies, memsets) with its duration and
# the idle gap before it, and writes the Chrome trace under DIR.  Run the two separately: tracing slows the host.
import json
import os
import statistics
import subprocess
import sys
import time

GAP_US = 8.0  # idle device time that separates two steps in a trace

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [os.path.join(ROOT, "rust-llkv_b200"), ROOT]
import numpy as np  # noqa: E402

from llkv_b200 import gpu, tpch  # noqa: E402


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                              text=True, timeout=30).stdout.strip()
    except Exception as e:  # (the numbers below still stand; the card is then unknown)
        return f"unknown ({e})"


def legs(ctx):
    n = tpch.lineitem_rows(10)
    t, snap = tpch.lineitem_table(n, seed=6, with_q1=True, with_mvcc=True)
    li = gpu.DeviceTable.from_host(ctx, t, chunk_rows=1 << 20)
    del t
    c0, _ = tpch.int64_table(10_000_000, seed=1, table_id=3)
    x = c0.columns[tpch.X_FIELD].values
    lo, hi = (int(v) for v in np.percentile(x[:1_000_000], [25, 75]).astype(np.int64))
    t0 = gpu.DeviceTable.from_host(ctx, c0, chunk_rows=1 << 20)
    return [li, t0], [
        ("q6", li, tpch.q6_filter(), tpch.q6_aggregates(), (), None, 0, 1),
        ("q1_mvcc", li, tpch.q1_filter(), tpch.q1_aggregates(), tpch.Q1_GROUP_BY, snap, 4, 64),
        ("config0", t0, tpch.between_filter(tpch.X_FIELD, lo, hi), tpch.sum_int64(tpch.X_FIELD), (), None, 0, 1),
    ]


def prepare(ctx, leg):
    name, dt, flt, specs, keys, snap, hint, cap = leg
    prog = gpu.Program(ctx, flt)
    dt.set_snapshot(snap)
    agg = gpu.Aggregation(dt, specs, keys, cardinality_hint=hint)
    for _ in range(6):  # compile, specialise, capture
        agg.execute(prog, snap is not None)
        agg.finalize_raw(cap)
    ctx.synchronize()
    return prog, agg


def time_steps(ctx, leg, steps):
    name, dt, flt, specs, keys, snap, hint, cap = leg
    prog, agg = prepare(ctx, leg)
    ex, fi, kms = [], [], []
    for _ in range(steps):
        t0 = time.perf_counter()
        agg.execute(prog, snap is not None)
        t1 = time.perf_counter()
        agg.finalize_raw(cap)
        t2 = time.perf_counter()
        ex.append((t1 - t0) * 1e6)
        fi.append((t2 - t1) * 1e6)
        kms.append(agg.run_info().last_kernel_ms * 1e3)
    info = agg.run_info()
    agg.destroy()
    prog.destroy()
    step = [a + b for a, b in zip(ex, fi)]
    med = statistics.median
    return {"leg": name, "steps": steps, "graph_replays": info.graph_replays, "execute_us": med(ex), "finalize_us": med(fi),
            "step_us": med(step), "kernel_us": med(kms), "step_minus_kernel_us": med([s - k for s, k in zip(step, kms)]),
            "step_mean_us": statistics.mean(step)}


def trace_steps(ctx, leg, out_dir, steps=20):
    import torch
    from torch.profiler import ProfilerActivity, profile
    name, dt, flt, specs, keys, snap, hint, cap = leg
    prog, agg = prepare(ctx, leg)
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        for _ in range(steps):
            agg.execute(prog, snap is not None)
            agg.finalize_raw(cap)
        ctx.synchronize()
    agg.destroy()
    prog.destroy()
    path = os.path.join(out_dir, f"exp_step_{name}.json")
    prof.export_chrome_trace(path)
    ev = json.load(open(path))
    ev = ev["traceEvents"] if isinstance(ev, dict) else ev
    dev = sorted((e for e in ev if e.get("ph") == "X" and e.get("cat") in ("kernel", "gpu_memcpy", "gpu_memset")), key=lambda e: e["ts"])
    # a step's nodes run back to back on the device; the host's finalize and the next launch call leave a longer idle gap
    steps_nodes, cur = [], []
    for e in dev:
        if cur and e["ts"] - (cur[-1]["ts"] + cur[-1]["dur"]) > GAP_US:
            steps_nodes.append(cur)
            cur = []
        cur.append(e)
    if cur:
        steps_nodes.append(cur)
    is_scan = lambda e: "lean" in e["name"] or "scan_kernel" in e["name"]
    steps_nodes = [s for s in steps_nodes[1:] if sum(map(is_scan, s)) == 1]  # (the first: profiler warm-up)
    rows = {}
    for nodes in steps_nodes:
        for k, e in enumerate(nodes):
            gap = e["ts"] - (nodes[k - 1]["ts"] + nodes[k - 1]["dur"]) if k else 0.0
            r = rows.setdefault(f"{k:02d} {e['cat']}: {e['name'][:60]}", [[], []])
            r[0].append(e["dur"])
            r[1].append(gap)
    med = statistics.median
    table = [{"node": k, "dur_us": med(v[0]), "gap_before_us": med(v[1]), "seen": len(v[0])} for k, v in sorted(rows.items())]
    span = [n[-1]["ts"] + n[-1]["dur"] - n[0]["ts"] for n in steps_nodes]
    scan = [sum(e["dur"] for e in n if is_scan(e)) for n in steps_nodes]
    return {"leg": name, "steps_traced": len(steps_nodes), "device_span_us": med(span) if span else None,
            "span_minus_scan_us": med([a - b for a, b in zip(span, scan)]) if span else None, "nodes": table, "trace": path}


def main():
    args = [a for a in sys.argv[1:]]
    out_dir = None
    if "--trace" in args:
        i = args.index("--trace")
        out_dir = args[i + 1]
        del args[i:i + 2]
        os.makedirs(out_dir, exist_ok=True)
    steps = int(args[0]) if args else 400
    print(json.dumps({"card": card()}), flush=True)
    if out_dir:
        import torch
        torch.cuda.init()
    ctx = gpu.Context(0)
    ctx.set_timing(True)
    tables, ls = legs(ctx)
    try:
        for leg in ls:
            r = trace_steps(ctx, leg, out_dir) if out_dir else time_steps(ctx, leg, steps)
            print(json.dumps(r), flush=True)
    finally:
        for t in tables:
            t.destroy()
        ctx.close()


if __name__ == "__main__":
    main()
