#!/usr/bin/env python
"""bench.py -- headline benchmark: the mplan2vdl-emitted TPC-H Q6 plan over synthetic SF100 lineitem
columns resident in HBM (BASELINE.json north_star), executed by libvdl_cuda.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--query q06|q01] [--sf 100] [--dump-outputs DIR]

One "step" = one execution of the plan over the whole (sharded) table: ONE launch of the fused scan-fold
kernel per GPU, whose last thread block [exchanges the partial tables with the other GPUs through peer memory
for N>1,] finalizes and writes the result to mapped host memory, and the host's wait for it.  Prints ONE JSON line (rank 0).  See DESIGN.md section 6 for what each
field means and how the roofline / cpu_baseline / e2e numbers are obtained.
"""
from __future__ import annotations

import argparse
import json
import os
import re
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

QUERIES = {
    # plan file, algorithmic bytes per lineitem row for the single-table plans (SURVEY.md section 8 d: distinct base
    # columns x stored width); for the join plans the bytes are summed over every table the plan loads
    "q06": ("q06.vdl", 28),
    "q01": ("q01.vdl", 52),
    "q03": ("q03.vdl", None),
    "q05": ("q05.vdl", None),
    "q12": ("q12.vdl", None),
    "q19": ("q19.vdl", None),
}


def algorithmic_bytes(cat, names, rows_of, rows_fact_here):
    """Sum over the distinct base columns the plan Loads of rows x stored width; pkey pseudo-columns only give a length."""
    from mplan2vdl_b200 import tpch
    total = 0
    for n in names:
        t, c = n.split(".", 1)
        if c == cat.tables[t].pkey_name:
            continue
        total += (rows_fact_here if t == tpch.FACT_TABLE else rows_of(t)) * cat.column(n).width
    return total
FALLBACK_HBM_GBS = 6650.0   # B200_PROFILING.md fallback, used only when MEASURED_PEAKS.json is absent


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    except Exception:
        return FALLBACK_HBM_GBS, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms during the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device: int):
        self.device, self.proc, self.path = device, None, None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.device), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200"], stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self) -> dict:
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if not self.proc:
            return out
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        try:
            for line in open(self.path):
                f = [x.strip() for x in line.split(",")]
                if len(f) < 9:
                    continue
                try:
                    sm.append(float(f[1])); mx.append(float(f[2]))
                except ValueError:
                    continue
                for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
            os.unlink(self.path)
        except Exception:
            pass
        if sm:
            out = {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}
        return out


def host_threads() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def cpu_oracle_rate(cat, query: str, sf: float, target_seconds: float = 12.0, max_rows: int = 59_986_052, steps: int = 1):
    """Time the CPU oracle (kind "port": the reference ships no executor) on a bounded sample of the same workload:
    the first `rows` lineitem rows of the same synthetic table.  Returns (rows/s, sample rows, threads, seconds list)."""
    max_rows = min(max_rows, CPU_ARM_MAX_ROWS)
    from mplan2vdl_b200 import synth, tpch
    from oracle.oracle import Oracle, gen_column
    text = tpch.plan_text(QUERIES[query][0])
    names = tpch.plan_columns(text)
    seed = synth.seed_for(sf)
    threads = host_threads()        # set explicitly: torchrun exports OMP_NUM_THREADS=1 to its workers

    def run(rows, reps):
        orc = Oracle()
        for n in names:
            orc.bind(n, gen_column(synth.column_spec(cat, n, sf), rows, 0, seed, threads))
        secs = []
        for _ in range(reps):
            orc.run(text, threads)
            secs.append(orc.seconds)
        return secs

    probe_rows = 2_000_000
    t = min(run(probe_rows, 2))
    rows = int(min(max_rows, max(probe_rows, probe_rows * target_seconds / max(t, 1e-6) / max(steps, 1))))
    if steps == 1:       # bounded sample, repeated until about target_seconds of CPU work have been timed
        steps = int(max(1, min(40, target_seconds / max(t * rows / probe_rows, 1e-6))))
    secs = run(rows, steps)
    return rows / statistics.median(secs), rows, threads, secs


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path.  orm011/mplan2vdl ships no executor
    (SURVEY.md section 0), so this arm times the CPU oracle -- the restatement of the Voodoo op semantics -- with all
    host threads on a bounded sample of the same workload."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from mplan2vdl_b200.meta import builtin_catalog
    cat = builtin_catalog()
    total = max(1, args.steps + args.warmup)
    rate, rows, threads, secs = cpu_oracle_rate(cat, args.query, args.sf, target_seconds=60.0, steps=total)
    timed = secs[args.warmup:] or secs
    ms = 1e3 * statistics.mean(timed)
    value = rows / (ms / 1e3)
    sample = f"first {rows} lineitem rows of the synthetic SF{args.sf:g} table, {len(timed)} timed runs of the op-at-a-time CPU oracle"
    line = {
        "impl": "reference", "metric": f"tpch_{args.query}_rows_per_s", "value": value, "unit": "rows/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "int64", "data": "synthetic",
        "config": workload_config(args),
        "cpu_baseline": {"value": value, "unit": "rows/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


L2_BYTES = 126e6
CPU_ARM_MAX_ROWS = 59_986_052


def check_parity(cat, query: str, sf: float, result: dict, chunk_rows: int = 40_000_000) -> dict:
    """BASELINE.md section 3: "parity check ... in the same run".  The CPU oracle over ALL rows of the workload, the fact
    table generated and consumed `chunk_rows` at a time (oracle/chunked.py), compared bit for bit with what the GPU returned."""
    import numpy as np
    from mplan2vdl_b200 import tpch
    from oracle import chunked
    t0 = time.perf_counter()
    text = tpch.plan_text(QUERIES[query][0])
    want, co = chunked.run_chunked(text, cat, sf, chunk_rows=chunk_rows, threads=host_threads())
    bad = [k for k in want if k not in result or not np.array_equal(np.asarray(result[k], dtype=np.int64), want[k])]
    bad += [k for k in result if k not in want]
    return {"status": "exact" if not bad else "MISMATCH", "against": "CPU oracle (oracle/vdl_oracle.c) over the whole table, chunked",
            "rows_checked": co.rows, "outputs_checked": len(want), "values_checked": int(sum(len(v) for v in want.values())),
            "mismatched_outputs": bad, "oracle_seconds": round(co.seconds, 2), "seconds": round(time.perf_counter() - t0, 2)}


DUMP_BYTES = 64 << 20


def dump_outputs(result: dict, out_dir: str, seed: int = 0) -> None:
    """Every result column as <out_dir>/<name>.npy in float64, so that two builds of the project can be compared output
    for output.  Integer results beyond 2**53 (fixed-point sums at large scale factors) are rounded to the nearest double,
    so a difference in their last units does not show.  Past DUMP_BYTES in all, every column keeps the same seeded sample
    of its rows, in row order."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    keep = max(1, (DUMP_BYTES // max(len(result), 1) - 128) // 8)      # 128: the .npy header
    for name, col in result.items():
        col = np.asarray(col)
        if len(col) > keep:
            col = col[np.sort(np.random.default_rng(seed).choice(len(col), keep, replace=False))]
        np.save(os.path.join(out_dir, re.sub(r"[^A-Za-z0-9_.-]", "_", name) + ".npy"), col.astype(np.float64))


def workload_config(args):
    """Identical for both arms (--impl ours / reference): a function of the command line only."""
    from mplan2vdl_b200 import synth, tpch
    from mplan2vdl_b200.meta import builtin_catalog
    cat = builtin_catalog()
    plan, bpr = QUERIES[args.query]
    names = tpch.plan_columns(tpch.plan_text(plan))
    rows_total = synth.table_rows(cat, "lineitem", args.sf)
    total_bytes = algorithmic_bytes(cat, names, lambda t: synth.table_rows(cat, t, args.sf), rows_total)
    return {"workload": f"TPC-H {args.query.upper()} SF{args.sf:g}: plans/{plan} (mplan2vdl Voodoo plan) over synthetic TPC-H columns "
                        "generated to the reference's bounds.csv",
            "lineitem_rows": rows_total, "algorithmic_bytes_per_lineitem_row": bpr, "algorithmic_bytes": total_bytes,
            "results": ("int64 columns" if args.int64_results else
                        "typed: a result column whose every value is a value of a 4-byte column (by provenance) crosses PCIe as int32, the others as int64"),
            "l2": ("inputs far exceed the 126 MB L2; no flush needed between steps" if total_bytes / max(args.gpus, 1) >= 4 * L2_BYTES else
                   "inputs per GPU are within 4x the 126 MB L2: between timed steps a 256 MB buffer is written, then a second 256 MB "
                   "buffer is read so that the flush's dirty lines are written back (both outside the per-step events)"),
            "cpu_arm": f"cpu_baseline / --impl reference time the op-at-a-time CPU oracle on a PREFIX of the same table (at most the first "
                       f"{min(CPU_ARM_MAX_ROWS, rows_total)} of {rows_total} lineitem rows per step) and report rows/s of that prefix: a scan "
                       "extrapolates linearly, but it is a sample, not the whole table",
            "e2e_storage": "e2e = host columns in the executor's narrow storage format (int32 wherever a column's exact min/max fit, e.g. Q6: "
                           "16 instead of 28 bytes per lineitem row on the wire and in HBM); the same measurement with every column in the "
                           "reference's widths (Types.hs:129-140) is reported as e2e_reference_storage; value / roofline use the reference widths",
            "parallelism": f"lineitem row-range sharded over {args.gpus} GPU(s), dimension tables replicated"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--query", default="q06", choices=sorted(QUERIES))
    ap.add_argument("--sf", type=float, default=100)
    ap.add_argument("--e2e-steps", type=int, default=2)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-parity", action="store_true", help="skip the whole-table CPU-oracle check of the result")
    ap.add_argument("--int64-results", action="store_true", help="every result column crosses PCIe as int64 (default: int32 where the values provably fit)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the result of the last timed step to DIR/<output>.npy "
                    "(float64, so integers beyond 2**53, such as Q1's fixed-point sums at SF100, are rounded; a seeded "
                    "sample of the rows when the result exceeds 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs: the reference arm runs on a prefix of the table, its result is not the workload's")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    if args.impl == "reference":
        run_reference(args)
        return

    import numpy as np
    import torch
    import __graft_entry__
    __graft_entry__.build()
    from mplan2vdl_b200 import synth, tpch
    from mplan2vdl_b200.executor import Context
    from mplan2vdl_b200.meta import builtin_catalog

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (libvdl_cuda has no CPU fallback)")
    torch.cuda.set_device(local)

    cat = builtin_catalog()
    plan_file, bytes_per_row = QUERIES[args.query]
    text = tpch.plan_text(plan_file)
    names = tpch.plan_columns(text)
    rows_total = synth.table_rows(cat, "lineitem", args.sf)

    ctx = Context(local)
    info = tpch.load_synthetic(ctx, cat, names, args.sf, rank=rank, world=world)
    rows_here = info["rows"]["lineitem"]
    bytes_here = algorithmic_bytes(cat, names, lambda t: synth.table_rows(cat, t, args.sf), rows_here)
    plan = ctx.plan(text)
    if not args.int64_results:
        plan.set_typed_outputs(True)         # result columns that are values of 4-byte columns travel as int32 (Q3: 28 of 44 MB)
    ext = torch.cuda.ExternalStream(ctx.stream, device=local)
    from mplan2vdl_b200.dist import ShardedPlan
    sharded = ShardedPlan(ctx, plan, rank, world, info["row_base"])
    def step(fetch=True):
        # fetch=False: the C call alone (vdl_plan_run: launches + wait until the results are in the library's pinned host
        # buffers); the arrays are wrapped once, after the loop -- no Python objects are built inside a timed region
        return sharded.step(copy=False, fetch=fetch)

    def barrier():
        ctx.synchronize()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    result = None
    for _ in range(args.warmup):
        result = step()
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    launches0 = ctx.launch_count
    kernel_ms = []
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    flush = bytes_here < 4 * L2_BYTES       # small inputs would be re-read from L2: evict them between steps
    flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device=f"cuda:{local}") if flush else None
    drain_buf = torch.zeros(256 << 20, dtype=torch.uint8, device=f"cuda:{local}") if flush else None
    barrier()
    t0 = time.perf_counter()
    if not flush:
        ev0.record(ext)
        for _ in range(args.steps):
            step(fetch=False)
        ev1.record(ext)
        barrier()
        dev_ms = ev0.elapsed_time(ev1)
        # the dominant kernel's own duration over THESE steps: the library records an event pair around every launch of it
        # (a ring of 64), read here, after the timed region, instead of synchronising on an event every step
        kern_mean, kern_min = plan.kernel_ms_stats(min(args.steps, 64))
        result = plan.outputs(False)
    else:                                   # per-step events; the flush runs between them, on the same stream
        dev_ms = 0.0
        for _ in range(args.steps):
            with torch.cuda.stream(ext):
                flush_buf.fill_(1)          # evicts the inputs ...
                drain_buf.sum()             # ... and reading a second buffer writes the flush's dirty lines back before the
                                            # timed step, so its reads do not share DRAM with 126 MB of write-backs
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(ext)
            step(fetch=False)
            b.record(ext)
            ctx.synchronize()
            dev_ms += a.elapsed_time(b)
            kernel_ms.append(plan.kernel_ms(0) if plan.num_fused else plan.probe_kernel_ms())
        barrier()
        result = plan.outputs(False)
        kern_mean, kern_min = statistics.mean(kernel_ms), min(kernel_ms)
    wall_ms = 1e3 * (time.perf_counter() - t0)
    # the views die with the next step; a sharded-tail plan's result is spread over the ranks: gathered here, outside the timing
    result = sharded.global_result() if sharded.tail_mode else {k: np.array(v, copy=True) for k, v in result.items()}
    launches = ctx.launch_count - launches0
    clocks = sampler.stop() if rank == 0 else {}
    if rank == 0 and args.dump_outputs:
        dump_outputs(result, args.dump_outputs)
    if world > 1:
        t = torch.tensor([dev_ms, kern_mean], dtype=torch.float64, device=f"cuda:{local}")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dev_ms = float(t[0])
    ms_per_step = dev_ms / args.steps
    value = rows_total / (ms_per_step / 1e3)
    fused = plan.num_fused > 0
    pstats = plan.stats()
    probed = pstats["probe_folds"] + pstats["probe_emits"] > 0
    if not fused and not probed:   # op-at-a-time plan: the "kernel" is the whole chain of per-op launches
        kern_mean = kern_min = ms_per_step

    # roofline of the dominant kernel (the fused scan): algorithmic bytes of THIS rank's shard / its mean duration
    peak, peak_kind = measured_peak()
    achieved = bytes_here / (kern_mean / 1e3) / 1e9
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": None,
                "peak_source": f"{peak_kind} copy bandwidth (MEASURED_PEAKS.json)" if peak_kind == "measured" else "fallback 6650 GB/s",
                "kernel": f"fused_scan_fold_kernel<{plan.shape(0)}>" if fused else ("probe_kernel (fused FK-join probe)" if probed else "op-at-a-time plan (all per-op kernels of one step)"),
                "kernel_ms": kern_mean, "kernel_ms_min": kern_min,
                "frac_of_8TBs_spec": achieved / 8000.0, "bytes_per_launch": bytes_here}
    # DRAM bytes ncu counted for one launch of this kernel (profiles/traffic.json, tools/update_traffic.py) -- reported only
    # while the sources that define THIS kernel's device code (mplan2vdl_b200.build.KERNEL_FAMILIES: the fused scan's or the
    # probe's .cu + .cuh files) still hash to what the capture was taken from, so a stale figure cannot ride along
    try:
        from mplan2vdl_b200.build import source_hash
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            tj = json.load(f)
        tr = tj.get("workloads", {}).get(f"{args.query}_sf{args.sf:g}")
        if tr and world == 1:
            fam = tr.get("family", "scan" if plan.num_fused else "probe")
            if tj.get("family_hashes", {}).get(fam) == source_hash(fam):
                roofline["traffic"] = tr["dram_bytes"]
                roofline["traffic_source"] = (f"ncu --set full, profiles/{tj.get('prefix')}_{args.query}_sf{args.sf:g}_dominant_kernel.txt ({tr.get('kernel')}); "
                                              f"the {fam} kernel's sources are unchanged since that capture (hash {source_hash(fam)})")
                # a selective plan (probe kernel) never touches most columns of the rows it rejects: the DRAM bytes ncu
                # counted are then the honest numerator, the all-columns algorithmic figure an upper bound
                roofline["dram_gbs_by_traffic"] = tr["dram_bytes"] / (kern_mean / 1e3) / 1e9
                roofline["frac_by_traffic"] = roofline["dram_gbs_by_traffic"] / peak
            else:
                roofline["traffic_source"] = f"profiles/traffic.json is older than the {fam} kernel's sources (hash differs): not reported"
    except Exception:
        pass

    # end to end through the public API with HOST buffers: H2D of every column + column analysis + (re)prepare + run + D2H of
    # the result, per step.  Two host storage formats, both timed:
    #   reference  every column in the reference's storage model (Types.hs:129-140: decimals / oids / string codes 8 bytes)
    #   narrow     the executor's own format (SURVEY.md App. G11 "narrower storage as a separately reported variant"):
    #              a column whose exact min / max (vdl_column_analyze at load time) fit int32 is kept as int32, on the host
    #              and in HBM -- lossless, the kernels sign-extend; fewer bytes cross PCIe and HBM
    # "e2e" (the headline) is the narrow format with its own byte counts; "e2e_reference_storage" is printed next to it.
    e2e = e2e_ref = None
    if not args.no_e2e:
        handles = [ctx.lookup(n) for n in names]
        widths = [synth.column_spec(cat, n, args.sf).width for n in names]
        nrows = [info["rows"][n.split(".")[0]] for n in names]

        def measure(handles, host, label):
            h2d = sum(b.numel() * b.element_size() for b in host)

            def e2e_step():
                for h, b, nr in zip(handles, host, nrows):
                    ctx.upload_into(h, b.data_ptr(), nr)     # new write generation: the plan re-analyses and re-prepares
                step(fetch=False)
                return plan.outputs(False)

            e2e_step()
            barrier()
            t0 = time.perf_counter()
            for _ in range(args.e2e_steps):
                r2 = e2e_step()
            barrier()
            e2e_s = (time.perf_counter() - t0) / args.e2e_steps
            if world > 1:
                t = torch.tensor([e2e_s], dtype=torch.float64, device=f"cuda:{local}")
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                e2e_s = float(t[0])
            if sharded.tail_mode:
                r2 = sharded.global_result()
            for k in result:
                assert np.array_equal(r2[k], result[k]), f"e2e ({label}) result differs from the device-resident result"
            d2h = sum(v.nbytes for v in result.values())
            return {"value": rows_total / e2e_s, "unit": "rows/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": 1e3 * e2e_s, "steps": args.e2e_steps, "timing": "host wall clock, barrier + synchronize both sides; "
                    "every step uploads all columns from pinned host memory, re-analyses them (min/max), re-prepares the scan and runs the plan",
                    "h2d_gbs": h2d / e2e_s / 1e9, "storage": label,
                    "bytes_per_lineitem_row_on_the_wire": round(sum(b.element_size() for b, n in zip(host, names) if n.startswith("lineitem.")), 1)}

        # exact statistics decide the narrow format (outside the timed region: the storage format is chosen at load time)
        narrow_w = []
        for h, w in zip(handles, widths):
            lo, hi = ctx.analyze(h)
            narrow_w.append(4 if (w == 4 or (lo >= -2**31 and hi < 2**31)) else 8)
        host = []
        for h, w, nr in zip(handles, widths, nrows):
            buf = torch.empty(nr, dtype=torch.int32 if w == 4 else torch.int64, pin_memory=True)
            ctx.download_into(h, buf.data_ptr(), nr)
            host.append(buf)
        e2e_ref = measure(handles, host, "reference (Types.hs widths)")
        host_n = []
        for n, b, w in zip(names, host, narrow_w):
            if b.element_size() == w:
                host_n.append(b)
            else:
                nb = torch.empty(b.numel(), dtype=torch.int32, pin_memory=True)
                nb.copy_(b)                                  # lossless by the statistics above
                host_n.append(nb)
        del host
        handles_n = []
        for n, b, nr in zip(names, host_n, nrows):          # same names, narrower columns: the plan re-binds by name
            ctx.drop_column(n)
            handles_n.append(ctx.alloc_column(n, b.element_size(), nr))
        e2e = measure(handles_n, host_n, "narrow (int32 where the column statistics allow)")
        e2e["kernel_ms"] = plan.kernel_ms(0) if plan.num_fused else plan.probe_kernel_ms()
        e2e["kernel"] = plan.shape(0) if plan.num_fused else "probe"
        del host_n

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        rate, srows, threads, secs = cpu_oracle_rate(cat, args.query, args.sf)
        cpu = {"value": rate, "unit": "rows/s", "cores": threads, "kind": "port",
               "sample": f"first {srows} lineitem rows of the same synthetic table; op-at-a-time CPU oracle (OpenMP), "
                         f"{len(secs)} runs, median {statistics.median(secs):.2f} s, total {sum(secs):.1f} s"}

    parity = None
    if rank == 0 and not args.no_parity:
        parity = check_parity(cat, args.query, args.sf, result)

    if rank == 0:
        line = {
            "metric": f"tpch_{args.query}_rows_per_s", "value": value, "unit": "rows/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "int64", "data": "synthetic", "config": workload_config(args),
            "combine": "none (single GPU)" if world == 1 else (("peer-memory exchange fused into the scan kernel's last thread block (NVLink stores + epoch flags), no collective"
                                                                  if plan.num_fused else "peer-memory exchange kernel after the probe pass (NVLink stores + epoch flags) + finalize, no collective")
                                                                 if sharded.peer_mode else
                                                                 ("sharded tail: every rank keeps the result slice of its rows; one all-gather of a boundary record per rank "
                                                                  "(run count, first / last key, first / last row of each output) merges the groups that straddle shards"
                                                                  if sharded.tail_mode else "NCCL all-gather of the partial tables / survivors + finalize")),
            "roofline": roofline,
            "cpu_baseline": cpu, "e2e": e2e, "e2e_reference_storage": e2e_ref, "gpu_launches": launches, "clocks": clocks,
            "wall_ms_per_step": wall_ms / args.steps, "result": {k: [int(x) for x in v[:8]] for k, v in result.items()},
            "plan": plan.stats(), "parity": parity,
        }
        print(json.dumps(line), flush=True)
    plan.close()
    ctx.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if parity and parity["status"] != "exact":
        raise SystemExit(f"bench.py: PARITY MISMATCH against the CPU oracle in outputs {parity['mismatched_outputs']}")


if __name__ == "__main__":
    main()
