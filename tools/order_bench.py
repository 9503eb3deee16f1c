#!/usr/bin/env python
"""ORDER BY / LIMIT on the GPU, measured in one run (writes JSON lines to --out and stdout):

  * Q3 at --sf (default 10; its lineitem, orders and customer columns are far above the 126 MB L2), ms per step, three
    plans alternated step by step: as the fixtures have it (no order), `revenue DESC, o_orderdate LIMIT 10`, and the same
    ORDER BY without a limit.  Typed outputs on, as bench.py runs it.  A step is vdl_plan_run (launches, the result copy
    and the wait), timed with CUDA events on the context's stream; warm-up steps are excluded.  The ordered results are
    checked against the unordered one ordered by numpy (np.lexsort, stable).
  * vdl_op_order alone over 1e6 / 1e7 / 1e8 rows, 1 and 3 keys, limit -1 and 10, and vdl_op_partition (the stable LSD radix
    sort it shares its passes with) on a 38-bit key at the same sizes.  1e6 rows of keys (8-20 MB) fit L2; 1e7 and 1e8 do
    not.

The device name and its power limit are recorded beside the numbers."""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
sys.path.insert(0, ROOT)


def device_info() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    name, power, clock = (q.stdout.strip().split(", ") + ["?", "?", "?"])[:3]
    return {"device": name, "power_limit": power, "max_sm_clock": clock}


def timed(ctx, ext, fn, reps: int, warmup: int = 1) -> list:
    """Per-call milliseconds from CUDA events on the context's stream around `fn` (which ends in a synchronise)."""
    import torch
    for _ in range(warmup):
        fn()
    ctx.synchronize()
    out = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(ext)
        fn()
        b.record(ext)
        ctx.synchronize()
        out.append(a.elapsed_time(b))
    return out


def stats(ms: list) -> dict:
    return {"ms_median": round(float(np.median(ms)), 4), "ms_min": round(float(min(ms)), 4), "ms_mean": round(float(np.mean(ms)), 4), "reps": len(ms)}


def q3_steps(ctx, ext, sf: float, steps: int, warmup: int, emit):
    from mplan2vdl_b200 import tpch
    from mplan2vdl_b200.meta import builtin_catalog
    from mplan2vdl_b200.executor import order_keys
    import torch
    cat = builtin_catalog()
    text = tpch.plan_text("q03.vdl")
    t0 = time.perf_counter()
    tpch.load_synthetic(ctx, cat, tpch.plan_columns(text), sf)
    keys = [("revenue", True), ("o_orderdate", False)]
    variants = {"no_order": None, "order_limit10": (keys, 10), "order_full": (keys, None)}
    plans = {}
    for name, o in variants.items():
        p = ctx.plan(text)
        p.set_typed_outputs(True)
        if o:
            p.set_order(*o)
        plans[name] = p
    results, ms = {}, {k: [] for k in plans}
    for _ in range(warmup):
        for name, p in plans.items():
            p.execute()
    ctx.synchronize()
    for _ in range(steps):
        for name, p in plans.items():            # alternated: the three see the same state of the machine
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(ext)
            p.execute()
            b.record(ext)
            ctx.synchronize()
            ms[name].append(a.elapsed_time(b))
    for name, p in plans.items():
        results[name] = {k: np.asarray(v, np.int64) for k, v in p.outputs().items()}
    plain = results["no_order"]
    names = list(plain)
    idx, desc = order_keys(names, keys)
    cols = [~plain[names[i]] if d else plain[names[i]] for i, d in zip(idx, desc)]
    perm = np.lexsort(cols[::-1])
    checks = {}
    for name, lim in (("order_limit10", 10), ("order_full", None)):
        p = perm if lim is None else perm[:lim]
        checks[name] = all(np.array_equal(results[name][k], plain[k][p]) for k in names)
    rows = len(plain[names[0]])
    out_bytes = {name: sum(v.nbytes for v in r.values()) for name, r in results.items()}
    for name in plans:
        emit({"bench": "q03_step", "sf": sf, "variant": name, "result_rows": len(results[name][names[0]]), "rows_unordered": rows,
              "result_bytes_host": out_bytes[name], "matches_reference": checks.get(name, True), **stats(ms[name])})
    for p in plans.values():
        p.close()
    for c in tpch.plan_columns(text):
        ctx.drop_column(c)
    return time.perf_counter() - t0


def op_bench(ctx, ext, sizes, reps: int, emit):
    rng = np.random.default_rng(1)
    for n in sizes:
        k38 = rng.integers(0, 1 << 38, n, dtype=np.int64)
        h38 = ctx.upload_column("ob.k38", k38)
        k1 = ctx.upload_column("ob.k1", rng.integers(0, 1 << 12, n, dtype=np.int64).astype(np.int32))
        k2 = ctx.upload_column("ob.k2", rng.integers(-(1 << 29), 1 << 29, n, dtype=np.int64))
        k3 = ctx.upload_column("ob.k3", rng.integers(0, 1 << 20, n, dtype=np.int64).astype(np.int32))
        for nkeys, (handles, desc, bits) in {1: ([h38], [True], 38), 3: ([k1, k2, k3], [False, True, False], 12 + 30 + 20)}.items():
            for limit in (None, 10):
                def run():
                    v = ctx.op_order(handles, desc, limit)
                    ctx.synchronize()
                    ctx.free(v)
                ms = timed(ctx, ext, run, reps)
                med = float(np.median(ms))
                emit({"bench": "op_order", "rows": n, "keys": nkeys, "packed_bits": bits, "limit": -1 if limit is None else limit,
                      "rows_per_s": round(n / (med / 1e3)), **stats(ms)})
            if n <= 10_000_000:             # correctness of the limited path at this size, against numpy
                v = ctx.op_order(handles, desc, 10)
                got = ctx.download(v)
                ctx.free(v)
                host = [ctx.download(h) for h in handles]
                cols = [~x if d else x for x, d in zip(host, desc)]
                assert np.array_equal(got, np.lexsort(cols[::-1])[:10]), (n, nkeys)

        def part():
            v = ctx.op_partition(h38, 0, 1, (1 << 38) - 1)
            ctx.synchronize()
            ctx.free(v)
        ms = timed(ctx, ext, part, reps)
        emit({"bench": "op_partition", "rows": n, "key_bits": 38, "rows_per_s": round(n / (float(np.median(ms)) / 1e3)), **stats(ms)})
        for c in ("ob.k38", "ob.k1", "ob.k2", "ob.k3"):
            ctx.drop_column(c)


def main() -> int:
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--sf", type=float, default=10.0)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--sizes", default="1000000,10000000,100000000")
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("order_bench.py: no CUDA device (the measurements are of the GPU)")
    from mplan2vdl_b200.executor import Context
    lines = []

    def emit(rec):
        rec = {**info, **rec}
        lines.append(rec)
        print(json.dumps(rec), flush=True)
    info = device_info()
    ctx = Context(0)
    ext = torch.cuda.ExternalStream(ctx.stream, device=0)
    q3_steps(ctx, ext, args.sf, args.steps, args.warmup, emit)
    op_bench(ctx, ext, [int(s) for s in args.sizes.split(",")], args.reps, emit)
    ctx.close()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("".join(json.dumps(r) + "\n" for r in lines))
    return 0


if __name__ == "__main__":
    sys.exit(main())
