#!/usr/bin/env python
"""ORDER BY over strings on the GPU, measured in one run (writes JSON lines to --out and stdout):

  * vdl_op_collate alone at 1e4 .. 1e7 rows over four heaps: the 3 l_returnflag codes, the 150 p_type strings, the 16,384
    p_name strings and the ~400 k s_name codes (int64 data drawn uniformly from the heap's entries), beside vdl_op_order
    on one int64 key of the same n.  Per call, CUDA events on the context's stream, warm-up excluded.
  * Q1, Q9 and Q16 at --sf (default 10), ms per step, two plans alternated step by step: as the fixtures have them (no
    order) and with TPC-H's ORDER BY on the keys' strings (tpch_queries.COLLATED_ORDER, tpch.collation_heaps), typed
    outputs on as bench.py runs them.  A step is vdl_plan_run (launches, the result copy and the wait).  The ordered
    result is checked against the unordered one sorted on the host by the keys' strings.

The device name and its power limit are recorded beside the numbers."""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from order_bench import device_info, stats, timed  # noqa: E402


def heaps(cat):
    """name -> (heap bytes, origin, the values a row may hold)"""
    from mplan2vdl_b200 import synth
    out = {}
    for name, col in (("l_returnflag_3", "lineitem.l_returnflag"), ("s_name_400k", "supplier.s_name")):
        heap, origin = synth.code_heap(cat, col)
        spec = synth.column_spec(cat, col, 10)
        out[name] = (heap, origin, spec.vmin + spec.stride * np.arange(spec.p0, dtype=np.int64))
    for name, col in (("p_type_150", "part.p_type"), ("p_name_16k", "part.p_name")):
        heap, offs = synth.string_heap(cat, col)
        out[name] = (heap, 0, offs)
    return out


def op_bench(ctx, ext, cat, sizes, reps: int, emit):
    rng = np.random.default_rng(3)
    for hname, (heap, origin, values) in heaps(cat).items():
        h = ctx.upload_column("cb.heap", heap)
        for n in sizes:
            d = ctx.upload_column("cb.data", values[rng.integers(0, len(values), n)])

            def run():
                v = ctx.op_collate(d, h, origin)
                ctx.synchronize()
                ctx.free(v)
            ms = timed(ctx, ext, run, reps, warmup=2)
            distinct = len(np.unique(ctx.download(d)))
            emit({"bench": "op_collate", "heap": hname, "heap_entries": len(values), "heap_bytes": len(heap), "rows": n,
                  "distinct_strings": distinct, "rows_per_s": round(n / (float(np.median(ms)) / 1e3)), **stats(ms)})
            ctx.drop_column("cb.data")
        ctx.drop_column("cb.heap")
    for n in sizes:
        k = ctx.upload_column("cb.key", rng.integers(-(1 << 62), 1 << 62, n, dtype=np.int64))

        def order():
            v = ctx.op_order([k], [False], None)
            ctx.synchronize()
            ctx.free(v)
        ms = timed(ctx, ext, order, reps, warmup=2)
        emit({"bench": "op_order", "keys": 1, "rows": n, "rows_per_s": round(n / (float(np.median(ms)) / 1e3)), **stats(ms)})
        ctx.drop_column("cb.key")


def host_order(cat, text, plain: dict, keys) -> np.ndarray:
    """The permutation that sorts `plain` by `keys` on the host: string keys by their bytes (ascending), numeric keys by
    value, ties in row order (Python's sort is stable)."""
    from mplan2vdl_b200 import synth, tpch
    from mplan2vdl_b200.executor import order_keys
    names = list(plain)
    idx, desc = order_keys(names, keys)
    recipes = tpch.collation_recipes(cat, text, keys)
    cols = []
    for (name, _d), i, d in zip(keys, idx, desc):
        vals = plain[names[i]]
        if name in recipes:
            assert not d, "string keys are ascending here"
            kind, q = recipes[name]
            heap, origin = (synth.string_heap(cat, q)[0], 0) if kind == "pool" else synth.code_heap(cat, q)
            hb = heap.tobytes()
            cols.append([hb[int(v) - origin:hb.index(b"\0", int(v) - origin)] for v in vals])
        else:
            cols.append([-int(v) if d else int(v) for v in vals])
    n = len(plain[names[0]])
    return np.asarray(sorted(range(n), key=lambda r: tuple(c[r] for c in cols)), np.int64)


def plan_steps(ctx, ext, cat, q: str, sf: float, steps: int, warmup: int, emit):
    import torch
    from mplan2vdl_b200 import tpch
    from mplan2vdl_b200.tpch_queries import COLLATED_ORDER
    text = tpch.plan_text(q + ".vdl")
    cols = tpch.plan_columns(text)
    tpch.load_synthetic(ctx, cat, cols, sf)
    keys, limit = COLLATED_ORDER[q]
    plans = {"no_order": ctx.plan(text), "collated": ctx.plan(text)}
    for p in plans.values():
        p.set_typed_outputs(True)
    plans["collated"].set_order(keys, limit, tpch.collation_heaps(ctx, cat, text, keys))
    ms = {k: [] for k in plans}
    for _ in range(warmup):
        for p in plans.values():
            p.execute()
    ctx.synchronize()
    for _ in range(steps):
        for name, p in plans.items():            # alternated: both see the same state of the machine
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(ext)
            p.execute()
            b.record(ext)
            ctx.synchronize()
            ms[name].append(a.elapsed_time(b))
    res = {name: {k: np.asarray(v, np.int64) for k, v in p.outputs().items()} for name, p in plans.items()}
    plain = res["no_order"]
    perm = host_order(cat, text, plain, keys)
    ok = all(np.array_equal(res["collated"][k], plain[k][perm]) for k in plain)
    rows = len(next(iter(plain.values())))
    for name in plans:
        emit({"bench": "plan_step", "plan": q, "sf": sf, "variant": name, "result_rows": rows,
              "matches_reference": ok if name == "collated" else True, **stats(ms[name])})
    for p in plans.values():
        p.close()
    for c in cols:
        ctx.drop_column(c)


def main() -> int:
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--sf", type=float, default=10.0)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--sizes", default="10000,100000,1000000,10000000")
    ap.add_argument("--plans", default="q01,q09,q16")
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("collate_bench.py: no CUDA device (the measurements are of the GPU)")
    from mplan2vdl_b200.executor import Context
    from mplan2vdl_b200.meta import builtin_catalog
    lines = []

    def emit(rec):
        rec = {**info, **rec}
        lines.append(rec)
        print(json.dumps(rec), flush=True)
    info = device_info()
    cat = builtin_catalog()
    ctx = Context(0)
    ext = torch.cuda.ExternalStream(ctx.stream, device=0)
    t0 = time.perf_counter()
    op_bench(ctx, ext, cat, [int(s) for s in args.sizes.split(",")], args.reps, emit)
    for q in filter(None, args.plans.split(",")):
        plan_steps(ctx, ext, cat, q, args.sf, args.steps, args.warmup, emit)
    ctx.close()
    print(f"collate_bench: {time.perf_counter() - t0:.1f} s", file=sys.stderr)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("".join(json.dumps(r) + "\n" for r in lines))
    return 0


if __name__ == "__main__":
    sys.exit(main())
