"""`mplan2vdl ... | python -m mplan2vdl_b200 [--sf 1] [--csv]` -- the place of the HTTP Voodoo server in the
reference pipeline (eval_query.sh:18-26): read the Voodoo program mplan2vdl printed (stdin or a file), execute it on
GPU 0 over synthetic TPC-H-shaped tables generated to the reference's bounds metadata, and print the server's JSON
(resolve.py:8-32) -- or, with --csv, what `resolve.py dictionary.csv` would print from it.  The translator drops ORDER BY
and LIMIT; --order-by / --limit / --tpch-order apply them on the GPU before the result is copied, and --collate orders
string-coded keys by their strings."""
from __future__ import annotations

import argparse
import os
import re
import sys
import time

from .tpch import STRING_TYPES   # storage types whose values are string-heap offsets or dictionary codes


def parse_order_by(spec: str) -> list:
    """'revenue:desc,o_orderdate' -> [("revenue", True), ("o_orderdate", False)]."""
    keys = []
    for part in (p.strip() for p in spec.split(",")):
        if not part:
            continue
        name, _, direction = part.partition(":")
        if direction.lower() not in ("", "asc", "desc"):
            raise ValueError(f"--order-by {part!r}: the direction is 'asc' or 'desc'")
        keys.append((name, direction.lower() == "desc"))
    return keys


def order_request(args, text: str, cat) -> tuple:
    """(keys, limit) the arguments ask for, checked against the plan's outputs and the catalogue before any device is
    opened.  Raises ValueError: an unknown or ambiguous name, a key whose output comes from a char / varchar column
    (with --collate: such a key that has no string heap)."""
    from .executor import order_keys
    from .tpch_queries import COLLATED_ORDER, ORDER
    keys, limit = parse_order_by(args.order_by), args.limit
    if limit is not None and limit < 0:
        raise ValueError("--limit must be >= 0")
    if args.tpch_order:
        if keys or limit is not None:
            raise ValueError("--tpch-order gives the ORDER BY and LIMIT itself: not with --order-by / --limit")
        q = os.path.basename(args.plan).split(".")[0]
        known = {**COLLATED_ORDER, **ORDER} if args.collate else ORDER
        if q not in known:
            what = "TPC-H ORDER BY" if args.collate else "numeric TPC-H ORDER BY"
            raise ValueError(f"--tpch-order: no {what} for plan {q!r} (known: {', '.join(sorted(known))})")
        keys, limit = known[q]
    if not keys:
        return keys, limit
    from .tpch import plan_outputs
    names = plan_outputs(text)
    try:
        idx, _ = order_keys(names, keys)
    except KeyError as e:
        raise ValueError(e.args[0]) from None
    if args.collate:
        from .tpch import collation_recipes
        collation_recipes(cat, text, keys)          # every string key has a heap, or ValueError
        return keys, limit
    for i in idx:
        parts = names[i].split("__")
        if len(parts) == 3:
            try:
                col = cat.column(f"{parts[1]}.{parts[2]}")
            except KeyError:
                continue
            if col.mtype in STRING_TYPES:
                raise ValueError(f"--order-by {names[i]}: a {col.mtype} column is held as string-heap offsets / dictionary codes, "
                                 "which do not sort in collation order")
    return keys, limit


def main(argv=None) -> int:
    ap = argparse.ArgumentParser(prog="python -m mplan2vdl_b200")
    ap.add_argument("plan", nargs="?", default="-", help="Voodoo program text (VdlFormat); '-' = stdin")
    ap.add_argument("--sf", type=float, default=1.0, help="scale factor of the synthetic tables")
    ap.add_argument("--csv", action="store_true", help="decode dictionary-coded outputs and print CSV (resolve.py)")
    ap.add_argument("--no-fuse", action="store_true", help="op-at-a-time execution only")
    ap.add_argument("--explain", action="store_true", help="print what the planner makes of the program (JSON) and stop: needs no GPU")
    ap.add_argument("--order-by", default="", help="ORDER BY, applied on the GPU: comma-separated output names or aliases "
                    "(the part before '__'), each optionally :asc or :desc; ties keep the plan's own order")
    ap.add_argument("--limit", type=int, default=None, help="LIMIT: only the first N rows (of the ordered result) are copied")
    ap.add_argument("--tpch-order", action="store_true", help="TPC-H's own ORDER BY / LIMIT of the plan (qNN.vdl) when its keys are numeric "
                    "(with --collate: string keys too)")
    ap.add_argument("--collate", action="store_true", help="order keys whose output comes from a char / varchar column by their "
                    "strings (byte order), not by their heap offsets / dictionary codes")
    args = ap.parse_args(argv)
    text = sys.stdin.read() if args.plan == "-" else open(args.plan).read()
    text = re.sub(r" ;;.*", "", text)          # the pipeline strips the --metadata suffix with sed (eval_query.sh:20)
    if args.explain:
        import json
        from .executor import explain
        sys.stdout.write(json.dumps(explain(text, fuse=not args.no_fuse), indent=1) + "\n")
        return 0

    from . import resolve, tpch
    from .executor import Context
    from .meta import builtin_catalog
    cat = builtin_catalog()
    try:
        order, limit = order_request(args, text, cat)
    except ValueError as e:
        ap.error(str(e))
    ctx = Context(0)
    tpch.load_synthetic(ctx, cat, tpch.plan_columns(text), args.sf)
    plan = ctx.plan(text, fuse=not args.no_fuse)
    if order or limit is not None:
        heaps = tpch.collation_heaps(ctx, cat, text, order) if args.collate else None
        plan.set_order(order, limit, heaps)
    t0 = time.perf_counter()
    out = plan.run()
    us = 1e6 * (time.perf_counter() - t0)
    doc = resolve.to_server_json(out, {"timeInMicrosecondsForPlan": us})
    sys.stdout.write(resolve.to_csv(resolve.resolve(doc, cat)) if args.csv else doc + "\n")
    plan.close()
    ctx.close()
    return 0


if __name__ == "__main__":
    sys.exit(main())
