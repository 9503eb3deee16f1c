"""Synthetic TPC-H-shaped tables resident in HBM, sharded the way the executor scales out:
the fact table (lineitem) by contiguous row range, dimension tables replicated (SURVEY.md section 8 e)."""
from __future__ import annotations

import os
import re

from . import synth
from .meta import Catalog

PLANS_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "plans")
FACT_TABLE = "lineitem"
SHARD_ALIGN = 4096      # shard boundaries are multiples of the largest scan tile so every shard starts tile-aligned


def plan_text(name: str) -> str:
    with open(os.path.join(PLANS_DIR, name)) as f:
        return f.read()


def plan_columns(text: str) -> list:
    """Qualified names of the columns a plan Loads (Vdl.hs:419-420 `Load,<table>.<col>`)."""
    seen = []
    for m in re.finditer(r"^\d+,Load,([\w.]+)", text, re.M):
        if m.group(1) not in seen:
            seen.append(m.group(1))
    return seen


def plan_outputs(text: str) -> list:
    """Output names of a plan in MaterializeCompact order: the Project each `MaterializeCompact,Id n` names (Vdl.hs:278-292)."""
    project = dict(re.findall(r"^(\d+),Project,([^,\s]+),", text, re.M))
    return [project[i] for i in re.findall(r"^\d+,MaterializeCompact,Id (\d+)", text, re.M)]


def shard_range(rows: int, rank: int, world: int) -> tuple:
    """(first global row, row count) of `rank`'s contiguous shard of a `rows`-row fact table."""
    per = -(-rows // world)
    per = -(-per // SHARD_ALIGN) * SHARD_ALIGN
    start = min(rows, rank * per)
    return start, max(0, min(rows, start + per) - start)


def load_synthetic(ctx, cat: Catalog, columns, sf: float, rank: int = 0, world: int = 1, rows_override: dict | None = None) -> dict:
    """Generate the named columns in place on ctx's GPU.  Returns {"row_base": int, "rows": {table: rows on this GPU}}."""
    seed = synth.seed_for(sf)
    rows_here, row_base = {}, 0
    heaps = {q[:-len(".heap")] for q in columns if synth.is_heap(q)}     # string columns whose heap a Like reads
    for q in columns:
        table = q.split(".")[0]
        if synth.is_heap(q):                               # the bytes of the heap: host-built (small), uploaded once
            heap, _ = synth.string_heap(cat, q[:-len(".heap")])
            ctx.upload_column(q, heap)
            continue
        total = (rows_override or {}).get(table, synth.table_rows(cat, table, sf))
        if table == FACT_TABLE:
            start, n = shard_range(total, rank, world)
            row_base = start
        else:
            start, n = 0, total
        if q in heaps:                                     # ... and its offsets column: pool entries drawn per global row
            ctx.upload_column(q, synth.string_offsets(cat, q, n, start, seed))
            rows_here[table] = n
            continue
        spec = synth.column_spec(cat, q, sf)
        if table in (rows_override or {}) and spec.kind == synth.FKDENSE:
            spec = synth.ColumnSpec(spec.name, spec.width, spec.kind, spec.vmin, spec.stride, spec.p0, total, spec.stream)
        ctx.fill_synthetic(q, spec, n, seed, start)
        rows_here[table] = n
    return {"row_base": row_base, "rows": rows_here}


# storage types whose values are string-heap offsets or dictionary codes, not a collation order
STRING_TYPES = ("char", "varchar")
# prefix of the name a code heap is uploaded under: no plan Loads it (Load names are [\w.]+), so it never meets a Like heap
CODE_HEAP_PREFIX = "collate:"


def collation_recipes(cat: Catalog, text: str, keys) -> dict:
    """{key name: ("pool", column) or ("codes", column)} for the ORDER BY `keys` of plan `text` whose output comes from a
    char / varchar column (keys as Plan.set_order takes them; numeric keys are left out).  "pool": the plan Loads the
    column's heap, so its values are offsets into synth.string_heap (origin 0); "codes": its values are dictionary codes,
    ordered through synth.code_heap.  Raises KeyError for an unknown name, ValueError for a string key with neither."""
    from .executor import order_keys
    names, loads = plan_outputs(text), plan_columns(text)
    out = {}
    for key in keys:
        name = key if isinstance(key, str) else key[0]
        (i,), _ = order_keys(names, [name])
        parts = names[i].split("__")
        if len(parts) != 3:
            continue
        q = f"{parts[1]}.{parts[2]}"
        try:
            col = cat.column(q)
        except KeyError:
            continue
        if col.mtype not in STRING_TYPES:
            continue
        if q + ".heap" in loads:
            out[name] = ("pool", q)
            continue
        spec = synth.column_spec(cat, q, 10)
        if spec.kind not in (synth.UNIFORM, synth.SEQ) or spec.stride < 2:
            raise ValueError(f"ORDER BY {names[i]}: no string heap for {q} (neither Loaded with its heap nor codes at a fixed stride)")
        out[name] = ("codes", q)
    return out


def collation_heaps(ctx, cat: Catalog, text: str, keys) -> dict:
    """The `heaps` mapping of Plan.set_order for the string keys among `keys` of plan `text` (collation_recipes): a
    pool heap the plan Loads is looked up (uploaded when absent), a code heap uploaded once under CODE_HEAP_PREFIX +
    column.  {} when no key is a string."""
    from .lib import VdlError
    out = {}
    for name, (kind, q) in collation_recipes(cat, text, keys).items():
        hname = q + ".heap" if kind == "pool" else CODE_HEAP_PREFIX + q
        origin = 0 if kind == "pool" else synth.column_spec(cat, q, 10).vmin       # code_heap's origin: the smallest code
        try:
            h = ctx.lookup(hname)
        except VdlError:                            # the bytes are built only when the heap is not on the device yet
            h = ctx.upload_column(hname, synth.string_heap(cat, q)[0] if kind == "pool" else synth.code_heap(cat, q)[0])
        out[name] = (h, origin)
    return out
