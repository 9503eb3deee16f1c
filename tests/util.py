"""Shared helpers for the parity tests: host columns from the synthetic recipe, via the oracle's generator."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

# The reference translator's own MonetDB plans and metadata files (tests/tpch10noorder of an orm011/mplan2vdl checkout)
# are not part of this repository.  The tests that translate them run when MPLAN2VDL_REFERENCE names such a checkout.
REFERENCE = os.environ.get("MPLAN2VDL_REFERENCE", "")
FIXTURES = os.path.join(REFERENCE, "tests", "tpch10noorder") if REFERENCE else ""
needs_reference = pytest.mark.skipif(not os.path.isdir(FIXTURES),
                                     reason="needs MPLAN2VDL_REFERENCE: a checkout of the reference translator (orm011/mplan2vdl)")

from mplan2vdl_b200 import synth  # noqa: E402
from oracle.oracle import Oracle, gen_column  # noqa: E402

Q6_COLS = ["l_quantity", "l_extendedprice", "l_discount", "l_shipdate"]
Q1_COLS = Q6_COLS + ["l_tax", "l_returnflag", "l_linestatus"]


def plan_text(name: str) -> str:
    with open(os.path.join(ROOT, "plans", name)) as f:
        return f.read()


def host_columns(cat, qualified_names, rows_by_table, sf=1, seed=None, row_offset=0):
    """{qualified: ndarray} generated on the host; rows_by_table overrides the SF cardinalities."""
    seed = synth.seed_for(sf) if seed is None else seed
    out = {}
    heaps = {q[:-len(".heap")] for q in qualified_names if synth.is_heap(q)}
    for q in qualified_names:
        t = q.split(".")[0]
        if synth.is_heap(q):                     # string heap of a Like (uint8 bytes) ...
            out[q] = synth.string_heap(cat, q[:-len(".heap")])[0]
        elif q in heaps:                         # ... and the offsets into it
            out[q] = synth.string_offsets(cat, q, rows_by_table[t], row_offset, seed)
        else:
            out[q] = gen_column(synth.column_spec(cat, q, sf), rows_by_table[t], row_offset, seed)
    return out


def run_oracle(plan, cols, threads=0):
    o = Oracle()
    for k, v in cols.items():
        o.bind(k, v)
    return o.run(plan, threads)


def assert_same(a: dict, b: dict):
    assert list(a.keys()) == list(b.keys())
    for k in a:
        np.testing.assert_array_equal(np.asarray(a[k], dtype=np.int64), np.asarray(b[k], dtype=np.int64), err_msg=k)


def run_gpu(plan, cols, fuse=True, ctx=None):
    """Upload host columns, run the plan through libvdl_cuda's C ABI, return ({name: array}, stats)."""
    from mplan2vdl_b200.executor import Context
    own = ctx is None
    ctx = ctx or Context(0)
    try:
        for k, v in cols.items():
            ctx.upload_column(k, v)
        p = ctx.plan(plan, fuse=fuse)
        out = p.run()
        stats = p.stats()
        stats["shape"] = p.shape(0) if stats["fused_scans"] else None
        p.close()
        for k in cols:
            ctx.drop_column(k)
        return out, stats
    finally:
        if own:
            ctx.close()


def q19_columns(cat, sf=0.01, seed=19):
    """Synthetic tables for Q19 with the string-coded columns redrawn from the codes the query mentions (plus a few
    others), so that its very selective predicate keeps some rows (the uniform recipe over [min, max] almost never
    hits 'DELIVER IN PERSON' x 'AIR' x three brands x twelve containers)."""
    from mplan2vdl_b200 import tpch
    text = plan_text("q19.vdl")
    rows = {t: synth.table_rows(cat, t, sf) for t in cat.tables}
    cols = host_columns(cat, tpch.plan_columns(text), rows, sf=sf)
    rng = np.random.default_rng(seed)
    D = cat.dictionary

    def draw(col, names, extra, n):
        codes = [D[col][x] for x in names] + extra
        return np.array(codes, dtype=np.int64)[rng.integers(0, len(codes), n)]
    n, npart = rows["lineitem"], rows["part"]
    cols["lineitem.l_shipinstruct"] = draw("lineitem.l_shipinstruct", ["DELIVER IN PERSON"], [24, 32], n)
    cols["lineitem.l_shipmode"] = draw("lineitem.l_shipmode", ["AIR", "MAIL"], [16], n)
    cols["part.p_brand"] = draw("part.p_brand", ["Brand#12", "Brand#23", "Brand#34"], [16, 32], npart)
    cols["part.p_container"] = draw("part.p_container", ["SM CASE", "SM BOX", "MED BAG", "MED PKG", "LG CASE", "LG PKG", "SM PKG", "LG BOX"], [8], npart)
    return text, cols


def golden_case(cat, q):
    """(plan text, host columns, committed answer) of query `q` at SF 0.01: tests/golden/tpch_sf0.01_answers.json, written
    by tools/make_golden_results.py from the SQL-level numpy evaluation (oracle/sqlref.py)."""
    import json
    from mplan2vdl_b200 import tpch
    with open(os.path.join(ROOT, "tests", "golden", "tpch_sf0.01_answers.json")) as f:
        g = json.load(f)
    sf = g["sf"]
    assert g["seed"] == synth.seed_for(sf)
    if q == "q19":
        text, cols = q19_columns(cat, sf=sf)
    else:
        text = plan_text(q + ".vdl")
        rows = {t: synth.table_rows(cat, t, sf) for t in cat.tables}
        cols = host_columns(cat, tpch.plan_columns(text), rows, sf=sf)
    return text, cols, {k: np.asarray(v, dtype=np.int64) for k, v in g["answers"][q].items()}
