"""--use_cross_product (MainFuns.hs:72, Mplan.hs:309-313): a plain join becomes a selection over the cross product of its
inputs (Vlite.hs:672-680), printed with CrossProductOuter / CrossProductInner (Vdl.hs:412-416).  Quadratic, so tiny tables:
the reference's 12.sql.mplan with the flag, against the direct numpy evaluation of the same mplan's relational IR read as a
VALUE join (tests/ir_eval.py) -- and the per-op semantics on hand-written vectors (Vlite.hs:283-292)."""
import os

import numpy as np
import pytest

import ir_eval
from mplan2vdl_b200 import mplan, tpch, vlite
from util import FIXTURES, assert_same, host_columns, needs_reference, run_gpu, run_oracle

PAIRS = "\n".join(["1,Load,a.x", "2,Load,b.y", "3,CrossProductOuter,Id 1,Id 2", "4,CrossProductInner,Id 1,Id 2",
                   "5,Gather,Id 1,Id 3,val", "6,Gather,Id 2,Id 4,val", "7,Multiply,val,Id 5,val,Id 6,val",
                   "8,Project,outer,Id 3,val", "9,MaterializeCompact,Id 8", "10,Project,inner,Id 4,val", "11,MaterializeCompact,Id 10",
                   "12,Project,prod,Id 7,val", "13,MaterializeCompact,Id 12", ""])
A, B = np.array([3, 5, 7, 11], dtype=np.int64), np.array([10, 100], dtype=np.int64)


def q12_like_plan(catalog):
    """Q12's shape without reading the fixture (the GPU box has no reference checkout): lineitem x orders on the order key."""
    from mplan2vdl_b200.vlite import Bin, CartesianProduct, GroupBy, Project, Ref, Select, Table
    li = Table("lineitem", [("lineitem.l_orderkey", None), ("lineitem.l_quantity", None)])
    od = Table("orders", [("orders.o_orderkey", None), ("orders.o_shippriority", None)])
    sel = Select(CartesianProduct(li, od), Bin("Eq", Ref("lineitem.l_orderkey"), Ref("orders.o_orderkey")))
    g = GroupBy(sel, [("orders.o_shippriority", None)], [(("FChoose", Ref("orders.o_shippriority")), None), (("FSum", Ref("lineitem.l_quantity")), "L1.L1")])
    return Project(g, [(Ref("orders.o_shippriority"), None), (Ref("L1"), "L1.qty")])


def small_tables(catalog, text, nli=300, nord=40, seed=5):
    cols = host_columns(catalog, tpch.plan_columns(text), {"lineitem": nli, "orders": nord}, sf=0.01)
    rng = np.random.default_rng(seed)
    if "orders.o_orderkey" in cols and "lineitem.l_orderkey" in cols:
        okeys = np.unique(cols["orders.o_orderkey"])
        pick = np.r_[okeys, [okeys.max() + 7]]                   # some lineitems match no order
        cols["lineitem.l_orderkey"] = pick[rng.integers(0, len(pick), nli)].astype(cols["lineitem.l_orderkey"].dtype)
    if "lineitem.lineitem_orders" in cols:                       # the FK index column: row ids of the (small) orders table, some beyond it
        cols["lineitem.lineitem_orders"] = (cols["lineitem.lineitem_orders"] % (nord + 5)).astype(cols["lineitem.lineitem_orders"].dtype)
    return cols


def test_oracle_cross_product_vectors():
    out = run_oracle(PAIRS, {"a.x": A, "b.y": B})
    np.testing.assert_array_equal(out["outer"], [0, 0, 1, 1, 2, 2, 3, 3])       # Vlite.hs:281-282
    np.testing.assert_array_equal(out["inner"], [0, 1, 0, 1, 0, 1, 0, 1])
    np.testing.assert_array_equal(out["prod"], np.outer(A, B).reshape(-1))


def test_translator_prints_the_cross_product_of_a_hand_built_join(catalog):
    text = vlite.translate(catalog, q12_like_plan(catalog))
    ops = [l.split(",")[1] for l in text.splitlines()]
    assert ops.count("CrossProductOuter") == 1 and ops.count("CrossProductInner") == 1
    cols = small_tables(catalog, text)
    out = run_oracle(text, cols)
    # value join, by hand
    li_k, li_q = cols["lineitem.l_orderkey"].astype(np.int64), cols["lineitem.l_quantity"].astype(np.int64)
    od_k, od_p = cols["orders.o_orderkey"].astype(np.int64), cols["orders.o_shippriority"].astype(np.int64)
    want = {}
    for k, q in zip(li_k, li_q):
        for p in od_p[od_k == k]:
            want[int(p)] = want.get(int(p), 0) + int(q)
    got = dict(zip((int(x) for x in list(out.values())[0]), (int(x) for x in list(out.values())[1])))
    assert got == want and want


@needs_reference
def test_fixture_12_with_the_flag_agrees_with_the_value_join(catalog):
    ir_eval.set_catalog(catalog)
    src = open(os.path.join(FIXTURES, "12.sql.mplan")).read()
    text = mplan.translate_mplan(catalog, src, cross_product=True)
    assert "CrossProductOuter" in text and "CrossProductInner" in text
    rel = mplan.relexpr_from_mplan(catalog, src)                  # the same mplan as a join, evaluated on VALUES
    names = tpch.plan_columns(text)
    allnames = names + [c for c in ir_eval.base_columns(rel) if c not in names]
    cols = small_tables(catalog, "\n".join(f"{i + 1},Load,{c}" for i, c in enumerate(allnames)) + "\n", nli=400, nord=60)
    # the uniform recipe almost never satisfies Q12's predicate: plant rows that do
    from mplan2vdl_b200.tpch_queries import day
    rng = np.random.default_rng(12)
    n = len(cols["lineitem.l_shipmode"])
    mode = np.array([catalog.dictionary["lineitem.l_shipmode"][m] for m in ("MAIL", "SHIP", "AIR")], dtype=np.int64)
    cols["lineitem.l_shipmode"] = mode[rng.integers(0, 3, n)].astype(cols["lineitem.l_shipmode"].dtype)
    receipt = rng.integers(day(1993, 11, 1), day(1995, 3, 1), n)
    cols["lineitem.l_receiptdate"] = receipt.astype(cols["lineitem.l_receiptdate"].dtype)
    cols["lineitem.l_commitdate"] = (receipt - rng.integers(-3, 9, n)).astype(cols["lineitem.l_commitdate"].dtype)
    cols["lineitem.l_shipdate"] = (receipt - rng.integers(2, 20, n)).astype(cols["lineitem.l_shipdate"].dtype)
    got = list(run_oracle(text, {k: cols[k] for k in names}).values())
    want = ir_eval.evaluate(cols, rel)
    assert len(got) == len(want) and len(want[0]) > 0
    # rows compared as a set: the dictionary's code for SHIP (160) lies outside the column's bounds.csv range (the storage
    # is one byte wide), so the masked group key orders the two groups differently from their raw codes
    og, ow = np.argsort(got[0], kind="stable"), np.argsort(want[0], kind="stable")
    for g, w in zip(got, want):
        np.testing.assert_array_equal(np.asarray(g)[og], np.asarray(w)[ow])


@pytest.mark.gpu
@pytest.mark.parametrize("fuse", [True, False])
def test_gpu_cross_product_matches_the_oracle(catalog, fuse):
    out, _ = run_gpu(PAIRS, {"a.x": A, "b.y": B}, fuse=fuse)
    assert_same(out, run_oracle(PAIRS, {"a.x": A, "b.y": B}))
    text = vlite.translate(catalog, q12_like_plan(catalog))
    cols = small_tables(catalog, text)
    got, _ = run_gpu(text, cols, fuse=fuse)
    assert_same(got, run_oracle(text, cols))


@pytest.mark.gpu
def test_gpu_cross_product_refuses_absurd_sizes():
    from mplan2vdl_b200.executor import Context
    ctx = Context(0)
    a = ctx.op_range(0, 1, 1 << 20)
    with pytest.raises(Exception, match="CrossProduct"):
        ctx.op_cross_product(a, a, False)
    ctx.close()
