"""Semijoins, the dim-side semijoin's Scatter with size hint, antijoins, joins against a single value and Like over string
heaps (SURVEY.md section 8 f3; Vlite.hs:691-713, 1010-1014, 1212-1232, 1117-1120): the reference's fixtures 04 / 09 / 11 /
14 / 15 / 16.sql.mplan translated by the restated
front end, interpreted by the CPU oracle, against the direct numpy evaluation of the relational IR (tests/ir_eval.py:
value joins, no Voodoo ops).  The GPU tests run the same programs through libvdl_cuda."""
import os

import numpy as np
import pytest

import ir_eval
from mplan2vdl_b200 import mplan, synth, tpch, tpch_queries, vlite
from mplan2vdl_b200.vlite import Bin, GroupBy, Join, Lit, Project, Ref, Select, Table
from util import FIXTURES, assert_same, host_columns, needs_reference, plan_text, run_oracle

SF = 0.01


def columns_for(catalog, text, rel, sf=SF, tweak=True):
    rows = {t: synth.table_rows(catalog, t, sf) for t in catalog.tables}
    names = tpch.plan_columns(text)
    allnames = names + [c for c in ir_eval.base_columns(rel) if c not in names]
    cols = host_columns(catalog, allnames, rows, sf=sf)
    if tweak and "nation.n_name" in cols:        # the recipe's nation names never hit 'GERMANY': plant it
        cols["nation.n_name"] = cols["nation.n_name"].copy()
        cols["nation.n_name"][[3, 7, 11]] = catalog.dictionary["nation.n_name"]["GERMANY"]
    return names, cols


@needs_reference
@pytest.mark.parametrize("n", ["01", "03", "04", "05", "06", "09", "10", "11", "12", "14", "15", "16", "18"])
def test_fixture_program_agrees_with_the_direct_evaluation_of_its_ir(catalog, n):
    ir_eval.set_catalog(catalog)
    rel = mplan.relexpr_from_mplan(catalog, open(os.path.join(FIXTURES, f"{n}.sql.mplan")).read())
    text = vlite.translate(catalog, rel)
    names, cols = columns_for(catalog, text, rel)
    if n == "18":       # HAVING sum(l_quantity) > 300 per order: the recipe's quantities rarely get there
        cols["lineitem.l_quantity"] = cols["lineitem.l_quantity"] * 3
    got = list(run_oracle(text, {k: cols[k] for k in names}).values())
    want = ir_eval.evaluate(cols, rel)
    assert len(got) == len(want)
    for k, (g, w) in enumerate(zip(got, want)):
        np.testing.assert_array_equal(g, w, err_msg=f"output {k}")
    if n in ("04", "09", "10", "11", "14", "15", "16", "18"):
        assert len(got[0]) > 0


def q4_like(catalog, lo=(1993, 7, 1), hi=(1993, 10, 1)):
    """Q4's shape, hand-built: orders[date range] semijoin lineitem[commit < receipt], count per priority."""
    D = tpch_queries.DATE
    orders = Select(Table("orders", [("orders.o_orderkey", None), ("orders.o_orderdate", None), ("orders.o_orderpriority", None)]),
                    tpch_queries.between(Lit(D, tpch_queries.day(*lo)), Ref("orders.o_orderdate"), Lit(D, tpch_queries.day(*hi))))
    li = Select(Table("lineitem", [("lineitem.l_orderkey", "L2.l_orderkey"), ("lineitem.l_commitdate", "L2.l_commitdate"), ("lineitem.l_receiptdate", "L2.l_receiptdate")]),
                Bin("Lt", Ref("L2.l_commitdate"), Ref("L2.l_receiptdate")))
    semi = Join(orders, li, [Bin("Eq", Ref("L2.l_orderkey"), Ref("orders.o_orderkey"))], "LeftSemi")
    g = GroupBy(semi, [("orders.o_orderpriority", None)], [(("FChoose", Ref("orders.o_orderpriority")), None), (("Count",), "L1.L1")])
    return Project(g, [(Ref("orders.o_orderpriority"), None), (Ref("L1"), "L1.order_count")])


def test_dim_side_semijoin_marks_row_zero_for_partnerless_fact_rows(catalog):
    """The place where the reference's graph is NOT the SQL: the Scatter positions of the dim-side semijoin are the
    uncleaned gather mask, so fact rows whose order is outside the date range write slot 0 (Vlite.hs:1214-1218).  The
    oracle interprets the graph; ir_eval restates exactly that; the SQL answer differs by that one order at most."""
    ir_eval.set_catalog(catalog)
    rel = q4_like(catalog)
    text = vlite.translate(catalog, rel)
    assert "Modulo" in text and text.count("FoldSelect") == 3      # orders select, lineitem select, qualified orders (the cleaning select is dead code)
    names, cols = columns_for(catalog, text, rel)
    got = run_oracle(text, {k: cols[k] for k in names})
    want = ir_eval.evaluate(cols, rel)
    np.testing.assert_array_equal(got["order_count"], want[1])
    # pure SQL: orders in range with at least one late lineitem
    od = cols["orders.o_orderdate"]
    sel = (od >= tpch_queries.day(1993, 7, 1)) & (od < tpch_queries.day(1993, 10, 1))
    late = cols["lineitem.l_commitdate"] < cols["lineitem.l_receiptdate"]
    hit = np.zeros(len(od), bool)
    hit[cols["lineitem.lineitem_orders"][late]] = True
    assert abs(int((sel & hit).sum()) - int(got["order_count"].sum())) <= 1


def test_semijoin_over_an_empty_dimension_selection_fails_loudly(catalog):
    """No order in the date range: dim' is empty, yet the partnerless fact rows still mark slot 0 of the (hint-sized)
    `qualified` vector, and gathering dim' at position 0 is out of range.  The graph the reference emits has no answer
    here; the executor reports it instead of inventing one."""
    from oracle.oracle import OracleError
    rel = q4_like(catalog, lo=(2001, 1, 1), hi=(2001, 2, 1))
    text = vlite.translate(catalog, rel)
    names, cols = columns_for(catalog, text, rel)
    with pytest.raises(OracleError, match="Gather"):
        run_oracle(text, {k: cols[k] for k in names})


def test_semijoin_with_no_fact_row_selected(catalog):
    ir_eval.set_catalog(catalog)
    rel = q4_like(catalog)
    text = vlite.translate(catalog, rel)
    names, cols = columns_for(catalog, text, rel)
    cols["lineitem.l_commitdate"] = cols["lineitem.l_receiptdate"] + 1          # nothing is late
    got = run_oracle(text, {k: cols[k] for k in names})
    assert all(len(v) == 0 for v in got.values())
    assert all(len(v) == 0 for v in ir_eval.evaluate(cols, rel))


@pytest.mark.gpu
@pytest.mark.parametrize("q", ["q04", "q11", "q15", "q09", "q14", "q16", "q20", "q10", "q18"])
@pytest.mark.parametrize("sf", [0.01, 0.1])
def test_gpu_runs_the_semijoin_programs(catalog, q, sf):
    from util import run_gpu
    text = plan_text(q + ".vdl")
    rows = {t: synth.table_rows(catalog, t, sf) for t in catalog.tables}
    cols = host_columns(catalog, tpch.plan_columns(text), rows, sf=sf)
    if "nation.n_name" in cols:
        cols["nation.n_name"] = cols["nation.n_name"].copy()
        cols["nation.n_name"][[3, 7, 11]] = catalog.dictionary["nation.n_name"]["GERMANY"]
        cols["nation.n_name"][[2, 5, 13, 17]] = catalog.dictionary["nation.n_name"]["CANADA"]
    if q == "q18":
        cols["lineitem.l_quantity"] = cols["lineitem.l_quantity"] * 3
    want = run_oracle(text, cols)
    assert len(next(iter(want.values()))) > 0 or q == "q20"     # (Q20's composite-FK chain is rarely satisfied by the uniform recipe)
    got, stats = run_gpu(text, cols)
    assert_same(got, want)
    got_u, _ = run_gpu(text, cols, fuse=False)
    assert_same(got_u, want)
