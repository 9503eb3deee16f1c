"""The translator's front half restated (mplan2vdl_b200/mplan.py: Scanner.x + Parser.y + Mplan.hs): the reference's own
fixtures tests/tpch10noorder/NN.sql.mplan must turn into exactly the checked-in Voodoo programs."""
import os

import pytest

from mplan2vdl_b200 import mplan, tpch_queries, vlite
from util import FIXTURES, host_columns, needs_reference, plan_text, run_oracle


@needs_reference
@pytest.mark.parametrize("n,plan", [("06", "q06.vdl"), ("03", "q03.vdl"), ("05", "q05.vdl"), ("12", "q12.vdl"), ("19", "q19.vdl"),
                                    ("04", "q04.vdl"), ("11", "q11.vdl"), ("15", "q15.vdl"), ("09", "q09.vdl"), ("14", "q14.vdl"), ("16", "q16.vdl"), ("20", "q20.vdl"), ("10", "q10.vdl"), ("18", "q18.vdl")])
def test_reference_fixture_translates_to_the_checked_in_program(catalog, n, plan):
    text = open(os.path.join(FIXTURES, f"{n}.sql.mplan")).read()
    assert mplan.translate_mplan(catalog, text) == plan_text(plan)      # q06.vdl is pinned by the reference README


@needs_reference
def test_q1_fixture_gives_the_same_ir_as_the_hand_built_one(catalog):
    text = open(os.path.join(FIXTURES, "01.sql.mplan")).read()
    gen = mplan.translate_mplan(catalog, text)
    assert gen == vlite.translate(catalog, tpch_queries.q01())
    assert gen.splitlines()[:82] == plan_text("q01.vdl").splitlines()[:82]      # SURVEY.md App. F (then duplicates, G10)


@needs_reference
def test_unsupported_fixtures_fail_loudly_with_the_construct_named(catalog):
    for n, what in [("13", "plain joins"), ("22", "IN operator"), ("21", "single complete FK"), ("17", "not known to be unique"),
                    ("02", "char literal"), ("07", "char literal"), ("08", "char literal")]:
        with pytest.raises((NotImplementedError, ValueError), match=what):
            mplan.translate_mplan(catalog, open(os.path.join(FIXTURES, f"{n}.sql.mplan")).read())


OWN_PLAN = """
# a plan in MonetDB's notation written for this test (comment lines, `|` indentation, chained comparison,
# date + interval folding, decimal casts, count(*) and avg):
project (
| group by (
| | select (
| | | table(sys.lineitem) [ lineitem.l_quantity NOT NULL, lineitem.l_discount NOT NULL, lineitem.l_shipdate NOT NULL, lineitem.l_linestatus NOT NULL ] COUNT
| | ) [ date "1995-06-01" <= lineitem.l_shipdate NOT NULL < sys.sql_add(date "1995-06-01", month_interval "6"), lineitem.l_discount NOT NULL >= decimal(15,2)[decimal(2,2) "3"] ]
| ) [ lineitem.l_linestatus NOT NULL ] [ lineitem.l_linestatus NOT NULL, sys.sum no nil (lineitem.l_quantity NOT NULL) as L1.L1, sys.count() NOT NULL as L2.L2, sys.avg no nil (double[lineitem.l_discount NOT NULL] as lineitem.l_discount) as L3.L3 ]
) [ lineitem.l_linestatus NOT NULL, L1 as L1.sum_qty, L2 as L2.cnt, L3 as L3.avg_disc ]
"""


def test_own_plan_parses_lowers_and_runs(catalog):
    rel = mplan.relexpr_from_mplan(catalog, OWN_PLAN)
    assert type(rel).__name__ == "Project" and type(rel.child).__name__ == "GroupBy"
    sel = rel.child.child
    assert sel.predicate.left.left.right.name == "lineitem.l_shipdate"
    assert sel.predicate.left.left.left.n == mplan.day_count("1995-06-01") and sel.predicate.left.right.right.n == mplan.day_count("1995-12-01")
    text = vlite.translate(catalog, rel)
    cols = host_columns(catalog, ["lineitem.l_quantity", "lineitem.l_discount", "lineitem.l_shipdate", "lineitem.l_linestatus"], {"lineitem": 20_000})
    out = run_oracle(text, cols)
    assert list(out) == ["l_linestatus__lineitem__l_linestatus", "sum_qty", "cnt", "avg_disc"]
    import numpy as np
    m = (cols["lineitem.l_shipdate"] >= mplan.day_count("1995-06-01")) & (cols["lineitem.l_shipdate"] < mplan.day_count("1995-12-01")) & (cols["lineitem.l_discount"] >= 3)
    for i, code in enumerate(out["l_linestatus__lineitem__l_linestatus"]):
        g = m & (cols["lineitem.l_linestatus"] == code)
        assert out["cnt"][i] == g.sum() and out["sum_qty"][i] == cols["lineitem.l_quantity"][g].sum()


def test_date_interval_folding():
    import datetime
    assert mplan.add_months_rollover(datetime.date(1994, 1, 1), 12) == datetime.date(1995, 1, 1)
    assert mplan.add_months_rollover(datetime.date(1994, 1, 31), 1) == datetime.date(1994, 3, 3)       # rolls over, like addGregorianMonthsRollOver
    assert mplan.day_count("1994-01-01") == 728294
