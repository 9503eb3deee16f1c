"""TPC-H queries as the relational IR Mplan.hs builds from the reference's fixtures
(tests/tpch10noorder/NN.sql.mplan), for the Vlite/Vdl restatement in vlite.py.

Literal encodings follow Mplan.hs: dates are day counts since 0000-01-01 (46-57; date.toordinal() + 365),
date +/- interval is folded at translation time (368-388), decimal literals keep their digits with the scale as
the decimal point (461-484), char literals are dictionary codes (41-44; dictionary.csv)."""
from __future__ import annotations

import datetime

from .vlite import Bin, Cast, GroupBy, Join, Lit, Project, Ref, Select, Table

DATE = ("date",)


def day(y, m, d) -> int:
    return datetime.date(y, m, d).toordinal() + 365


def dec(point, n):
    return Lit(("dec", point), n)


ONE_2 = Cast(2, dec(0, 1))       # decimal(15,2)[tinyint "1"]  -> 100


def between(lo, x, hi, first="Leq", second="Lt"):      # sc P.Interval (Mplan.hs:505-518)
    return Bin("LogAnd", Bin(first, lo, x), Bin(second, x, hi))


def conj(*es):                                          # conjunction (552-559)
    out = es[0]
    for e in es[1:]:
        out = Bin("LogAnd", out, e)
    return out


def li(*cols):
    return [("lineitem." + c, None) for c in cols]


def q06():
    """06.sql.mplan:14-20."""
    t = Table("lineitem", li("l_quantity", "l_extendedprice", "l_discount", "l_shipdate"))
    pred = conj(
        between(Lit(DATE, day(1994, 1, 1)), Ref("lineitem.l_shipdate"), Lit(DATE, day(1995, 1, 1))),
        between(Cast(2, Bin("Sub", Cast(2, dec(2, 6)), dec(2, 1))), Ref("lineitem.l_discount"),
                Cast(2, Bin("Add", Cast(2, dec(2, 6)), dec(2, 1))), "Leq", "Leq"),
        Bin("Lt", Ref("lineitem.l_quantity"), Cast(2, dec(0, 24))))
    g = GroupBy(Select(t, pred), [], [(("FSum", Bin("Mul", Ref("lineitem.l_extendedprice"), Ref("lineitem.l_discount"))), "L1.L1")])
    return Project(g, [(Ref("L1"), "L1.revenue")])


def q01():
    """01.sql.mplan:23-29.  1998-12-01 - 7776000000 ms = 1998-09-02."""
    t = Table("lineitem", li("l_quantity", "l_extendedprice", "l_discount", "l_tax", "l_returnflag", "l_linestatus", "l_shipdate"))
    s = Select(t, Bin("Leq", Ref("lineitem.l_shipdate"), Lit(DATE, day(1998, 9, 2))))
    ep, disc, tax = Ref("lineitem.l_extendedprice"), Ref("lineitem.l_discount"), Ref("lineitem.l_tax")
    disc_price = Bin("Mul", ep, Bin("Sub", ONE_2, disc))
    g = GroupBy(s, [("lineitem.l_returnflag", None), ("lineitem.l_linestatus", None)], [
        (("FChoose", Ref("lineitem.l_returnflag")), None), (("FChoose", Ref("lineitem.l_linestatus")), None),
        (("FSum", Ref("lineitem.l_quantity")), "L1.L1"), (("FSum", ep), "L2.L2"), (("FSum", disc_price), "L3.L3"),
        (("FSum", Bin("Mul", disc_price, Bin("Add", ONE_2, tax))), "L4.L4"),
        (("Avg", Cast(None, Ref("lineitem.l_quantity"))), "L5.L5"), (("Avg", Cast(None, ep)), "L6.L6"),
        (("Avg", Cast(None, disc)), "L7.L7"), (("Count",), "L10.L10")])
    return Project(g, [(Ref("lineitem.l_returnflag"), None), (Ref("lineitem.l_linestatus"), None), (Ref("L1"), "L1.sum_qty"),
                       (Ref("L2"), "L2.sum_base_price"), (Ref("L3"), "L3.sum_disc_price"), (Ref("L4"), "L4.sum_charge"),
                       (Ref("L5"), "L5.avg_qty"), (Ref("L6"), "L6.avg_price"), (Ref("L7"), "L7.avg_disc"), (Ref("L10"), "L10.count_order")])


def q03(catalog):
    """03.sql.mplan:24-40: (orders[o_orderdate < d] JOIN customer[BUILDING]) JOIN lineitem[l_shipdate > d], group by 3 keys."""
    d = Lit(DATE, day(1995, 3, 15))
    orders = Select(Table("orders", [("orders.o_orderdate", None), ("orders.o_shippriority", None), ("orders.%TID%", None),
                                     ("orders.orders_customer", "orders.%orders_customer")]),
                    Bin("Lt", Ref("orders.o_orderdate"), d))
    building = Lit(("str", "customer.c_mktsegment"), catalog.dictionary["customer.c_mktsegment"]["BUILDING"])
    customer = Select(Table("customer", [("customer.c_mktsegment", None), ("customer.%TID%", None)]),
                      Bin("Eq", Ref("customer.c_mktsegment"), building))
    j1 = Join(orders, customer, [Bin("Eq", Ref("orders.%orders_customer"), Ref("customer.%TID%"))])
    lineitem = Select(Table("lineitem", li("l_orderkey", "l_extendedprice", "l_discount", "l_shipdate") +
                            [("lineitem.lineitem_orders", "lineitem.%lineitem_orders")]),
                      Bin("Gt", Ref("lineitem.l_shipdate"), d))
    j2 = Join(j1, lineitem, [Bin("Eq", Ref("lineitem.%lineitem_orders"), Ref("orders.%TID%"))])
    revenue = Bin("Mul", Ref("lineitem.l_extendedprice"), Bin("Sub", ONE_2, Ref("lineitem.l_discount")))
    g = GroupBy(j2, [("lineitem.l_orderkey", None), ("orders.o_shippriority", None), ("orders.o_orderdate", None)],
                [(("FChoose", Ref("lineitem.l_orderkey")), None), (("FChoose", Ref("orders.o_orderdate")), None),
                 (("FChoose", Ref("orders.o_shippriority")), None), (("FSum", revenue), "L1.L1")])
    return Project(g, [(Ref("lineitem.l_orderkey"), None), (Ref("L1"), "L1.revenue"), (Ref("orders.o_orderdate"), None),
                       (Ref("orders.o_shippriority"), None)])


def q05(catalog):
    """05.sql.mplan:27-50: lineitem -> orders[1994] -> customer -> supplier (c_nationkey = s_nationkey) -> nation -> region['ASIA']."""
    orders = Select(Table("orders", [("orders.o_orderdate", None), ("orders.%TID%", None), ("orders.orders_customer", "orders.%orders_customer")]),
                    between(Lit(DATE, day(1994, 1, 1)), Ref("orders.o_orderdate"), Lit(DATE, day(1995, 1, 1))))
    lineitem = Table("lineitem", li("l_extendedprice", "l_discount") + [("lineitem.lineitem_orders", "lineitem.%lineitem_orders"),
                                                                        ("lineitem.lineitem_supplier", "lineitem.%lineitem_supplier")])
    j1 = Join(lineitem, orders, [Bin("Eq", Ref("lineitem.%lineitem_orders"), Ref("orders.%TID%"))])
    j2 = Join(j1, Table("customer", [("customer.c_nationkey", None), ("customer.%TID%", None)]),
              [Bin("Eq", Ref("orders.%orders_customer"), Ref("customer.%TID%"))])
    supplier = Table("supplier", [("supplier.s_nationkey", None), ("supplier.%TID%", None), ("supplier.supplier_nation", "supplier.%supplier_nation")])
    j3 = Join(j2, supplier, [Bin("Eq", Ref("lineitem.%lineitem_supplier"), Ref("supplier.%TID%")),
                             Bin("Eq", Ref("customer.c_nationkey"), Ref("supplier.s_nationkey"))])
    nation = Table("nation", [("nation.n_name", None), ("nation.%TID%", None), ("nation.nation_region", "nation.%nation_region")])
    j4 = Join(j3, nation, [Bin("Eq", Ref("supplier.%supplier_nation"), Ref("nation.%TID%"))])
    asia = Lit(("str", "region.r_name"), catalog.dictionary["region.r_name"]["ASIA"])
    region = Select(Table("region", [("region.r_name", None), ("region.%TID%", None)]), Bin("Eq", Ref("region.r_name"), asia))
    j5 = Join(j4, region, [Bin("Eq", Ref("nation.%nation_region"), Ref("region.%TID%"))])
    revenue = Bin("Mul", Ref("lineitem.l_extendedprice"), Bin("Sub", ONE_2, Ref("lineitem.l_discount")))
    g = GroupBy(j5, [("nation.n_name", None)], [(("FChoose", Ref("nation.n_name")), None), (("FSum", revenue), "L1.L1")])
    return Project(g, [(Ref("nation.n_name"), None), (Ref("L1"), "L1.revenue")])


QUERIES = {"q06": lambda cat: q06(), "q01": lambda cat: q01(), "q03": q03, "q05": q05}

# TPC-H's ORDER BY / LIMIT of the checked-in plans whose sort keys are all numeric outputs, which the fixtures
# (tpch10noorder) drop and the executor applies on request (Plan.set_order, --tpch-order): plan -> (keys, limit), keys as
# (output name or alias, descending).  The other plans order by a string-coded output (n_name, l_returnflag, ...): their
# values are heap offsets or dictionary codes, not a collation order.
ORDER = {
    "q03": ([("revenue", True), ("o_orderdate__orders__o_orderdate", False)], 10),
    "q05": ([("revenue", True)], None),
    "q10": ([("revenue", True)], 20),
    "q11": ([("value", True)], None),
    "q18": ([("o_totalprice__orders__o_totalprice", True), ("o_orderdate__orders__o_orderdate", False)], 100),
}

# TPC-H's ORDER BY of the checked-in plans whose sort keys include a string-coded output, applied with the keys' strings
# (Plan.set_order's heaps, tpch.collation_heaps, --tpch-order --collate): plan -> (keys, limit) as in ORDER.
COLLATED_ORDER = {
    "q01": ([("l_returnflag", False), ("l_linestatus", False)], None),
    "q04": ([("o_orderpriority", False)], None),
    "q09": ([("nation", False), ("o_year", True)], None),
    "q12": ([("l_shipmode", False)], None),
    "q16": ([("supplier_cnt", True), ("p_brand", False), ("p_type", False), ("p_size", False)], None),
    "q20": ([("s_name", False)], None),
}
