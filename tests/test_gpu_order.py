"""ORDER BY / LIMIT on the GPU: vdl_op_order against the numpy reference (tests/test_order.py) over row counts around the
radix tile, key counts 1..8, int32 / int64 / virtual range keys, heavy duplicates, packed widths beyond 64 bits and the
select path's limits; plans ordered by vdl_plan_set_order against the CPU oracle's unordered result ordered by the
reference, for op-at-a-time, fused-scan and probe-fold outputs, on one GPU and on two ranks of vdl_comm."""
import ctypes as C

import numpy as np
import pytest

from mplan2vdl_b200 import synth, tpch
from mplan2vdl_b200.tpch_queries import ORDER
from test_order import I64_MAX, I64_MIN, reference_order
from util import Q1_COLS, Q6_COLS, host_columns, plan_text, run_oracle

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    from mplan2vdl_b200.executor import Context
    c = Context(0)
    yield c
    c.close()


def key_sets(n, rng):
    """name -> ([(host values, dtype or 'range' (from, step))], descending)"""
    i32 = lambda a: a.astype(np.int32)                                     # noqa: E731
    return {
        "one_int64": ([rng.integers(-2**62, 2**62, n)], [False]),
        "two_dups": ([i32(rng.integers(0, 4, n)), rng.integers(-50, 50, n)], [True, False]),
        "three_range": ([i32(rng.integers(-3, 3, n)), ("range", 1000, -7), rng.integers(0, 2**20, n)], [False, True, False]),
        "eight_wide": ([rng.integers(-2**21, 2**21, n) if k % 2 else i32(rng.integers(-2**20, 2**20, n)) for k in range(8)],
                       [bool(k % 3 == 1) for k in range(8)]),
        "int64_limits": ([rng.choice(np.array([I64_MIN, I64_MAX, 0, -1], np.int64), n), rng.integers(0, 2**40, n)], [True, False]),
        "constant_then_dups": ([np.full(n, 42, np.int64), i32(rng.integers(0, 3, n))], [True, True]),
    }


def upload_keys(ctx, spec, n, tag):
    """(handles, host values as int64, column names, range handles)"""
    handles, host, names, ranges = [], [], [], []
    for j, k in enumerate(spec):
        if isinstance(k, tuple):
            _, start, step = k
            ranges.append(ctx.op_range(start, step, n))
            handles.append(ranges[-1])
            host.append(start + step * np.arange(n, dtype=np.int64))
        else:
            name = f"ord.{tag}_{j}"
            handles.append(ctx.upload_column(name, np.ascontiguousarray(k)))
            names.append(name)
            host.append(k.astype(np.int64))
    return handles, host, names, ranges


@pytest.mark.parametrize("n", [0, 1, 4095, 4096, 4097, 1_000_003])
def test_op_order_matches_the_reference(ctx, n):
    rng = np.random.default_rng(n)
    for tag, (spec, desc) in key_sets(n, rng).items():
        handles, host, names, ranges = upload_keys(ctx, spec, n, tag)
        want = reference_order(host, desc, -1)
        for limit in (-1, 0, 1, 10, 4096, n + 1):
            v = ctx.op_order(handles, desc, None if limit < 0 else limit)
            got = ctx.download(v)
            ctx.free(v)
            np.testing.assert_array_equal(got, want if limit < 0 else want[:limit], err_msg=f"{tag} n={n} limit={limit}")
        for h in ranges:
            ctx.free(h)
        for x in names:
            ctx.drop_column(x)


def test_select_refines_past_the_first_digit(ctx):
    """Over 4096 rows share the top digit of the packed key: the select must look at further digits to keep few candidates,
    and ties among them still come out in row order."""
    rng = np.random.default_rng(7)
    n = 300_000
    k = (np.int64(5) << 32) + rng.integers(0, 2**20, n)
    k[rng.integers(0, n, 100)] = (np.int64(200) << 32)             # a few rows widen the range: one top digit holds the rest
    k[rng.integers(0, n, 3000)] = (np.int64(5) << 32) + 17         # duplicates at the low end
    h = ctx.upload_column("ord.refine", k)
    for desc in (False, True):
        want = reference_order([k], [desc], -1)
        for limit in (1, 10, 100, 5000):
            v = ctx.op_order([h], [desc], limit)
            np.testing.assert_array_equal(ctx.download(v), want[:limit], err_msg=f"desc={desc} limit={limit}")
            ctx.free(v)
    ctx.drop_column("ord.refine")


def test_op_order_rejects_unequal_lengths(ctx):
    from mplan2vdl_b200.lib import VdlError
    a, b = ctx.op_range(0, 1, 10), ctx.op_range(0, 1, 11)
    with pytest.raises(VdlError, match="key 1 has 11 rows"):
        ctx.op_order([a, b], [0, 0], None)
    assert ctx.download(ctx.op_order([], None, 3)).tolist() == [0, 1, 2]


# ---- plans ----------------------------------------------------------------------------------------------------------
def ordered_reference(want: dict, keys, limit):
    from mplan2vdl_b200.executor import order_keys
    names = list(want)
    idx, desc = order_keys(names, keys)
    n = len(want[names[0]])
    perm = reference_order([want[names[i]] for i in idx], desc, -1 if limit is None else limit, n=n)
    return {k: np.asarray(v, np.int64)[perm] for k, v in want.items()}


def same(got: dict, want: dict, what=""):
    assert list(got) == list(want)
    for k in want:
        np.testing.assert_array_equal(np.asarray(got[k], np.int64), want[k], err_msg=f"{what} {k}")


def tpch_columns(catalog, text, sf):
    rows = {t: synth.table_rows(catalog, t, sf) for t in catalog.tables}
    return host_columns(catalog, tpch.plan_columns(text), rows, sf=sf)


CASES = [
    ("q03", None, True, 0.02),
    ("q10", None, True, 0.02),
    ("q18", None, True, 0.05),                                               # (no order passes HAVING on these tables: empty)
    ("q05", ([("revenue", True)], 2), True, 0.02),                             # probe fold groups: host-resident outputs
    ("q01", ([("sum_qty", True), ("count_order", False)], 2), True, 0.01),     # fused scan + post ops: host-resident outputs
    ("q03", ([("revenue", False), ("l_orderkey", True)], None), False, 0.01),  # op-at-a-time only, full order
]


@pytest.mark.parametrize("q,order,fuse,sf", CASES)
@pytest.mark.parametrize("typed", [False, True])
def test_plans_ordered_like_the_reference(catalog, ctx, q, order, fuse, sf, typed):
    keys, limit = order or ORDER[q]
    text = plan_text(q + ".vdl")
    cols = tpch_columns(catalog, text, sf)
    plain = run_oracle(text, cols)
    want = ordered_reference(plain, keys, limit)
    for k, v in cols.items():
        ctx.upload_column(k, v)
    try:
        plan = ctx.plan(text, fuse=fuse)
        plan.set_typed_outputs(typed)
        plan.set_order(keys, limit)
        for step in range(2):
            same(plan.run(), want, f"{q} step {step}")
        plan.set_order([], None)
        off = plan.run()
        ref = ctx.plan(text, fuse=fuse)
        ref.set_typed_outputs(typed)
        never = ref.run()
        for k in never:
            assert off[k].dtype == never[k].dtype and np.array_equal(off[k], never[k]), k
        same(off, {k: np.asarray(v, np.int64) for k, v in plain.items()}, f"{q} order off")
        ref.close()
        plan.close()
    finally:
        for k in cols:
            ctx.drop_column(k)


def test_order_and_sharded_tail_exclude_each_other(catalog, ctx):
    from mplan2vdl_b200.lib import VdlError
    text = plan_text("q03.vdl")
    cols = tpch_columns(catalog, text, 0.002)
    for k, v in cols.items():
        ctx.upload_column(k, v)
    try:
        plan = ctx.plan(text)
        plan.tail_enable(True)
        with pytest.raises(VdlError, match="sharded tail"):
            plan.set_order([("revenue", True)], 10)
        plan.tail_enable(False)
        plan.set_order([], 5)
        with pytest.raises(VdlError, match="sharded tail"):
            plan.tail_enable(True)
        plan.set_order([], None)
        plan.tail_enable(True)
        plan.close()
    finally:
        for k in cols:
            ctx.drop_column(k)


def test_unequal_output_lengths_and_bad_key_index_fail_with_the_message(ctx):
    from mplan2vdl_b200.lib import VdlError
    ctx.upload_column("ul.a", np.arange(5, dtype=np.int64))
    ctx.upload_column("ul.b", np.arange(7, dtype=np.int64))
    plan = ctx.plan("1,Load,ul.a\n2,Project,first,Id 1,val\n3,MaterializeCompact,Id 2\n"
                    "4,Load,ul.b\n5,Project,second,Id 4,val\n6,MaterializeCompact,Id 5\n")
    plan.set_order([("first", True)], None)
    with pytest.raises(VdlError, match="first has 5 rows, second has 7"):
        plan.run()
    with pytest.raises(VdlError, match="out of range"):
        plan._set_order([2], [False], -1)
    plan.set_order([], None)
    out = plan.run()
    assert out["first"].tolist() == list(range(5)) and out["second"].tolist() == list(range(7))
    plan.close()
    ctx.drop_column("ul.a")
    ctx.drop_column("ul.b")


@pytest.mark.parametrize("query,colnames,keys", [("q01.vdl", Q1_COLS, [("sum_charge", True)]), ("q06.vdl", Q6_COLS, [("revenue", False)])])
def test_comm_ranks_order_their_global_result(catalog, query, colnames, keys):
    from mplan2vdl_b200 import lib as L_
    from mplan2vdl_b200.executor import order_keys
    from test_gpu_comm import outputs, upload
    L = L_.load()
    rows, text, world = 70_001, plan_text(query), 2
    names = ["lineitem." + c for c in colnames]
    plain = run_oracle(text, host_columns(catalog, names, {"lineitem": rows}))
    limit = 3 if query == "q01.vdl" else None
    want = ordered_reference(plain, keys, limit)
    idx, desc = order_keys(list(plain), keys)
    comm = C.c_void_p()
    assert L.vdl_comm_init_all(world, (C.c_int * world)(0, 0), C.byref(comm)) == 0
    bases = []
    for r in range(world):
        start, n = tpch.shard_range(rows, r, world)
        c = C.c_void_p(L.vdl_comm_ctx(comm, r))
        for k, v in host_columns(catalog, names, {"lineitem": n}, row_offset=start).items():
            upload(L, c, k, np.ascontiguousarray(v))
        bases.append(start)
    cp = C.c_void_p()
    assert L.vdl_comm_plan_load(comm, text.encode(), L_.VDL_PLAN_FUSE, (C.c_int64 * world)(*bases), C.byref(cp)) == 0, L.vdl_comm_last_error(comm)
    for r in range(world):
        p = C.c_void_p(L.vdl_comm_plan_rank(cp, r))
        k = len(idx)
        assert L.vdl_plan_set_order(p, k, (C.c_int * k)(*idx), (C.c_int * k)(*[int(d) for d in desc]), -1 if limit is None else limit) == 0
    for _ in range(3):
        assert L.vdl_comm_plan_run(cp) == 0, L.vdl_comm_last_error(comm)
        for r in range(world):
            same(outputs(L, C.c_void_p(L.vdl_comm_plan_rank(cp, r))), want, f"rank {r}")
    L.vdl_comm_plan_destroy(cp)
    L.vdl_comm_destroy(comm)


def test_cli_tpch_order_q03(capsys):
    import csv
    import io
    import os
    from mplan2vdl_b200 import __main__ as cli
    path = os.path.join(tpch.PLANS_DIR, "q03.vdl")

    def rows(argv):
        assert cli.main(argv) == 0
        r = list(csv.reader(io.StringIO(capsys.readouterr().out)))
        return r[0], r[1:]
    head, plain = rows([path, "--sf", "0.01", "--csv"])
    head2, ordered = rows([path, "--sf", "0.01", "--csv", "--tpch-order"])
    assert head == head2 and len(ordered) == 10 and len(plain) > 10
    rev, date = head.index(".revenue"), head.index(".o_orderdate__orders__o_orderdate")
    want = sorted(plain, key=lambda r: (-int(r[rev]), int(r[date])))[:10]      # sorted() is stable: ties in plan order
    assert ordered == want
