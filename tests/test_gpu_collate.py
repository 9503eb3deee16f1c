"""ORDER BY over strings on the GPU: vdl_op_collate against the numpy reference (tests/test_collate.py) over row counts
around the select tile, on hand-made heaps (long strings that share a prefix and first differ at byte 63, 64 or 65, bytes
>= 0x80, duplicates at different offsets, offsets aligned to 1..8 bytes), the synthetic p_type / p_name pools and a code
heap below zero; the TPC-H plans ordered by their string keys (vdl_plan_set_order_heap) against the CPU oracle's result
ordered by the reference, on one GPU and on two ranks of vdl_comm; the command line."""
import ctypes as C

import numpy as np
import pytest

from mplan2vdl_b200 import synth, tpch
from mplan2vdl_b200.tpch_queries import COLLATED_ORDER
from test_collate import build_heap, reference_collate
from test_gpu_order import ordered_reference, same, tpch_columns
from test_order import reference_order
from util import plan_text, run_oracle

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    from mplan2vdl_b200.executor import Context
    c = Context(0)
    yield c
    c.close()


def long_strings():
    """Strings of 0..200 bytes: a shared 80-byte prefix with bytes >= 0x80, cut or changed at bytes 63, 64 and 65 (the edge
    of the first 8-word chunk), short ASCII strings and the empty string."""
    p = bytes(1 + (0x80 + 37 * i) % 255 for i in range(200))
    out = [b"", b"A", b"AB", b"\x7f", b"\x80", b"\xff", p, p[:63], p[:64], p[:65], p[:66]]
    for at in (63, 64, 65):
        for c in (b"\x01", b"A", b"\x90", b"\xfe"):
            out.append(p[:at] + c + p[at + 1:at + 20])
    return out


def datasets(catalog, n, rng):
    """name -> (values, heap bytes, origin)"""
    out = {}
    three, offs3 = build_heap([b"N", b"R", b"A"], stride=24, start=16)
    out["three_int64"] = (offs3[rng.integers(0, 3, n)], three, 0)
    strings = long_strings()
    for align in (1, 2, 4, 8):                    # offsets aligned to 2^a, a = 0..3; every string twice (duplicates)
        # zero bytes after a string (to the next multiple of 2^a) end it as its NUL would
        heap, offs = build_heap([s + bytes(-(len(s) + 1) % align) for s in strings + strings], start=align)
        vals = offs[rng.integers(0, len(offs), n)]
        out[f"long_align{align}"] = (vals.astype(np.int32) if align in (1, 4) else vals, heap, 0)
    for col in ("part.p_type", "part.p_name"):
        heap, _ = synth.string_heap(catalog, col)
        out[col] = (synth.string_offsets(catalog, col, n, 17, 99), heap, 0)
    heap, origin = synth.code_heap(catalog, "orders.o_orderpriority")
    out["o_orderpriority_codes"] = ((origin + 8 * rng.integers(0, 30, n)).astype(np.int32), heap, origin)
    heap, origin = synth.code_heap(catalog, "supplier.s_name")             # ~400 k codes, many equal strings
    out["s_name_codes"] = (origin + 8 * rng.integers(0, len(heap) // 8, n), heap, origin)
    return out


@pytest.mark.parametrize("n", [0, 1, 4095, 4096, 4097, 1_000_003])
def test_op_collate_matches_the_reference(catalog, ctx, n):
    rng = np.random.default_rng(n)
    for name, (vals, heap, origin) in datasets(catalog, n, rng).items():
        d = ctx.upload_column("coll.data", np.ascontiguousarray(vals))
        h = ctx.upload_column("coll.heap", heap)
        try:
            v = ctx.op_collate(d, h, origin)
            got = ctx.download(v)
            ctx.free(v)
            np.testing.assert_array_equal(got, reference_collate(vals, heap, origin), err_msg=f"{name} n={n}")
        finally:
            ctx.drop_column("coll.data")
            ctx.drop_column("coll.heap")


def test_op_collate_reports_an_offset_past_the_heap(ctx):
    from mplan2vdl_b200.lib import VdlError
    heap, offs = build_heap([b"B", b"A"], stride=8)
    d = ctx.upload_column("coll.bad", np.array([offs[0], len(heap) + 8, offs[1]], np.int64))
    h = ctx.upload_column("coll.badheap", heap)
    ctx.free(ctx.op_collate(d, h, 0))
    probe = "1,Load,coll.bad\n2,Project,out,Id 1,val\n3,MaterializeCompact,Id 2\n"
    with pytest.raises(VdlError) as e:               # the range error, at the next check
        ctx.plan(probe).run()
    assert e.value.code == 5
    assert ctx.plan(probe).run()["out"].tolist() == [0, len(heap) + 8, 8]      # reported once, the context still works
    with pytest.raises(VdlError, match="string heap"):
        ctx.op_collate(d, d, 0)
    ctx.drop_column("coll.bad")
    ctx.drop_column("coll.badheap")


# ---- plans ----------------------------------------------------------------------------------------------------------
def collated_reference(catalog, text, want: dict, keys, limit):
    """The oracle's unordered result ordered by `keys`, string keys by the reference ranks of their strings."""
    from mplan2vdl_b200.executor import order_keys
    names = list(want)
    recipes = tpch.collation_recipes(catalog, text, keys)
    idx, desc = order_keys(names, keys)
    cols = []
    for (name, _d), i in zip(keys, idx):
        vals = np.asarray(want[names[i]], np.int64)
        if name in recipes:
            kind, q = recipes[name]
            heap, origin = (synth.string_heap(catalog, q)[0], 0) if kind == "pool" else synth.code_heap(catalog, q)
            vals = reference_collate(vals, heap, origin)
        cols.append(vals)
    perm = reference_order(cols, desc, -1 if limit is None else limit, n=len(want[names[0]]))
    return {k: np.asarray(v, np.int64)[perm] for k, v in want.items()}


CASES = [(q, lim) for q in sorted(COLLATED_ORDER) for lim in (None, 3)]


@pytest.mark.parametrize("q,limit", CASES)
def test_plans_ordered_by_their_strings(catalog, ctx, q, limit):
    keys = COLLATED_ORDER[q][0]
    text, sf = plan_text(q + ".vdl"), 0.01
    cols = tpch_columns(catalog, text, sf)
    plain = run_oracle(text, cols)
    want = collated_reference(catalog, text, plain, keys, limit)
    for k, v in cols.items():
        ctx.upload_column(k, v)
    heaps = {}
    try:
        plan = ctx.plan(text)
        heaps = tpch.collation_heaps(ctx, catalog, text, keys)
        plan.set_order(keys, limit, heaps)
        for step in range(2):
            same(plan.run(), want, f"{q} step {step}")
        # heaps cleared one by one: the keys compare by their codes again
        for k in range(len(keys)):
            plan._set_order_heap(k, 0, 0)
        same(plan.run(), ordered_reference(plain, keys, limit), f"{q} heaps cleared")
        plan.set_order(keys, limit, heaps)
        plan.set_order(keys, limit)                  # a later set_order clears every heap
        same(plan.run(), ordered_reference(plain, keys, limit), f"{q} set_order again")
        plan.set_order([], None)
        off = plan.run()
        ref = ctx.plan(text)
        never = ref.run()
        for k in never:
            assert off[k].dtype == never[k].dtype and np.array_equal(off[k], never[k]), k
        ref.close()
        plan.close()
    finally:
        for k in cols:
            ctx.drop_column(k)
        for _name, (kind, col) in tpch.collation_recipes(catalog, text, keys).items():
            if kind == "codes":
                ctx.drop_column(tpch.CODE_HEAP_PREFIX + col)


def test_set_order_heap_refuses_a_bad_key_or_heap(ctx):
    from mplan2vdl_b200.lib import VdlError
    ctx.upload_column("sh.a", np.arange(5, dtype=np.int64))
    h = ctx.upload_column("sh.heap", np.zeros(8, np.uint8))
    plan = ctx.plan("1,Load,sh.a\n2,Project,a,Id 1,val\n3,MaterializeCompact,Id 2\n")
    plan.set_order(["a"])
    with pytest.raises(VdlError, match="out of range"):
        plan._set_order_heap(1, h, 0)
    with pytest.raises(VdlError, match="not a string heap"):
        plan._set_order_heap(0, ctx.lookup("sh.a"), 0)
    plan.close()
    ctx.drop_column("sh.a")
    ctx.drop_column("sh.heap")


def test_comm_ranks_order_q12_by_its_strings(catalog):
    from mplan2vdl_b200 import lib as L_
    from mplan2vdl_b200.executor import order_keys
    from test_gpu_comm import outputs, upload
    L = L_.load()
    text, sf, world = plan_text("q12.vdl"), 0.02, 2
    keys, limit = COLLATED_ORDER["q12"]
    rows = {t: synth.table_rows(catalog, t, sf) for t in catalog.tables}
    cols = host_columns_for(catalog, text, rows, sf)
    plain = run_oracle(text, cols)
    want = collated_reference(catalog, text, plain, keys, limit)
    idx, desc = order_keys(list(plain), keys)
    heap, origin = synth.code_heap(catalog, "lineitem.l_shipmode")
    comm = C.c_void_p()
    assert L.vdl_comm_init_all(world, (C.c_int * world)(0, 0), C.byref(comm)) == 0
    bases, heap_of = [], []
    for r in range(world):
        start, n = tpch.shard_range(rows["lineitem"], r, world)
        c = C.c_void_p(L.vdl_comm_ctx(comm, r))
        for k, v in cols.items():
            upload(L, c, k, np.ascontiguousarray(v[start:start + n] if k.startswith("lineitem.") else v))
        upload(L, c, "collate:lineitem.l_shipmode", heap)
        hv = C.c_int32()
        assert L.vdl_column_lookup(c, b"collate:lineitem.l_shipmode", C.byref(hv)) == 0
        heap_of.append(hv.value)
        bases.append(start)
    cp = C.c_void_p()
    assert L.vdl_comm_plan_load(comm, text.encode(), L_.VDL_PLAN_FUSE, (C.c_int64 * world)(*bases), C.byref(cp)) == 0, L.vdl_comm_last_error(comm)
    for r in range(world):
        p = C.c_void_p(L.vdl_comm_plan_rank(cp, r))
        k = len(idx)
        assert L.vdl_plan_set_order(p, k, (C.c_int * k)(*idx), (C.c_int * k)(*[int(d) for d in desc]), -1) == 0
        assert L.vdl_plan_set_order_heap(p, 0, heap_of[r], origin) == 0
    for _ in range(3):
        assert L.vdl_comm_plan_run(cp) == 0, L.vdl_comm_last_error(comm)
        for r in range(world):
            same(outputs(L, C.c_void_p(L.vdl_comm_plan_rank(cp, r))), want, f"rank {r}")
    L.vdl_comm_plan_destroy(cp)
    L.vdl_comm_destroy(comm)


def host_columns_for(catalog, text, rows, sf):
    from util import host_columns
    return host_columns(catalog, tpch.plan_columns(text), rows, sf=sf)


def test_cli_q01_collated_prints_a_before_n_before_r(capsys):
    import csv
    import io
    import os
    from mplan2vdl_b200 import __main__ as cli
    path = os.path.join(tpch.PLANS_DIR, "q01.vdl")
    assert cli.main([path, "--sf", "0.01", "--csv", "--tpch-order", "--collate"]) == 0
    r = list(csv.reader(io.StringIO(capsys.readouterr().out)))
    head, rows = r[0], r[1:]
    flag = [i for i, h in enumerate(head) if "l_returnflag" in h][0]
    got = [row[flag] for row in rows]
    assert set(got) == {"A", "N", "R"} and got == sorted(got), got
