"""ORDER BY over strings (vdl_op_collate, vdl_plan_set_order_heap, Plan.set_order(heaps=), --collate) without a GPU: the
numpy reference the GPU tests compare against, checked on hand cases and against Python's own sort; the synthetic code
heaps; the collated TPC-H orders; the command line's parsing, which happens before a device is opened."""
import os

import numpy as np
import pytest

from mplan2vdl_b200 import synth, tpch
from mplan2vdl_b200.executor import Plan
from mplan2vdl_b200.tpch_queries import COLLATED_ORDER, ORDER

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def heap_strings(values, heap, origin=0) -> list:
    """The NUL-terminated byte string each value points to (heap byte value - origin)."""
    h = np.asarray(heap, np.uint8).tobytes()
    out = []
    for v in np.asarray(values, np.int64):
        off = int(v) - origin
        assert 0 <= off < len(h), f"offset {off} outside a heap of {len(h)} bytes"
        end = h.index(b"\0", off)
        out.append(h[off:end])
    return out


def reference_collate(values, heap, origin=0):
    """vdl_op_collate in numpy: rank of each row's string among the distinct strings of `values` (unsigned byte order, a
    proper prefix first: numpy's fixed-width byte strings, whose padding is NUL, compare that way)."""
    values = np.asarray(values, np.int64)
    if len(values) == 0:
        return np.zeros(0, np.int64)
    offs, inv = np.unique(values, return_inverse=True)
    strs = heap_strings(offs, heap, origin)
    width = max(1, max(len(s) for s in strs))
    _, rank = np.unique(np.array(strs, dtype=f"S{width}"), return_inverse=True)
    return rank.reshape(-1).astype(np.int64)[inv.reshape(-1)]


def build_heap(strings, stride=None, start=0):
    """(heap bytes, offset of each string): strings laid out from `start`, each NUL-terminated, padded to `stride` (None:
    back to back)."""
    parts, offs, at = [bytes(start)], [], start
    for s in strings:
        b = s + b"\0"
        if stride:
            b = b.ljust(stride, b"\0")
        offs.append(at)
        parts.append(b)
        at += len(b)
    return np.frombuffer(b"".join(parts), np.uint8).copy(), np.array(offs, np.int64)


def python_ranks(strings):
    distinct = sorted(set(strings))
    return [distinct.index(s) for s in strings]


def test_prefix_high_bytes_and_empty_string():
    heap, offs = build_heap([b"ABC", b"AB", b"", b"\x7f", b"\x80", b"\xff\x01", b"A"])
    got = reference_collate(offs, heap)
    # '' < 'A' < 'AB' < 'ABC' < 0x7F < 0x80 < 0xFF 0x01
    np.testing.assert_array_equal(got, [3, 2, 0, 4, 5, 6, 1])


def test_equal_strings_at_different_offsets_share_a_rank():
    heap, offs = build_heap([b"R", b"N", b"R", b"A", b"N"], stride=8)
    vals = offs[[0, 1, 2, 3, 4, 2, 0]]
    np.testing.assert_array_equal(reference_collate(vals, heap), [2, 1, 2, 0, 1, 2, 2])


def test_origin_shifts_the_offsets():
    heap, offs = build_heap([b"N", b"R", b"A"], stride=24)
    codes = offs - 16                                        # codes from -16 on: heap byte 0 stands for -16
    np.testing.assert_array_equal(reference_collate(codes[[2, 0, 1, 0]], heap, origin=-16), [0, 1, 2, 1])
    assert reference_collate([], heap).shape == (0,)


@pytest.mark.parametrize("seed", range(6))
def test_reference_agrees_with_python_sort(seed):
    rng = np.random.default_rng(seed)
    alphabet = np.array([1, 2, 0x41, 0x42, 0x7F, 0x80, 0xFE, 0xFF], np.uint8)
    strings = [bytes(rng.choice(alphabet, int(rng.integers(0, 80)))) for _ in range(int(rng.integers(1, 60)))]
    heap, offs = build_heap(strings)
    rows = rng.integers(0, len(strings), 500)
    want = python_ranks([strings[i] for i in rows])
    np.testing.assert_array_equal(reference_collate(offs[rows], heap), want)


# ---- code heaps ----------------------------------------------------------------------------------------------------
CODE_COLUMNS = ["lineitem.l_returnflag", "lineitem.l_linestatus", "orders.o_orderpriority", "lineitem.l_shipmode",
                "nation.n_name", "part.p_brand", "supplier.s_name", "region.r_name", "customer.c_mktsegment"]


@pytest.mark.parametrize("col", CODE_COLUMNS)
def test_code_heap_covers_every_drawable_code(catalog, col):
    spec = synth.column_spec(catalog, col, 10)
    heap, origin = synth.code_heap(catalog, col)
    assert origin == spec.vmin
    rows = spec.p0 if spec.kind == synth.UNIFORM else synth.table_rows(catalog, col.split(".")[0], 10)
    codes = spec.vmin + spec.stride * np.arange(rows, dtype=np.int64)
    for c in codes:
        off = int(c) - origin
        assert 0 <= off and off + spec.stride <= len(heap)
        assert 0 in heap[off:off + spec.stride], f"{col}: code {c} has no NUL inside its stride"
    for s, code in catalog.dictionary.get(col, {}).items():
        if (code - spec.vmin) % spec.stride == 0 and spec.vmin <= code < spec.vmin + len(heap):
            assert heap_strings([code], heap, origin)[0] == s.encode()[:spec.stride - 1]
    # the column itself is drawn as before: its values are the codes of the recipe
    from oracle.oracle import gen_column
    n = min(1000, synth.table_rows(catalog, col.split(".")[0], 10))
    v = gen_column(spec, n, 0, synth.seed_for(10))
    assert set(np.unique(v).tolist()) <= set(codes.tolist())
    assert len(heap_strings(v, heap, origin)) == n


def test_code_heap_names_the_dictionary_strings(catalog):
    heap, origin = synth.code_heap(catalog, "lineitem.l_returnflag")
    assert origin == 16 and heap_strings([16, 40, 64], heap, origin) == [b"N", b"R", b"A"]
    heap, origin = synth.code_heap(catalog, "orders.o_orderpriority")
    assert origin == -128 and heap_strings([40, 104], heap, origin) == [b"1-URGEN", b"2-HIGH"]
    assert synth.code_heap(catalog, "orders.o_orderpriority")[0].tobytes() == heap.tobytes()     # deterministic
    with pytest.raises(ValueError, match="no code heap"):
        synth.code_heap(catalog, "lineitem.l_quantity")


# ---- collated TPC-H orders -----------------------------------------------------------------------------------------
def test_collated_orders_resolve_and_have_heaps(catalog):
    from mplan2vdl_b200.executor import order_keys
    assert set(COLLATED_ORDER) == {"q01", "q04", "q09", "q12", "q16", "q20"}
    assert not set(COLLATED_ORDER) & set(ORDER)
    for q, (keys, limit) in COLLATED_ORDER.items():
        text = tpch.plan_text(q + ".vdl")
        names = tpch.plan_outputs(text)
        idx, _ = order_keys(names, keys)
        recipes = tpch.collation_recipes(catalog, text, keys)
        assert recipes, q
        for (name, _d), i in zip(keys, idx):
            parts = names[i].split("__")
            string = len(parts) == 3 and catalog.column(f"{parts[1]}.{parts[2]}").mtype in ("char", "varchar")
            assert (name in recipes) == string, (q, name)
    assert tpch.collation_recipes(catalog, tpch.plan_text("q16.vdl"), ["p_type"]) == {"p_type": ("pool", "part.p_type")}
    assert tpch.collation_recipes(catalog, tpch.plan_text("q01.vdl"), ["l_returnflag", "sum_qty"]) == \
        {"l_returnflag": ("codes", "lineitem.l_returnflag")}


# ---- Plan.set_order(heaps=) without a device -----------------------------------------------------------------------
class NamesOnlyPlan(Plan):
    def __init__(self, names):
        self.names, self.sent, self.heaps, self.h = names, None, [], None

    def output_names(self):
        return self.names

    def _set_order(self, idx, desc, limit):
        self.sent = (idx, desc, limit)
        self.heaps = []

    def _set_order_heap(self, key, heap, origin):
        self.heaps.append((key, heap, origin))

    def close(self):
        pass


Q16 = ["p_brand__part__p_brand", "p_type__part__p_type", "p_size__part__p_size", "supplier_cnt"]


def test_heaps_name_keys_by_alias_or_full_name():
    p = NamesOnlyPlan(Q16)
    p.set_order([("supplier_cnt", True), "p_brand", "p_type"], None, {"p_type__part__p_type": 7, "p_brand": (9, -16)})
    assert p.sent == ([3, 0, 1], [True, False, False], -1)
    assert sorted(p.heaps) == [(1, 9, -16), (2, 7, 0)]
    p.set_order(["p_brand"])
    assert p.sent == ([0], [False], -1) and p.heaps == []


def test_a_heap_for_a_name_that_is_not_a_key_raises_before_anything_is_set():
    p = NamesOnlyPlan(Q16)
    with pytest.raises(KeyError, match="not among the keys"):
        p.set_order(["p_brand"], 3, {"p_type": 5})
    with pytest.raises(KeyError, match="no output"):
        p.set_order(["p_brand"], 3, {"p_nothing": 5})
    assert p.sent is None and p.heaps == []


# ---- command line --------------------------------------------------------------------------------------------------
def request(argv):
    from mplan2vdl_b200 import __main__ as cli
    from mplan2vdl_b200.meta import builtin_catalog
    import argparse
    ap = argparse.ArgumentParser()
    ap.add_argument("plan")
    ap.add_argument("--order-by", default="")
    ap.add_argument("--limit", type=int, default=None)
    ap.add_argument("--tpch-order", action="store_true")
    ap.add_argument("--collate", action="store_true")
    args = ap.parse_args([os.path.join(ROOT, argv[0])] + argv[1:])
    text = open(args.plan).read()
    return cli.order_request(args, text, builtin_catalog())


def test_collate_accepts_string_keys():
    assert request(["plans/q05.vdl", "--order-by", "n_name:desc", "--collate"]) == ([("n_name", True)], None)
    assert request(["plans/q16.vdl", "--order-by", "p_type,p_brand", "--limit", "3", "--collate"]) == \
        ([("p_type", False), ("p_brand", False)], 3)
    with pytest.raises(ValueError, match="char column"):
        request(["plans/q05.vdl", "--order-by", "n_name:desc"])


def test_collate_with_numeric_keys_changes_nothing():
    for argv in (["plans/q03.vdl", "--order-by", "revenue:desc", "--limit", "10"], ["plans/q03.vdl", "--tpch-order"]):
        assert request(argv + ["--collate"]) == request(argv)


@pytest.mark.parametrize("q", sorted(COLLATED_ORDER))
def test_tpch_order_collate_resolves_the_string_plans(q):
    assert request([f"plans/{q}.vdl", "--tpch-order", "--collate"]) == COLLATED_ORDER[q]
    with pytest.raises(ValueError, match="no numeric TPC-H ORDER BY"):
        request([f"plans/{q}.vdl", "--tpch-order"])


@pytest.mark.parametrize("argv,message", [
    (["plans/q05.vdl", "--order-by", "n_name:desc"], "char column"),
    (["plans/q06.vdl", "--tpch-order", "--collate"], "no TPC-H ORDER BY"),
    (["plans/q16.vdl", "--order-by", "nothing", "--collate"], "no output"),
])
def test_cli_refuses_before_opening_a_device(argv, message, capsys, monkeypatch):
    from mplan2vdl_b200 import __main__ as cli
    from mplan2vdl_b200 import executor

    def no_device(*a, **k):
        raise AssertionError("a device was opened")
    monkeypatch.setattr(executor, "Context", no_device)
    with pytest.raises(SystemExit) as e:
        cli.main([os.path.join(ROOT, argv[0])] + argv[1:])
    assert e.value.code == 2
    assert message in capsys.readouterr().err


def test_collation_heaps_build_bytes_only_for_heaps_not_on_the_device(catalog, monkeypatch):
    """A heap already on the device is looked up, not rebuilt; a code heap is uploaded under a name no plan Loads, with
    code_heap's origin."""
    from mplan2vdl_b200.lib import VdlError

    class FakeCtx:
        def __init__(self, present):
            self.present, self.uploaded = dict(present), []

        def lookup(self, name):
            if name not in self.present:
                raise VdlError(3, f"{name} is not registered")
            return self.present[name]

        def upload_column(self, name, arr):
            self.uploaded.append((name, arr.tobytes()))
            self.present[name] = 100 + len(self.present)
            return self.present[name]

    text = tpch.plan_text("q16.vdl")
    keys = COLLATED_ORDER["q16"][0]
    ctx = FakeCtx({"part.p_type.heap": 7})
    heaps = tpch.collation_heaps(ctx, catalog, text, keys)
    code, origin = synth.code_heap(catalog, "part.p_brand")
    assert heaps == {"p_type": (7, 0), "p_brand": (101, origin)}
    assert ctx.uploaded == [(tpch.CODE_HEAP_PREFIX + "part.p_brand", code.tobytes())]

    def no_build(*a, **k):
        raise AssertionError("heap bytes built for a heap already on the device")
    monkeypatch.setattr(synth, "code_heap", no_build)
    monkeypatch.setattr(synth, "string_heap", no_build)
    assert tpch.collation_heaps(ctx, catalog, text, keys) == heaps
