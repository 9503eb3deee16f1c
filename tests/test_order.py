"""ORDER BY / LIMIT (vdl_op_order, vdl_plan_set_order, Plan.set_order, --order-by / --limit / --tpch-order) without a GPU:
the numpy reference the GPU tests compare against, checked on hand cases and against Python's own sort; name resolution;
the command line's parsing and its refusal of string-coded keys, which happens before a device is opened."""
import numpy as np
import pytest

from mplan2vdl_b200.executor import Plan, order_keys

I64_MIN, I64_MAX = np.iinfo(np.int64).min, np.iinfo(np.int64).max


def reference_order(keys, descending, limit, n=None):
    """Positions 0..n-1 ordered lexicographically over `keys` (signed int64; ~x for a descending key, exact at the int64
    limits), ties in row order; the first `limit` (limit < 0: all).  No keys: row order (n gives the length)."""
    cols = [~np.asarray(k, np.int64) if d else np.asarray(k, np.int64) for k, d in zip(keys, descending)]
    perm = np.lexsort(cols[::-1]) if cols else np.arange(n, dtype=np.int64)
    return perm if limit < 0 else perm[:limit]


def python_order(keys, descending, limit):
    n = len(keys[0])
    rows = sorted(range(n), key=lambda i: tuple(-int(k[i]) if d else int(k[i]) for k, d in zip(keys, descending)) + (i,))
    return np.array(rows if limit < 0 else rows[:limit], dtype=np.int64)


def test_ties_keep_row_order():
    k = np.array([3, 1, 3, 1, 2, 3], np.int64)
    np.testing.assert_array_equal(reference_order([k], [False], -1), [1, 3, 4, 0, 2, 5])
    np.testing.assert_array_equal(reference_order([k], [True], -1), [0, 2, 5, 4, 1, 3])


@pytest.mark.parametrize("desc", [False, True])
def test_int64_limits(desc):
    k = np.array([0, I64_MAX, I64_MIN, -1, I64_MAX, I64_MIN, 1], np.int64)
    got = reference_order([k], [desc], -1)
    want = [2, 5, 3, 0, 6, 1, 4] if not desc else [1, 4, 6, 0, 3, 2, 5]
    np.testing.assert_array_equal(got, want)


def test_constant_keys_and_second_key():
    c = np.full(5, 7, np.int64)
    k = np.array([2, 0, 2, 1, 0], np.int64)
    np.testing.assert_array_equal(reference_order([c], [True], -1), np.arange(5))
    np.testing.assert_array_equal(reference_order([c, k], [False, True], -1), [0, 2, 3, 1, 4])


def test_no_keys_is_limit_in_row_order():
    np.testing.assert_array_equal(reference_order([], [], 3, n=10), [0, 1, 2])
    np.testing.assert_array_equal(reference_order([], [], 30, n=10), np.arange(10))


@pytest.mark.parametrize("limit", [0, 1, 6, 7, 100])
def test_limits(limit):
    k = np.array([5, -5, 0, 5, 9, -5], np.int64)
    full = [1, 5, 2, 0, 3, 4]
    np.testing.assert_array_equal(reference_order([k], [False], limit), full[:limit])


@pytest.mark.parametrize("seed", range(8))
def test_reference_agrees_with_python_sort(seed):
    rng = np.random.default_rng(seed)
    n, nk = int(rng.integers(1, 300)), int(rng.integers(1, 9))
    keys = [rng.choice(np.array([I64_MIN, I64_MAX, -1, 0, 1, 2**40], np.int64), n) if rng.random() < 0.3
            else rng.integers(-4, 4, n).astype(np.int64) for _ in range(nk)]
    desc = [bool(rng.integers(0, 2)) for _ in range(nk)]
    limit = int(rng.integers(-1, n + 2))
    np.testing.assert_array_equal(reference_order(keys, desc, limit), python_order(keys, desc, limit))


# ---- name resolution (Plan.set_order without a device) ---------------------------------------------------------------
class NamesOnlyPlan(Plan):
    """A Plan whose outputs are only names: set_order resolves them and records what it would pass to the library."""

    def __init__(self, names):
        self.names, self.sent, self.h = names, None, None

    def output_names(self):
        return self.names

    def _set_order(self, idx, desc, limit):
        self.sent = (idx, desc, limit)

    def close(self):
        pass


Q3 = ["l_orderkey__lineitem__l_orderkey", "revenue", "o_orderdate__orders__o_orderdate", "o_shippriority__orders__o_shippriority"]


def test_alias_and_full_name():
    p = NamesOnlyPlan(Q3)
    p.set_order([("revenue", True), "o_orderdate"], limit=10)
    assert p.sent == ([1, 2], [True, False], 10)
    p.set_order([("o_orderdate__orders__o_orderdate", 1), ("l_orderkey", False)])
    assert p.sent == ([2, 0], [True, False], -1)
    p.set_order([], None)
    assert p.sent == ([], [], -1)


def test_unknown_and_ambiguous_names_raise_before_anything_is_set():
    p = NamesOnlyPlan(["a__t__x", "a__t__y", "b"])
    with pytest.raises(KeyError, match="no output"):
        p.set_order(["c"])
    with pytest.raises(KeyError, match="more than one"):
        p.set_order(["b", "a"])
    assert p.sent is None
    p.set_order(["a__t__y"])             # the full name is unique
    assert p.sent == ([1], [False], -1)
    assert order_keys(["x__t__x", "x"], ["x"]) == ([1], [False])     # an exact name wins over an alias


# ---- command line --------------------------------------------------------------------------------------------------
def test_parse_order_by():
    from mplan2vdl_b200.__main__ import parse_order_by
    assert parse_order_by("revenue:desc,o_orderdate") == [("revenue", True), ("o_orderdate", False)]
    assert parse_order_by(" a:ASC , b:Desc ,") == [("a", False), ("b", True)]
    assert parse_order_by("") == []
    with pytest.raises(ValueError, match="asc"):
        parse_order_by("revenue:down")


@pytest.mark.parametrize("argv,message", [
    (["plans/q05.vdl", "--order-by", "n_name:desc"], "char column"),
    (["plans/q10.vdl", "--order-by", "revenue,c_name"], "varchar column"),
    (["plans/q03.vdl", "--order-by", "nothing"], "no output"),
    (["plans/q06.vdl", "--tpch-order"], "no numeric TPC-H ORDER BY"),
    (["plans/q03.vdl", "--tpch-order", "--limit", "5"], "not with"),
    (["plans/q03.vdl", "--limit", "-1"], ">= 0"),
])
def test_cli_refuses_before_opening_a_device(argv, message, capsys, monkeypatch):
    import os

    from mplan2vdl_b200 import __main__ as cli
    from mplan2vdl_b200 import executor

    def no_device(*a, **k):
        raise AssertionError("a device was opened")
    monkeypatch.setattr(executor, "Context", no_device)
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    argv = [os.path.join(root, argv[0])] + argv[1:]
    with pytest.raises(SystemExit) as e:
        cli.main(argv)
    assert e.value.code == 2
    assert message in capsys.readouterr().err


def test_tpch_orders_name_numeric_outputs_of_the_plans(catalog):
    from mplan2vdl_b200 import tpch
    from mplan2vdl_b200.tpch_queries import ORDER
    for q, (keys, limit) in ORDER.items():
        names = tpch.plan_outputs(tpch.plan_text(q + ".vdl"))
        idx, _ = order_keys(names, keys)
        for i in idx:
            parts = names[i].split("__")
            if len(parts) == 3:
                assert catalog.column(f"{parts[1]}.{parts[2]}").mtype not in ("char", "varchar"), (q, names[i])
    assert ORDER["q03"][1] == 10 and ORDER["q10"][1] == 20 and ORDER["q18"][1] == 100
