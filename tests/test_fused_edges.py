"""The fused select -> map -> fold scan against a plain reference of its descriptor, at the edges of its int32 proofs.

vdl_fused_prepare picks one of several kernel families for a descriptor -- the generic kernel, the static shapes
sel3_sum2 / sel1_key2_sum5 (vdl_shapes.cuh), the NVRTC-specialised kernel with shared-memory tables or with register
slots -- and decides from the column statistics how each value is computed: an affine term in 32 bits (FF_NARROW), an
8-byte predicate column compared on its low words (mode 2), a register-slot sum kept in 32 bits (RK_N32) or as a
32x32+64 multiply-add (RK_MADW).  Every family must give the same answer as the descriptor's definition
(include/vdl_cuda.h), which `reference` below states with wrapping uint64 numpy.  The CPU tests anchor that reference to
the oracle through plan texts; the GPU tests run each descriptor on every family that can take it, with data placed on
both sides of each proof's boundary: raw 8-byte values beyond int32 whose shifted values fit, min/max exactly at the
int32 limits and one beyond, more keys than register slots, row counts around the tile size, and the rows a thread
folds per tile in the register-slot kernels."""
import ctypes as C
import re

import numpy as np
import pytest

from util import assert_same, run_gpu, run_oracle

I32_MIN, I32_MAX = -2**31, 2**31 - 1
I64_MIN, I64_MAX = -2**63, 2**63 - 1
M64 = 2**64 - 1
SUM, MIN, MAX, CHOOSE, COUNT = 0, 1, 2, 3, 4
ADD, SUBTRACT, MULTIPLY, DIVIDE, MODULO = 6, 7, 9, 10, 11
P_FOLD, P_POST, P_CONST = 0, 1, 2
ROWID, CONST = -2, -1
RK_WIDE, RK_N32, RK_FIRST, RK_MADW = 0, 1, 2, 3


def T(col, shr=0, a=0, b=1):
    """An affine term a + b * (column >> shr) (column -2: the global row id, -1: the constant a)."""
    return (col, shr, a, b)


def spec(cols, preds=(), keys=(), key_mask=-1, domain=1, folds=(), posts=(), row_base=0):
    """A fused-scan descriptor over host columns: preds (col, shr, lo, hi); keys (term, shl); folds (op, [terms]);
    posts (op, (kind, value), (kind, value))."""
    return dict(cols=list(cols), preds=list(preds), keys=list(keys), key_mask=key_mask, domain=domain, folds=list(folds),
                posts=list(posts), row_base=row_base)


# ---------------------------------------------------------------------------------------------------- the reference
def _wrap(x):
    x &= M64
    return x - (1 << 64) if x >> 63 else x


def _binop(op, a, b):
    """binop_apply (oracle/vdl_oracle.c) on Python ints: wrapping arithmetic, C division, x / 0 = 0, x / -1 = -x."""
    if op == ADD:
        return _wrap(a + b)
    if op == SUBTRACT:
        return _wrap(a - b)
    if op == MULTIPLY:
        return _wrap(a * b)
    if op == DIVIDE:
        if b == 0:
            return 0
        if b == -1:
            return _wrap(-a)
        q = abs(a) // abs(b)
        return q if (a < 0) == (b < 0) else -q
    if op == MODULO:
        if b in (0, -1):
            return 0
        r = abs(a) % abs(b)
        return -r if a < 0 else r
    raise ValueError(op)


def _term(s, t, rows):
    col, shr, a, b = t
    if col == CONST:
        return np.full(rows, a, np.int64)
    if col == ROWID:
        leaf = np.arange(rows, dtype=np.int64) + np.int64(s["row_base"])
    else:
        leaf = s["cols"][col][:rows].astype(np.int64) >> np.int64(shr)
    return (np.uint64(a & M64) + np.uint64(b & M64) * leaf.view(np.uint64)).view(np.int64)


def reference(s, rows):
    """What vdl_fused_desc means (include/vdl_cuda.h): ([one int64 array per fold], [one per post op]), one entry per
    key that saw a selected row, ascending key order."""
    sel = np.ones(rows, bool)
    for col, shr, lo, hi in s["preds"]:
        v = s["cols"][col][:rows].astype(np.int64) >> np.int64(shr)
        sel &= (v >= np.int64(lo)) & (v <= np.int64(hi))
    key = np.zeros(rows, np.uint64)
    for t, shl in s["keys"]:
        key |= _term(s, t, rows).view(np.uint64) << np.uint64(shl)
    key = (key & np.uint64(s["key_mask"] & M64)).view(np.int64)
    rowsel = np.flatnonzero(sel)
    ks = key[rowsel]
    assert ((ks >= 0) & (ks < s["domain"])).all(), "the descriptor's keys must lie in [0, domain)"
    order = np.argsort(ks, kind="stable")            # selected rows by key, ascending row order inside a key
    srows, ks = rowsel[order], ks[order]
    _, starts = np.unique(ks, return_index=True)
    n = len(starts)
    folds = []
    for op, factors in s["folds"]:
        if op == COUNT:
            folds.append(np.diff(np.append(starts, len(ks))).astype(np.int64))
            continue
        val = np.ones(rows, np.uint64)
        for t in factors:
            val = val * _term(s, t, rows).view(np.uint64)
        val = val[srows]
        if n == 0:
            folds.append(np.zeros(0, np.int64))
        elif op == SUM:
            folds.append(np.add.reduceat(val, starts).view(np.int64))
        elif op == MIN:
            folds.append(np.minimum.reduceat(val.view(np.int64), starts))
        elif op == MAX:
            folds.append(np.maximum.reduceat(val.view(np.int64), starts))
        elif op == CHOOSE:
            folds.append(val.view(np.int64)[starts])
        else:
            raise ValueError(op)
    posts = []
    for op, (ak, av), (bk, bv) in s["posts"]:
        def operand(kind, v, g):
            return v if kind == P_CONST else int((folds if kind == P_FOLD else posts)[v][g])
        posts.append(np.array([_binop(op, operand(ak, av, g), operand(bk, bv, g)) for g in range(n)], dtype=np.int64))
    return folds, posts


# ---------------------------------------------------------------------------------------------------- plan texts
# Each plan states a descriptor in the form the fusion pass rewrites (Vlite.hs:721-730, 1048-1098); _plan_cases pairs it with
# that descriptor over the columns in the order given.
SHIFTED_PRED = """1,Load,t.x
2,Project,val,Id 1,x
3,RangeV,val,1,Id 2,0
4,BitShift,val,Id 2,val,Id 3,val
5,RangeV,val,1073741823,Id 2,0
6,Greater,val,Id 4,val,Id 5,val
7,RangeV,val,0,Id 6,1
8,FoldSelect,val,Id 7,val,Id 6,val
9,Gather,Id 2,Id 8,val
10,RangeV,val,0,Id 9,0
11,FoldSum,val,Id 10,val,Id 9,val
12,Project,s,Id 11,val
13,MaterializeCompact,Id 12
14,RangeV,val,1,Id 9,0
15,FoldSum,val,Id 10,val,Id 14,val
16,Project,c,Id 15,val
17,MaterializeCompact,Id 16
"""

SHIFTED_VALUE = """1,Load,t.x
2,Project,val,Id 1,x
3,Load,t.y
4,Project,val,Id 3,y
5,RangeV,val,0,Id 4,0
6,Greater,val,Id 4,val,Id 5,val
7,RangeV,val,0,Id 6,1
8,FoldSelect,val,Id 7,val,Id 6,val
9,Gather,Id 2,Id 8,val
10,RangeV,val,4,Id 9,0
11,BitShift,val,Id 9,val,Id 10,val
12,RangeV,val,0,Id 11,0
13,FoldSum,val,Id 12,val,Id 11,val
14,Project,s,Id 13,val
15,MaterializeCompact,Id 14
"""

# key = (((k >> 30) << 3) | ((j >> 2) - 1)) & 63, sorted by Partition + Scatter as plans/q01.vdl does
SHIFTED_KEY = """1,Load,t.k
2,Project,val,Id 1,k
3,Load,t.j
4,Project,val,Id 3,j
5,Load,t.v
6,Project,val,Id 5,v
7,RangeV,val,0,Id 6,0
8,Greater,val,Id 6,val,Id 7,val
9,RangeV,val,0,Id 8,1
10,FoldSelect,val,Id 9,val,Id 8,val
11,Gather,Id 2,Id 10,val
12,RangeV,val,30,Id 11,0
13,BitShift,val,Id 11,val,Id 12,val
14,RangeV,val,0,Id 13,0
15,RangeV,val,3,Id 13,0
16,Subtract,val,Id 14,val,Id 15,val
17,BitShift,val,Id 13,val,Id 16,val
18,Gather,Id 4,Id 10,val
19,RangeV,val,2,Id 18,0
20,BitShift,val,Id 18,val,Id 19,val
21,RangeV,val,1,Id 20,0
22,Subtract,val,Id 20,val,Id 21,val
23,BitwiseOr,val,Id 17,val,Id 22,val
24,RangeV,val,63,Id 23,0
25,BitwiseAnd,val,Id 23,val,Id 24,val
26,RangeV,val,0,Id 25,1
27,RangeC,val,0,64,1
28,Partition,val,Id 25,val,Id 27,val
29,Scatter,Id 25,Id 26,val,Id 28,val
30,Gather,Id 6,Id 10,val
31,RangeV,val,0,Id 30,1
32,Scatter,Id 30,Id 31,val,Id 28,val
33,FoldSum,val,Id 29,val,Id 32,val
34,Project,s,Id 33,val
35,MaterializeCompact,Id 34
36,RangeV,val,1,Id 30,0
37,RangeV,val,0,Id 36,1
38,Scatter,Id 36,Id 37,val,Id 28,val
39,FoldSum,val,Id 29,val,Id 38,val
40,Project,c,Id 39,val
41,MaterializeCompact,Id 40
"""


def _plan_cases(rows=1000, seed=0):
    """(name, plan text, {column: array}, descriptor, output names); the descriptor's columns in dict order."""
    rng = np.random.default_rng(seed)
    x = rng.integers(2**31, 2**32, rows, dtype=np.int64)                       # x >> 1 fits int32, x does not
    pred = ("shifted_pred", SHIFTED_PRED, {"t.x": x},
            spec([x], preds=[(0, 1, 2**30, I64_MAX)], folds=[(SUM, [T(0)]), (SUM, [])]), ["s", "c"])
    x = rng.integers(2**31, 2**35, rows, dtype=np.int64)                       # x >> 4 fits int32, x does not
    y = rng.integers(-3, 4, rows).astype(np.int32)
    value = ("shifted_value", SHIFTED_VALUE, {"t.x": x, "t.y": y},
             spec([x, y], preds=[(1, 0, 1, I64_MAX)], folds=[(SUM, [T(0, 4)])]), ["s"])
    k = rng.integers(2**40, 2**48, rows, dtype=np.int64)                       # k >> 30 fits int32, k does not; bit 32 of k is a key bit
    j = rng.integers(4, 36, rows).astype(np.int32)
    v = rng.integers(-5, 1000, rows, dtype=np.int64)
    key = ("shifted_key", SHIFTED_KEY, {"t.k": k, "t.j": j, "t.v": v},
           spec([k, j, v], preds=[(2, 0, 1, I64_MAX)], keys=[(T(0, 30), 3), (T(1, 2, -1), 0)], key_mask=63, domain=64,
                folds=[(SUM, [T(2)]), (COUNT, [])]), ["s", "c"])
    return [pred, value, key]


@pytest.mark.parametrize("case", range(3), ids=["shifted_pred", "shifted_value", "shifted_key"])
def test_reference_matches_oracle_on_plans(case):
    name, text, cols, s, outs = _plan_cases()[case]
    want = run_oracle(text, cols)
    folds, _ = reference(s, len(next(iter(cols.values()))))
    assert list(want) == outs
    assert_same(want, dict(zip(outs, folds)))
    if name == "shifted_pred":
        assert len(want["c"]) == 1 and want["c"][0] == 1000      # every row passes: (x >> 1) > 2^30 - 1 for x >= 2^31


def test_reference_definitions():
    """The reference's own edges, spelled out: wrapping products and sums, MIN / MAX of wrapped products, CHOOSE = the
    first selected row of a key, row ids from row_base, empty keys dropped, post ops with binop_apply's division."""
    c = np.array([I64_MIN, I64_MAX, 3, -7, 2**62], np.int64)
    g = np.array([1, 1, 3, 3, 1], np.int32)
    s = spec([c, g], preds=[(0, 63, -1, 0)], keys=[(T(1), 0)], key_mask=3, domain=4, row_base=2**40,
             folds=[(SUM, [T(0), T(0)]), (MIN, [T(0), T(CONST, 0, 2)]), (MAX, [T(0)]), (CHOOSE, [T(ROWID, 0, 1, 3)]),
                    (COUNT, [])],
             posts=[(DIVIDE, (P_FOLD, 2), (P_CONST, -1)), (MODULO, (P_FOLD, 1), (P_CONST, -1)),
                    (DIVIDE, (P_FOLD, 1), (P_CONST, 0)), (DIVIDE, (P_POST, 0), (P_CONST, -7)), (MODULO, (P_FOLD, 2), (P_CONST, 10))])
    folds, posts = reference(s, 5)
    sq = [_wrap(v * v) for v in c.tolist()]
    assert folds[0].tolist() == [_wrap(sq[0] + sq[1] + sq[4]), _wrap(sq[2] + sq[3])]
    assert folds[1].tolist() == [min(_wrap(2 * v) for v in (I64_MIN, I64_MAX, 2**62)), -14]
    assert folds[2].tolist() == [I64_MAX, 3]
    assert folds[3].tolist() == [1 + 3 * 2**40, 1 + 3 * (2**40 + 2)]
    assert folds[4].tolist() == [3, 2]
    assert posts[0].tolist() == [-I64_MAX, -3]
    assert posts[1].tolist() == [0, 0] and posts[2].tolist() == [0, 0]
    assert posts[3].tolist() == [I64_MAX // 7, 0] and posts[4].tolist() == [I64_MAX % 10, 3]
    empty = spec([c], preds=[(0, 0, 5, 4)], folds=[(SUM, [T(0)])])
    assert [len(f) for f in reference(empty, 5)[0]] == [0]


def test_plans_fuse_to_one_scan():
    """The plan-level GPU tests below are only about the fused scan if the planner fuses these plans."""
    from mplan2vdl_b200.executor import explain
    for name, text, cols, s, _ in _plan_cases(rows=10):
        fs = explain(text)["fused_scans"]
        assert len(fs) == 1, name
        assert fs[0]["predicates"] == len(s["preds"]) and fs[0]["key_parts"] == len(s["keys"]), (name, fs)
        assert fs[0]["domain"] == s["domain"], (name, fs)


# ---------------------------------------------------------------------------------------------------- GPU: families
# environment switches read by vdl_fused_prepare, and what each family asserts about the kernel it got
SWITCHES = ["VDL_GENERIC_ONLY", "VDL_SCAN_JIT", "VDL_SCAN_JIT_MIN_ROWS", "VDL_NO_REGISTER_SLOTS", "VDL_RS_GEOMETRY",
            "VDL_RS_ALL_SLOTS", "VDL_DEBUG_SHAPE", "VDL_DEBUG_JIT"]
FAMILIES = {
    "generic": {"VDL_GENERIC_ONLY": "1"},
    "static": {"VDL_SCAN_JIT": "0"},
    "static_tables": {"VDL_SCAN_JIT": "0", "VDL_NO_REGISTER_SLOTS": "1"},
    "jit_tables": {"VDL_SCAN_JIT_MIN_ROWS": "0", "VDL_NO_REGISTER_SLOTS": "1"},
    "jit_rs_352x4": {"VDL_SCAN_JIT_MIN_ROWS": "0", "VDL_RS_GEOMETRY": "352,4"},
    "jit_rs_352x2": {"VDL_SCAN_JIT_MIN_ROWS": "0", "VDL_RS_GEOMETRY": "352,2"},
    "jit_rs_480x2": {"VDL_SCAN_JIT_MIN_ROWS": "0", "VDL_RS_GEOMETRY": "480,2"},
}
RS_FAMILIES = ["jit_rs_352x4", "jit_rs_352x2", "jit_rs_480x2"]
SHAPE_LINE = re.compile(r"\[vdl\] fused scan: shape=(\S+)( \(register slots\))? nc=(\d+) r=(\d+)")
ACC_RK = re.compile(r"ACC_RK\[K_MAX_ACC\] = \{([^}]*)\}")


@pytest.fixture(scope="module")
def ctx():
    from mplan2vdl_b200.executor import Context
    c = Context(0)                       # one context for the module: its NVRTC cache serves every case
    yield c
    c.close()


@pytest.fixture(scope="module")
def sm_count():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def _family(monkeypatch, family):
    for k in SWITCHES:
        monkeypatch.delenv(k, raising=False)
    for k, v in FAMILIES[family].items():
        monkeypatch.setenv(k, v)
    monkeypatch.setenv("VDL_DEBUG_SHAPE", "1")
    monkeypatch.setenv("VDL_DEBUG_JIT", "1")


class Uploaded:
    """The columns of a spec registered in the context (dropped on close)."""
    _n = 0

    def __init__(self, ctx, s):
        Uploaded._n += 1
        self.ctx, self.names = ctx, [f"edge{Uploaded._n}.c{i}" for i in range(len(s["cols"]))]
        self.handles = [ctx.upload_column(n, np.ascontiguousarray(a)) for n, a in zip(self.names, s["cols"])]

    def close(self):
        for n in self.names:
            self.ctx.drop_column(n)


def _desc(s, handles, rows):
    from mplan2vdl_b200 import lib as L_
    d = L_.FusedDesc()
    d.rows, d.row_base, d.ncolumns = rows, s["row_base"], len(handles)
    for i, h in enumerate(handles):
        d.column[i] = h
    d.npreds = len(s["preds"])
    for i, p in enumerate(s["preds"]):
        d.pred[i] = L_.RangePred(*p)
    d.nkeys = len(s["keys"])
    for i, (t, shl) in enumerate(s["keys"]):
        d.key[i].e = L_.Affine(*t)
        d.key[i].shl = shl
    d.key_mask, d.domain, d.nfolds = s["key_mask"], s["domain"], len(s["folds"])
    for i, (op, factors) in enumerate(s["folds"]):
        d.fold[i].op, d.fold[i].nfactors = op, len(factors)
        for t, f in enumerate(factors):
            d.fold[i].factor[t] = L_.Affine(*f)
    d.nposts = len(s["posts"])
    for q, (op, (ak, av), (bk, bv)) in enumerate(s["posts"]):
        d.post[q] = L_.PostOp(op, ak, bk, 0, av, bv)
    return d


class Scan:
    """A prepared fused scan: the kernel it got (shape name, register slots, geometry, ACC_RK of a run-time shape)."""

    def __init__(self, ctx, capfd, s, handles, rows):
        capfd.readouterr()
        self.ctx, self.s, self.rows = ctx, s, rows
        self.d = _desc(s, handles, rows)
        self.f = C.c_void_p()
        ctx.check(ctx.L.vdl_fused_prepare(ctx.h, C.byref(self.d), C.byref(self.f)))
        self.shape = ctx.L.vdl_fused_shape_name(self.f).decode()
        err = capfd.readouterr().err
        m = SHAPE_LINE.findall(err)
        assert m, err
        shape, rs, nc, r = m[-1]
        assert shape == self.shape
        self.rs, self.nc, self.r = bool(rs), int(nc), int(r)
        rk = ACC_RK.findall(err)
        self.acc_rk = [int(x) for x in rk[-1].split(",")] if rk and self.rs else None

    def launch(self):
        """One single-GPU step (the scan kernel's last CTA finalizes): ([fold results], [post results])."""
        L, f = self.ctx.L, self.f
        self.ctx.check(L.vdl_fused_launch_ex(f, 1))
        data, n = C.POINTER(C.c_int64)(), C.c_int64()
        folds, posts = [], []
        for i in range(len(self.s["folds"])):
            self.ctx.check(L.vdl_fused_result_host(f, i, C.byref(data), C.byref(n)))
            folds.append(np.ctypeslib.as_array(data, shape=(n.value,)).copy() if n.value else np.zeros(0, np.int64))
        for q in range(len(self.s["posts"])):
            self.ctx.check(L.vdl_fused_post_host(f, q, C.byref(data), C.byref(n)))
            posts.append(np.ctypeslib.as_array(data, shape=(n.value,)).copy() if n.value else np.zeros(0, np.int64))
        return folds, posts

    def close(self):
        self.ctx.L.vdl_fused_destroy(self.f)


def _expect_family(scan, family, expect):
    """expect: the static shape name the case matches ("generic" if none) for the static families; "rs" / "tables" for
    the run-time shapes."""
    if family == "generic":
        assert scan.shape == "generic" and not scan.rs
    elif family.startswith("static"):
        assert scan.shape == expect
        assert scan.rs == (family == "static" and expect == "sel1_key2_sum5")
    else:
        assert scan.shape.startswith("jit:"), (family, scan.shape)
        assert scan.rs == (expect == "rs" and family in RS_FAMILIES), (family, expect)
        if scan.rs:
            assert (scan.nc, scan.r) == tuple(int(x) for x in FAMILIES[family]["VDL_RS_GEOMETRY"].split(","))


def _check(ctx, capfd, s, rows, family, expect, handles):
    scan = Scan(ctx, capfd, s, handles, rows)
    try:
        _expect_family(scan, family, expect)
        want_f, want_p = reference(s, rows)
        for step in range(2):             # the epilogue reset the table and the ticket: the second step is a fresh one
            got_f, got_p = scan.launch()
            for i, (g, w) in enumerate(zip(got_f, want_f)):
                np.testing.assert_array_equal(g, w, err_msg=f"{family} step {step} fold {i} ({scan.shape})")
            for q, (g, w) in enumerate(zip(got_p, want_p)):
                np.testing.assert_array_equal(g, w, err_msg=f"{family} step {step} post {q} ({scan.shape})")
        return scan
    finally:
        scan.close()


def _cases(n=40_000, seed=1):
    """name -> (spec, {family: expectation}) of the descriptor matrix."""
    rng = np.random.default_rng(seed)
    out = {}
    TABLES = {"generic": None, "jit_tables": "tables"}
    RS = dict(TABLES, **{f: "rs" for f in RS_FAMILIES})

    def ends(a, lo, hi):
        a[:2] = lo, hi
        return a
    # Q6 structure (sel3_sum2): int32 predicate column, two 8-byte columns whose min / max are exactly the int32 limits
    c0 = ends(rng.integers(I32_MIN, I32_MAX, n, endpoint=True).astype(np.int32), I32_MIN, I32_MAX)
    c1 = ends(rng.integers(I32_MIN, I32_MAX, n, endpoint=True), I32_MIN, I32_MAX)
    c2 = ends(rng.integers(-1000, 1000, n, endpoint=True), -1000, 1000)
    q6 = spec([c0, c1, c2], preds=[(0, 0, -2**40, 2**40), (1, 0, I32_MIN, I32_MAX // 2), (2, 0, -500, I64_MAX)],
              folds=[(SUM, [T(1), T(2)]), (COUNT, [])])
    out["q6_int32_limits"] = (q6, {"generic": None, "static": "sel3_sum2", "static_tables": "sel3_sum2", "jit_tables": "tables"})
    c1b = c1.copy()
    c1b[5] = I32_MAX + 1                               # one value beyond: neither the low-word compare nor FF_NARROW
    c2b = c2.copy()
    c2b[6] = I32_MIN - 1
    out["q6_one_beyond"] = (dict(q6, cols=[c0, c1b, c2b]), {"generic": None, "static": "generic", "static_tables": "generic",
                                                            "jit_tables": "tables"})
    # Q1 structure (sel1_key2_sum5): all 32 keys present, more than the 8 register slots
    date = rng.integers(0, 1000, n).astype(np.int32)
    rf = 8 * rng.integers(2, 10, n) + rng.integers(0, 8, n)
    ls = 8 * rng.integers(2, 6, n) + rng.integers(0, 8, n)
    qty, price = rng.integers(1, 51, n), rng.integers(90_000, 10_000_000, n)
    disc, tax = rng.integers(0, 11, n), rng.integers(0, 9, n)
    q1 = spec([date, rf, ls, qty, price, disc, tax], preds=[(0, 0, 100, 900)],
              keys=[(T(1, 3, -8, 4), 0), (T(2, 3, -2), 0)], key_mask=31, domain=32,
              folds=[(CHOOSE, [T(1)]), (CHOOSE, [T(2)]), (SUM, [T(3)]), (SUM, [T(4)]), (SUM, [T(4), T(5, 0, 100, -1)]),
                     (SUM, [T(4), T(5, 0, 100, -1), T(6, 0, 100)]), (SUM, [T(5)]), (COUNT, [])],
              posts=[(DIVIDE, (P_FOLD, 2), (P_FOLD, 7)), (DIVIDE, (P_FOLD, 3), (P_FOLD, 7))])
    out["q1_32_keys"] = (q1, dict(RS, static="sel1_key2_sum5", static_tables="sel1_key2_sum5"))
    # the same with only 4 of the 32 keys present, as TPC-H Q1's four flag / status pairs: the second step of _check
    # launches the 4-slot variant of the static and of the run-time compiled register-slot kernels (own generator: the
    # other cases keep their data)
    rng4 = np.random.default_rng([seed, 4])
    pair = rng4.choice(np.array([(2, 2), (3, 2), (3, 3), (4, 2)]), n)
    rf4, ls4 = 8 * pair[:, 0] + rng4.integers(0, 8, n), 8 * pair[:, 1] + rng4.integers(0, 8, n)
    out["q1_4_keys"] = (dict(q1, cols=[date, rf4, ls4, qty, price, disc, tax]),
                        dict(RS, static="sel1_key2_sum5", static_tables="sel1_key2_sum5"))
    # shifted 8-byte columns whose raw values do not fit int32: predicates (mode 2), factors (FF_NARROW)
    x = rng.integers(2**31, 2**48, n)
    x2 = rng.integers(2**31, 2**32, n)
    out["shifted_pred_and_factor"] = (
        spec([x, x2], preds=[(0, 20, 2**11 + 5, 2**27), (1, 1, 2**30 + 2**28, I64_MAX)],
             folds=[(SUM, [T(0, 20)]), (COUNT, []), (MAX, [T(1, 1, -3, 5)]), (MIN, [T(0, 24, 7, -1)])]), TABLES)
    # shifted key parts: (k >> 20) & 0x3FFF needs bits 32, 33 of k; a domain of 16384 (the largest) above gmax
    k = rng.integers(2**31, 2**48, n)
    y = rng.integers(2**31, 2**40, n)
    v = rng.integers(-2**20, 2**20, n).astype(np.int32)
    out["shifted_key_16384"] = (
        spec([k, y, v], keys=[(T(0, 20), 0)], key_mask=0x3FFF, domain=16384,
             folds=[(SUM, [T(2)]), (COUNT, []), (SUM, [T(1, 12, 5, 3)]), (MAX, [T(1, 12)])]), TABLES)
    # (k >> 28) & 63 with k in [2^40, 2^48): the low word keeps 4 correct key bits; the register-slot kernels need a
    # 32-bit key, so these descriptors run on shared-memory tables
    k2 = rng.integers(2**40, 2**48, n)
    out["shifted_key_64"] = (spec([k2, v], keys=[(T(0, 28), 0)], key_mask=63, domain=64,
                                  folds=[(SUM, [T(1)]), (COUNT, [])]), {f: "tables" for f in RS} | {"generic": None})
    # all 64 keys of a domain of 64 (overflow of the 8 register slots), MIN / MAX over the whole int32 range, b = -1
    # on INT32_MIN (which must not narrow)
    kk = rng.integers(0, 64, n).astype(np.int32)
    kk[:64] = np.arange(64)
    w = ends(rng.integers(I32_MIN, I32_MAX, n, endpoint=True).astype(np.int32), I32_MIN, I32_MAX)
    out["keys_64_of_64"] = (spec([kk, w], keys=[(T(0), 0)], key_mask=63, domain=64,
                                 folds=[(SUM, [T(1)]), (MIN, [T(1)]), (MAX, [T(1, 0, 0, -1)]), (COUNT, [])]), RS)
    # narrowing at the exact edges, products that wrap int64, MIN / MAX over INT64_MIN / INT64_MAX, post ops
    g4 = rng.integers(0, 4, n).astype(np.int32)
    g4[:8] = [0, 1, 2, 3, 0, 1, 2, 3]
    cw = rng.integers(I64_MIN, I64_MAX, n, endpoint=True)
    cw[:4], cw[4:8] = I64_MIN, I64_MAX
    zo = rng.integers(0, 2, n)
    out["narrow_edges_posts"] = (
        spec([g4, c0, c1, zo, cw], keys=[(T(0), 0)], key_mask=3, domain=4,
             folds=[(SUM, [T(1, 0, 0, -1)]), (SUM, [T(2, 0, I32_MAX, 1)]), (SUM, [T(3, 0, I32_MIN, I32_MAX)]),
                    (MIN, [T(4)]), (MAX, [T(4)]), (SUM, [T(4), T(4)]), (COUNT, [])],
             posts=[(DIVIDE, (P_FOLD, 3), (P_CONST, 0)), (DIVIDE, (P_FOLD, 3), (P_CONST, -1)),
                    (MODULO, (P_FOLD, 3), (P_CONST, -1)), (MODULO, (P_FOLD, 3), (P_CONST, 0)),
                    (MODULO, (P_FOLD, 4), (P_CONST, 7)), (DIVIDE, (P_POST, 1), (P_FOLD, 6)),
                    (SUBTRACT, (P_POST, 5), (P_FOLD, 0)), (DIVIDE, (P_FOLD, 5), (P_FOLD, 2))]), RS)
    # predicate bounds: the whole int64 range, int32 bounds partly outside int32, int32 shifts beyond 31, mode-2
    # values exactly at the clamped bounds
    a32 = ends(rng.integers(I32_MIN, I32_MAX, n, endpoint=True).astype(np.int32), I32_MIN, I32_MAX)
    b64 = ends(rng.integers(-1000, 1000, n, endpoint=True), -1000, 1000)
    out["pred_bounds"] = (
        spec([a32, b64], preds=[(0, 0, I64_MIN, I64_MAX), (1, 0, -2**40, 999), (0, 35, -1, -1), (0, 31, -1, 0), (1, 0, -1000, I64_MAX)],
             folds=[(SUM, [T(1)]), (COUNT, []), (MIN, [T(0, 33, 1, 1)])]), TABLES)
    out["pred_clamped_to_edge"] = (spec([a32, b64], preds=[(1, 0, -2**40, -1000), (0, 0, I32_MIN, 2**40)],
                                        folds=[(SUM, [T(1)]), (COUNT, [])]), TABLES)
    # predicates no row can pass: the scan is not launched, the (identity) table finalizes to no group
    for name, p in [("pred_int32_above", (0, 0, 2**40, 2**41)), ("pred_int32_below", (0, 0, I64_MIN, -2**40)),
                    ("pred_lo_gt_hi", (1, 0, 5, 4))]:
        out[name] = (spec([a32, b64], preds=[p], folds=[(SUM, [T(1)]), (COUNT, [])]), {"generic": None, "static": "generic"})
    # FoldChoose and row ids near 2^40
    g8 = rng.integers(0, 8, n).astype(np.int32)
    out["choose_rowid_2p40"] = (
        spec([g8, c2], keys=[(T(0), 0)], key_mask=7, domain=8, row_base=2**40 - 1000,
             folds=[(CHOOSE, [T(ROWID, 0, 1, 3)]), (CHOOSE, [T(1)]), (MIN, [T(ROWID)]), (SUM, [T(ROWID), T(1)]), (COUNT, [])]), RS)
    return out


CASES = list(_cases(n=64).keys())


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES)
def test_descriptor_matrix(case, ctx, capfd, monkeypatch):
    s, families = _cases()[case]
    up = Uploaded(ctx, s)
    try:
        for family, expect in families.items():
            _family(monkeypatch, family)
            _check(ctx, capfd, s, len(s["cols"][0]), family, expect, up.handles)
    finally:
        up.close()


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["q6_int32_limits", "q1_32_keys", "keys_64_of_64"])
def test_row_counts_around_tiles(case, ctx, capfd, monkeypatch, sm_count):
    """0, 1, tile_rows - 1, tile_rows, tile_rows + 1, sm_count tiles, and sm_count tiles plus a tail tile (the one staged
    with plain loads), for the tile size each family chose."""
    n_max = sm_count * 2048 + 1000
    s, families = _cases(n=n_max, seed=3)[case]
    up = Uploaded(ctx, s)
    try:
        for family, expect in families.items():
            _family(monkeypatch, family)
            probe = Scan(ctx, capfd, s, up.handles, 1)
            tile = probe.nc * probe.r
            probe.close()
            for rows in sorted({0, 1, tile - 1, tile, tile + 1, sm_count * tile, sm_count * tile + tile // 3 + 1}):
                assert rows <= n_max
                _check(ctx, capfd, s, rows, family, expect, up.handles)
    finally:
        up.close()


# ---------------------------------------------------------------------------------------------------- GPU: RS proofs
def _rs_pattern(nc, r, tiles, value):
    """Rows of `tiles` tiles of nc*r rows.  Per tile, the first half of the warps select every row (dense: folded in
    place, r rows per thread) and the other warps select the rows of 23 of their 32 lanes (queued, then dealt to all
    threads): a thread of a dense warp folds about 1.3 r rows per tile, more than r but at most 2 r."""
    nw = nc // 32
    ctid = np.arange(nc * r) % nc
    sel = ((ctid // 32) < (nw + 1) // 2) | ((ctid % 32) < 23)
    p = np.tile(sel.astype(np.int32), tiles)
    rows = len(p)
    return [p, np.zeros(rows, np.int32), np.full(rows, value, np.int32)]


@pytest.mark.gpu
@pytest.mark.parametrize("geometry", RS_FAMILIES)
def test_rs_n32_bound(geometry, ctx, capfd, monkeypatch, sm_count):
    """RK_N32 keeps a register-slot SUM in 32 bits when tiles_per_cta * 2 * R * max|value| <= INT32_MAX: at the largest
    value that proof allows the sum must be RK_N32, one above it must not, and at the value a bound of R rows per tile
    would allow (which the queue share of a dense warp's threads exceeds) the result must still be exact."""
    nc, r = (int(x) for x in FAMILIES[geometry]["VDL_RS_GEOMETRY"].split(","))
    tiles_per_cta = 3
    bound = tiles_per_cta * 2 * r
    m = I32_MAX // bound
    _family(monkeypatch, geometry)
    names = {}
    for value in (m, m + 1, I32_MAX // (tiles_per_cta * r)):
        cols = _rs_pattern(nc, r, tiles_per_cta * sm_count, value)
        s = spec(cols, preds=[(0, 0, 1, 1)], keys=[(T(1), 0)], key_mask=1, domain=2, folds=[(SUM, [T(2)]), (COUNT, [])])
        up = Uploaded(ctx, s)
        try:
            scan = _check(ctx, capfd, s, len(cols[0]), geometry, "rs", up.handles)
            names[value] = (scan.shape, scan.acc_rk[0])
        finally:
            up.close()
    assert names[m][1] == RK_N32, names
    assert names[m + 1][1] != RK_N32 and names[m + 1][0] != names[m][0], names
    assert names[I32_MAX // (tiles_per_cta * r)][1] != RK_N32, names


@pytest.mark.gpu
@pytest.mark.parametrize("geometry", RS_FAMILIES)
def test_rs_madw_bound(geometry, ctx, capfd, monkeypatch, sm_count):
    """RK_MADW multiplies two factors proved to lie in [0, 2^31): maxima of exactly 2^31 - 1 qualify, 2^31 does not
    (for either factor); the int64 sums of ~2^62 products wrap."""
    nc, r = (int(x) for x in FAMILIES[geometry]["VDL_RS_GEOMETRY"].split(","))
    rows = sm_count * nc * r + 777
    rng = np.random.default_rng(11)
    _family(monkeypatch, geometry)
    got = {}
    for xmax, ymax in ((I32_MAX, I32_MAX), (I32_MAX, 2**31), (2**31, I32_MAX)):
        g = rng.integers(0, 6, rows).astype(np.int32)
        x = rng.integers(2**30, xmax, rows, endpoint=True)
        y = rng.integers(2**30, ymax, rows, endpoint=True)
        x[0], y[1] = xmax, ymax
        s = spec([g, x, y], keys=[(T(0), 0)], key_mask=7, domain=8, folds=[(SUM, [T(1), T(2)]), (COUNT, [])])
        up = Uploaded(ctx, s)
        try:
            scan = _check(ctx, capfd, s, rows, geometry, "rs", up.handles)
            got[(xmax, ymax)] = (scan.shape, scan.acc_rk[0])
        finally:
            up.close()
    assert got[(I32_MAX, I32_MAX)][1] == RK_MADW, got
    assert got[(I32_MAX, 2**31)][1] == RK_WIDE and got[(2**31, I32_MAX)][1] == RK_WIDE, got
    assert got[(I32_MAX, 2**31)][0] != got[(I32_MAX, I32_MAX)][0], got


# ---------------------------------------------------------------------------------------------------- GPU: plans
@pytest.mark.gpu
@pytest.mark.parametrize("jit", [False, True], ids=["default", "jit"])
@pytest.mark.parametrize("case", range(3), ids=["shifted_pred", "shifted_value", "shifted_key"])
def test_plans_with_shifted_wide_columns(case, jit, monkeypatch):
    for k in SWITCHES:
        monkeypatch.delenv(k, raising=False)
    if jit:
        monkeypatch.setenv("VDL_SCAN_JIT_MIN_ROWS", "0")
    name, text, cols, s, outs = _plan_cases(rows=50_000, seed=5)[case]
    want = run_oracle(text, cols)
    assert_same(want, dict(zip(outs, reference(s, 50_000)[0])))
    fused, stats = run_gpu(text, cols, fuse=True)
    assert stats["fused_scans"] == 1, stats
    assert stats["shape"].startswith("jit:") == jit, stats
    assert_same(fused, want)
    unfused, _ = run_gpu(text, cols, fuse=False)
    assert_same(unfused, want)
