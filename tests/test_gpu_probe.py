"""The fused FK-join probe kernels through their C entry points (vdl_probe_*), against a numpy evaluation of the
same leaf / term / predicate descriptor: fold mode (small key domain) and emit mode (dense ordered output).  Every case
runs through both kernels: the interpreter and the kernel compiled at run time for the descriptor."""
import ctypes as C

import numpy as np
import pytest

from mplan2vdl_b200 import lib as vlib

pytestmark = pytest.mark.gpu

SUM, MIN, MAX, CHOOSE, COUNT = range(5)


def term(leaf, a=0, b=1, shr=0):
    return vlib.Term(leaf, shr, a, b)


def product(*terms):
    p = vlib.Product()
    p.nfactors = len(terms)
    for i, t in enumerate(terms):
        p.factor[i] = t
    return p


def tables(n, n1, n2, seed):
    rng = np.random.default_rng(seed)
    fk1 = np.sort(rng.integers(0, n1, n)).astype(np.int64)           # clustered like lineitem -> orders
    return {
        "f.fk1": fk1,
        "f.v": rng.integers(1, 1000, n).astype(np.int64),
        "f.x": rng.integers(0, 5, n).astype(np.int32),
        "d1.a": rng.integers(0, 100, n1).astype(np.int32),
        "d1.fk2": rng.integers(0, n2, n1).astype(np.int64),
        "d1.x": rng.integers(0, 5, n1).astype(np.int64),
        "d2.b": (8 * rng.integers(2, 12, n2)).astype(np.int64),
    }


KERNELS = ["interpreter", "jit"]


def use_kernel(kernel, monkeypatch):
    """VDL_PROBE_JIT=0 keeps the interpreter; VDL_PROBE_JIT_MIN_ROWS=0 compiles the descriptor at every size.  With
    VDL_DEBUG_JIT the compiled source is printed, which shows that the kernel named by the parameter is the one that ran."""
    monkeypatch.delenv("VDL_PROBE_JIT", raising=False)
    monkeypatch.delenv("VDL_PROBE_JIT_MIN_ROWS", raising=False)
    monkeypatch.setenv("VDL_PROBE_JIT_MIN_ROWS" if kernel == "jit" else "VDL_PROBE_JIT", "0")
    monkeypatch.setenv("VDL_DEBUG_JIT", "1")


def assert_kernel_ran(kernel, capfd):
    err = capfd.readouterr().err
    assert ("[vdl jit] probe:" in err) == (kernel == "jit") and "runs instead" not in err, err[-2000:]


@pytest.fixture(params=KERNELS)
def kernel(request, monkeypatch, capfd):
    use_kernel(request.param, monkeypatch)
    yield request.param
    assert_kernel_ran(request.param, capfd)


def run_probe(ctx, desc):
    L = ctx.L
    h = C.c_void_p()
    ctx.check(L.vdl_probe_prepare(ctx.h, C.byref(desc), C.byref(h)))
    ctx.check(L.vdl_probe_run(h))
    return h


@pytest.mark.parametrize("n", [1, 1000, 1024, 1025, 300_007])
def test_probe_fold_matches_numpy(n, kernel):
    from mplan2vdl_b200.executor import Context
    ctx = Context(0)
    t = tables(n, max(1, n // 4), 50, n)
    hv = {k: ctx.upload_column(k, v) for k, v in t.items()}
    d = vlib.ProbeDesc()
    d.rows, d.row_base = n, 7
    leaves = [("f.fk1", -1), ("d1.a", 0), ("d1.fk2", 0), ("d2.b", 2), ("f.v", -1), ("f.x", -1), ("d1.x", 0)]
    d.nleaves = len(leaves)
    for i, (c, par) in enumerate(leaves):
        d.leaf[i] = vlib.Leaf(hv[c], par)
    d.npreds = 3
    d.pred[0] = vlib.ProbePred(0, 0, term(1), term(-1), 10, 79)                 # 10 <= a[fk1] <= 79
    d.pred[1] = vlib.ProbePred(1, 0, term(5), term(6), 0, 0)                    # f.x == d1.x[fk1]
    d.pred[2] = vlib.ProbePred(0, 0, term(3, shr=3), term(-1), 3, 10)           # 3 <= (b >> 3) <= 10
    d.nkeys, d.key_mask, d.domain = 1, 15, 16
    d.key[0] = term(3, a=-2, shr=3)                                             # (b >> 3) - 2
    d.key_shl[0] = 0
    folds = [(SUM, product(term(4), term(1, a=100, b=-1))), (COUNT, product()), (MIN, product(term(4))), (MAX, product(term(1))),
             (CHOOSE, product(term(3))), (SUM, product(term(-2)))]
    d.nfolds = len(folds)
    for i, (op, pr) in enumerate(folds):
        d.fold[i] = vlib.ProbeFold(op, 0, pr)
    d.nposts = 1
    d.post[0] = vlib.PostOp(10, vlib.VDL_POST_FOLD, vlib.VDL_POST_FOLD, 0, 0, 1)   # Divide(fold 0, fold 1)
    h = run_probe(ctx, d)

    a, x1, fk2 = t["d1.a"][t["f.fk1"]].astype(np.int64), t["d1.x"][t["f.fk1"]], t["d1.fk2"][t["f.fk1"]]
    b = t["d2.b"][fk2]
    sel = (a >= 10) & (a <= 79) & (t["f.x"] == x1) & ((b >> 3) >= 3) & ((b >> 3) <= 10)
    key = ((b >> 3) - 2) & 15
    rowid = 7 + np.arange(n, dtype=np.int64)
    want = [[] for _ in range(len(folds) + 1)]
    for k in sorted(set(key[sel].tolist())):
        m = sel & (key == k)
        s0 = int((t["f.v"][m] * (100 - a[m])).sum())
        want[0].append(s0); want[1].append(int(m.sum())); want[2].append(int(t["f.v"][m].min())); want[3].append(int(a[m].max()))
        want[4].append(int(b[m][0])); want[5].append(int(rowid[m].sum())); want[6].append(int(s0 / int(m.sum())))
    for i in range(len(folds) + 1):
        data, ln = C.POINTER(C.c_int64)(), C.c_int64()
        ctx.check(ctx.L.vdl_probe_result_host(h, i, C.byref(data), C.byref(ln)))
        got = [data[j] for j in range(ln.value)]
        assert got == want[i], (i, got, want[i])
    ctx.L.vdl_probe_destroy(h)
    ctx.close()


@pytest.mark.parametrize("n", [1, 1024, 5000, 1_000_003])
def test_probe_emit_is_the_dense_foldselect_order(n, kernel):
    from mplan2vdl_b200.executor import Context
    ctx = Context(0)
    t = tables(n, max(1, n // 3), 20, n + 1)
    hv = {k: ctx.upload_column(k, v) for k, v in t.items()}
    d = vlib.ProbeDesc()
    d.rows, d.row_base = n, 0
    leaves = [("f.fk1", -1), ("d1.a", 0), ("f.v", -1)]
    d.nleaves = len(leaves)
    for i, (c, par) in enumerate(leaves):
        d.leaf[i] = vlib.Leaf(hv[c], par)
    d.npreds = 1
    d.pred[0] = vlib.ProbePred(0, 0, term(1), term(-1), 0, 29)
    d.nemits = 3
    d.emit[0] = product(term(-2))
    d.emit[1] = product(term(2), term(1, a=1))
    d.emit[2] = product(term(0))
    h = run_probe(ctx, d)
    a = t["d1.a"][t["f.fk1"]].astype(np.int64)
    sel = np.nonzero(a <= 29)[0]
    want = [sel, t["f.v"][sel] * (1 + a[sel]), t["f.fk1"][sel]]
    for k in range(3):
        v = C.c_int32()
        ctx.check(ctx.L.vdl_probe_emit_take(h, k, C.byref(v)))
        np.testing.assert_array_equal(ctx.download(v.value), want[k])
        ctx.free(v.value)
    ctx.L.vdl_probe_destroy(h)
    ctx.close()


def test_probe_reports_lookup_index_out_of_range(monkeypatch, capfd):
    from mplan2vdl_b200.executor import Context
    from mplan2vdl_b200.lib import VdlError
    for kernel in KERNELS:
        use_kernel(kernel, monkeypatch)
        ctx = Context(0)
        f = ctx.upload_column("f.fk", np.array([0, 1, 5], dtype=np.int64))
        dcol = ctx.upload_column("d.a", np.array([1, 2], dtype=np.int64))
        d = vlib.ProbeDesc()
        d.rows, d.nleaves = 3, 2
        d.leaf[0], d.leaf[1] = vlib.Leaf(f, -1), vlib.Leaf(dcol, 0)
        d.nkeys, d.domain, d.key_mask, d.nfolds = 0, 1, -1, 1
        d.fold[0] = vlib.ProbeFold(SUM, 0, product(term(1)))
        h = run_probe(ctx, d)
        data, ln = C.POINTER(C.c_int64)(), C.c_int64()
        with pytest.raises(VdlError):
            ctx.check(ctx.L.vdl_probe_result_host(h, 0, C.byref(data), C.byref(ln)))
        ctx.L.vdl_probe_destroy(h)
        ctx.close()
        assert_kernel_ran(kernel, capfd)
