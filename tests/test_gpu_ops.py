"""Per-op parity on the GPU: every Voodoo op through libvdl_cuda's C ABI against the CPU oracle."""
import numpy as np
import pytest

import test_oracle_ops as K
from util import run_gpu, run_oracle

pytestmark = pytest.mark.gpu
I64 = np.int64


def both(plan, **cols):
    cols = {"t." + k: np.asarray(v) for k, v in cols.items()}
    want = run_oracle(plan, cols)
    for fuse in (False, True):
        got, _ = run_gpu(plan, cols, fuse=fuse)
        assert list(got) == list(want)
        for k in want:
            np.testing.assert_array_equal(got[k], want[k], err_msg=f"{k} fuse={fuse}")
    return want


@pytest.mark.parametrize("op", ["Add", "Subtract", "Multiply", "Divide", "Modulo", "Greater", "Equals", "LogicalAnd",
                                "LogicalOr", "BitwiseAnd", "BitwiseOr", "BitShift"])
def test_binary_kat_and_random(op):
    both(K.binop_plan(op), a=K.A, b=K.B)
    rng = np.random.default_rng(11)
    n = 1_000_003
    a = rng.integers(-2**62, 2**62, n).astype(I64)
    b = rng.integers(-70, 70, n).astype(I64) if op == "BitShift" else rng.integers(-2**40, 2**40, n).astype(I64)
    b[::97] = 0
    both(K.binop_plan(op), a=a, b=b)


def test_int32_columns_and_ranges():
    both(K.binop_plan("Add"), a=np.array([-5, 7, 2**31 - 1], dtype=np.int32), b=np.array([2**40, 1, 1], dtype=I64))
    plan = ("1,Load,t.a\n2,Project,val,Id 1,a\n3,RangeV,val,10,Id 2,3\n4,RangeC,val,-1,4,2\n"
            "5,Project,rv,Id 3,val\n6,MaterializeCompact,Id 5\n7,Project,rc,Id 4,val\n8,MaterializeCompact,Id 7\n")
    both(plan, a=np.zeros(3, I64))


@pytest.mark.parametrize("n,density", [(6, 0.5), (4095, 0.3), (4096, 0.0), (4097, 1.0), (1_000_003, 0.02), (3_000_000, 0.9)])
def test_fold_select_gather(n, density):
    rng = np.random.default_rng(n)
    p = (rng.random(n) < density).astype(I64) * rng.integers(1, 5, n)
    x = rng.integers(-10**15, 10**15, n).astype(I64)
    r = both(K.SELECT, p=p, x=x)
    assert len(r["pos"]) == int((p != 0).sum())


@pytest.mark.parametrize("op", ["FoldSum", "FoldMin", "FoldMax", "FoldChoose", "FoldCount"])
def test_folds(op):
    both(K.FOLD.format(op=op), g=np.array([5, 5, 9, 2, 2, 2, 5], I64), x=np.array([1, 2, 3, 4, 5, 6, 7], I64))
    both(K.FOLD.format(op=op), g=np.zeros(0, I64), x=np.zeros(0, I64))
    rng = np.random.default_rng(5)
    for n, ngroups in ((1_000_003, 50), (300_007, 200_000), (70_001, 1)):
        g = np.sort(rng.integers(0, ngroups, n)).astype(I64)
        x = rng.integers(-2**62, 2**62, n).astype(I64)     # sums wrap
        both(K.FOLD.format(op=op), g=g, x=x)


@pytest.mark.parametrize("n,nkeys", [(7, 4), (4096, 4), (100_003, 4), (1_000_003, 4)])
def test_partition_scatter(n, nkeys):
    rng = np.random.default_rng(n)
    k = rng.integers(-2, nkeys + 3, n).astype(I64)
    r = both(K.PART, k=k)
    assert np.all(np.diff(np.clip(r["sorted"], 0, 4)) >= 0)
    assert sorted(r["perm"].tolist()) == list(range(n))


def test_partition_wide_keys_multi_pass():
    plan = K.PART.replace("3,RangeC,val,0,4,1", "3,RangeC,val,0,274877906944,1")    # 2^38 pivots (Q3's composite key)
    rng = np.random.default_rng(3)
    k = rng.integers(0, 2**38, 200_003).astype(I64)
    r = both(plan, k=k)
    np.testing.assert_array_equal(r["sorted"], np.sort(k))


# The radix sort that Partition shares with Order: its first pass takes the row ids from the positions, so ties (here
# also the clamped buckets below the first pivot and above the last) check that it is stable.
@pytest.mark.parametrize("n", [1, 4095, 4097, 200_003])                   # around the radix sort's 4096-row tiles
@pytest.mark.parametrize("keys", ["unique", "ties", "ordered"])
@pytest.mark.parametrize("pfrom,pcount,pstep", [
    pytest.param(0, 256, 1, id="count256"),           # the first count past the counting partition: 2 passes
    pytest.param(-5000, 70_000, 1, id="count70000"),  # 3 passes
    pytest.param(0, 2**38, 1, id="count2e38"),        # Q3's composite key: 5 passes
    pytest.param(7, 10, 3, id="step3")])              # a non-unit step takes the radix sort at any count
def test_partition_radix_sort_stable(pfrom, pcount, pstep, keys, n):
    plan = K.PART.replace("3,RangeC,val,0,4,1", f"3,RangeC,val,{pfrom},{pcount},{pstep}")
    rng = np.random.default_rng(n)
    last = pfrom + (pcount - 1) * pstep
    if keys == "unique":
        k = pfrom + rng.permutation(n).astype(I64) * max(1, pcount * pstep // n)
    else:       # few distinct values, with some at or below the first pivot and above the last (the clamped buckets)
        pool = np.array([np.iinfo(I64).min, pfrom - 1, pfrom, pfrom + 1, pfrom + pstep * (pcount // 2), last, last + 1,
                         np.iinfo(I64).max], I64)
        k = pool[rng.integers(0, len(pool), n)]
        if keys == "ordered":
            k = np.sort(k)
    r = both(plan, k=k)
    d = k.astype(np.uint64) - np.uint64(pfrom % 2**64)                  # bucket = pivots below the key
    b = np.where(k <= pfrom, 0, np.minimum((d + np.uint64(pstep - 1)) // np.uint64(pstep), np.uint64(pcount)))
    np.testing.assert_array_equal(r["sorted"], k[np.argsort(b, kind="stable")])


def test_scatter_index_space():
    plan = ("1,Load,t.p\n2,Project,val,Id 1,p\n3,RangeV,val,0,Id 2,1\n4,FoldSelect,val,Id 3,val,Id 2,val\n"
            "5,RangeV,val,1,Id 4,0\n6,RangeV,val,0,Id 5,1\n7,Scatter,Id 5,Id 6,val,Id 4,val\n"
            "8,Project,valid,Id 7,val\n9,MaterializeCompact,Id 8\n"
            "10,Scatter,Id 6,Id 6,val,Id 4,val\n11,Project,inv,Id 10,val\n12,MaterializeCompact,Id 11\n")
    rng = np.random.default_rng(1)
    both(plan, p=np.array([0, 1, 0, 0, 1, 1], I64))
    both(plan, p=(rng.random(500_001) < 0.4).astype(I64))


def test_errors_are_reported_not_fatal():
    from mplan2vdl_b200.executor import Context
    from mplan2vdl_b200.lib import VdlError
    ctx = Context(0)
    with pytest.raises(VdlError):
        ctx.plan("1,Load,t.a\n2,Semisort,Id 1\n")                       # unsupported op
    with pytest.raises(VdlError):
        ctx.plan("1,Load,t.a\n2,Project,val,Id 1,a\n3,MaterializeCompact,Id 2\n").run()   # unbound column
    ctx.upload_column("t.x", np.arange(3, dtype=I64))
    ctx.upload_column("t.i", np.array([0, 3], I64))
    with pytest.raises(VdlError):                                         # gather out of range
        ctx.plan("1,Load,t.x\n2,Project,val,Id 1,x\n3,Load,t.i\n4,Project,val,Id 3,i\n5,Gather,Id 2,Id 4,val\n6,MaterializeCompact,Id 5\n").run()
    # the context is still usable afterwards
    out = ctx.plan("1,Load,t.x\n2,Project,out,Id 1,val\n3,MaterializeCompact,Id 2\n").run()
    np.testing.assert_array_equal(out["out"], [0, 1, 2])
    ctx.close()


def test_op_map_register_program():
    """vdl_op_map directly: one launch for ((a + 7*i) * b > c) | t[a & 3], against numpy."""
    from mplan2vdl_b200.executor import Context
    from mplan2vdl_b200.lib import VdlError
    rng = np.random.default_rng(5)
    n = 100_003
    a = rng.integers(-2**40, 2**40, n).astype(I64)
    b = rng.integers(-2**20, 2**20, n).astype(np.int32)
    c = rng.integers(-2**60, 2**60, n).astype(I64)
    t = np.array([0, 8, 16, 32], I64)
    ctx = Context(0)
    try:
        va, vb, vc, vt = (ctx.upload_column(f"t.{k}", v) for k, v in (("a", a), ("b", b), ("c", c), ("t", t)))
        prog = [("Load", 0, 0, 0), ("Range", 1, 0, 1), ("Add", 1, 0, 1), ("Load", 2, 0, 1), ("Multiply", 1, 1, 2), ("Load", 2, 0, 2),
                ("Greater", 1, 1, 2), ("Range", 2, 2, 0), ("BitwiseAnd", 0, 0, 2), ("Gather", 0, 0, 0), ("BitwiseOr", 3, 1, 0)]
        out = ctx.download(ctx.op_map(prog, [va, vb, vc], [vt], imms=[0, 7, 3]))
        i = np.arange(n, dtype=I64)
        want = (((a + 7 * i) * b.astype(I64)) > c).astype(I64) | t[a & 3]
        np.testing.assert_array_equal(out, want)
        with pytest.raises(VdlError):          # register 5 is read before anything wrote it
            ctx.op_map([("Load", 0, 0, 0), ("Add", 1, 0, 5)], [va])
        with pytest.raises(VdlError):          # inputs of different lengths
            ctx.op_map([("Load", 0, 0, 0), ("Load", 1, 0, 1), ("Add", 1, 0, 1)], [va, vt])
        # a Gather instruction out of range: value 0 and the context's error flag, which the next plan run reports
        out = ctx.download(ctx.op_map([("Load", 0, 0, 0), ("Gather", 1, 0, 0)], [vc], [vt]))
        np.testing.assert_array_equal(out, np.where((c >= 0) & (c < 4), t[np.clip(c, 0, 3)], 0))
        with pytest.raises(VdlError):
            ctx.plan("1,Load,t.t\n2,Project,val,Id 1,t\n3,RangeV,val,0,Id 2,1\n4,Gather,Id 2,Id 3,val\n5,Project,o,Id 4,val\n6,MaterializeCompact,Id 5\n").run()
    finally:
        ctx.close()


MAP_PLAN = (
    "1,Load,t.a\n2,Project,val,Id 1,a\n3,Load,t.b\n4,Project,val,Id 3,b\n"
    "5,RangeV,val,100,Id 2,0\n6,Greater,val,Id 2,val,Id 5,val\n"                    # a > 100
    "7,RangeV,val,7,Id 6,0\n8,Equals,val,Id 4,val,Id 7,val\n"                        # b == 7 (constant as long as an interior node)
    "9,LogicalOr,val,Id 6,val,Id 8,val\n"
    "10,Multiply,val,Id 2,val,Id 4,val\n11,Add,val,Id 10,val,Id 10,val\n"            # shared interior node
    "12,Multiply,val,Id 11,val,Id 9,val\n"
    "13,Load,t.k\n14,Project,val,Id 13,k\n15,Load,t.d\n16,Project,val,Id 15,d\n17,Gather,Id 16,Id 14,val\n"
    "18,Add,val,Id 12,val,Id 17,val\n"
    "19,RangeV,val,0,Id 18,1\n20,FoldSelect,val,Id 19,val,Id 9,val\n21,Gather,Id 18,Id 20,val\n"   # node 9 also feeds a FoldSelect: materialised
    "22,Project,out,Id 18,val\n23,MaterializeCompact,Id 22\n24,Project,sel,Id 21,val\n25,MaterializeCompact,Id 24\n")


@pytest.mark.parametrize("n", [0, 1, 1000, 300_007])
def test_map_clusters_in_plans(n):
    """Chains of elementwise ops / gathers in the op-at-a-time remainder run as vdl_op_map launches (build_clusters);
    nodes something outside the chain consumes are still materialised."""
    rng = np.random.default_rng(n)
    cols = dict(a=rng.integers(0, 200, n).astype(I64), b=rng.integers(0, 10, n).astype(I64), k=rng.integers(0, 50, n).astype(I64),
                d=rng.integers(-2**50, 2**50, 50).astype(I64))
    both(MAP_PLAN, **cols)
    _, stats = run_gpu(MAP_PLAN, {"t." + k: v for k, v in cols.items()}, fuse=True)
    assert stats["map_clusters"] >= 2 and stats["map_nodes"] >= 8, stats
    _, stats0 = run_gpu(MAP_PLAN, {"t." + k: v for k, v in cols.items()}, fuse=False)
    assert stats0["map_clusters"] == 0 and (n == 0 or stats0["launches"] > stats["launches"])


def test_map_cluster_gather_out_of_range():
    from mplan2vdl_b200.lib import VdlError
    cols = {"t.a": np.arange(10, dtype=I64), "t.b": np.arange(10, dtype=I64), "t.k": np.array([0, 1, 2, 3, 4, 5, 6, 7, 8, 50], I64), "t.d": np.arange(50, dtype=I64)}
    with pytest.raises(VdlError):
        run_gpu(MAP_PLAN, cols, fuse=True)


@pytest.mark.parametrize("n", [1000, 70_001])      # interpreter / run-time specialised kernel (>= 65536 rows)
def test_map_binary_semantics_match_per_op_kernels(n):
    """Every binary op through vdl_op_map (both of its kernels) against vdl_op_binary, which the oracle pins, on edge
    values: INT64_MIN / -1, division and modulo by 0, shifts by 0, +-63, +-64, +-70."""
    from mplan2vdl_b200.executor import Context
    from mplan2vdl_b200.lib import BINARY_OPS
    rng = np.random.default_rng(n)
    edge = np.array([0, 1, -1, 2, -2, 63, -63, 64, -64, 70, -70, 2**62, -2**62, 2**63 - 1, -2**63, 12345, -98765], I64)
    a = np.concatenate([np.repeat(edge, len(edge)), rng.integers(-2**63, 2**63 - 1, n, dtype=I64)])
    b = np.concatenate([np.tile(edge, len(edge)), rng.integers(-80, 80, n, dtype=I64)])
    ctx = Context(0)
    try:
        va, vb = ctx.upload_column("t.a", a), ctx.upload_column("t.b", b)
        for op in BINARY_OPS:
            want = ctx.download(ctx.op_binary(op, va, vb))
            got = ctx.download(ctx.op_map([("Load", 0, 0, 0), ("Load", 1, 0, 1), (op, 2, 0, 1), ("Range", 3, 0, 0), ("Add", 2, 2, 3)], [va, vb], imms=[0]))
            np.testing.assert_array_equal(got, want, err_msg=op)
    finally:
        ctx.close()


@pytest.mark.parametrize("pat", ["PROMO%", "%BRASS", "%green%", "%Customer%Complaints%", "%", "", "_", "__", "a,b", "%r%r%", "forest gree_", "%N"])
def test_like_kat_and_pool(pat, catalog):
    """vdl_op_like against the oracle: the hand-written strings of tests/test_oracle_ops.py, then a million rows drawn from the
    synthetic p_type / p_name heaps."""
    from mplan2vdl_b200 import synth
    offs, heap = K.like_columns(K.STRINGS)
    both(K.LIKE.format(pat=pat), **{"s": offs, "s.heap": heap})
    for col in ("part.p_type", "part.p_name"):
        h, _ = synth.string_heap(catalog, col)
        o = synth.string_offsets(catalog, col, 1_000_003, 17, 99)
        both(K.LIKE.format(pat=pat), **{"s": o, "s.heap": h})


def test_like_rejects_a_bad_offset_and_a_heap_is_only_a_dictionary():
    from mplan2vdl_b200.executor import Context
    from mplan2vdl_b200.lib import VdlError
    offs, heap = K.like_columns(K.STRINGS)
    ctx = Context(0)
    h = ctx.upload_column("t.s.heap", heap)
    d = ctx.upload_column("t.s", np.array([0, len(heap) + 5], dtype=I64))
    with pytest.raises(VdlError):
        ctx.op_binary("Add", h, h)                 # a byte vector is not a numeric operand
    out = ctx.op_like(d, h, "%")
    with pytest.raises(VdlError):                  # offset past the heap: range error at the plan's check
        p = ctx.plan(K.LIKE.format(pat="%"))
        p.run()
    ctx.free(out)
    ctx.close()
