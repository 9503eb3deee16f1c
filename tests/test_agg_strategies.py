"""--aggserial / --aggshuffle / --agghierarchical -g GRAIN (MainFuns.hs:61-65, 139-147; getScatterMask Vlite.hs:1082-1098;
make2LevelFold Vlite.hs:1173-1194).  The restated translator prints all three graph shapes; the CPU oracle interprets the
two-level Folds literally in the dense model; the GPU tests run them through libvdl_cuda fused (the planner collapses a
provably refining level 1) and op-at-a-time (vdl_op_fold evaluates level 2 itself)."""
import numpy as np
import pytest

from mplan2vdl_b200 import synth, tpch, tpch_queries, vlite
from util import FIXTURES, assert_same, host_columns, needs_reference, run_gpu, run_oracle

SF = 0.01
QUERIES = ["q06", "q01", "q03", "q05"]


def program(catalog, q, strategy):
    return vlite.translate(catalog, tpch_queries.QUERIES[q](catalog), strategy)


def columns(catalog, text, sf=SF, rows_override=None):
    rows = {t: synth.table_rows(catalog, t, sf) for t in catalog.tables}
    rows.update(rows_override or {})
    return host_columns(catalog, tpch.plan_columns(text), rows, sf=sf)


def test_shuffle_strategy_only_adds_shuffle_statements(catalog):
    serial, shuffle = program(catalog, "q01", "serial"), program(catalog, "q01", "shuffle")
    assert "Shuffle" not in serial and "Shuffle" in shuffle
    strip = lambda t: [",".join(l.split(",")[1:3]) for l in t.splitlines() if ",Shuffle," not in l]
    assert [l.split(",")[1] for l in serial.splitlines()] == [l.split(",")[1] for l in shuffle.splitlines() if ",Shuffle," not in l]
    assert len(strip(serial)) == len(strip(shuffle))


def test_hierarchical_strategy_prints_two_folds_per_aggregate(catalog):
    serial, hier = program(catalog, "q01", "serial"), program(catalog, "q01", ("hierarchical", 2))
    nfold = lambda t: sum(1 for l in t.splitlines() if l.split(",")[1] in ("FoldSum", "FoldChoose", "FoldMin", "FoldMax"))
    assert nfold(hier) == 2 * nfold(serial)
    # (pos >> log2 grain) & 1 (Vlite.hs:1188): the grain is the shift count
    assert any(l.split(",")[1] == "RangeV" and l.split(",")[3] == "2" for l in hier.splitlines())


@pytest.mark.parametrize("q", QUERIES)
@pytest.mark.parametrize("strategy", ["shuffle", ("hierarchical", 0), ("hierarchical", 2), ("hierarchical", 13)])
def test_oracle_gives_the_serial_answer_when_level_one_refines_the_groups(catalog, q, strategy):
    """With the partition's index space as small as the reference infers it (G2: `count` of a Scatter = the largest
    position its metadata allows = the pivot count), a big grain makes level1par constant and a small one composes it below
    the group key; either way the level-1 runs refine the groups and the answer is the serial one."""
    serial, text = program(catalog, q, "serial"), program(catalog, q, strategy)
    cols = columns(catalog, serial)
    want = run_oracle(serial, cols)
    got = run_oracle(text, cols)
    assert_same(got, want)
    assert all(len(v) for v in want.values())


def test_oracle_interprets_a_non_refining_level_one_literally():
    """Hand-written vectors: level-1 groups that straddle a group boundary.  Dense model: level-1 run k is credited to the
    group at its first row (the sparse Voodoo vector keeps the level-1 result at that row: Vdl.hs:255-264)."""
    g = np.array([2, 2, 2, 3, 3, 3, 3, 5], dtype=np.int64)
    d = np.array([1, 2, 3, 4, 5, 6, 7, 8], dtype=np.int64) * 10
    text = "\n".join([
        "1,Load,t.g", "2,Load,t.d",
        "3,RangeV,val,0,Id 1,1", "4,RangeV,val,1,Id 1,0", "5,BitShift,val,Id 3,val,Id 4,val",      # pos >> 1
        "6,BitwiseAnd,val,Id 5,val,Id 4,val",                                                       # & 1: 0 0 1 1 0 0 1 1
        "7,BitwiseOr,val,Id 1,val,Id 6,val",                                                        # 2 2 3 3 3 3 3 5
        "8,FoldSum,val,Id 7,val,Id 2,val",                                                          # 30, 250, 80
        "9,FoldSum,val,Id 1,val,Id 8,val",                                                          # g at the run heads (rows 0, 2, 7): 2, 2, 5
        "10,Project,s,Id 9,val", "11,MaterializeCompact,Id 10", ""])
    out = run_oracle(text, {"t.g": g, "t.d": d})
    np.testing.assert_array_equal(out["s"], [280, 80])          # the serial answer would be 60, 220, 80


@pytest.mark.gpu
@pytest.mark.parametrize("fuse", [True, False])
def test_gpu_non_refining_level_one_matches_the_oracle(fuse):
    g = np.array([2, 2, 2, 3, 3, 3, 3, 5], dtype=np.int64)
    d = np.array([1, 2, 3, 4, 5, 6, 7, 8], dtype=np.int64) * 10
    text = "\n".join([
        "1,Load,t.g", "2,Load,t.d", "3,RangeV,val,0,Id 1,1", "4,RangeV,val,1,Id 1,0", "5,BitShift,val,Id 3,val,Id 4,val",
        "6,BitwiseAnd,val,Id 5,val,Id 4,val", "7,BitwiseOr,val,Id 1,val,Id 6,val", "8,FoldSum,val,Id 7,val,Id 2,val",
        "9,FoldSum,val,Id 1,val,Id 8,val", "10,Project,s,Id 9,val", "11,MaterializeCompact,Id 10", ""])
    out, _ = run_gpu(text, {"t.g": g, "t.d": d}, fuse=fuse)
    np.testing.assert_array_equal(out["s"], [280, 80])


@pytest.mark.gpu
@pytest.mark.parametrize("q", QUERIES)
@pytest.mark.parametrize("strategy", ["shuffle", ("hierarchical", 0), ("hierarchical", 2), ("hierarchical", 13)])
def test_gpu_runs_every_strategy(catalog, q, strategy):
    text = program(catalog, q, strategy)
    rows = {"lineitem": 300_007} if q in ("q06", "q01") else None      # the join plans keep the FK columns inside their tables
    cols = columns(catalog, text, rows_override=rows)
    want = run_oracle(text, cols)
    fused, fstats = run_gpu(text, cols, fuse=True)
    assert_same(fused, want)
    plain, _ = run_gpu(text, cols, fuse=False)
    assert_same(plain, want)
    if q == "q06" or (q == "q01" and (strategy == "shuffle" or strategy[1] < 13)):
        # Shuffle is an alias; a level 1 that provably refines the groups collapses: the plan is ONE fused scan again.  (Q1 with
        # a grain above the 32 slots the reference's metadata gives the sorted vector: level1par is inferred constant, the keys
        # are OR-ed without a shift, nothing is provable and both Folds run op-at-a-time -- literally.)
        assert fstats["fused_scans"] == 1, fstats


@pytest.mark.parametrize("q", ["q01", "q05"])
def test_goffset_shifts_the_group_key_and_nothing_else(catalog, q):
    """--goffset (MainFuns.hs:67; makeCompositeKey Vlite.hs:1125-1131): the synthesized key gets an offset before its size
    hint; the groups, their order and every aggregate stay what they were."""
    rel = tpch_queries.QUERIES[q](catalog)
    serial, shifted = vlite.translate(catalog, rel), vlite.translate(catalog, rel, goffset=3)
    assert shifted != serial and "Add" in [l.split(",")[1] for l in shifted.splitlines()]
    cols = columns(catalog, serial)
    assert_same(run_oracle(shifted, cols), run_oracle(serial, cols))


def test_without_the_cleanup_passes_the_program_is_longer_and_means_the_same(catalog):
    rel = tpch_queries.QUERIES["q06"](catalog)
    clean, raw = vlite.translate(catalog, rel), vlite.translate(catalog, rel, apply_cleanup_passes=False)
    assert len(raw.splitlines()) > len(clean.splitlines())
    cols = columns(catalog, clean)
    assert_same(run_oracle(raw, cols), run_oracle(clean, cols))


@needs_reference
def test_catalogue_from_the_four_metadata_files_is_the_built_in_one(catalog):
    from mplan2vdl_b200 import mplan
    from mplan2vdl_b200.meta import load_metadata_files
    d = FIXTURES
    cat = load_metadata_files(f"{d}/bounds.csv", f"{d}/storage.csv", f"{d}/schema.msqldump", f"{d}/dictionary.csv")
    for n in ("01", "05", "16"):
        src = open(f"{d}/{n}.sql.mplan").read()
        assert mplan.translate_mplan(cat, src) == mplan.translate_mplan(catalog, src)
