"""Row-range sharding on the GPU: N ranks emulated on one device (one context per rank), their partial tables
concatenated the way the NCCL all-gather lays them out, merged by the finalize kernel."""
import numpy as np
import pytest

from mplan2vdl_b200 import tpch
from util import Q1_COLS, Q6_COLS, assert_same, host_columns, plan_text, run_oracle

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("query,colnames", [("q06.vdl", Q6_COLS), ("q01.vdl", Q1_COLS)])
@pytest.mark.parametrize("world", [2, 3])
def test_emulated_ranks_merge_to_the_whole_table_answer(catalog, query, colnames, world):
    import torch
    from mplan2vdl_b200.dist import DeviceView
    from mplan2vdl_b200.executor import Context
    rows, text = 50_000, plan_text(query)
    names = ["lineitem." + c for c in colnames]
    want = run_oracle(text, host_columns(catalog, names, {"lineitem": rows}))
    ctxs, plans, tables = [], [], []
    for rank in range(world):
        start, n = tpch.shard_range(rows, rank, world)
        ctx = Context(0)
        for k, v in host_columns(catalog, names, {"lineitem": n}, row_offset=start).items():
            ctx.upload_column(k, v)
        plan = ctx.plan(text)
        plan.set_row_base(start)
        plan.run_local()
        assert plan.num_fused == 1
        ptr, cnt = plan.partials(0)
        ctx.synchronize()
        tables.append(torch.as_tensor(DeviceView(ptr, cnt), device="cuda:0").clone())
        ctxs.append(ctx)
        plans.append(plan)
    gathered = torch.cat(tables)
    torch.cuda.synchronize()
    for rank in range(world):          # every rank finalizes from the same gathered buffer and gets the global answer
        got = plans[rank].finish([gathered.data_ptr()], world)
        assert_same(got, want)
    for p, c in zip(plans, ctxs):
        p.close()
        c.close()


def test_empty_shard_is_harmless(catalog):
    """More ranks than aligned row blocks: trailing ranks own zero rows."""
    import torch
    from mplan2vdl_b200.dist import DeviceView
    from mplan2vdl_b200.executor import Context
    rows, world, text = 5000, 3, plan_text("q06.vdl")
    names = ["lineitem." + c for c in Q6_COLS]
    want = run_oracle(text, host_columns(catalog, names, {"lineitem": rows}))
    tables, keep = [], []
    for rank in range(world):
        start, n = tpch.shard_range(rows, rank, world)
        ctx = Context(0)
        for k, v in host_columns(catalog, names, {"lineitem": n}, row_offset=start).items():
            ctx.upload_column(k, v)
        plan = ctx.plan(text)
        plan.set_row_base(start)
        plan.run_local()
        ptr, cnt = plan.partials(0)
        ctx.synchronize()
        tables.append(torch.as_tensor(DeviceView(ptr, cnt), device="cuda:0").clone())
        keep.append((ctx, plan))
    assert tpch.shard_range(rows, 2, world)[1] == 0
    gathered = torch.cat(tables)
    torch.cuda.synchronize()
    assert_same(keep[0][1].finish([gathered.data_ptr()], world), want)


@pytest.mark.parametrize("query,colnames", [("q06.vdl", Q6_COLS), ("q01.vdl", Q1_COLS)])
@pytest.mark.parametrize("world", [2, 4])
def test_peer_memory_exchange_emulated_ranks(catalog, query, colnames, world):
    """The fused combine: every rank's scan kernel stores its partial table into all ranks' exchange buffers, waits
    for the others' epoch flags and finalizes -- one launch per rank and step, no collective.  Ranks are emulated by
    one context (stream) each on the same GPU, driven from one host thread each; several steps to cover both buffer
    parities; the last rank owns an empty shard when the rows do not split."""
    import threading
    from mplan2vdl_b200.executor import Context
    rows, text = 40_000, plan_text(query)
    names = ["lineitem." + c for c in colnames]
    want = run_oracle(text, host_columns(catalog, names, {"lineitem": rows}))
    ctxs, plans = [], []
    for rank in range(world):
        start, n = tpch.shard_range(rows, rank, world)
        ctx = Context(0)
        for k, v in host_columns(catalog, names, {"lineitem": n}, row_offset=start).items():
            ctx.upload_column(k, v)
        plan = ctx.plan(text)
        plan.set_row_base(start)
        plan.run_local()                    # prepares the scan (all allocations happen here, none while peers spin)
        ctx.synchronize()
        ctxs.append(ctx)
        plans.append(plan)
    bufs = [ctxs[r].ipc_alloc(plans[r].exchange_bytes(0, world)) for r in range(world)]
    for r in range(world):
        plans[r].set_peers(0, r, world, bufs)
    for step in range(3):
        results, errors = [None] * world, []

        def work(r):
            try:
                results[r] = plans[r].run()
            except Exception as e:          # pragma: no cover
                errors.append(e)
        threads = [threading.Thread(target=work, args=(r,)) for r in range(world)]
        for t in threads:
            t.start()
        for t in threads:
            t.join(60)
        assert not errors, errors
        for r in range(world):
            assert_same(results[r], want)
    for r in range(world):
        plans[r].close()
        ctxs[r].ipc_free(bufs[r])
        ctxs[r].close()


@pytest.mark.parametrize("world,sf", [(2, 0.01), (3, 0.01), (4, 0.002)])      # (4, 0.002): the last rank's shard is empty
def test_fk_join_plan_sharded_through_probe_partials(catalog, world, sf):
    """Q5 (one probe fold group): lineitem row-range sharded, dimension tables replicated; the per-rank partial tables
    (FoldChoose values included) are concatenated like an all-gather and merged by every rank's finalize."""
    import torch
    from mplan2vdl_b200 import synth
    from mplan2vdl_b200.dist import DeviceView
    from mplan2vdl_b200.executor import Context
    text = plan_text("q05.vdl")
    names = tpch.plan_columns(text)
    rows = {t: synth.table_rows(catalog, t, sf) for t in catalog.tables}
    cols = host_columns(catalog, names, rows, sf=sf)
    want = run_oracle(text, cols)
    assert len(want["revenue"]) > 0 or sf < 0.01
    assert sf >= 0.01 or tpch.shard_range(rows["lineitem"], world - 1, world)[1] == 0
    ctxs, plans, tables = [], [], []
    for rank in range(world):
        start, n = tpch.shard_range(rows["lineitem"], rank, world)
        ctx = Context(0)
        for k, v in cols.items():
            ctx.upload_column(k, v[start:start + n] if k.startswith("lineitem.") else v)
        plan = ctx.plan(text)
        plan.set_row_base(start)
        plan.run_local()
        assert plan.num_fused == 0 and plan.num_partials == 1
        ptr, cnt = plan.partials(0)
        ctx.synchronize()
        tables.append(torch.as_tensor(DeviceView(ptr, cnt), device="cuda:0").clone())
        ctxs.append(ctx)
        plans.append(plan)
    gathered = torch.cat(tables)
    torch.cuda.synchronize()
    for rank in range(world):
        assert_same(plans[rank].finish([gathered.data_ptr()], world), want)
    for p, c in zip(plans, ctxs):
        p.close()
        c.close()


def test_peer_exchange_times_out_instead_of_hanging(catalog, monkeypatch):
    """A rank whose peer never launches the step must come back with an error, not spin forever."""
    from mplan2vdl_b200.executor import Context
    from mplan2vdl_b200.lib import VdlError
    monkeypatch.setenv("VDL_PEER_TIMEOUT_MS", "200")
    rows, text = 20_000, plan_text("q06.vdl")
    names = ["lineitem." + c for c in Q6_COLS]
    ctx = Context(0)
    for k, v in host_columns(catalog, names, {"lineitem": rows}).items():
        ctx.upload_column(k, v)
    plan = ctx.plan(text)
    plan.run_local()
    ctx.synchronize()
    bufs = [ctx.ipc_alloc(plan.exchange_bytes(0, 2)) for _ in range(2)]      # "rank 1" exists only as a buffer
    plan.set_peers(0, 0, 2, bufs)
    with pytest.raises(VdlError, match="peer GPU never delivered"):
        plan.run()
    plan.close()
    for b in bufs:
        ctx.ipc_free(b)
    ctx.close()


@pytest.mark.parametrize("q", ["q05.vdl", "q12.vdl"])
@pytest.mark.parametrize("world,sf", [(2, 0.01), (4, 0.01), (4, 0.002)])       # (4, 0.002): the last rank's shard is empty
def test_probe_fold_plans_combine_over_peer_memory(catalog, q, world, sf):
    """FK-join plans whose Folds run on the probe kernel: each rank's partial table crosses to every rank's exchange
    buffer inside a kernel (fold_exchange_kernel), the finalize merges them -- vdl_plan_run returns the global result on
    every rank, no collective, no host round trip.  Emulated ranks (one context + host thread each), three steps."""
    import threading
    from mplan2vdl_b200 import synth
    from mplan2vdl_b200.executor import Context
    text = plan_text(q)
    rows = {t: synth.table_rows(catalog, t, sf) for t in catalog.tables}
    cols = host_columns(catalog, tpch.plan_columns(text), rows, sf=sf)
    want = run_oracle(text, cols)
    ctxs, plans = [], []
    for rank in range(world):
        start, n = tpch.shard_range(rows["lineitem"], rank, world)
        ctx = Context(0)
        for k, v in cols.items():
            ctx.upload_column(k, v[start:start + n] if k.startswith("lineitem.") else v)
        plan = ctx.plan(text)
        plan.set_row_base(start)
        plan.run_local()
        ctx.synchronize()
        assert plan.num_fused == 0 and plan.num_partials == 1 and plan.num_emits == 0
        ctxs.append(ctx)
        plans.append(plan)
    bufs = [ctxs[r].ipc_alloc(plans[r].exchange_bytes(0, world)) for r in range(world)]
    for r in range(world):
        plans[r].set_peers(0, r, world, bufs)
    for step in range(3):
        results, errors = [None] * world, []

        def work(r):
            try:
                results[r] = plans[r].run()
            except Exception as e:          # pragma: no cover
                errors.append(e)
        threads = [threading.Thread(target=work, args=(r,)) for r in range(world)]
        for t in threads:
            t.start()
        for t in threads:
            t.join(60)
        assert not errors, errors
        for r in range(world):
            assert_same(results[r], want)
    for r in range(world):
        plans[r].close()
        ctxs[r].ipc_free(bufs[r])
        ctxs[r].close()


def test_probe_peer_exchange_times_out_instead_of_hanging(catalog, monkeypatch):
    from mplan2vdl_b200 import synth
    from mplan2vdl_b200.executor import Context
    from mplan2vdl_b200.lib import VdlError
    monkeypatch.setenv("VDL_PEER_TIMEOUT_MS", "200")
    text = plan_text("q12.vdl")
    rows = {t: synth.table_rows(catalog, t, 0.002) for t in catalog.tables}
    ctx = Context(0)
    for k, v in host_columns(catalog, tpch.plan_columns(text), rows, sf=0.002).items():
        ctx.upload_column(k, v)
    plan = ctx.plan(text)
    plan.run_local()
    ctx.synchronize()
    bufs = [ctx.ipc_alloc(plan.exchange_bytes(0, 2)) for _ in range(2)]      # "rank 1" exists only as a buffer
    plan.set_peers(0, 0, 2, bufs)
    with pytest.raises(VdlError, match="peer GPU never delivered"):
        plan.run()
    plan.close()
    for b in bufs:
        ctx.ipc_free(b)
    ctx.close()


@pytest.mark.parametrize("q", ["q03.vdl", "q19.vdl"])
@pytest.mark.parametrize("world,sf", [(2, 0.01), (3, 0.01), (4, 0.002)])       # (4, 0.002): the last rank's shard is empty
def test_emit_plans_sharded_by_exchanging_survivors(catalog, q, world, sf):
    """Plans whose probe passes EMIT vectors (Q3: high-cardinality group-by; Q19: an OR above the join): every rank
    probes its lineitem shard, the survivors are concatenated in rank order (what dist.gather_survivors does with
    all-gathers) and every rank evaluates the remaining ops on the global vectors."""
    import torch
    from mplan2vdl_b200 import synth
    from mplan2vdl_b200.dist import DeviceView
    from mplan2vdl_b200.executor import Context
    from util import q19_columns
    text = plan_text(q)
    if q == "q19.vdl":
        text, cols = q19_columns(catalog, sf=sf)
    else:
        rows_all = {t: synth.table_rows(catalog, t, sf) for t in catalog.tables}
        cols = host_columns(catalog, tpch.plan_columns(text), rows_all, sf=sf)
    nli = len(cols["lineitem.lineitem_l_orderkey_l_linenumber_pkey"])
    want = run_oracle(text, cols)
    assert len(next(iter(want.values()))) > 0 or sf < 0.01
    ctxs, plans = [], []
    for rank in range(world):
        start, n = tpch.shard_range(nli, rank, world)
        ctx = Context(0)
        for k, v in cols.items():
            ctx.upload_column(k, v[start:start + n] if k.startswith("lineitem.") else v)
        plan = ctx.plan(text)
        plan.set_row_base(start)
        plan.run_local()
        ctxs.append(ctx)
        plans.append(plan)
    nem = plans[0].num_emits
    assert nem >= 1 and plans[0].num_partials == 0
    keep = []
    for i in range(nem):
        parts = []
        for rank in range(world):
            ptr, n = plans[rank].emit(i)
            parts.append(torch.as_tensor(DeviceView(ptr, n), device="cuda:0").clone() if n else torch.empty(0, dtype=torch.int64, device="cuda:0"))
        g = torch.cat(parts)
        keep.append(g)
        torch.cuda.synchronize()
        for rank in range(world):
            plans[rank].emit_replace(i, g.data_ptr() if g.numel() else 0, g.numel())
    for rank in range(world):
        assert_same(plans[rank].finish([], world), want)
    for p, c in zip(plans, ctxs):
        p.close()
        c.close()
