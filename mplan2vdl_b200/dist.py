"""Row-range sharded execution: one process per GPU, torch.distributed for the plumbing.

Two ways to combine the per-rank partial aggregate tables:
* peer memory (default on GPUs): every rank owns a small exchange buffer that all ranks map (CUDA IPC); the LAST
  thread block of each rank's scan kernel stores its table into every peer's buffer over NVLink, publishes an epoch
  flag, waits for the other ranks' flags, merges and finalizes.  One kernel launch per GPU and step, no collective
  library on the data path (include/vdl_cuda.h, "multi-GPU combine over peer memory").  A probe pass in fold mode
  combines with the same code in two more launches: probe_choose_kernel, then the one-block fold_exchange_kernel
  (exchange, merge, finalize), which also serves a scan rank with an empty shard.
* all-gather (gloo on CPUs in the tests, NCCL if peer mapping is unavailable or VDL_NO_PEER is set), described next.

The fact table is split by contiguous row range (tpch.shard_range), dimension tables are replicated, every rank
runs the same plan on its shard (vdl_plan_run_local), the per-rank partial aggregate tables -- [accumulators x key
domain] int64, a few bytes to a few KB -- are all-gathered (NCCL over NVLink on GPUs), and every rank merges them in
fold_finalize_kernel (vdl_plan_finish): SUM/MIN/MAX accumulators combine by their op, FoldChoose takes the value
from the rank that holds the smallest first row, empty groups are dropped after the merge.  There is no other
data-path collective: the scan itself never leaves the GPU that owns the rows.

Plans that EMIT survivors (Q3, Q19) and whose outputs are all Folds by runs of one groups vector run their whole tail on
the shard (vdl_plan_tail_*): every rank keeps the slice of the result that belongs to its rows, and only a boundary record
per rank -- run count, first / last key, first / last row of every output, a few dozen int64 -- is all-gathered so that the
groups straddling shard boundaries are merged into the rank where they start (merge_tail_boundaries).  The survivors never
move; the result stays sharded (ShardedPlan.global_result concatenates it when somebody wants it in one place).  Anything
else that emits falls back to all-gathering the survivors and evaluating the tail on every rank.
"""
from __future__ import annotations

import torch


class DeviceView:
    """Library-owned device memory exposed through __cuda_array_interface__ so torch can wrap it without a copy."""

    def __init__(self, ptr: int, n_int64: int):
        self.__cuda_array_interface__ = {"shape": (n_int64,), "typestr": "<i8", "data": (ptr, False), "version": 2}


def gather_survivors(local: torch.Tensor, world: int, group=None) -> torch.Tensor:
    """All-gather vectors of DIFFERENT lengths (each rank's surviving rows of an emitted vector) into their
    concatenation in rank order: lengths first, then the vectors padded to the longest."""
    import torch.distributed as dist
    n = torch.tensor([local.numel()], dtype=torch.int64, device=local.device)
    lens = torch.empty(world, dtype=torch.int64, device=local.device)
    if local.is_cuda:
        dist.all_gather_into_tensor(lens, n, group=group)
    else:
        parts = list(lens.view(world, 1).unbind(0))
        dist.all_gather(parts, n, group=group)
    lens = lens.tolist()
    width = max(max(lens), 1)
    padded = torch.zeros(width, dtype=local.dtype, device=local.device)
    padded[:local.numel()] = local
    out = torch.empty(world * width, dtype=local.dtype, device=local.device)
    if local.is_cuda:
        dist.all_gather_into_tensor(out, padded, group=group)
    else:
        parts = list(out.view(world, width).unbind(0))
        dist.all_gather(parts, padded, group=group)
    return torch.cat([out[r * width:r * width + lens[r]] for r in range(world)]) if sum(lens) else out[:0]


def gather_partial_tables(local: torch.Tensor, world: int, group=None) -> torch.Tensor:
    """All-gather one rank-local partial table (1-D int64 tensor, CPU/gloo or CUDA/nccl) into [world * n]."""
    import torch.distributed as dist
    out = torch.empty(world * local.numel(), dtype=local.dtype, device=local.device)
    if local.is_cuda:
        dist.all_gather_into_tensor(out, local, group=group)
    else:                                   # gloo has no all_gather_into_tensor for every build: use the list form
        parts = list(out.view(world, -1).unbind(0))
        dist.all_gather(parts, local, group=group)
    return out


FOLD_SUM, FOLD_MIN, FOLD_MAX, FOLD_CHOOSE, FOLD_COUNT = range(5)


def merge_tail_boundaries(recs, ops, rank):
    """recs[r] = [sorted, runs, first key, last key, first row of every output ..., last row of every output ...] of rank
    r's local result.  Returns None when the shards' keys are not globally in order (the caller falls back to moving the
    survivors), else (drop_first, last_row): drop_first -- this rank's first group continues a group that starts on an
    earlier rank; last_row -- the values of this rank's last group after merging the following ranks' share of it, or
    None when nothing changes.  FoldChoose keeps the value of the rank where the group starts (first of the run, G6)."""
    k = len(ops)
    live = [r for r in range(len(recs)) if recs[r][1] > 0]
    if any(not recs[r][0] for r in live):
        return None
    for a, b in zip(live, live[1:]):
        if recs[a][3] > recs[b][2]:
            return None
    if rank not in live:
        return False, None
    at = live.index(rank)
    me = recs[rank]
    drop_first = at > 0 and recs[live[at - 1]][3] == me[2]
    if me[1] == 1 and drop_first:                      # my only group belongs to an earlier rank
        return True, None
    last, changed = list(me[4 + k:4 + 2 * k]), False
    for r in live[at + 1:]:
        if recs[r][2] != me[3]:
            break
        first = recs[r][4:4 + k]
        for i, op in enumerate(ops):
            if op in (FOLD_SUM, FOLD_COUNT):
                last[i] = (last[i] + first[i] + 2 ** 63) % 2 ** 64 - 2 ** 63      # int64 wrap-around, as the kernels add
            elif op == FOLD_MIN:
                last[i] = min(last[i], first[i])
            elif op == FOLD_MAX:
                last[i] = max(last[i], first[i])
        changed = True
        if recs[r][1] > 1:                             # the group ends inside rank r
            break
    return drop_first, (last if changed else None)


def check_shardable(plan, world: int, fact_table: str):
    """Row-range sharding of a plan that emits survivors is implemented for ONE probe pass over the sharded fact table
    (Q3, Q19).  A pass over a replicated dimension table would emit the same rows on every rank, and a semijoin's dimension
    side needs matches from every rank's fact rows (Q4, Q20): refused loudly rather than miscomputed."""
    if world > 1 and plan.num_emits > 0:
        tables = plan.emit_tables()
        if len(tables) != 1 or tables[0] != fact_table:
            raise NotImplementedError(f"plan with probe emit passes over {tables} cannot be row-range sharded on {fact_table!r}: "
                                      "run it on one GPU")


class ShardedPlan:
    """A plan executed over this rank's shard; step() returns the global result on every rank."""

    def __init__(self, ctx, plan, rank: int, world: int, row_base: int, group=None, peer: bool | None = None, fact_table: str = "lineitem"):
        import os
        check_shardable(plan, world, fact_table)
        self.ctx, self.plan, self.rank, self.world, self.group = ctx, plan, rank, world, group
        plan.set_row_base(row_base)
        self._stream = torch.cuda.ExternalStream(ctx.stream, device=ctx.device) if world > 1 else None
        self._gathered = []
        self._want_peer = world > 1 and (peer if peer is not None else not os.environ.get("VDL_NO_PEER"))
        self.peer_mode = False
        self.peer_fallback = None          # why the peer-memory combine is not in use (None: it is, or was never wanted)
        self._mine, self._opened = [], []
        # sharded tail: decided from the plan's shape alone, so every rank decides alike
        self.tail_ops = plan.tail_info() if world > 1 and plan.num_emits > 0 and not os.environ.get("VDL_NO_TAIL") else None
        self.tail_mode = self.tail_ops is not None
        if self.tail_mode:
            plan.tail_enable(True)
        self._tail_slice, self._tb = None, None

    def _tail_buffers(self):
        """Allocated once: the record as a ctypes array over a pinned tensor, its device copy, the gathered records."""
        import ctypes
        import torch.distributed as dist
        n = 4 + 2 * len(self.tail_ops)
        cuda = torch.cuda.is_available() and dist.get_backend(self.group) == "nccl"
        host = torch.zeros(n, dtype=torch.int64, pin_memory=cuda)
        rec = (ctypes.c_int64 * n).from_address(host.data_ptr())
        allhost = torch.zeros(self.world * n, dtype=torch.int64, pin_memory=cuda)
        dev = torch.zeros(n, dtype=torch.int64, device=f"cuda:{self.ctx.device}") if cuda else None
        alldev = torch.zeros(self.world * n, dtype=torch.int64, device=f"cuda:{self.ctx.device}") if cuda else None
        self._tb = (n, cuda, host, rec, allhost, dev, alldev)
        return self._tb

    def _step_tail(self):
        """Whole plan on the shard, then the boundary records of all ranks; returns False when the shards turn out not to be
        globally ordered (every rank sees the same records, so every rank falls back together)."""
        import torch.distributed as dist
        n, cuda, host, rec, allhost, dev, alldev = self._tb or self._tail_buffers()
        self.plan.execute()                              # probe pass + tail on this rank's rows, outputs in pinned memory
        self.plan.tail_boundary(rec)                     # straight into the pinned tensor
        if cuda:
            dev.copy_(host, non_blocking=True)
            dist.all_gather_into_tensor(alldev, dev, group=self.group)
            allhost.copy_(alldev, non_blocking=True)
            torch.cuda.current_stream().synchronize()
        else:
            parts = list(allhost.view(self.world, n).unbind(0))
            dist.all_gather(parts, host, group=self.group)
        merged = merge_tail_boundaries(allhost.view(self.world, n).tolist(), self.tail_ops, self.rank)
        if merged is None:
            return False
        self.plan.tail_apply(*merged)
        self._tail_slice = None                          # wrapped on demand (outputs())
        return True

    def outputs(self) -> dict:
        """This rank's share of the last step's result: the global result when the plan combines partial tables, the slice
        for this rank's rows in sharded-tail mode (views of the library's pinned buffers, valid until the next step)."""
        return self.plan.outputs(False)

    def global_result(self) -> dict:
        """The whole result on every rank (copies).  Sharded-tail plans gather their slices in rank order."""
        import numpy as np
        if not self.tail_mode:
            return {k: np.array(v, copy=True) for k, v in self.plan.outputs(False).items()}
        import torch.distributed as dist
        parts = [None] * self.world
        dist.all_gather_object(parts, {k: np.array(v, copy=True) for k, v in self.plan.outputs(False).items()}, group=self.group)
        return {k: np.concatenate([p[k] for p in parts]) for k in parts[0]}

    def _setup_peers(self) -> bool:
        """Allocate / exchange / map the exchange buffers (after the scans exist, i.e. after one step).  Collective:
        EVERY rank takes part in every all_gather_object and in the final MIN all_reduce whatever failed locally (a
        rank that left the sequence early would leave the others in a mismatched collective: a hang), the ranks agree
        once on success, and on failure everything opened or allocated so far is released again."""
        import torch.distributed as dist
        ok, ptr_lists, why = 1, [], ""
        for i in range(self.plan.num_partials):       # fused scans, then probe fold groups
            mine, blob = None, None
            if ok:
                try:
                    mine = self.ctx.ipc_alloc(self.plan.exchange_bytes(i, self.world))
                    self._mine.append(mine)
                    blob = self.ctx.ipc_export(mine)
                except Exception as e:
                    ok, why = 0, f"partial table {i}: {e}"
            handles = [None] * self.world
            dist.all_gather_object(handles, blob, group=self.group)       # None = "this rank could not export"
            if ok and any(h is None for h in handles):
                ok, why = 0, f"partial table {i}: a peer could not export its buffer"
            if not ok:
                continue
            ptrs = []
            try:
                for r, h in enumerate(handles):
                    if r == self.rank:
                        ptrs.append(mine)
                    else:
                        ptrs.append(self.ctx.ipc_open(h))
                        self._opened.append(ptrs[-1])
                ptr_lists.append(ptrs)
            except Exception as e:
                ok, why = 0, f"partial table {i}: {e}"
        flag = torch.tensor([ok], device=f"cuda:{self.ctx.device}" if torch.cuda.is_available() else "cpu")
        dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=self.group)
        if int(flag.item()) == 0:
            self.peer_fallback = why or "a peer rank could not map the exchange buffers"
            print(f"[vdl] rank {self.rank}: peer-memory exchange unavailable ({self.peer_fallback}); using the all-gather path", flush=True)
            self.close()                                 # unmap / free what this rank did manage to set up
            return False
        for i, ptrs in enumerate(ptr_lists):
            self.plan.set_peers(i, self.rank, self.world, ptrs)
        dist.barrier(group=self.group)
        return True

    def step(self, copy: bool = True, fetch: bool = True) -> dict:
        """copy=False: the arrays are views of pinned host buffers owned by the library, valid until the next step.
        fetch=False: run the step only (the results are on the host when it returns; plan.outputs() reads them)."""
        if self.world == 1 or self.peer_mode:
            if not fetch:
                return self.plan.execute()
            return self.plan.run(copy)                  # one launch per fused scan: its last thread block finalizes
        if self.tail_mode:
            if self._step_tail():
                return self.plan.outputs(copy) if fetch else None
            self.tail_mode = False                      # shards not globally ordered: move the survivors instead
            self.plan.tail_enable(False)
        out = self._step_all_gather(copy)
        if self._want_peer:                             # the scans exist now: switch to the peer-memory combine
            self._want_peer = False                     # (plans that emit survivors keep the all-gather path)
            self.peer_mode = self.plan.num_partials > 0 and self.plan.num_emits == 0 and self._setup_peers()
        return out

    def _step_all_gather(self, copy: bool = True) -> dict:
        self.plan.run_local()
        ptrs = []
        with torch.cuda.stream(self._stream):           # NCCL is ordered after the scan on the library's stream
            for i in range(self.plan.num_partials):
                ptr, n = self.plan.partials(i)
                local = torch.as_tensor(DeviceView(ptr, n), device=f"cuda:{self.ctx.device}")
                g = gather_partial_tables(local, self.world, self.group)
                if len(self._gathered) <= i:
                    self._gathered.append(None)
                self._gathered[i] = g                   # keep alive until finish() has consumed it
                ptrs.append(g.data_ptr())
            self._survivors = []
            for i in range(self.plan.num_emits):        # plans that emit vectors: every rank continues on ALL survivors
                ptr, n = self.plan.emit(i)
                local = torch.as_tensor(DeviceView(ptr, n), device=f"cuda:{self.ctx.device}") if n else \
                    torch.empty(0, dtype=torch.int64, device=f"cuda:{self.ctx.device}")
                g = gather_survivors(local, self.world, self.group)
                self._survivors.append(g)
                self.plan.emit_replace(i, g.data_ptr() if g.numel() else 0, g.numel())
            self._stream.synchronize()                  # the gathered vectors are complete before the library reads them
        return self.plan.finish(ptrs, self.world, copy)

    def close(self):
        for p in self._opened:
            try:
                self.ctx.ipc_close(p)
            except Exception:
                pass
        for p in self._mine:
            try:
                self.ctx.ipc_free(p)
            except Exception:
                pass
        self._opened, self._mine = [], []
