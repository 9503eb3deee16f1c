"""Host-side executor front end: what a caller of the missing Voodoo server would use.

The reference's own pipeline (eval_query.sh:10-26) was: translate the mplan to a Voodoo program, POST
the text to the server, get ``{"results": {tmpN: {".<outname>": [ints]}}}`` back and decode it with
resolve.py.  Here the program text goes to ``Context.plan(text)`` and ``Plan.run()`` returns
``{outname: int64 array}`` in MaterializeCompact order; ``mplan2vdl_b200.resolve`` decodes it.
Everything below is a thin layer over the C ABI (include/vdl_cuda.h) -- no computation happens in Python.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import lib as _lib
from .lib import VDL_I32, VDL_I64, VDL_PLAN_FUSE, VdlError


class Context:
    """One per GPU (vdl_ctx).  Owns the registered columns."""

    def __init__(self, device: int = 0):
        self.L = _lib.load()
        h = C.c_void_p()
        rc = self.L.vdl_ctx_create(device, C.byref(h))
        if rc:
            raise VdlError(rc, self.L.vdl_last_error(None).decode())
        self.h = h
        self.device = device
        self._keepalive = {}

    def close(self):
        if getattr(self, "h", None):
            self.L.vdl_ctx_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def check(self, rc: int):
        if rc:
            raise VdlError(rc, self.L.vdl_last_error(self.h).decode())

    # ---- columns -----------------------------------------------------------------------------
    def alloc_column(self, name: str, width: int, rows: int) -> int:
        v = C.c_int32()
        self.check(self.L.vdl_column_alloc(self.h, name.encode(), width, rows, C.byref(v)))
        return v.value

    def upload_column(self, name: str, arr: np.ndarray) -> int:
        """Allocate + host->device copy of an int32/int64 numpy column (uint8: the bytes of a string heap, `<col>.heap`)."""
        if arr.dtype not in (np.int32, np.int64, np.uint8):
            raise TypeError(f"{name}: columns are int32 or int64 (uint8 for a string heap), got {arr.dtype}")
        arr = np.ascontiguousarray(arr)
        v = self.alloc_column(name, arr.dtype.itemsize, arr.shape[0])
        self.check(self.L.vdl_column_upload(self.h, v, arr.ctypes.data, arr.shape[0]))
        return v

    def upload_into(self, v: int, host_ptr: int, rows: int):
        """Host->device copy into an existing column (host memory may be pinned: then the copy is a straight DMA)."""
        self.check(self.L.vdl_column_upload(self.h, v, host_ptr, rows))

    def touch(self, v: int):
        """Tell the library that the column's memory was written behind its back (bound tensors, device_ptr())."""
        self.check(self.L.vdl_column_touch(self.h, v))

    def generation(self, v: int) -> int:
        g = C.c_uint64()
        self.check(self.L.vdl_vec_generation(self.h, v, C.byref(g)))
        return g.value

    def analyze(self, v: int):
        """Exact (min, max) of a column, computed on the device and cached until the column is written again."""
        lo, hi = C.c_int64(), C.c_int64()
        self.check(self.L.vdl_column_analyze(self.h, v, C.byref(lo), C.byref(hi)))
        return lo.value, hi.value

    def download_into(self, v: int, host_ptr: int, rows: int):
        """Device->host copy of a column in its stored type."""
        self.check(self.L.vdl_column_download(self.h, v, host_ptr, rows))

    def device_ptr(self, v: int) -> int:
        return self.L.vdl_vec_device_ptr(self.h, v) or 0

    def bind_tensor(self, name: str, tensor) -> int:
        """Register a CUDA torch tensor (int32/int64, contiguous) as a column without copying."""
        import torch
        if tensor.dtype not in (torch.int32, torch.int64) or not tensor.is_cuda or not tensor.is_contiguous():
            raise TypeError(f"{name}: need a contiguous CUDA int32/int64 tensor")
        v = C.c_int32()
        n = tensor.numel()
        self.check(self.L.vdl_column_bind(self.h, name.encode(), tensor.element_size(), n, n, tensor.data_ptr(), C.byref(v)))
        self._keepalive[name] = tensor
        return v.value

    def fill_synthetic(self, name: str, spec, rows: int, seed: int, row_offset: int = 0) -> int:
        """Allocate `rows` of column `name` and generate global rows [row_offset, row_offset+rows) in place."""
        v = self.alloc_column(name, spec.width, rows)
        self.check(self.L.vdl_column_fill_synthetic(self.h, v, seed & (2**64 - 1), spec.stream, spec.kind, spec.vmin,
                                                    spec.stride, spec.p0, spec.p1, row_offset))
        return v

    def drop_column(self, name: str):
        self.check(self.L.vdl_column_drop(self.h, name.encode()))
        self._keepalive.pop(name, None)

    def lookup(self, name: str) -> int:
        v = C.c_int32()
        self.check(self.L.vdl_column_lookup(self.h, name.encode(), C.byref(v)))
        return v.value

    # ---- vectors / per-op API ----------------------------------------------------------------
    def download(self, v: int) -> np.ndarray:
        n = C.c_int64()
        self.check(self.L.vdl_vec_len(self.h, v, C.byref(n)))
        out = np.empty(n.value, dtype=np.int64)
        self.check(self.L.vdl_vec_download(self.h, v, out.ctypes.data, n.value))
        return out

    def free(self, v: int):
        self.check(self.L.vdl_vec_free(self.h, v))

    def _out(self, fn, *args) -> int:
        v = C.c_int32()
        self.check(fn(self.h, *args, C.byref(v)))
        return v.value

    def op_range(self, start: int, step: int, length: int) -> int:
        return self._out(self.L.vdl_op_range, start, step, length)

    def op_binary(self, op: str, a: int, b: int) -> int:
        return self._out(self.L.vdl_op_binary, _lib.BINARY_OPS.index(op), a, b)

    def op_map(self, program, inputs, tables=(), imms=()) -> int:
        """One launch for a register program over row-aligned `inputs` (vdl_op_map).  program: (op, dst, a, b) with op a
        binary op name, "Load" (b = input), "Range" (a, b = indices into imms: from, step) or "Gather" (a = register
        holding the position, b = table)."""
        d = _lib.MapDesc()
        d.ninputs, d.ntables, d.ninstrs, d.nimms = len(inputs), len(tables), len(program), len(imms)
        special = {"Gather": _lib.VDL_MAP_GATHER, "Load": _lib.VDL_MAP_LOAD, "Range": _lib.VDL_MAP_RANGE}
        for t, (op, dst, a, b) in enumerate(program):
            d.instr[t] = _lib.MapInstr(special[op] if op in special else _lib.BINARY_OPS.index(op), dst, a, b)
        for k, v in enumerate(imms):
            d.imm[k] = v
        ins = (C.c_int32 * max(1, len(inputs)))(*inputs)
        tabs = (C.c_int32 * max(1, len(tables)))(*tables)
        return self._out(self.L.vdl_op_map, C.byref(d), ins, tabs)

    def op_like(self, data: int, heap: int, pattern: str) -> int:
        return self._out(self.L.vdl_op_like, data, heap, pattern.encode())

    def op_cross_product(self, left: int, right: int, inner: bool) -> int:
        return self._out(self.L.vdl_op_cross_product, left, right, int(inner))

    def op_fold_select(self, pred: int) -> int:
        return self._out(self.L.vdl_op_fold_select, pred)

    def op_gather(self, src: int, pos: int) -> int:
        return self._out(self.L.vdl_op_gather, src, pos)

    def op_scatter(self, src: int, pos: int, out_len: int) -> int:
        return self._out(self.L.vdl_op_scatter, src, pos, out_len)

    def op_partition(self, data: int, pivot_from: int, pivot_step: int, pivot_count: int) -> int:
        return self._out(self.L.vdl_op_partition, data, pivot_from, pivot_step, pivot_count)

    def op_fold(self, op: str, groups: int, data: int) -> int:
        return self._out(self.L.vdl_op_fold, _lib.FOLD_OPS.index(op), groups, data)

    def op_collate(self, data: int, heap: int, origin: int = 0) -> int:
        """Collation rank of every row's string (vdl_op_collate): the string of row i starts at heap byte data[i] - origin;
        the rank is the number of distinct strings of `data` that sort before it (unsigned byte order, prefixes first)."""
        return self._out(self.L.vdl_op_collate, data, heap, origin)

    def op_order(self, keys, descending=None, limit: int | None = None) -> int:
        """Positions that order the rows of the key vectors (vdl_op_order): lexicographic over `keys`, signed int64, key i
        descending when descending[i]; ties keep row order; the first `limit` of them (None: all)."""
        k = len(keys)
        ks = (C.c_int32 * max(1, k))(*keys)
        ds = (C.c_int * max(1, k))(*[int(bool(d)) for d in (descending or [0] * k)])
        return self._out(self.L.vdl_op_order, k, ks, ds, -1 if limit is None else limit)

    # ---- peer-addressable buffers (multi-GPU combine without a collective library) ------------
    def ipc_alloc(self, nbytes: int) -> int:
        p = C.c_void_p()
        self.check(self.L.vdl_ipc_alloc(self.h, nbytes, C.byref(p)))
        return p.value

    def ipc_export(self, ptr: int) -> bytes:
        buf = C.create_string_buffer(64)
        self.check(self.L.vdl_ipc_export(self.h, C.c_void_p(ptr), buf))
        return buf.raw

    def ipc_open(self, handle: bytes) -> int:
        p = C.c_void_p()
        self.check(self.L.vdl_ipc_open(self.h, handle, C.byref(p)))
        return p.value

    def ipc_close(self, ptr: int):
        self.check(self.L.vdl_ipc_close(self.h, C.c_void_p(ptr)))

    def ipc_free(self, ptr: int):
        self.check(self.L.vdl_ipc_free(self.h, C.c_void_p(ptr)))

    # ---- misc --------------------------------------------------------------------------------
    def synchronize(self):
        self.check(self.L.vdl_ctx_synchronize(self.h))

    @property
    def stream(self) -> int:
        return self.L.vdl_ctx_stream(self.h) or 0

    @property
    def launch_count(self) -> int:
        return self.L.vdl_ctx_launch_count(self.h)

    def plan(self, text: str, fuse: bool = True) -> "Plan":
        return Plan(self, text, fuse)


def order_keys(names, keys) -> tuple:
    """(output indices, descending flags) of ORDER BY `keys` over outputs `names`.  A key is a name or (name, descending); a
    name is a full output name or its alias, the part before the first '__' (``o_orderdate`` for
    ``o_orderdate__orders__o_orderdate``).  Raises KeyError for a name that matches no output or more than one."""
    idx, desc = [], []
    for key in keys:
        name, d = (key, False) if isinstance(key, str) else (key[0], bool(key[1]))
        hits = [i for i, n in enumerate(names) if n == name]
        if not hits:
            hits = [i for i, n in enumerate(names) if n.split("__", 1)[0] == name]
        if len(hits) != 1:
            raise KeyError(f"ORDER BY {name!r}: {'no output' if not hits else 'more than one output'} of "
                           f"{list(names)} has that name or alias")
        idx.append(hits[0])
        desc.append(d)
    return idx, desc


def explain(text: str, fuse: bool = True) -> dict:
    """What the planner makes of a program (vdl_plan_explain): no GPU, no columns needed.  Raises VdlError for a program
    the parser or the planner rejects."""
    import json
    L = _lib.load()
    buf = C.create_string_buffer(1 << 16)
    rc = L.vdl_plan_explain(text.encode(), VDL_PLAN_FUSE if fuse else 0, buf, len(buf))
    doc = json.loads(buf.value.decode()) if buf.value else {}
    if rc:
        raise VdlError(rc, doc.get("message", "vdl_plan_explain failed"))
    return doc


class Plan:
    """A loaded Voodoo program (vdl_plan)."""

    def __init__(self, ctx: Context, text: str, fuse: bool = True):
        self.ctx, self.L = ctx, ctx.L
        h = C.c_void_p()
        ctx.check(self.L.vdl_plan_load(ctx.h, text.encode(), VDL_PLAN_FUSE if fuse else 0, C.byref(h)))
        self.h = h

    def close(self):
        if getattr(self, "h", None) and getattr(self.ctx, "h", None):
            self.L.vdl_plan_destroy(self.h)
        self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def stats(self) -> dict:
        s, n, f, l = C.c_int(), C.c_int(), C.c_int(), C.c_int64()
        self.ctx.check(self.L.vdl_plan_stats(self.h, C.byref(s), C.byref(n), C.byref(f), C.byref(l)))
        pf, pe, pv = C.c_int(), C.c_int(), C.c_int()
        self.ctx.check(self.L.vdl_plan_probe_stats(self.h, C.byref(pf), C.byref(pe), C.byref(pv)))
        mc, mn = C.c_int(), C.c_int()
        self.ctx.check(self.L.vdl_plan_map_stats(self.h, C.byref(mc), C.byref(mn)))
        return {"statements": s.value, "nodes": n.value, "fused_scans": f.value, "launches": l.value,
                "probe_folds": pf.value, "probe_emits": pe.value, "emitted_vectors": pv.value,
                "map_clusters": mc.value, "map_nodes": mn.value}

    def set_row_base(self, row_base: int):
        self.ctx.check(self.L.vdl_plan_set_row_base(self.h, row_base))

    def exchange_bytes(self, i: int, world: int) -> int:
        n = C.c_int64()
        self.ctx.check(self.L.vdl_plan_exchange_bytes(self.h, i, world, C.byref(n)))
        return n.value

    def set_peers(self, i: int, rank: int, world: int, ptrs):
        """Exchange buffers (device pointers valid on THIS GPU) of all ranks for fused scan i; run() then returns the
        global result on every rank with one kernel launch per GPU."""
        arr = (C.c_void_p * world)(*ptrs)
        self.ctx.check(self.L.vdl_plan_set_peers(self.h, i, rank, world, arr))

    def run_local(self):
        self.ctx.check(self.L.vdl_plan_run_local(self.h))

    @property
    def num_fused(self) -> int:
        return self.L.vdl_plan_num_fused(self.h)

    @property
    def num_emits(self) -> int:
        """Vectors emitted by probe passes (sharded runs exchange them between run_local() and finish())."""
        return self.L.vdl_plan_num_emits(self.h)

    def emit(self, i: int):
        p, n = C.c_void_p(), C.c_int64()
        self.ctx.check(self.L.vdl_plan_emit(self.h, i, C.byref(p), C.byref(n)))
        return p.value or 0, n.value

    def emit_replace(self, i: int, ptr: int, n: int):
        self.ctx.check(self.L.vdl_plan_emit_replace(self.h, i, C.c_void_p(ptr), n))

    def emit_tables(self) -> list:
        """The table each probe emit group walks (vdl_plan_emit_group_table)."""
        out = []
        for g in range(self.stats()["probe_emits"]):
            name = C.c_char_p()
            self.ctx.check(self.L.vdl_plan_emit_group_table(self.h, g, C.byref(name)))
            out.append(name.value.decode())
        return out

    def tail_info(self):
        """None, or the fold op (VDL_FOLD_*: 0 Sum, 1 Min, 2 Max, 3 Choose, 4 Count) of every output when all of them are
        Folds by runs of one groups vector: the plan's tail can then run on a row-range shard (vdl_plan_tail_info)."""
        n = self.L.vdl_plan_num_outputs(self.h)
        ok, ops = C.c_int(), (C.c_int * max(n, 1))()
        self.ctx.check(self.L.vdl_plan_tail_info(self.h, C.byref(ok), ops, n))
        return [ops[i] for i in range(n)] if ok.value else None

    def tail_enable(self, on: bool = True):
        self.ctx.check(self.L.vdl_plan_tail_enable(self.h, int(on)))

    def tail_boundary(self, into=None):
        """[keys in order, runs, first key, last key, first row of every output ..., last row of every output ...] of the
        last run (after tail_enable).  `into`: a ctypes int64 array to fill instead of building a list."""
        n = 4 + 2 * self.L.vdl_plan_num_outputs(self.h)
        rec = into if into is not None else (C.c_int64 * n)()
        self.ctx.check(self.L.vdl_plan_tail_boundary(self.h, rec, len(rec)))
        return rec if into is not None else list(rec)

    def tail_apply(self, drop_first: bool, last_row=None):
        """The boundary merge's verdict for this rank (vdl_plan_tail_apply): outputs() then returns the rank's slice."""
        arr = None
        if last_row is not None:
            arr = (C.c_int64 * len(last_row))(*last_row)
        self.ctx.check(self.L.vdl_plan_tail_apply(self.h, int(drop_first), arr))

    @property
    def num_partials(self) -> int:
        """Partial aggregate tables of a sharded run: the fused scans, then the probe fold groups."""
        return self.L.vdl_plan_num_partials(self.h)

    def partials(self, i: int):
        """(device pointer, number of int64) of partial table i (finish() takes the gathered buffers in this order)."""
        p, n = C.c_void_p(), C.c_int64()
        self.ctx.check(self.L.vdl_plan_partials(self.h, i, C.byref(p), C.byref(n)))
        return p.value, n.value

    def shape(self, i: int = 0) -> str:
        """Which scan-kernel instantiation fused scan i uses: "generic" or a static shape name."""
        f = C.c_void_p()
        self.ctx.check(self.L.vdl_plan_fused(self.h, i, C.byref(f)))
        return self.L.vdl_fused_shape_name(f).decode()

    def kernel_ms(self, i: int = 0) -> float:
        f = C.c_void_p()
        self.ctx.check(self.L.vdl_plan_fused(self.h, i, C.byref(f)))
        ms = C.c_float()
        self.ctx.check(self.L.vdl_fused_last_kernel_ms(f, C.byref(ms)))
        return ms.value

    def kernel_ms_stats(self, n: int):
        """(mean, min) duration in ms of the plan's dominant kernel over the last n runs (events recorded by the library)."""
        a, b = C.c_float(), C.c_float()
        self.ctx.check(self.L.vdl_plan_kernel_ms_stats(self.h, n, C.byref(a), C.byref(b)))
        return a.value, b.value

    def probe_kernel_ms(self) -> float:
        ms = C.c_float()
        self.ctx.check(self.L.vdl_plan_probe_kernel_ms(self.h, C.byref(ms)))
        return ms.value

    def finish(self, gathered_ptrs=None, nranks: int = 1, copy: bool = True) -> dict:
        arr = None
        if gathered_ptrs is not None:
            arr = (C.c_void_p * len(gathered_ptrs))(*gathered_ptrs)
        self.ctx.check(self.L.vdl_plan_finish(self.h, arr, nranks))
        return self.outputs(copy)

    def run(self, copy: bool = True) -> dict:
        self.ctx.check(self.L.vdl_plan_run(self.h))
        return self.outputs(copy)

    def execute(self):
        """vdl_plan_run alone: when it returns the results are in the library's pinned host buffers (outputs() wraps them
        as arrays).  What a host that steps a plan repeatedly calls -- no Python objects are built per step."""
        rc = self.L.vdl_plan_run(self.h)
        if rc:
            self.ctx.check(rc)

    def set_typed_outputs(self, on: bool = True):
        """Result columns whose values provably fit travel as int32 (vdl_plan_set_typed_outputs); outputs() then returns
        int32 arrays for them."""
        self.ctx.check(self.L.vdl_plan_set_typed_outputs(self.h, int(on)))

    def output_names(self) -> list:
        """The output names in MaterializeCompact order (known from loading: no run needed)."""
        names = []
        for i in range(self.L.vdl_plan_num_outputs(self.h)):
            name = C.c_char_p()
            self.ctx.check(self.L.vdl_plan_output_typed(self.h, i, C.byref(name), None, None, None))
            names.append(name.value.decode())
        return names

    def set_order(self, keys, limit: int | None = None, heaps=None):
        """ORDER BY `keys` LIMIT `limit`, applied on the device to every later run before the results are copied
        (vdl_plan_set_order).  keys: [name or (name, descending)], names as `order_keys` resolves them; ([], None) turns
        the order off.  heaps: {key name or alias: heap handle or (heap handle, origin)}: that key compares by the strings
        its values point to in the heap (vdl_plan_set_order_heap, vdl_op_collate), not by the values themselves.  An
        unknown or ambiguous name, or a heap name that is not among the keys, raises before anything is set."""
        names = self.output_names()
        idx, desc = order_keys(names, keys)
        by_key = []
        for name, h in (heaps or {}).items():
            (i,), _ = order_keys(names, [name])
            if i not in idx:
                raise KeyError(f"ORDER BY heap {name!r}: {names[i]} is not among the keys {[names[j] for j in idx]}")
            h, origin = h if isinstance(h, tuple) else (h, 0)
            by_key.append((idx.index(i), int(h), int(origin)))
        self._set_order(idx, desc, -1 if limit is None else limit)
        for k, h, origin in by_key:
            self._set_order_heap(k, h, origin)

    def _set_order(self, idx, desc, limit: int):
        k = len(idx)
        self.ctx.check(self.L.vdl_plan_set_order(self.h, k, (C.c_int * max(1, k))(*idx),
                                                 (C.c_int * max(1, k))(*[int(d) for d in desc]), limit))

    def _set_order_heap(self, key: int, heap: int, origin: int):
        self.ctx.check(self.L.vdl_plan_set_order_heap(self.h, key, heap, origin))

    def outputs(self, copy: bool = True) -> dict:
        """{output name: int64 (or, with typed outputs, int32) array}.  copy=False returns views of the library's pinned host
        buffers, valid until the plan runs again or is closed."""
        out = {}
        for i in range(self.L.vdl_plan_num_outputs(self.h)):
            name, data, n, dt = C.c_char_p(), C.c_void_p(), C.c_int64(), C.c_int()
            self.ctx.check(self.L.vdl_plan_output_typed(self.h, i, C.byref(name), C.byref(data), C.byref(n), C.byref(dt)))
            if n.value:
                ctype = C.c_int32 if dt.value == 4 else C.c_int64
                arr = np.ctypeslib.as_array(C.cast(data, C.POINTER(ctype)), shape=(n.value,))
            else:
                arr = np.zeros(0, np.int64)
            out[name.value.decode()] = arr.copy() if copy and n.value else arr
        return out
