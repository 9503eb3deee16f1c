"""ctypes binding of libvdl_cuda's C ABI (include/vdl_cuda.h).

The product path has no CPU fallback: if the CUDA library is missing this module raises.
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
SO = os.path.join(HERE, "libvdl_cuda.so")

VDL_U8, VDL_I32, VDL_I64 = 1, 4, 8
VDL_PLAN_FUSE = 1
BINARY_OPS = ["LogicalAnd", "LogicalOr", "BitwiseAnd", "BitwiseOr", "BitShift", "Equals", "Add", "Subtract",
              "Greater", "Multiply", "Divide", "Modulo"]
FOLD_OPS = ["FoldSum", "FoldMin", "FoldMax", "FoldChoose", "FoldCount"]
VDL_MAX_COLS, VDL_MAX_PREDS, VDL_MAX_KEYS, VDL_MAX_AGGS, VDL_MAX_FACTORS, VDL_MAX_POSTS = 12, 8, 4, 8, 3, 8
VDL_POST_FOLD, VDL_POST_POST, VDL_POST_CONST = 0, 1, 2
VDL_MAX_ORDER_KEYS = 8


class VdlError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"libvdl_cuda error {code}: {msg}")
        self.code = code


class Affine(C.Structure):
    _fields_ = [("column", C.c_int32), ("shr", C.c_int32), ("a", C.c_int64), ("b", C.c_int64)]


class RangePred(C.Structure):
    _fields_ = [("column", C.c_int32), ("shr", C.c_int32), ("lo", C.c_int64), ("hi", C.c_int64)]


class KeyPart(C.Structure):
    _fields_ = [("e", Affine), ("shl", C.c_int32), ("pad", C.c_int32)]


class FoldSpec(C.Structure):
    _fields_ = [("op", C.c_int32), ("nfactors", C.c_int32), ("factor", Affine * VDL_MAX_FACTORS)]


class PostOp(C.Structure):
    _fields_ = [("op", C.c_int32), ("a_kind", C.c_int32), ("b_kind", C.c_int32), ("pad", C.c_int32),
                ("a", C.c_int64), ("b", C.c_int64)]


class FusedDesc(C.Structure):
    _fields_ = [("rows", C.c_int64), ("row_base", C.c_int64), ("ncolumns", C.c_int32),
                ("column", C.c_int32 * VDL_MAX_COLS), ("npreds", C.c_int32), ("pred", RangePred * VDL_MAX_PREDS),
                ("nkeys", C.c_int32), ("key", KeyPart * VDL_MAX_KEYS), ("key_mask", C.c_int64), ("domain", C.c_int64),
                ("nfolds", C.c_int32), ("fold", FoldSpec * VDL_MAX_AGGS),
                ("nposts", C.c_int32), ("post", PostOp * VDL_MAX_POSTS)]


VDL_MAX_LEAVES, VDL_MAX_PROBE_PREDS, VDL_MAX_EMITS, VDL_MAX_INDICATORS, VDL_MAX_MORE_RANGES = 24, 12, 8, 4, 3


class Leaf(C.Structure):
    _fields_ = [("column", C.c_int32), ("parent", C.c_int32)]


class Term(C.Structure):
    _fields_ = [("leaf", C.c_int32), ("shr", C.c_int32), ("a", C.c_int64), ("b", C.c_int64)]


class ProbePred(C.Structure):
    _fields_ = [("kind", C.c_int32), ("cmp", C.c_int32), ("t", Term), ("u", Term), ("lo", C.c_int64), ("hi", C.c_int64),
                ("nmore", C.c_int32), ("pad", C.c_int32), ("lo_more", C.c_int64 * VDL_MAX_MORE_RANGES), ("hi_more", C.c_int64 * VDL_MAX_MORE_RANGES)]


class Product(C.Structure):
    _fields_ = [("nfactors", C.c_int32), ("pad", C.c_int32), ("factor", Term * VDL_MAX_FACTORS)]


class ProbeFold(C.Structure):
    _fields_ = [("op", C.c_int32), ("pad", C.c_int32), ("value", Product)]


class ProbeDesc(C.Structure):
    _fields_ = [("rows", C.c_int64), ("row_base", C.c_int64), ("nleaves", C.c_int32), ("npreds", C.c_int32),
                ("leaf", Leaf * VDL_MAX_LEAVES), ("pred", ProbePred * VDL_MAX_PROBE_PREDS),
                ("nkeys", C.c_int32), ("nfolds", C.c_int32), ("key", Term * VDL_MAX_KEYS), ("key_shl", C.c_int32 * VDL_MAX_KEYS),
                ("key_mask", C.c_int64), ("domain", C.c_int64), ("fold", ProbeFold * VDL_MAX_AGGS),
                ("nposts", C.c_int32), ("nemits", C.c_int32), ("post", PostOp * VDL_MAX_POSTS), ("emit", Product * VDL_MAX_EMITS),
                ("nindicators", C.c_int32), ("pad2", C.c_int32), ("indicator", ProbePred * VDL_MAX_INDICATORS)]


VDL_MAP_MAX_INPUTS, VDL_MAP_MAX_TABLES, VDL_MAP_MAX_INSTRS, VDL_MAP_MAX_IMMS, VDL_MAP_MAX_REGS = 48, 8, 160, 32, 32
VDL_MAP_GATHER, VDL_MAP_LOAD, VDL_MAP_RANGE = 16, 17, 18


class MapInstr(C.Structure):
    _fields_ = [("op", C.c_int16), ("dst", C.c_int16), ("a", C.c_int16), ("b", C.c_int16)]


class MapDesc(C.Structure):
    _fields_ = [("ninputs", C.c_int32), ("ntables", C.c_int32), ("ninstrs", C.c_int32), ("nimms", C.c_int32),
                ("instr", MapInstr * VDL_MAP_MAX_INSTRS), ("imm", C.c_int64 * VDL_MAP_MAX_IMMS)]


# every symbol include/vdl_cuda.h declares: (name, restype, argtypes)
_P, _I, _L = C.c_void_p, C.c_int, C.c_int64
SYMBOLS = [
    ("vdl_abi_version", _I, []),
    ("vdl_abi_sizeof_fused_desc", _I, []),
    ("vdl_ctx_create", _I, [_I, C.POINTER(_P)]),
    ("vdl_ctx_destroy", _I, [_P]),
    ("vdl_last_error", C.c_char_p, [_P]),
    ("vdl_ctx_stream", _P, [_P]),
    ("vdl_ctx_synchronize", _I, [_P]),
    ("vdl_ctx_launch_count", _L, [_P]),
    ("vdl_column_alloc", _I, [_P, C.c_char_p, _I, _L, C.POINTER(C.c_int32)]),
    ("vdl_column_bind", _I, [_P, C.c_char_p, _I, _L, _L, _P, C.POINTER(C.c_int32)]),
    ("vdl_column_touch", _I, [_P, C.c_int32]),
    ("vdl_vec_generation", _I, [_P, C.c_int32, C.POINTER(C.c_uint64)]),
    ("vdl_column_upload", _I, [_P, C.c_int32, _P, _L]),
    ("vdl_column_download", _I, [_P, C.c_int32, _P, _L]),
    ("vdl_column_fill_synthetic", _I, [_P, C.c_int32, C.c_uint64, C.c_uint64, _I, _L, _L, _L, _L, _L]),
    ("vdl_column_analyze", _I, [_P, C.c_int32, C.POINTER(_L), C.POINTER(_L)]),
    ("vdl_column_lookup", _I, [_P, C.c_char_p, C.POINTER(C.c_int32)]),
    ("vdl_column_drop", _I, [_P, C.c_char_p]),
    ("vdl_vec_len", _I, [_P, C.c_int32, C.POINTER(_L)]),
    ("vdl_vec_dtype", _I, [_P, C.c_int32, C.POINTER(_I)]),
    ("vdl_vec_index_space", _I, [_P, C.c_int32, C.POINTER(_L)]),
    ("vdl_vec_device_ptr", _P, [_P, C.c_int32]),
    ("vdl_vec_download", _I, [_P, C.c_int32, _P, _L]),
    ("vdl_vec_free", _I, [_P, C.c_int32]),
    ("vdl_op_range", _I, [_P, _L, _L, _L, C.POINTER(C.c_int32)]),
    ("vdl_op_binary", _I, [_P, _I, C.c_int32, C.c_int32, C.POINTER(C.c_int32)]),
    ("vdl_op_map", _I, [_P, C.POINTER(MapDesc), C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(C.c_int32)]),
    ("vdl_abi_sizeof_map_desc", _I, []),
    ("vdl_jit_selftest", _I, [C.c_char_p, _I]),
    ("vdl_scan_jit_selftest", _I, [C.c_char_p, _I]),
    ("vdl_probe_jit_selftest", _I, [C.c_char_p, _I]),
    ("vdl_op_like", _I, [_P, C.c_int32, C.c_int32, C.c_char_p, C.POINTER(C.c_int32)]),
    ("vdl_op_cross_product", _I, [_P, C.c_int32, C.c_int32, _I, C.POINTER(C.c_int32)]),
    ("vdl_op_fold_select", _I, [_P, C.c_int32, C.POINTER(C.c_int32)]),
    ("vdl_op_gather", _I, [_P, C.c_int32, C.c_int32, C.POINTER(C.c_int32)]),
    ("vdl_op_scatter", _I, [_P, C.c_int32, C.c_int32, _L, C.POINTER(C.c_int32)]),
    ("vdl_op_partition", _I, [_P, C.c_int32, _L, _L, _L, C.POINTER(C.c_int32)]),
    ("vdl_op_fold", _I, [_P, _I, C.c_int32, C.c_int32, C.POINTER(C.c_int32)]),
    ("vdl_op_order", _I, [_P, _I, C.POINTER(C.c_int32), C.POINTER(_I), _L, C.POINTER(C.c_int32)]),
    ("vdl_op_collate", _I, [_P, C.c_int32, C.c_int32, _L, C.POINTER(C.c_int32)]),
    ("vdl_fused_prepare", _I, [_P, C.POINTER(FusedDesc), C.POINTER(_P)]),
    ("vdl_fused_launch", _I, [_P]),
    ("vdl_fused_partials", _I, [_P, C.POINTER(_P), C.POINTER(_L)]),
    ("vdl_fused_finalize", _I, [_P, _P, _I]),
    ("vdl_fused_num_groups", _I, [_P, C.POINTER(_L)]),
    ("vdl_fused_result", _I, [_P, _I, C.POINTER(C.c_int32)]),
    ("vdl_fused_launch_ex", _I, [_P, _I]),
    ("vdl_fused_result_host", _I, [_P, _I, C.POINTER(C.POINTER(_L)), C.POINTER(_L)]),
    ("vdl_fused_post_host", _I, [_P, _I, C.POINTER(C.POINTER(_L)), C.POINTER(_L)]),
    ("vdl_fused_shape_name", C.c_char_p, [_P]),
    ("vdl_fused_destroy", _I, [_P]),
    ("vdl_fused_last_kernel_ms", _I, [_P, C.POINTER(C.c_float)]),
    ("vdl_fused_kernel_ms_stats", _I, [_P, _I, C.POINTER(C.c_float), C.POINTER(C.c_float)]),
    ("vdl_probe_kernel_ms_stats", _I, [_P, _I, C.POINTER(C.c_float), C.POINTER(C.c_float)]),
    ("vdl_plan_kernel_ms_stats", _I, [_P, _I, C.POINTER(C.c_float), C.POINTER(C.c_float)]),
    ("vdl_plan_load", _I, [_P, C.c_char_p, _I, C.POINTER(_P)]),
    ("vdl_plan_stats", _I, [_P, C.POINTER(_I), C.POINTER(_I), C.POINTER(_I), C.POINTER(_L)]),
    ("vdl_plan_explain", _I, [C.c_char_p, _I, C.c_char_p, _I]),
    ("vdl_probe_exchange_bytes", _I, [_P, _I, C.POINTER(_L)]),
    ("vdl_probe_set_peers", _I, [_P, _I, _I, C.POINTER(_P)]),
    ("vdl_abi_sizeof_probe_desc", _I, []),
    ("vdl_probe_prepare", _I, [_P, C.POINTER(ProbeDesc), C.POINTER(_P)]),
    ("vdl_probe_run", _I, [_P]),
    ("vdl_probe_result_host", _I, [_P, _I, C.POINTER(C.POINTER(_L)), C.POINTER(_L)]),
    ("vdl_probe_emit_take", _I, [_P, _I, C.POINTER(C.c_int32)]),
    ("vdl_probe_last_kernel_ms", _I, [_P, C.POINTER(C.c_float)]),
    ("vdl_probe_destroy", _I, [_P]),
    ("vdl_plan_num_emits", _I, [_P]),
    ("vdl_plan_emit_group_table", _I, [_P, _I, C.POINTER(C.c_char_p)]),
    ("vdl_plan_emit", _I, [_P, _I, C.POINTER(_P), C.POINTER(_L)]),
    ("vdl_plan_emit_replace", _I, [_P, _I, _P, _L]),
    ("vdl_plan_tail_info", _I, [_P, _P, _P, _I]),
    ("vdl_plan_tail_enable", _I, [_P, _I]),
    ("vdl_plan_tail_boundary", _I, [_P, _P, _I]),
    ("vdl_plan_tail_apply", _I, [_P, _I, _P]),
    ("vdl_plan_num_partials", _I, [_P]),
    ("vdl_plan_partials", _I, [_P, _I, C.POINTER(_P), C.POINTER(_L)]),
    ("vdl_probe_run_ex", _I, [_P, _I]),
    ("vdl_probe_partials", _I, [_P, C.POINTER(_P), C.POINTER(_L)]),
    ("vdl_probe_finalize", _I, [_P, _P, _I]),
    ("vdl_plan_probe_stats", _I, [_P, C.POINTER(_I), C.POINTER(_I), C.POINTER(_I)]),
    ("vdl_plan_map_stats", _I, [_P, C.POINTER(_I), C.POINTER(_I)]),
    ("vdl_plan_probe_kernel_ms", _I, [_P, C.POINTER(C.c_float)]),
    ("vdl_plan_set_row_base", _I, [_P, _L]),
    ("vdl_plan_exchange_bytes", _I, [_P, _I, _I, C.POINTER(_L)]),
    ("vdl_plan_set_peers", _I, [_P, _I, _I, _I, C.POINTER(_P)]),
    ("vdl_fused_exchange_bytes", _I, [_P, _I, C.POINTER(_L)]),
    ("vdl_fused_set_peers", _I, [_P, _I, _I, C.POINTER(_P)]),
    ("vdl_ipc_alloc", _I, [_P, _L, C.POINTER(_P)]),
    ("vdl_ipc_export", _I, [_P, _P, C.c_char_p]),
    ("vdl_ipc_open", _I, [_P, C.c_char_p, C.POINTER(_P)]),
    ("vdl_ipc_close", _I, [_P, _P]),
    ("vdl_ipc_free", _I, [_P, _P]),
    ("vdl_plan_run_local", _I, [_P]),
    ("vdl_plan_num_fused", _I, [_P]),
    ("vdl_plan_fused", _I, [_P, _I, C.POINTER(_P)]),
    ("vdl_plan_finish", _I, [_P, C.POINTER(_P), _I]),
    ("vdl_plan_run", _I, [_P]),
    ("vdl_plan_launch", _I, [_P]),
    ("vdl_comm_init_all", _I, [_I, C.POINTER(_I), C.POINTER(_P)]),
    ("vdl_comm_size", _I, [_P]),
    ("vdl_comm_ctx", _P, [_P, _I]),
    ("vdl_comm_last_error", C.c_char_p, [_P]),
    ("vdl_comm_destroy", _I, [_P]),
    ("vdl_comm_plan_load", _I, [_P, C.c_char_p, _I, C.POINTER(_L), C.POINTER(_P)]),
    ("vdl_comm_plan_rank", _P, [_P, _I]),
    ("vdl_comm_plan_run", _I, [_P]),
    ("vdl_comm_plan_destroy", _I, [_P]),
    ("vdl_plan_num_outputs", _I, [_P]),
    ("vdl_plan_output", _I, [_P, _I, C.POINTER(C.c_char_p), C.POINTER(C.POINTER(_L)), C.POINTER(_L)]),
    ("vdl_plan_set_typed_outputs", _I, [_P, _I]),
    ("vdl_plan_output_typed", _I, [_P, _I, C.POINTER(C.c_char_p), C.POINTER(_P), C.POINTER(_L), C.POINTER(_I)]),
    ("vdl_plan_set_order", _I, [_P, _I, C.POINTER(_I), C.POINTER(_I), _L]),
    ("vdl_plan_set_order_heap", _I, [_P, _I, C.c_int32, _L]),
    ("vdl_plan_destroy", _I, [_P]),
]

_lib = None


def load():
    """dlopen libvdl_cuda.so and type every entry point.  Raises if the library is not built."""
    global _lib
    if _lib is None:
        if not os.path.exists(SO):
            raise ImportError(f"{SO} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                              "(there is no CPU fallback)")
        L = C.CDLL(SO)
        for name, res, args in SYMBOLS:
            fn = getattr(L, name)
            fn.restype, fn.argtypes = res, args
        if L.vdl_abi_sizeof_probe_desc() != C.sizeof(ProbeDesc):
            raise RuntimeError("vdl_probe_desc layout mismatch between lib.py and libvdl_cuda.so")
        if L.vdl_abi_sizeof_map_desc() != C.sizeof(MapDesc):
            raise ImportError("vdl_map_desc layout mismatch between lib.py and libvdl_cuda.so")
        if L.vdl_abi_sizeof_fused_desc() != C.sizeof(FusedDesc):
            raise ImportError("vdl_fused_desc layout mismatch between lib.py and libvdl_cuda.so")
        _lib = L
    return _lib
