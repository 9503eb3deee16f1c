{-# LANGUAGE ForeignFunctionInterface #-}
-- | Raw FFI bindings to libvdl_cuda (include/vdl_cuda.h), the B200 executor for the Voodoo programs mplan2vdl
-- emits.  SOURCE ONLY: this image has no GHC, so this module has never been compiled; it mirrors, call for call,
-- the ctypes binding in mplan2vdl_b200/lib.py that IS exercised by the test-suite.
--
-- Every import is `safe`: the calls block (kernel launches + stream synchronisation) and must not stall the
-- Haskell runtime's capability.  Handles: VdlCtx / VdlPlan / VdlFused are opaque pointers; vectors are Int32
-- handles owned by the context.
module VdlCuda where

import Data.Int (Int32, Int64)
import Data.Word (Word64)
import Foreign.C.String (CString)
import Foreign.C.Types (CFloat (..), CInt (..))
import Foreign.Ptr (Ptr)

data VdlCtx
data VdlPlan
data VdlFused
data VdlProbe
data VdlComm      -- vdl_comm: one context per GPU of the box, peer access enabled (single-process multi-GPU)
data VdlCommPlan  -- vdl_comm_plan: one loaded program per rank, exchange buffers wired
data VdlFusedDesc  -- vdl_fused_desc / vdl_probe_desc: marshalled with Foreign.Storable by the caller (layouts in vdl_cuda.h)
data VdlProbeDesc
data VdlMapDesc   -- vdl_map_desc: marshalled with Foreign.Storable by the caller (layout in vdl_cuda.h)
type VdlVec = Int32

-- status codes (vdl_cuda.h)
vdlOk, vdlEInval, vdlECuda, vdlENotFound, vdlEUnsupported, vdlERange, vdlENoMem, vdlEStale :: CInt
vdlOk = 0; vdlEInval = 1; vdlECuda = 2; vdlENotFound = 3; vdlEUnsupported = 4; vdlERange = 5; vdlENoMem = 6; vdlEStale = 7

-- storage types: Types.hs sizeOf SInt32 = 4, SInt64 / SDecimal = 8
vdlI32, vdlI64 :: CInt
vdlI32 = 4; vdlI64 = 8

foreign import ccall safe "vdl_abi_version" c_vdl_abi_version :: IO CInt
foreign import ccall safe "vdl_ctx_create" c_vdl_ctx_create :: CInt -> Ptr (Ptr VdlCtx) -> IO CInt
foreign import ccall safe "vdl_ctx_destroy" c_vdl_ctx_destroy :: Ptr VdlCtx -> IO CInt
foreign import ccall safe "vdl_last_error" c_vdl_last_error :: Ptr VdlCtx -> IO CString

-- columns: what `Load n` (Vlite.hs Vx) binds
foreign import ccall safe "vdl_column_alloc" c_vdl_column_alloc :: Ptr VdlCtx -> CString -> CInt -> Int64 -> Ptr VdlVec -> IO CInt
foreign import ccall safe "vdl_column_touch" c_vdl_column_touch :: Ptr VdlCtx -> VdlVec -> IO CInt
foreign import ccall safe "vdl_vec_generation" c_vdl_vec_generation :: Ptr VdlCtx -> VdlVec -> Ptr Word64 -> IO CInt
foreign import ccall safe "vdl_column_upload" c_vdl_column_upload :: Ptr VdlCtx -> VdlVec -> Ptr () -> Int64 -> IO CInt
foreign import ccall safe "vdl_column_fill_synthetic" c_vdl_column_fill_synthetic
  :: Ptr VdlCtx -> VdlVec -> Word64 -> Word64 -> CInt -> Int64 -> Int64 -> Int64 -> Int64 -> Int64 -> IO CInt
foreign import ccall safe "vdl_column_lookup" c_vdl_column_lookup :: Ptr VdlCtx -> CString -> Ptr VdlVec -> IO CInt
foreign import ccall safe "vdl_vec_index_space" c_vdl_vec_index_space :: Ptr VdlCtx -> VdlVec -> Ptr Int64 -> IO CInt
foreign import ccall safe "vdl_vec_len" c_vdl_vec_len :: Ptr VdlCtx -> VdlVec -> Ptr Int64 -> IO CInt
foreign import ccall safe "vdl_vec_download" c_vdl_vec_download :: Ptr VdlCtx -> VdlVec -> Ptr Int64 -> Int64 -> IO CInt
foreign import ccall safe "vdl_vec_free" c_vdl_vec_free :: Ptr VdlCtx -> VdlVec -> IO CInt

-- one entry point per Vx constructor (Vlite.hs:102-116)
foreign import ccall safe "vdl_op_range" c_vdl_op_range :: Ptr VdlCtx -> Int64 -> Int64 -> Int64 -> Ptr VdlVec -> IO CInt
foreign import ccall safe "vdl_op_binary" c_vdl_op_binary :: Ptr VdlCtx -> CInt -> VdlVec -> VdlVec -> Ptr VdlVec -> IO CInt
foreign import ccall safe "vdl_op_like" c_vdl_op_like :: Ptr VdlCtx -> VdlVec -> VdlVec -> CString -> Ptr VdlVec -> IO CInt
foreign import ccall safe "vdl_op_cross_product" c_vdl_op_cross_product :: Ptr VdlCtx -> VdlVec -> VdlVec -> CInt -> Ptr VdlVec -> IO CInt
foreign import ccall safe "vdl_op_fold_select" c_vdl_op_fold_select :: Ptr VdlCtx -> VdlVec -> Ptr VdlVec -> IO CInt
foreign import ccall safe "vdl_op_map" c_vdl_op_map :: Ptr VdlCtx -> Ptr VdlMapDesc -> Ptr VdlVec -> Ptr VdlVec -> Ptr VdlVec -> IO CInt
foreign import ccall safe "vdl_jit_selftest" c_vdl_jit_selftest :: CString -> CInt -> IO CInt
foreign import ccall safe "vdl_probe_jit_selftest" c_vdl_probe_jit_selftest :: CString -> CInt -> IO CInt
foreign import ccall safe "vdl_scan_jit_selftest" c_vdl_scan_jit_selftest :: CString -> CInt -> IO CInt
foreign import ccall unsafe "vdl_abi_sizeof_map_desc" c_vdl_abi_sizeof_map_desc :: IO CInt
foreign import ccall safe "vdl_op_gather" c_vdl_op_gather :: Ptr VdlCtx -> VdlVec -> VdlVec -> Ptr VdlVec -> IO CInt
foreign import ccall safe "vdl_op_scatter" c_vdl_op_scatter :: Ptr VdlCtx -> VdlVec -> VdlVec -> Int64 -> Ptr VdlVec -> IO CInt
foreign import ccall safe "vdl_op_partition" c_vdl_op_partition :: Ptr VdlCtx -> VdlVec -> Int64 -> Int64 -> Int64 -> Ptr VdlVec -> IO CInt
foreign import ccall safe "vdl_op_fold" c_vdl_op_fold :: Ptr VdlCtx -> CInt -> VdlVec -> VdlVec -> Ptr VdlVec -> IO CInt
foreign import ccall safe "vdl_op_order" c_vdl_op_order :: Ptr VdlCtx -> CInt -> Ptr VdlVec -> Ptr CInt -> Int64 -> Ptr VdlVec -> IO CInt
foreign import ccall safe "vdl_op_collate" c_vdl_op_collate :: Ptr VdlCtx -> VdlVec -> VdlVec -> Int64 -> Ptr VdlVec -> IO CInt

-- whole programs: the text Vdl.vdlFromVexps prints
foreign import ccall safe "vdl_plan_load" c_vdl_plan_load :: Ptr VdlCtx -> CString -> CInt -> Ptr (Ptr VdlPlan) -> IO CInt
foreign import ccall safe "vdl_plan_set_row_base" c_vdl_plan_set_row_base :: Ptr VdlPlan -> Int64 -> IO CInt
foreign import ccall safe "vdl_plan_run" c_vdl_plan_run :: Ptr VdlPlan -> IO CInt
foreign import ccall safe "vdl_plan_run_local" c_vdl_plan_run_local :: Ptr VdlPlan -> IO CInt
foreign import ccall safe "vdl_plan_finish" c_vdl_plan_finish :: Ptr VdlPlan -> Ptr (Ptr ()) -> CInt -> IO CInt
foreign import ccall safe "vdl_plan_num_outputs" c_vdl_plan_num_outputs :: Ptr VdlPlan -> IO CInt
foreign import ccall safe "vdl_plan_output" c_vdl_plan_output :: Ptr VdlPlan -> CInt -> Ptr CString -> Ptr (Ptr Int64) -> Ptr Int64 -> IO CInt
foreign import ccall safe "vdl_plan_set_typed_outputs" c_vdl_plan_set_typed_outputs :: Ptr VdlPlan -> CInt -> IO CInt
foreign import ccall safe "vdl_plan_output_typed" c_vdl_plan_output_typed :: Ptr VdlPlan -> CInt -> Ptr CString -> Ptr (Ptr ()) -> Ptr Int64 -> Ptr CInt -> IO CInt
foreign import ccall safe "vdl_plan_set_order" c_vdl_plan_set_order :: Ptr VdlPlan -> CInt -> Ptr CInt -> Ptr CInt -> Int64 -> IO CInt
foreign import ccall safe "vdl_plan_set_order_heap" c_vdl_plan_set_order_heap :: Ptr VdlPlan -> CInt -> VdlVec -> Int64 -> IO CInt
foreign import ccall safe "vdl_plan_destroy" c_vdl_plan_destroy :: Ptr VdlPlan -> IO CInt

-- multi-GPU combine over peer memory (vdl_cuda.h "multi-GPU combine over peer memory"): after vdl_plan_set_peers,
-- vdl_plan_run returns the GLOBAL result on every rank with one kernel launch per GPU and no collective library
foreign import ccall safe "vdl_plan_exchange_bytes" c_vdl_plan_exchange_bytes :: Ptr VdlPlan -> CInt -> CInt -> Ptr Int64 -> IO CInt
foreign import ccall safe "vdl_plan_set_peers" c_vdl_plan_set_peers :: Ptr VdlPlan -> CInt -> CInt -> CInt -> Ptr (Ptr ()) -> IO CInt
foreign import ccall safe "vdl_ipc_alloc" c_vdl_ipc_alloc :: Ptr VdlCtx -> Int64 -> Ptr (Ptr ()) -> IO CInt
foreign import ccall safe "vdl_ipc_export" c_vdl_ipc_export :: Ptr VdlCtx -> Ptr () -> CString -> IO CInt      -- 64-byte handle
foreign import ccall safe "vdl_ipc_open" c_vdl_ipc_open :: Ptr VdlCtx -> CString -> Ptr (Ptr ()) -> IO CInt
foreign import ccall safe "vdl_ipc_close" c_vdl_ipc_close :: Ptr VdlCtx -> Ptr () -> IO CInt
foreign import ccall safe "vdl_ipc_free" c_vdl_ipc_free :: Ptr VdlCtx -> Ptr () -> IO CInt

-- what the fusion passes did with a loaded program (Folds on the fused scan; FK-join Folds / vectors on the probe kernel)
foreign import ccall safe "vdl_plan_stats" c_vdl_plan_stats :: Ptr VdlPlan -> Ptr CInt -> Ptr CInt -> Ptr CInt -> Ptr Int64 -> IO CInt
foreign import ccall safe "vdl_plan_explain" c_vdl_plan_explain :: CString -> CInt -> CString -> CInt -> IO CInt
foreign import ccall safe "vdl_probe_exchange_bytes" c_vdl_probe_exchange_bytes :: Ptr VdlProbe -> CInt -> Ptr Int64 -> IO CInt
foreign import ccall safe "vdl_probe_set_peers" c_vdl_probe_set_peers :: Ptr VdlProbe -> CInt -> CInt -> Ptr (Ptr ()) -> IO CInt
foreign import ccall safe "vdl_plan_map_stats" c_vdl_plan_map_stats :: Ptr VdlPlan -> Ptr CInt -> Ptr CInt -> IO CInt
foreign import ccall safe "vdl_plan_probe_stats" c_vdl_plan_probe_stats :: Ptr VdlPlan -> Ptr CInt -> Ptr CInt -> Ptr CInt -> IO CInt

-- sharded runs of FK-join plans: partial tables of every fused scan / probe fold group, and the vectors probe passes emit
foreign import ccall safe "vdl_plan_num_partials" c_vdl_plan_num_partials :: Ptr VdlPlan -> IO CInt
foreign import ccall safe "vdl_plan_partials" c_vdl_plan_partials :: Ptr VdlPlan -> CInt -> Ptr (Ptr ()) -> Ptr Int64 -> IO CInt
foreign import ccall safe "vdl_plan_num_emits" c_vdl_plan_num_emits :: Ptr VdlPlan -> IO CInt
foreign import ccall safe "vdl_plan_emit_group_table" c_vdl_plan_emit_group_table :: Ptr VdlPlan -> CInt -> Ptr CString -> IO CInt
foreign import ccall safe "vdl_plan_emit" c_vdl_plan_emit :: Ptr VdlPlan -> CInt -> Ptr (Ptr ()) -> Ptr Int64 -> IO CInt
foreign import ccall safe "vdl_plan_emit_replace" c_vdl_plan_emit_replace :: Ptr VdlPlan -> CInt -> Ptr () -> Int64 -> IO CInt
foreign import ccall safe "vdl_plan_tail_info" c_vdl_plan_tail_info :: Ptr VdlPlan -> Ptr CInt -> Ptr CInt -> CInt -> IO CInt
foreign import ccall safe "vdl_plan_tail_enable" c_vdl_plan_tail_enable :: Ptr VdlPlan -> CInt -> IO CInt
foreign import ccall safe "vdl_plan_tail_boundary" c_vdl_plan_tail_boundary :: Ptr VdlPlan -> Ptr Int64 -> CInt -> IO CInt
foreign import ccall safe "vdl_plan_tail_apply" c_vdl_plan_tail_apply :: Ptr VdlPlan -> CInt -> Ptr Int64 -> IO CInt

-- fused scan / FK-join probe / remaining context, column and plan entry points (tools/gen_hs_imports.py keeps this list
-- in step with include/vdl_cuda.h; tests/test_abi.py checks that every declaration has an import)
foreign import ccall safe "vdl_abi_sizeof_fused_desc" c_vdl_abi_sizeof_fused_desc :: IO CInt
foreign import ccall safe "vdl_ctx_stream" c_vdl_ctx_stream :: Ptr VdlCtx -> IO (Ptr ())
foreign import ccall safe "vdl_ctx_synchronize" c_vdl_ctx_synchronize :: Ptr VdlCtx -> IO CInt
foreign import ccall safe "vdl_ctx_launch_count" c_vdl_ctx_launch_count :: Ptr VdlCtx -> IO Int64
foreign import ccall safe "vdl_column_bind" c_vdl_column_bind :: Ptr VdlCtx -> CString -> CInt -> Int64 -> Int64 -> Ptr () -> Ptr VdlVec -> IO CInt
foreign import ccall safe "vdl_column_download" c_vdl_column_download :: Ptr VdlCtx -> VdlVec -> Ptr () -> Int64 -> IO CInt
foreign import ccall safe "vdl_column_analyze" c_vdl_column_analyze :: Ptr VdlCtx -> VdlVec -> Ptr Int64 -> Ptr Int64 -> IO CInt
foreign import ccall safe "vdl_column_drop" c_vdl_column_drop :: Ptr VdlCtx -> CString -> IO CInt
foreign import ccall safe "vdl_vec_dtype" c_vdl_vec_dtype :: Ptr VdlCtx -> VdlVec -> Ptr CInt -> IO CInt
foreign import ccall safe "vdl_vec_device_ptr" c_vdl_vec_device_ptr :: Ptr VdlCtx -> VdlVec -> IO (Ptr ())
foreign import ccall safe "vdl_fused_prepare" c_vdl_fused_prepare :: Ptr VdlCtx -> Ptr VdlFusedDesc -> Ptr (Ptr VdlFused) -> IO CInt
foreign import ccall safe "vdl_fused_launch" c_vdl_fused_launch :: Ptr VdlFused -> IO CInt
foreign import ccall safe "vdl_fused_launch_ex" c_vdl_fused_launch_ex :: Ptr VdlFused -> CInt -> IO CInt
foreign import ccall safe "vdl_fused_partials" c_vdl_fused_partials :: Ptr VdlFused -> Ptr (Ptr ()) -> Ptr Int64 -> IO CInt
foreign import ccall safe "vdl_fused_finalize" c_vdl_fused_finalize :: Ptr VdlFused -> Ptr () -> CInt -> IO CInt
foreign import ccall safe "vdl_fused_num_groups" c_vdl_fused_num_groups :: Ptr VdlFused -> Ptr Int64 -> IO CInt
foreign import ccall safe "vdl_fused_result" c_vdl_fused_result :: Ptr VdlFused -> CInt -> Ptr VdlVec -> IO CInt
foreign import ccall safe "vdl_fused_result_host" c_vdl_fused_result_host :: Ptr VdlFused -> CInt -> Ptr (Ptr Int64) -> Ptr Int64 -> IO CInt
foreign import ccall safe "vdl_fused_post_host" c_vdl_fused_post_host :: Ptr VdlFused -> CInt -> Ptr (Ptr Int64) -> Ptr Int64 -> IO CInt
foreign import ccall safe "vdl_fused_shape_name" c_vdl_fused_shape_name :: Ptr VdlFused -> IO CString
foreign import ccall safe "vdl_fused_destroy" c_vdl_fused_destroy :: Ptr VdlFused -> IO CInt
foreign import ccall safe "vdl_fused_exchange_bytes" c_vdl_fused_exchange_bytes :: Ptr VdlFused -> CInt -> Ptr Int64 -> IO CInt
foreign import ccall safe "vdl_fused_set_peers" c_vdl_fused_set_peers :: Ptr VdlFused -> CInt -> CInt -> Ptr (Ptr ()) -> IO CInt
foreign import ccall safe "vdl_fused_last_kernel_ms" c_vdl_fused_last_kernel_ms :: Ptr VdlFused -> Ptr CFloat -> IO CInt
foreign import ccall safe "vdl_abi_sizeof_probe_desc" c_vdl_abi_sizeof_probe_desc :: IO CInt
foreign import ccall safe "vdl_probe_prepare" c_vdl_probe_prepare :: Ptr VdlCtx -> Ptr VdlProbeDesc -> Ptr (Ptr VdlProbe) -> IO CInt
foreign import ccall safe "vdl_probe_run" c_vdl_probe_run :: Ptr VdlProbe -> IO CInt
foreign import ccall safe "vdl_probe_run_ex" c_vdl_probe_run_ex :: Ptr VdlProbe -> CInt -> IO CInt
foreign import ccall safe "vdl_probe_partials" c_vdl_probe_partials :: Ptr VdlProbe -> Ptr (Ptr ()) -> Ptr Int64 -> IO CInt
foreign import ccall safe "vdl_probe_finalize" c_vdl_probe_finalize :: Ptr VdlProbe -> Ptr () -> CInt -> IO CInt
foreign import ccall safe "vdl_probe_result_host" c_vdl_probe_result_host :: Ptr VdlProbe -> CInt -> Ptr (Ptr Int64) -> Ptr Int64 -> IO CInt
foreign import ccall safe "vdl_probe_emit_take" c_vdl_probe_emit_take :: Ptr VdlProbe -> CInt -> Ptr VdlVec -> IO CInt
foreign import ccall safe "vdl_probe_last_kernel_ms" c_vdl_probe_last_kernel_ms :: Ptr VdlProbe -> Ptr CFloat -> IO CInt
foreign import ccall safe "vdl_probe_destroy" c_vdl_probe_destroy :: Ptr VdlProbe -> IO CInt
foreign import ccall safe "vdl_plan_probe_kernel_ms" c_vdl_plan_probe_kernel_ms :: Ptr VdlPlan -> Ptr CFloat -> IO CInt
foreign import ccall safe "vdl_plan_num_fused" c_vdl_plan_num_fused :: Ptr VdlPlan -> IO CInt
foreign import ccall safe "vdl_plan_fused" c_vdl_plan_fused :: Ptr VdlPlan -> CInt -> Ptr (Ptr VdlFused) -> IO CInt

-- several GPUs driven from this one process (SURVEY.md section 8 b/e): the partial tables are exchanged inside the scan kernels
foreign import ccall safe "vdl_plan_launch" c_vdl_plan_launch :: Ptr VdlPlan -> IO CInt
foreign import ccall safe "vdl_comm_init_all" c_vdl_comm_init_all :: CInt -> Ptr CInt -> Ptr (Ptr VdlComm) -> IO CInt
foreign import ccall safe "vdl_comm_size" c_vdl_comm_size :: Ptr VdlComm -> IO CInt
foreign import ccall safe "vdl_comm_ctx" c_vdl_comm_ctx :: Ptr VdlComm -> CInt -> IO (Ptr VdlCtx)
foreign import ccall safe "vdl_comm_last_error" c_vdl_comm_last_error :: Ptr VdlComm -> IO CString
foreign import ccall safe "vdl_comm_destroy" c_vdl_comm_destroy :: Ptr VdlComm -> IO CInt
foreign import ccall safe "vdl_comm_plan_load" c_vdl_comm_plan_load :: Ptr VdlComm -> CString -> CInt -> Ptr Int64 -> Ptr (Ptr VdlCommPlan) -> IO CInt
foreign import ccall safe "vdl_comm_plan_rank" c_vdl_comm_plan_rank :: Ptr VdlCommPlan -> CInt -> IO (Ptr VdlPlan)
foreign import ccall safe "vdl_comm_plan_run" c_vdl_comm_plan_run :: Ptr VdlCommPlan -> IO CInt
foreign import ccall safe "vdl_comm_plan_destroy" c_vdl_comm_plan_destroy :: Ptr VdlCommPlan -> IO CInt
foreign import ccall safe "vdl_fused_kernel_ms_stats" c_vdl_fused_kernel_ms_stats :: Ptr VdlFused -> CInt -> Ptr CFloat -> Ptr CFloat -> IO CInt
foreign import ccall safe "vdl_probe_kernel_ms_stats" c_vdl_probe_kernel_ms_stats :: Ptr VdlProbe -> CInt -> Ptr CFloat -> Ptr CFloat -> IO CInt
foreign import ccall safe "vdl_plan_kernel_ms_stats" c_vdl_plan_kernel_ms_stats :: Ptr VdlPlan -> CInt -> Ptr CFloat -> Ptr CFloat -> IO CInt
