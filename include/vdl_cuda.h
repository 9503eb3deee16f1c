/*
 * vdl_cuda.h -- C ABI of libvdl_cuda, the B200 (sm_100a) executor for the Voodoo dataflow
 * graphs that orm011/mplan2vdl emits.
 *
 * What this boundary replaces.  mplan2vdl prints the Voodoo program to stdout
 * (MainFuns.hs:155-157) and an external Voodoo server, which is not in the reference
 * repository, received it over HTTP and answered with JSON (eval_query.sh:18-26,
 * resolve.py:8-32).  libvdl_cuda is that missing executor as an in-process library:
 *   - vdl_plan_load() takes exactly the text `Vdl.vdlFromVexps` produces
 *     (Vdl.hs:410-453 toVoodooList, 455-477 printLine, 490-495), so the existing
 *     stdout/wire format is a valid input unchanged;
 *   - the per-op entry points (vdl_op_*) are one call per constructor of the
 *     emitter's op set `Vd`/`Voodop` (Vdl.hs:32-44, 110-131) -- what a Haskell
 *     `Exec` module walking `[Vexp]` after MainFuns.hs:186 binds with
 *     `foreign import ccall safe` (see INTEGRATION.md and hs/VdlCuda.hs);
 *   - vdl_fused_scan_fold() is the single-launch select->map->fold kernel that the
 *     fusion peephole (same `Vx -> Maybe Vexp` shape as Vlite.hs:1295-1340) targets.
 *
 * Conventions: every call returns 0 on success and a VDL_E* code otherwise and never
 * throws or aborts across the ABI; vdl_last_error(ctx) gives the message.  Device buffers
 * are owned by the library and referenced by opaque handles.  Calls on one context are
 * serialised by the caller; different contexts (GPUs) may be driven from different host
 * threads.  All calls may block: bind them as `safe` FFI calls.  Plain pointers and sizes
 * only -- no torch or C++ types.
 */
#ifndef VDL_CUDA_H
#define VDL_CUDA_H

#ifndef __CUDACC_RTC__     /* (the library compiles some kernels at run time with NVRTC, which has no system headers) */
#include <stdint.h>
#endif

#ifdef __cplusplus
extern "C" {
#endif

#define VDL_ABI_VERSION 1

/* status codes */
enum {
  VDL_OK = 0,
  VDL_EINVAL = 1,      /* bad argument / malformed plan text */
  VDL_ECUDA = 2,       /* CUDA runtime error (message has the cudaError string) */
  VDL_ENOTFOUND = 3,   /* Load of a column that is not registered */
  VDL_EUNSUPPORTED = 4,/* op or plan shape outside what is supported (Semisort; a cross product beyond 2^33 pairs) */
  VDL_ERANGE = 5,      /* Gather/Scatter position out of range */
  VDL_ENOMEM = 6,
  VDL_ESTALE = 7       /* a prepared scan / probe was launched after one of its columns was rewritten or dropped */
};

/* storage types (reference Types.hs:66-89: SInt32 4 B; SInt64/SDecimal 8 B); VDL_U8: the bytes of a string heap,
 * `Load,<table>.<col>.heap` (Vdl.hs:244-247) -- such a vector can only be the dictionary argument of vdl_op_like or
 * vdl_op_collate */
enum { VDL_U8 = 1, VDL_I32 = 4, VDL_I64 = 8 };

/* binary elementwise ops, in the order of `Voodop` (Vdl.hs:110-123) */
enum {
  VDL_LOGICAL_AND = 0, VDL_LOGICAL_OR, VDL_BITWISE_AND, VDL_BITWISE_OR, VDL_BITSHIFT, VDL_EQUALS,
  VDL_ADD, VDL_SUBTRACT, VDL_GREATER, VDL_MULTIPLY, VDL_DIVIDE, VDL_MODULO
};
/* folds (Vdl.hs:124-129; FoldSelect has its own entry point) */
enum { VDL_FOLD_SUM = 0, VDL_FOLD_MIN = 1, VDL_FOLD_MAX = 2, VDL_FOLD_CHOOSE = 3, VDL_FOLD_COUNT = 4 };

/* synthetic column kinds (mplan2vdl_b200/synth.py; SURVEY.md Appendix D) */
enum { VDL_SYNTH_UNIFORM = 0, VDL_SYNTH_SEQ = 1, VDL_SYNTH_FKDENSE = 2 };

typedef struct vdl_ctx vdl_ctx;     /* one per device */
typedef struct vdl_plan vdl_plan;   /* a loaded Voodoo program */
typedef int32_t vdl_vec;            /* handle of a device vector (>0); columns are vectors too */

/* ---- context ---------------------------------------------------------------------- */
int vdl_abi_version(void);
/* sizeof(vdl_fused_desc) as this library was compiled, so FFI bindings can check their layout. */
int vdl_abi_sizeof_fused_desc(void);
int vdl_ctx_create(int device, vdl_ctx **out);
int vdl_ctx_destroy(vdl_ctx *ctx);
const char *vdl_last_error(vdl_ctx *ctx);
/* The CUDA stream every kernel of this context is launched on (a cudaStream_t), so callers
 * can time with events on the launching stream or order their own work after it. */
void *vdl_ctx_stream(vdl_ctx *ctx);
int vdl_ctx_synchronize(vdl_ctx *ctx);
/* Kernels launched by this context since creation (bench.py's gpu_launches). */
int64_t vdl_ctx_launch_count(vdl_ctx *ctx);

/* ---- columns: what `Load,<table>.<col>` binds (Vdl.hs:161-168, 419-420) --------------- */
/* Allocate a named column of `rows` values of `dtype` in HBM (padded for 16-byte bulk copies). */
int vdl_column_alloc(vdl_ctx *ctx, const char *name, int dtype, int64_t rows, vdl_vec *out);
/* Register caller-owned device memory (e.g. a torch tensor) as a named column; the memory must
 * stay valid while registered and be 16-byte aligned; after writing to it call vdl_column_touch (the library
 * caches column statistics and bakes proofs derived from them into prepared scans).  capacity_rows >= rows is
 * how many rows may be read past the logical end (bulk copies round the tail up to 16 bytes). */
int vdl_column_bind(vdl_ctx *ctx, const char *name, int dtype, int64_t rows, int64_t capacity_rows,
                    void *device_ptr, vdl_vec *out);
/* The caller wrote to the column's memory behind the library's back: renew its write generation (below). */
int vdl_column_touch(vdl_ctx *ctx, vdl_vec col);
/* Write generation of a vector: unique within the context, renewed by creation, vdl_column_upload,
 * vdl_column_fill_synthetic and vdl_column_touch.  Prepared scans / probes record (handle, generation) of their
 * columns -- the role bounds.csv plays for the reference's inferBounds (Vlite.hs:417-467) is played by statistics of
 * the data itself, so the proofs must follow the data: a plan re-analyses and re-prepares when a pair changed, and a
 * direct vdl_fused_launch / vdl_probe_run on a stale object fails with VDL_ESTALE instead of computing with old proofs. */
int vdl_vec_generation(vdl_ctx *ctx, vdl_vec v, uint64_t *generation);
/* Host -> device copy of a whole column (pageable or pinned host memory). */
int vdl_column_upload(vdl_ctx *ctx, vdl_vec col, const void *host, int64_t rows);
/* Device -> host copy of a whole column in its stored type (the inverse of vdl_column_upload). */
int vdl_column_download(vdl_ctx *ctx, vdl_vec col, void *host, int64_t rows);
/* Fill rows [0, rows) of `col` with the counter-based synthetic recipe for global rows
 * [row_offset, row_offset+rows): a shard generates its own row range in place. */
int vdl_column_fill_synthetic(vdl_ctx *ctx, vdl_vec col, uint64_t seed, uint64_t stream, int kind,
                              int64_t vmin, int64_t stride, int64_t p0, int64_t p1, int64_t row_offset);
/* Exact minimum / maximum of a column, computed on the device once and cached until the column is written
 * again -- the executor's own copy of what the reference reads from bounds.csv (Config.hs:57).  The fused scan
 * uses it to compare 8-byte predicate columns in 32 bits when every value fits. */
int vdl_column_analyze(vdl_ctx *ctx, vdl_vec col, int64_t *vmin, int64_t *vmax);
int vdl_column_lookup(vdl_ctx *ctx, const char *name, vdl_vec *out);
int vdl_column_drop(vdl_ctx *ctx, const char *name);

/* ---- vectors ----------------------------------------------------------------------- */
int vdl_vec_len(vdl_ctx *ctx, vdl_vec v, int64_t *len);
int vdl_vec_dtype(vdl_ctx *ctx, vdl_vec v, int *dtype);
/* The length of the vector the values of `v` index into, when the library knows it (App. G2): positions from FoldSelect /
 * pos_ / Partition index their input's row space, a Gather or a Scatter keeps the space of its source's values, `p % k`
 * (the scatter size hint, Vlite.hs:1117-1120) indexes k slots; -1 when unknown.  This is the explicit output length a
 * caller passes to vdl_op_scatter (the reference's metadata `count = posmax`, Vlite.hs:316-320, is not usable for that). */
int vdl_vec_index_space(vdl_ctx *ctx, vdl_vec v, int64_t *len);
void *vdl_vec_device_ptr(vdl_ctx *ctx, vdl_vec v);
/* Device -> host copy of v as int64 (int32 columns are sign-extended); `capacity` in elements. */
int vdl_vec_download(vdl_ctx *ctx, vdl_vec v, int64_t *host, int64_t capacity);
int vdl_vec_free(vdl_ctx *ctx, vdl_vec v);

/* ---- per-op entry points: one per Voodoo op, explicit lengths (SURVEY.md section 2.3) -- */
/* RangeV / RangeC (Vdl.hs:428-434): out[i] = from + i*step, i < len. */
int vdl_op_range(vdl_ctx *ctx, int64_t from, int64_t step, int64_t len, vdl_vec *out);
/* Elementwise binary op (Vdl.hs:436-439); a and b have equal length. */
int vdl_op_binary(vdl_ctx *ctx, int op, vdl_vec a, vdl_vec b, vdl_vec *out);
/* A tree of elementwise ops, Gathers and Ranges over vectors of ONE length in one launch: what the same chain of
 * vdl_op_binary / vdl_op_gather / vdl_op_range calls computes, without materialising the intermediates (the plan
 * executor groups the op-at-a-time remainder of a plan this way).  A register program is run per row i:
 *   VDL_LOGICAL_AND..VDL_MODULO   reg[dst] = op(reg[a], reg[b])
 *   VDL_MAP_LOAD                  reg[dst] = inputs[b][i]
 *   VDL_MAP_RANGE                 reg[dst] = imm[a] + i * imm[b]
 *   VDL_MAP_GATHER                reg[dst] = tables[b][reg[a]]   (out of range: 0 and the context's error flag, like vdl_op_gather)
 * All inputs have the result's length (an input no instruction loads is only a length witness); tables have any
 * length.  The result is the register written by the last instruction. */
#define VDL_MAP_MAX_INPUTS 48
#define VDL_MAP_MAX_TABLES 8
#define VDL_MAP_MAX_INSTRS 160
#define VDL_MAP_MAX_IMMS 32
#define VDL_MAP_MAX_REGS 32
#define VDL_MAP_GATHER 16
#define VDL_MAP_LOAD 17
#define VDL_MAP_RANGE 18
typedef struct vdl_map_instr { int16_t op, dst, a, b; } vdl_map_instr;
typedef struct vdl_map_desc {
  int32_t ninputs, ntables, ninstrs, nimms;
  vdl_map_instr instr[VDL_MAP_MAX_INSTRS];
  int64_t imm[VDL_MAP_MAX_IMMS];
} vdl_map_desc;
int vdl_op_map(vdl_ctx *ctx, const vdl_map_desc *desc, const vdl_vec *inputs, const vdl_vec *tables, vdl_vec *out);
int vdl_abi_sizeof_map_desc(void);
/* Host-only check of the run-time specialisation of vdl_op_map (no GPU needed): generates the CUDA C of a program that
 * uses every instruction, compiles it with NVRTC for sm_100a.  VDL_OK, VDL_ENOTFOUND (no NVRTC here: the interpreting
 * kernel is used) or VDL_ECUDA with NVRTC's log. */
int vdl_jit_selftest(char *log, int log_capacity);
/* Like (Vlite.hs:1010-1014 -> Vdl.hs:244-247, 444-447): out[i] = 1 if the NUL-terminated string at byte offset data[i] of
 * the string heap matches the SQL LIKE pattern (`%` any run of bytes, `_` any one byte, no escape character,
 * case-sensitive), else 0.  An offset outside the heap raises the context's range error (VDL_ERANGE at the next check). */
#define VDL_LIKE_MAX_PATTERN 128
int vdl_op_like(vdl_ctx *ctx, vdl_vec data, vdl_vec heap, const char *pattern, vdl_vec *out);
/* CrossProductOuter (inner = 0) / CrossProductInner (inner = 1): Vlite.hs:89-93 `crossp`, 283-292; printed by Vdl.hs:412-416;
 * joins under --use_cross_product (Mplan.hs:309-313).  The positions into `left` resp. `right` of the |left| x |right|
 * pairs, left-major: out[i] = i / |right| resp. i % |right|.  Only the lengths of the arguments matter.  Quadratic by
 * definition: refused above 2^33 pairs. */
int vdl_op_cross_product(vdl_ctx *ctx, vdl_vec left, vdl_vec right, int inner, vdl_vec *out);
/* FoldSelect with fold = pos_ pred (Vlite.hs:721-730): ascending positions of non-zero pred. */
int vdl_op_fold_select(vdl_ctx *ctx, vdl_vec pred, vdl_vec *out);
/* Gather (Vdl.hs:438): out[i] = src[pos[i]]. */
int vdl_op_gather(vdl_ctx *ctx, vdl_vec src, vdl_vec pos, vdl_vec *out);
/* Scatter (Vdl.hs:441-442): out[pos[i]] = src[i], unwritten = 0; out_len explicit (App. G2). */
int vdl_op_scatter(vdl_ctx *ctx, vdl_vec src, vdl_vec pos, int64_t out_len, vdl_vec *out);
/* Partition (Vdl.hs:266-269) with pivots RangeC(pivot_from, pivot_count, pivot_step): destination
 * positions of the stable sort of rows by bucket(data) = number of pivots below data[i]. */
int vdl_op_partition(vdl_ctx *ctx, vdl_vec data, int64_t pivot_from, int64_t pivot_step,
                     int64_t pivot_count, vdl_vec *out);
/* FoldSum/Min/Max/Choose/Count (Vdl.hs:255-264): one output per run of equal consecutive groups. */
int vdl_op_fold(vdl_ctx *ctx, int fold_op, vdl_vec groups, vdl_vec data, vdl_vec *out);
/* ORDER BY / LIMIT, which the emitter cannot express: positions 0..n-1 of the nkeys key vectors (equal length n) ordered
 * lexicographically over the keys compared as signed int64 (int32 sign-extended, ranges read as their values), key i
 * descending when descending[i] != 0 (descending may be NULL: all ascending); ties keep row order (stable).  out has
 * min(limit, n) entries (limit < 0: n); gathering any vector of length n by it gives its rows in that order.  nkeys = 0:
 * positions 0..limit-1 (limit >= 0; the caller knows n).  Keys of unequal length: VDL_EINVAL. */
#define VDL_MAX_ORDER_KEYS 8
int vdl_op_order(vdl_ctx *ctx, int nkeys, const vdl_vec *keys, const int *descending, int64_t limit, vdl_vec *out);
/* Collation rank of every row's string: the string of row i starts at heap[data[i] - origin] and ends at its NUL.
 * out[i] (int64) = number of distinct strings in `data` that sort before it.  Strings compare byte by byte as unsigned
 * char, and a proper prefix sorts first (C strcmp, MonetDB's byte order for UTF-8).  Equal strings at different offsets
 * get one rank.  An offset outside [0, heap length), or a string with no NUL before the heap ends, raises the context's
 * range error (VDL_ERANGE at the next check), as vdl_op_like does.  heap must be VDL_U8; data is int32 or int64.
 * origin is the value heap byte 0 stands for (0: the offsets of a Load,<t>.<c>.heap column); dictionary codes reach
 * below zero.  Ranking a string column turns it into a key vdl_op_order sorts in collation order. */
int vdl_op_collate(vdl_ctx *ctx, vdl_vec data, vdl_vec heap, int64_t origin, vdl_vec *out);

/* ---- fused select -> map -> fold -------------------------------------------------------
 * One launch that scans up to VDL_MAX_COLS columns of one table, applies a conjunction of range
 * predicates, computes a small bit-packed group key and folds products of affine column terms
 * per key.  This is what the fusion pass rewrites
 *   Fold(op, groups, f(Gather(c_i, FoldSelect(pos_ p, p)) ...))            (Vlite.hs:721-730)
 * and its Partition/Scatter-sorted grouped form (Vlite.hs:1048-1098) into. */
#define VDL_MAX_COLS 12
#define VDL_MAX_PREDS 8
#define VDL_MAX_KEYS 4
#define VDL_MAX_AGGS 8
#define VDL_MAX_FACTORS 3
#define VDL_MAX_POSTS 8

typedef struct {          /* value = a + b * (column[row] >> shr); column < 0: the constant a;   */
  int32_t column;         /* column == -2: the global row id (row_base + row)                      */
  int32_t shr;
  int64_t a, b;
} vdl_affine;

typedef struct { int32_t column, shr; int64_t lo, hi; } vdl_range_pred;  /* lo <= (col>>shr) <= hi */
typedef struct { vdl_affine e; int32_t shl, pad; } vdl_key_part;         /* (e) << shl, parts OR-ed */
typedef struct {
  int32_t op;             /* VDL_FOLD_SUM / MIN / MAX / CHOOSE / COUNT */
  int32_t nfactors;       /* value = product of factors (empty product = 1) */
  vdl_affine factor[VDL_MAX_FACTORS];
} vdl_fold_spec;

/* Elementwise epilogue over the fold results (AVG = Divide(FoldSum x, FoldSum 1), Vlite.hs:1038-1041): post op i
 * = op(a, b) per group, evaluated inside the finalize kernel; an operand is a fold's result, an earlier post op's
 * result, or a constant. */
enum { VDL_POST_FOLD = 0, VDL_POST_POST = 1, VDL_POST_CONST = 2 };
typedef struct { int32_t op, a_kind, b_kind, pad; int64_t a, b; } vdl_post_op;   /* op: a VDL_* binary op */

typedef struct {
  int64_t rows;                       /* rows of this shard */
  int64_t row_base;                   /* global row id of this shard's row 0 */
  int32_t ncolumns;
  vdl_vec column[VDL_MAX_COLS];       /* registered columns of one table, equal length */
  int32_t npreds;
  vdl_range_pred pred[VDL_MAX_PREDS];
  int32_t nkeys;                      /* 0: one group (key 0) */
  vdl_key_part key[VDL_MAX_KEYS];
  int64_t key_mask;                   /* key &= key_mask (Vlite.hs:1111-1115 size hint); -1: none */
  int64_t domain;                     /* keys are in [0, domain) */
  int32_t nfolds;
  vdl_fold_spec fold[VDL_MAX_AGGS];
  int32_t nposts;
  vdl_post_op post[VDL_MAX_POSTS];
} vdl_fused_desc;

typedef struct vdl_fused vdl_fused;   /* a prepared fused scan (device tables, launch geometry) */

int vdl_fused_prepare(vdl_ctx *ctx, const vdl_fused_desc *desc, vdl_fused **out);
/* Launch the scan over this shard; leaves the partial table [nacc][domain] of int64 in HBM. */
int vdl_fused_launch(vdl_fused *f);
/* mode 1 (single GPU): the scan kernel's last thread block also finalizes (as vdl_fused_finalize(f, NULL, 1) would),
 * so a step is one launch; mode 2: the same after the peer-memory exchange below; mode 0 = vdl_fused_launch. */
int vdl_fused_launch_ex(vdl_fused *f, int self_finalize);
/* The partial table for the multi-GPU combine: device pointer and its size in int64 elements. */
int vdl_fused_partials(vdl_fused *f, void **device_ptr, int64_t *n_int64);
/* Merge `nranks` partial tables laid out back to back at `all_partials` (an all-gather result; pass
 * NULL and 1 to use this shard's own table), drop empty groups and produce one vector per fold,
 * ascending key order -- the dense-model output of the Folds (G1, G14). */
int vdl_fused_finalize(vdl_fused *f, const void *all_partials, int nranks);
int vdl_fused_num_groups(vdl_fused *f, int64_t *ngroups);   /* synchronises */
int vdl_fused_result(vdl_fused *f, int fold_index, vdl_vec *out);
/* Host copy of one fold's result (pinned memory, valid until the next launch).  The group count, the error
 * counter and all fold results of a scan come back in ONE device->host copy. */
int vdl_fused_result_host(vdl_fused *f, int fold_index, const int64_t **data, int64_t *len);
/* The same for post op `post_index` of the descriptor. */
int vdl_fused_post_host(vdl_fused *f, int post_index, const int64_t **data, int64_t *len);
/* Host-only check of the run-time specialisation of the fused scan (no GPU needed): prints the shape-traits class of a
 * grouped descriptor and compiles the scan kernel over it with NVRTC for sm_100a.  Return codes as vdl_jit_selftest. */
int vdl_scan_jit_selftest(char *log, int log_capacity);
/* The same for the FK-join probe: a descriptor printed as CUDA C (one straight-line function per predicate stage). */
int vdl_probe_jit_selftest(char *log, int log_capacity);
/* Which instantiation of the scan kernel runs: "jit:<hash>" (the shape of this descriptor, compiled at run time), the name of
 * a precompiled static shape, or "generic". */
const char *vdl_fused_shape_name(vdl_fused *f);
int vdl_fused_destroy(vdl_fused *f);
/* ---- multi-GPU combine over peer memory (NVLink / NVSwitch), no collective library on the data path -------------
 * Every rank owns an exchange buffer of vdl_fused_exchange_bytes() in device memory that its peers can address
 * (same process: the pointer itself; one process per GPU: vdl_ipc_export on the owner, vdl_ipc_open on the peers).
 * After vdl_fused_set_peers(), vdl_fused_launch_ex(f, 2) runs the whole step as ONE kernel per GPU: the last thread
 * block of the scan stores this rank's partial table into every peer's buffer, publishes a per-rank epoch flag
 * (release, system scope), waits for the flags of all ranks, merges the tables and finalizes -- every rank ends up
 * with the global result.  All ranks must launch the same steps in the same order. */
#define VDL_MAX_RANKS 16
#define VDL_IPC_HANDLE_BYTES 64
int vdl_fused_exchange_bytes(vdl_fused *f, int world, int64_t *bytes);
int vdl_fused_set_peers(vdl_fused *f, int rank, int world, void *const *peer_buffers);
int vdl_ipc_alloc(vdl_ctx *ctx, int64_t bytes, void **device_ptr);            /* zero-filled cudaMalloc memory */
int vdl_ipc_export(vdl_ctx *ctx, void *device_ptr, unsigned char handle[VDL_IPC_HANDLE_BYTES]);
int vdl_ipc_open(vdl_ctx *ctx, const unsigned char handle[VDL_IPC_HANDLE_BYTES], void **device_ptr);
int vdl_ipc_close(vdl_ctx *ctx, void *device_ptr);
int vdl_ipc_free(vdl_ctx *ctx, void *device_ptr);

/* Duration of the last vdl_fused_launch's scan kernel alone, CUDA events on the context stream. */
int vdl_fused_last_kernel_ms(vdl_fused *f, float *ms);
/* Mean and minimum of the scan kernel's duration over the last n launches (n <= 64): the library records an event pair
 * around every launch, so a timed loop reads the durations afterwards instead of synchronising every step. */
int vdl_fused_kernel_ms_stats(vdl_fused *f, int n, float *mean_ms, float *min_ms);

/* ---- fused FK-join probe ----------------------------------------------------------------
 * One pass over a fact-table shard that follows foreign-key index columns into dimension columns, applies
 * the predicates of the whole join chain (handleGatherJoin / deduceMasks, Vlite.hs:1199-1280) and either
 * folds per group key or emits the surviving rows' expressions as dense vectors in row order.
 *   leaf       value(row) = column[ parent < 0 ? row : value of leaf `parent` (row) ]   (parent precedes the leaf)
 *   term       a + b * (leaf >> shr);  leaf -1: the constant a;  leaf -2: the global row id;
 *              leaf -3-k: 1 if indicator predicate k holds at the row, else 0 (CASE WHEN ... THEN 1 ELSE 0)
 *   predicate  kind 0: t in [lo, hi] or in one of the nmore further ranges [lo_more[i], hi_more[i]] (IN lists, <>);
 *              kind 1: t cmp u, cmp = VDL_CMP_*;  evaluated in order, the first failure rejects the row */
#define VDL_MAX_LEAVES 24
#define VDL_MAX_PROBE_PREDS 12
#define VDL_MAX_EMITS 8
#define VDL_MAX_INDICATORS 4
#define VDL_MAX_MORE_RANGES 3
enum { VDL_CMP_EQ = 0, VDL_CMP_NE, VDL_CMP_GT, VDL_CMP_GE, VDL_CMP_LT, VDL_CMP_LE };
typedef struct { vdl_vec column; int32_t parent; } vdl_leaf;
typedef struct { int32_t leaf, shr; int64_t a, b; } vdl_term;
typedef struct {
  int32_t kind, cmp;
  vdl_term t, u;
  int64_t lo, hi;
  int32_t nmore, pad;
  int64_t lo_more[VDL_MAX_MORE_RANGES], hi_more[VDL_MAX_MORE_RANGES];
} vdl_probe_pred;
typedef struct { int32_t nfactors, pad; vdl_term factor[VDL_MAX_FACTORS]; } vdl_product;
typedef struct { int32_t op, pad; vdl_product value; } vdl_probe_fold;       /* op: VDL_FOLD_* */
typedef struct {
  int64_t rows, row_base;
  int32_t nleaves, npreds;
  vdl_leaf leaf[VDL_MAX_LEAVES];
  vdl_probe_pred pred[VDL_MAX_PROBE_PREDS];
  /* fold mode (nfolds > 0): key = OR of (term << shl) & key_mask in [0, domain); nkeys == 0: one group */
  int32_t nkeys, nfolds;
  vdl_term key[VDL_MAX_KEYS];
  int32_t key_shl[VDL_MAX_KEYS];
  int64_t key_mask, domain;
  vdl_probe_fold fold[VDL_MAX_AGGS];
  int32_t nposts, nemits;
  vdl_post_op post[VDL_MAX_POSTS];
  /* emit mode (nemits > 0): one dense int64 vector per expression, surviving rows in ascending row order */
  vdl_product emit[VDL_MAX_EMITS];
  int32_t nindicators, pad2;
  vdl_probe_pred indicator[VDL_MAX_INDICATORS];   /* predicates used as 0/1 values (their terms may not be indicators) */
} vdl_probe_desc;
typedef struct vdl_probe vdl_probe;
/* Peer-memory combine for a probe in fold mode (same protocol and buffer layout as vdl_fused_set_peers; the table has
 * (nfolds + 2) * domain int64): after vdl_probe_set_peers, vdl_probe_run_ex(p, 2) leaves the GLOBAL result on every rank. */
int vdl_probe_exchange_bytes(vdl_probe *p, int world, int64_t *bytes);
int vdl_probe_set_peers(vdl_probe *p, int rank, int world, void *const *peer_buffers);
int vdl_abi_sizeof_probe_desc(void);
int vdl_probe_prepare(vdl_ctx *ctx, const vdl_probe_desc *desc, vdl_probe **out);
int vdl_probe_run(vdl_probe *p);                 /* asynchronous on the context stream */
/* Sharded fact table, fold mode: run without finalizing, all-gather the partial tables ([nfolds + 2][domain] int64 each)
 * with any transport, then merge + finalize (NULL, 1 = this rank alone). */
int vdl_probe_run_ex(vdl_probe *p, int finalize);
int vdl_probe_partials(vdl_probe *p, void **device_ptr, int64_t *n_int64);
int vdl_probe_finalize(vdl_probe *p, const void *all_partials, int nranks);
/* fold mode: host copy of fold `index` (0..nfolds-1) or post op (nfolds..); one vector entry per existing key */
int vdl_probe_result_host(vdl_probe *p, int index, const int64_t **data, int64_t *len);
/* emit mode: take ownership of the k-th emitted vector (synchronises for its length) */
int vdl_probe_emit_take(vdl_probe *p, int k, vdl_vec *out);
int vdl_probe_last_kernel_ms(vdl_probe *p, float *ms);
int vdl_probe_kernel_ms_stats(vdl_probe *p, int n, float *mean_ms, float *min_ms);
int vdl_probe_destroy(vdl_probe *p);

/* ---- whole plans: the text mplan2vdl prints (Vdl.hs:410-453) ---------------------------- */
enum { VDL_PLAN_FUSE = 1 };           /* flags: run the select->map->fold fusion pass */
int vdl_plan_load(vdl_ctx *ctx, const char *vdl_text, int flags, vdl_plan **out);
/* EXPLAIN: what the planner makes of a program, as JSON in `out` -- statements, nodes after CSE, the fused scans (table,
 * columns, predicates, key parts, domain, folds, post ops), probe fold and emit groups, map clusters, Folds left for
 * op-at-a-time evaluation, whether the tail is mergeable across shards.  Needs no context, no column and no device: binding
 * happens at run time.  A program the parser or the planner rejects gives {"error": code, "message": ...} and that code. */
int vdl_plan_explain(const char *vdl_text, int flags, char *out, int capacity);
/* Statements parsed, distinct nodes after structural CSE (App. G10), fused scans, kernel launches
 * of the last run. */
int vdl_plan_stats(vdl_plan *p, int *statements, int *nodes, int *fused_scans, int64_t *launches);
/* Sharded run of a plan whose probe passes EMIT vectors (high-cardinality group-bys: Q3): after vdl_plan_run_local every
 * rank holds its shard's survivors; concatenate them over the ranks in rank order (= global row order; any transport) and
 * substitute the result before vdl_plan_finish, which then evaluates the remaining ops on the global vectors. */
int vdl_plan_num_emits(vdl_plan *p);
/* The table whose rows probe emit group `group` (0 .. emit_groups - 1 of vdl_plan_probe_stats) walks.  Sharding by row range
 * is only meaningful when that is the sharded fact table: a pass over a replicated dimension table emits the same survivors on
 * every rank (mplan2vdl_b200/dist.py refuses such plans instead of miscomputing them). */
int vdl_plan_emit_group_table(vdl_plan *p, int group, const char **table);
int vdl_plan_emit(vdl_plan *p, int i, void **device_ptr, int64_t *len);              /* synchronises */
int vdl_plan_emit_replace(vdl_plan *p, int i, void *device_ptr, int64_t len);        /* caller-owned device memory */
/* Sharded TAIL: when every output of the plan is an op-at-a-time Fold by runs of ONE groups vector -- a constant (a single
 * SUM over a join's survivors: Q19) or keys sorted by their own Partition (Vlite.hs:1057-1060, the high-cardinality
 * group-by of Q3) -- a rank can run the whole plan on its row-range shard (vdl_plan_run): its outputs are the slice of the
 * global result that belongs to its rows, except that its first group may continue the previous rank's last one.
 * vdl_plan_tail_info: is the plan of that shape, and the fold op of every output (VDL_FOLD_*).  After vdl_plan_tail_enable,
 * every vdl_plan_run also records what vdl_plan_tail_boundary returns: rec = { keys were in order (Partition = identity) or
 * constant, number of runs, first key, last key, first row of every output ..., last row of every output ... } (4 + 2 x
 * outputs values).  Exchanging these records lets the ranks merge the straddling groups -- SUM adds, MIN / MAX compare,
 * FoldChoose keeps the earlier rank's value -- without moving the survivors (mplan2vdl_b200/dist.py
 * merge_tail_boundaries); vdl_plan_tail_apply writes the merged last row and / or gives up the first row (a group that
 * starts on an earlier rank), after which vdl_plan_output returns this rank's slice of the global result.  (Only meaningful
 * when the plan's one probe emit pass walks the sharded table: vdl_plan_emit_group_table.) */
int vdl_plan_tail_info(vdl_plan *p, int *mergeable, int *fold_ops, int cap);
int vdl_plan_tail_enable(vdl_plan *p, int on);
int vdl_plan_tail_boundary(vdl_plan *p, int64_t *rec, int cap);
int vdl_plan_tail_apply(vdl_plan *p, int drop_first, const int64_t *last_row);
/* FK-join plans: Folds run by the probe kernel, probe passes in emit mode, vectors those materialise. */
int vdl_plan_probe_stats(vdl_plan *p, int *fold_groups, int *emit_groups, int *emitted_vectors);
/* Map clusters of the op-at-a-time remainder: how many vdl_op_map launches stand for how many plan nodes. */
int vdl_plan_map_stats(vdl_plan *p, int *clusters, int *nodes_covered);
int vdl_plan_probe_kernel_ms(vdl_plan *p, float *ms);   /* sum over the probe passes of the last run; synchronises */
/* Dominant-kernel time of the last n runs (first fused scan, else the sum over the probe passes): mean and minimum. */
int vdl_plan_kernel_ms_stats(vdl_plan *p, int n, float *mean_ms, float *min_ms);
/* Phase 1: everything up to and including the fused scans (local shard). */
/* Global row id of this shard's row 0 (row-range sharding of the fact table; default 0). */
int vdl_plan_set_row_base(vdl_plan *p, int64_t row_base);
int vdl_plan_run_local(vdl_plan *p);
int vdl_plan_num_fused(vdl_plan *p);
/* Partial aggregate tables of a sharded run, in the order vdl_plan_finish expects the gathered buffers: the fused scans,
 * then the probe fold groups. */
int vdl_plan_num_partials(vdl_plan *p);
int vdl_plan_partials(vdl_plan *p, int i, void **device_ptr, int64_t *n_int64);
/* Sharded execution without a collective library: exchange buffers of partial table `index` (numbered like
 * vdl_plan_partials: fused scans, then probe fold groups) on every rank (see vdl_fused_set_peers / vdl_probe_set_peers);
 * once every partial table has its peers, vdl_plan_run() returns the GLOBAL result on every rank.  The size comes from
 * vdl_plan_exchange_bytes() once the plan has run at least once (vdl_plan_run_local). */
int vdl_plan_exchange_bytes(vdl_plan *p, int index, int world, int64_t *bytes);
int vdl_plan_set_peers(vdl_plan *p, int index, int rank, int world, void *const *peer_buffers);
int vdl_plan_fused(vdl_plan *p, int i, vdl_fused **out);
/* Phase 2: finalize the fused scans (optionally from all-gathered partials, one buffer per fused scan,
 * NULL entries / nranks 1 for single GPU), run the remaining ops, copy outputs to the host. */
int vdl_plan_finish(vdl_plan *p, const void *const *all_partials, int nranks);
/* vdl_plan_run_local + vdl_plan_finish for one GPU. */
int vdl_plan_run(vdl_plan *p);
/* The launches of vdl_plan_run without the wait (asynchronous on the context's stream); vdl_plan_finish(p, NULL, 1) then
 * awaits the results.  With peers set, issue every rank's vdl_plan_launch before awaiting any rank. */
int vdl_plan_launch(vdl_plan *p);
int vdl_plan_num_outputs(vdl_plan *p);
/* Output i in MaterializeCompact order: name (the Project's <out>, Vdl.hs:278-292), host int64 data. */
int vdl_plan_output(vdl_plan *p, int i, const char **name, const int64_t **data, int64_t *len);
/* Typed result columns.  The reference's result is text (the server's JSON, resolve.py:8-32), so the width a column
 * crosses PCIe in is the executor's choice: with typed outputs on, an op-at-a-time output whose every value is a value of
 * a 4-byte column -- by provenance: a probe pass emitting a plain column, Gather, Scatter, FoldChoose / FoldMin / FoldMax of
 * such a vector -- is narrowed on the device and copied as int32 (Q3 SF10: 28 instead of 44 MB per run).
 * vdl_plan_output_typed returns dtype 4 (int32 data) or 8 (int64); vdl_plan_output fails for a column delivered as int32. */
int vdl_plan_set_typed_outputs(vdl_plan *p, int on);
int vdl_plan_output_typed(vdl_plan *p, int i, const char **name, const void **data, int64_t *len, int *dtype);
/* ORDER BY key_output[0..nkeys) (output indices, descending[i] = 1: DESC) LIMIT limit, applied to every later
 * vdl_plan_run / vdl_plan_finish before the results are copied to the host (vdl_op_order's order: ties keep the plan's own
 * row order; nkeys = 0 with limit >= 0: the first `limit` rows).  nkeys = 0 and limit < 0: off (the default).  The outputs
 * must then all have one length (vdl_plan_finish fails with VDL_EINVAL naming two that differ); vdl_plan_output reports the
 * limited length.  Excludes the sharded tail (a rank holds only a slice of the result): with vdl_plan_tail_enable(p, 1)
 * in force this fails with VDL_EUNSUPPORTED, and so does that call while an order is set. */
int vdl_plan_set_order(vdl_plan *p, int nkeys, const int *key_output, const int *descending, int64_t limit);
/* Key k of the order set by vdl_plan_set_order compares by the strings its output's values point to in `heap`
 * (vdl_op_collate's contract, with `origin`).  heap = 0 clears it.  A later vdl_plan_set_order clears every heap.  The
 * outputs keep their values (offsets or codes): only the row order follows the strings.  A key index outside the current
 * order, or a heap that is not VDL_U8: VDL_EINVAL. */
int vdl_plan_set_order_heap(vdl_plan *p, int key, vdl_vec heap, int64_t origin);
int vdl_plan_destroy(vdl_plan *p);

/* ---- several GPUs of one box driven from ONE process (SURVEY.md section 8 b, e) ----------------------------------------
 * A communicator owns one context per rank (devices[r], or device r when NULL; the same device may appear twice: ranks
 * emulated on one GPU), with peer access enabled between the devices.  The caller registers rank r's row-range shard of the
 * fact table -- and the replicated dimension tables -- with vdl_comm_ctx(c, r) under the usual column names, loads the
 * program once for all ranks and runs it: one scan-kernel launch per GPU, whose last thread block exchanges the partial
 * aggregate tables with the peers over NVLink and finalizes (no collective library on the data path); every rank's plan
 * then holds the GLOBAL result (vdl_comm_plan_rank + vdl_plan_output).  What mplan2vdl_b200/dist.py does for
 * one-process-per-GPU launches (torchrun, CUDA IPC handles); this is the form a single Haskell host binds. */
typedef struct vdl_comm vdl_comm;
typedef struct vdl_comm_plan vdl_comm_plan;
int vdl_comm_init_all(int nranks, const int *devices, vdl_comm **out);
int vdl_comm_size(vdl_comm *c);
vdl_ctx *vdl_comm_ctx(vdl_comm *c, int rank);
const char *vdl_comm_last_error(vdl_comm *c);
int vdl_comm_destroy(vdl_comm *c);
/* row_base[r]: global row id of rank r's first fact row (NULL: 0 everywhere). */
int vdl_comm_plan_load(vdl_comm *c, const char *vdl_text, int flags, const int64_t *row_base, vdl_comm_plan **out);
vdl_plan *vdl_comm_plan_rank(vdl_comm_plan *p, int rank);
int vdl_comm_plan_run(vdl_comm_plan *p);
int vdl_comm_plan_destroy(vdl_comm_plan *p);

#ifdef __cplusplus
}
#endif
#endif /* VDL_CUDA_H */
