// Internal declarations shared by the translation units of libvdl_cuda (not part of the ABI).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include <functional>
#include <string>
#include <unordered_map>
#include <vector>

#include "vdl_device.cuh"      // vdl_cuda.h, i64 / u64, XDesc, FinDesc, the device code shared with the run-time compiled kernels

// A device vector.  Columns are vectors with a name.  Ranges (RangeV/RangeC) are kept virtual:
// no HBM traffic until a consumer needs the values.
struct Vec {
  void *ptr = nullptr;
  int dtype = VDL_I64;      // VDL_I32 / VDL_I64
  i64 len = 0;
  i64 cap_rows = 0;         // rows that may be read (>= len; bulk copies round the tail up to 16 B)
  bool owned = false;
  bool live = false;
  bool is_range = false;
  bool is_perm = false;        // a Partition result: a permutation of 0..len-1, so a Scatter by it writes every slot
  bool narrow32 = false;       // every value is a value of a 4-byte column (provenance: probe emit of a plain leaf, Gather,
                               // Scatter, FoldChoose / Min / Max of such a vector): a result column can travel as int32
  i64 from = 0, step = 0;
  i64 domain = -1;          // length of the vector these values index into; -1 unknown (App. G2)
  bool has_stats = false;   // vmin/vmax computed on the device by vdl_column_analyze (invalidated by writes)
  i64 vmin = 0, vmax = 0;
  // Write generation: unique within the context (taken from vdl_ctx::gen_counter) and renewed by every write the
  // library can see (creation, upload, synthetic fill, vdl_column_touch).  A prepared scan / probe records
  // (handle, generation) of its columns: a different pair means other data, another allocation or a recycled handle.
  u64 gen = 0;
  // a Fold result remembers the groups vector it was folded by: a Fold over these results with row-space groups (level 2
  // of a hierarchical fold, Vlite.hs:1181-1192) groups them by the groups value at each level-1 run's head
  vdl_vec fold_groups = 0;
  u64 fold_groups_gen = 0;
  std::string name;
};

#define VDL_EVENT_RING 64

struct vdl_ctx {
  int device = 0;
  cudaStream_t stream = nullptr;
  cudaStream_t copy_stream = nullptr;   // device->host copies of plan outputs, overlapped with the evaluation of the next output
  cudaEvent_t copy_event = nullptr;
  int sm_count = 148;
  int smem_optin = 0;
  std::vector<Vec> vecs;    // handle = index, 0 unused
  std::unordered_map<std::string, int> columns;
  std::string err;
  i64 launches = 0;
  int *d_errflag = nullptr; // device-side error counter (Gather/Scatter range checks)
  void *scratch = nullptr;  // reusable scratch for scans / histograms
  size_t scratch_bytes = 0;
  void *h_mail = nullptr, *d_mail = nullptr;   // 64 B of mapped pinned memory: scalars the host waits for (read_scalar)
  void *jit = nullptr;      // vdl_jit.cu: the run-time compiled map, scan and probe kernels
  u64 gen_counter = 0;      // source of Vec::gen
};

int vdl_fail(vdl_ctx *ctx, int code, const char *fmt, ...);
int vdl_cuda_fail(vdl_ctx *ctx, cudaError_t e, const char *what);
#define VDL_CUDA(ctx, call)                                       \
  do {                                                            \
    cudaError_t e__ = (call);                                     \
    if (e__ != cudaSuccess) return vdl_cuda_fail(ctx, e__, #call); \
  } while (0)
#define VDL_TRY(call)            \
  do {                           \
    int rc__ = (call);           \
    if (rc__) return rc__;       \
  } while (0)

// vector table
int vec_new(vdl_ctx *ctx, int dtype, i64 len, vdl_vec *out);              // allocates HBM
int vec_new_range(vdl_ctx *ctx, i64 from, i64 step, i64 len, vdl_vec *out);
Vec *vec_get(vdl_ctx *ctx, vdl_vec v);                                    // nullptr + error if invalid or a string heap
Vec *vec_get_any(vdl_ctx *ctx, vdl_vec v);                                // string heaps (VDL_U8) too
void vec_written(vdl_ctx *ctx, Vec *v);                                   // new generation, statistics dropped
// (handle, generation) of a live stored vector, or false
bool vec_identity(vdl_ctx *ctx, vdl_vec v, u64 *gen);
int scratch_reserve(vdl_ctx *ctx, size_t bytes);
int check_errflag(vdl_ctx *ctx, const char *what);                        // synchronises
// Host copy of a device scalar (<= 64 bytes) once the stream has reached this point.  A one-thread kernel stores it to
// mapped host memory, so the read never queues on the copy engine behind a bulk device->host copy of another stream
// (plan outputs); synchronises the context's stream.
int read_scalar(vdl_ctx *ctx, const void *device_src, void *host_dst, int bytes);
int vec_narrow_copy(vdl_ctx *ctx, vdl_vec src, vdl_vec *out);   // vdl_ops.cu: int64 -> int32 copy of a vector whose values fit

// Wait until a kernel has published `seq` in mapped pinned host memory (its last store, after a system-scope fence):
// a short spin on the word instead of cudaStreamSynchronize, whose wake-up costs 10-20 us -- several percent of a
// 0.3 ms step on 8 GPUs.  Falls back to synchronising the stream (errors surface there) after ~20 ms.
int wait_published(vdl_ctx *ctx, const volatile i64 *word, i64 seq);

Operand operand_of(const Vec &v);
inline bool vec_is_narrow(const Vec &v) { return v.narrow32 || (v.dtype == VDL_I32 && !v.is_range); }

int vdl_jit_map_launch(vdl_ctx *ctx, const MapArgs &m, i64 *out, i64 n, int blocks);   // 1 launched, 0 use the interpreter, <0 error
void vdl_jit_destroy(vdl_ctx *ctx);
// vdl_jit.cu: NVRTC compile of `src` for sm_100a against the headers embedded in the library.  VDL_OK (the image in
// *cubin, if given), VDL_ENOTFOUND when NVRTC is not installed, VDL_ECUDA when it rejected the source (NVRTC's log in
// *log, its status in *status, if given).  Needs no GPU.
int vdl_jit_compile(const std::string &src, std::string *log, std::vector<char> *cubin = nullptr, int *status = nullptr);
// The kernel `name` of the source `source()` returns, compiled and loaded once per context and cached under `key`;
// `source` is called on a miss only.  Takes `smem` bytes of dynamic shared memory when that is over the default 48 KB.
// nullptr: NVRTC is missing, compilation or loading failed (also cached: no retry), or the attribute could not be set.
cudaKernel_t vdl_jit_kernel(vdl_ctx *ctx, const std::string &key, const char *name, size_t smem, const std::function<std::string()> &source);

// Do the columns a prepared scan / probe was built from still hold what they held at prepare time?  (The statistics
// proofs -- int32 narrowing, 32-bit accumulators, the static shape -- and the device pointers are baked in.)
bool vdl_fused_current(vdl_fused *f);
bool vdl_probe_current(vdl_probe *p);

// Event pairs around the dominant kernel of the last VDL_EVENT_RING launches: durations are read AFTER a timed loop
// instead of synchronising on an event every step.
struct KernelTimer {
  cudaEvent_t ev0[VDL_EVENT_RING] = {nullptr}, ev1[VDL_EVENT_RING] = {nullptr};
  long n = 0;                        // launches timed so far
  void create();
  void destroy();
  int begin(vdl_ctx *ctx);
  int end(vdl_ctx *ctx);
  int last_ms(vdl_ctx *ctx, float *ms);
  int stats(vdl_ctx *ctx, int count, float *mean_ms, float *min_ms);   // over the last count (<= VDL_EVENT_RING) launches
};

// The error messages of a fold family (the fused scan, the probe in fold mode) for its FoldCombine.
struct FoldTexts {
  const char *nranks;       // printf format of an nranks without gathered tables
  const char *no_peers;     // peer exchange before set_peers
  const char *unfinalized;  // results fetched before a finalize
  const char *timeout;      // a peer never delivered its table
  const char *range;        // printf format of the number of rows out of range
};

// Combine of a fold family's per-rank partial tables [rows][domain] into the fold results: this rank's table, the merge
// (FinDesc: finalize_block), the peer-memory exchange (XDesc: exchange_block), the result buffer the finalize publishes
// into mapped pinned memory, and its fetch on the host (vdl_combine.cu).
struct FoldCombine {
  vdl_ctx *ctx = nullptr;
  const FoldTexts *texts = nullptr;
  i64 *table = nullptr;              // this rank's partial table, fd.part_stride int64
  FinDesc fd;                        // out / post_out / ngroups point into d_out, hmirror into h_out
  XDesc xd;                          // world 0: no peer exchange configured
  i64 *d_out = nullptr;              // [nout + npost][domain] results, then [ngroups, errors]
  i64 *h_out = nullptr;              // mapped pinned mirror (+ [seq]: the publication word)
  bool finalized = false;            // the last step published results (else it left its table for an external combine)
  bool table_clean = false;          // the table holds the fold identities (the family's init, or a finalize that reset it)
  i64 ngroups = -1;                  // -1 until fetch has read the published results

  // fd's layout fields (nacc, nchoose, cnt_idx, first_idx, out_kind, out_idx, acc_op, post, reset_table) are the
  // family's; this sets the rest and loads the combine kernels (not lazily behind a peer's spinning exchange).
  int allocate(vdl_ctx *c, const FoldTexts *t, i64 *tab, i64 part_stride, i64 domain, int nout, int npost);
  void release();
  int exchange_bytes(int world, int64_t *bytes) const;
  int set_peers(int rank, int world, void *const *peer_buffers);
  int partials(void **device_ptr, int64_t *n_int64) const;
  int next_epoch();                                     // before a step that exchanges over peer memory
  int finalize(const void *all_partials, int nranks);   // merge gathered tables (null, 1: this rank's own)
  int exchange();                                       // this rank's table to the peers, then the merge: one launch
  int fetch();
  int result_host(int index, const int64_t **data, int64_t *len);   // index over the nout results, then the npost
};
FoldCombine *vdl_fused_combine(vdl_fused *f);
FoldCombine *vdl_probe_combine(vdl_probe *p);   // fold mode only

