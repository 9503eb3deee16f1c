// Combine of per-rank partial tables, shared by the fused scan (vdl_fused.cu) and the FK-join probe in fold mode
// (vdl_probe.cu): the external all-gather finalize, the peer-memory exchange, the fetch of the published results, and
// the event ring both families time their dominant kernel with.
#include <stdlib.h>
#include <string.h>

#include <algorithm>

#include "vdl_internal.h"

// Merge of gathered tables (or this rank's own): an external finalize, or a single-GPU step with nothing to scan.
__global__ void __launch_bounds__(256, 1) fold_finalize_kernel(const __grid_constant__ FinDesc f) {
  __shared__ int warp_cnt[8];
  __shared__ i64 running;
  finalize_block<256>(f, f.parts, f.nranks, threadIdx.x, warp_cnt, &running);
}

// Peer-memory combine in one block: this rank's table (FoldChoose values included) to slot [parity][rank] of every
// rank's exchange buffer, the epoch published, the other ranks' flags awaited, then the merge of the `world` tables
// that arrived in this rank's own buffer.  A peer that never arrives: error flag after the timeout, never a hang.
__global__ void __launch_bounds__(256, 1) fold_exchange_kernel(const __grid_constant__ FinDesc f, const __grid_constant__ XDesc x, const i64 *table,
                                                               int *errflag) {
  __shared__ int warp_cnt[8];
  __shared__ i64 running;
  const i64 *parts = exchange_block<256>(x, table, errflag, threadIdx.x);
  finalize_block<256>(f, parts, x.world, threadIdx.x, warp_cnt, &running);
}

int FoldCombine::allocate(vdl_ctx *c, const FoldTexts *t, i64 *tab, i64 part_stride, i64 domain, int nout, int npost) {
  ctx = c;
  texts = t;
  table = tab;
  memset(&xd, 0, sizeof xd);
  const size_t nb = ((size_t)(nout + npost) * domain + 3) * sizeof(i64);
  i64 *mapped = nullptr;
  if (cudaMalloc(&d_out, nb) != cudaSuccess || cudaHostAlloc(&h_out, nb, cudaHostAllocMapped) != cudaSuccess ||
      cudaHostGetDevicePointer(&mapped, h_out, 0) != cudaSuccess)
    return VDL_ENOMEM;
  memset(h_out, 0, nb);        // (the publication word must not start out looking like a finished step)
  fd.part_stride = part_stride;
  fd.domain = domain;
  fd.nout = nout;
  fd.npost = npost;
  for (int o = 0; o < nout; o++) fd.out[o] = d_out + (size_t)o * domain;
  for (int q = 0; q < npost; q++) fd.post_out[q] = d_out + (size_t)(nout + q) * domain;
  fd.ngroups = d_out + (size_t)(nout + npost) * domain;
  fd.errflag = ctx->d_errflag;
  fd.hmirror = mapped;
  fd.parts = table;
  fd.nranks = 1;
  // Load the kernels a step may launch NOW: CUDA loads lazily, and loading can wait for running kernels, so a first
  // launch of a finalize behind a peer's spinning exchange kernel would stall the host until the exchange times out
  // (seen when one host thread drives several ranks).
  cudaFuncAttributes fa;
  cudaFuncGetAttributes(&fa, fold_finalize_kernel);
  cudaFuncGetAttributes(&fa, fold_exchange_kernel);
  cudaGetLastError();
  return VDL_OK;
}

void FoldCombine::release() {
  if (d_out) cudaFree(d_out);
  if (h_out) cudaFreeHost(h_out);
  d_out = h_out = nullptr;
}

int FoldCombine::exchange_bytes(int world, int64_t *bytes) const {
  if (!bytes || world < 1 || world > VDL_MAX_RANKS) return VDL_EINVAL;
  *bytes = ((int64_t)2 * world * fd.part_stride + 2 * world) * (int64_t)sizeof(i64);
  return VDL_OK;
}

int FoldCombine::set_peers(int rank, int world, void *const *peer_buffers) {
  if (!peer_buffers || world < 1 || world > VDL_MAX_RANKS || rank < 0 || rank >= world) return VDL_EINVAL;
  memset(&xd, 0, sizeof xd);
  xd.rank = rank;
  xd.world = world;
  xd.stride = fd.part_stride;
  xd.timeout_ns = 10000000000ull;                     // 10 s; VDL_PEER_TIMEOUT_MS overrides (tests)
  if (const char *e = getenv("VDL_PEER_TIMEOUT_MS")) xd.timeout_ns = (u64)atoll(e) * 1000000ull;
  for (int r = 0; r < world; r++) {
    if (!peer_buffers[r]) return vdl_fail(ctx, VDL_EINVAL, "set_peers: buffer of rank %d is null", r);
    xd.peer[r] = (i64 *)peer_buffers[r];
  }
  return VDL_OK;
}

int FoldCombine::partials(void **device_ptr, int64_t *n_int64) const {
  if (!device_ptr || !n_int64) return VDL_EINVAL;
  *device_ptr = table;
  *n_int64 = fd.part_stride;
  return VDL_OK;
}

int FoldCombine::next_epoch() {
  if (xd.world < 1) return vdl_fail(ctx, VDL_EINVAL, "%s", texts->no_peers);
  xd.epoch++;
  return VDL_OK;
}

int FoldCombine::finalize(const void *all_partials, int nranks) {
  if (nranks < 1 || (nranks > 1 && !all_partials)) return vdl_fail(ctx, VDL_EINVAL, texts->nranks, nranks);
  VDL_CUDA(ctx, cudaSetDevice(ctx->device));
  fd.parts = all_partials ? (const i64 *)all_partials : table;
  fd.nranks = nranks;
  fd.seq++;
  fold_finalize_kernel<<<1, 256, 0, ctx->stream>>>(fd);
  ctx->launches++;
  VDL_CUDA(ctx, cudaGetLastError());
  finalized = true;
  ngroups = -1;
  if (fd.reset_table) table_clean = true;
  return VDL_OK;
}

int FoldCombine::exchange() {
  fd.seq++;
  fold_exchange_kernel<<<1, 256, 0, ctx->stream>>>(fd, xd, table, ctx->d_errflag);
  ctx->launches++;
  VDL_CUDA(ctx, cudaGetLastError());
  return VDL_OK;
}

// The finalize wrote the group count, the error counter and every result straight into h_out (mapped): wait for its
// publication word, no copy.
int FoldCombine::fetch() {
  if (!finalized) return vdl_fail(ctx, VDL_EINVAL, "%s", texts->unfinalized);
  if (ngroups >= 0) return VDL_OK;
  const size_t tail = (size_t)(fd.nout + fd.npost) * fd.domain;
  VDL_TRY(wait_published(ctx, h_out + tail + 2, fd.seq));
  const i64 err = h_out[tail + 1];
  if (err) {
    cudaMemsetAsync(ctx->d_errflag, 0, sizeof(int), ctx->stream);
    if (err >= (1 << 20)) return vdl_fail(ctx, VDL_ECUDA, "%s", texts->timeout);
    return vdl_fail(ctx, VDL_ERANGE, texts->range, (long long)err);
  }
  ngroups = h_out[tail];
  return VDL_OK;
}

int FoldCombine::result_host(int index, const int64_t **data, int64_t *len) {
  if (!data || !len || index < 0 || index >= fd.nout + fd.npost) return VDL_EINVAL;
  VDL_TRY(fetch());
  *data = h_out + (size_t)index * fd.domain;
  *len = ngroups;
  return VDL_OK;
}

// ------------------------------------------------------------------------------ event ring
void KernelTimer::create() {
  for (int i = 0; i < VDL_EVENT_RING; i++) { cudaEventCreate(&ev0[i]); cudaEventCreate(&ev1[i]); }
}

void KernelTimer::destroy() {
  for (int i = 0; i < VDL_EVENT_RING; i++) { if (ev0[i]) cudaEventDestroy(ev0[i]); if (ev1[i]) cudaEventDestroy(ev1[i]); }
}

int KernelTimer::begin(vdl_ctx *ctx) {
  VDL_CUDA(ctx, cudaEventRecord(ev0[n % VDL_EVENT_RING], ctx->stream));
  return VDL_OK;
}

int KernelTimer::end(vdl_ctx *ctx) {
  VDL_CUDA(ctx, cudaEventRecord(ev1[n % VDL_EVENT_RING], ctx->stream));
  n++;
  return VDL_OK;
}

int KernelTimer::last_ms(vdl_ctx *ctx, float *ms) {
  const int i = (int)((n - 1) % VDL_EVENT_RING);
  VDL_CUDA(ctx, cudaEventSynchronize(ev1[i]));
  VDL_CUDA(ctx, cudaEventElapsedTime(ms, ev0[i], ev1[i]));
  return VDL_OK;
}

int KernelTimer::stats(vdl_ctx *ctx, int count, float *mean_ms, float *min_ms) {
  count = (int)std::min<long>(std::min<long>(count, VDL_EVENT_RING), n);
  double sum = 0;
  float mn = 1e30f;
  for (int k = 1; k <= count; k++) {
    const int i = (int)((n - k) % VDL_EVENT_RING);
    float ms = 0;
    VDL_CUDA(ctx, cudaEventSynchronize(ev1[i]));
    VDL_CUDA(ctx, cudaEventElapsedTime(&ms, ev0[i], ev1[i]));
    sum += ms;
    mn = std::min(mn, ms);
  }
  if (mean_ms) *mean_ms = (float)(sum / count);
  if (min_ms) *min_ms = mn;
  return VDL_OK;
}
