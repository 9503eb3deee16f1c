// Streaming-read microbenchmark used to pick the data path of the fused scan (DESIGN.md section 4):
//   ldg   : grid-stride 128-bit loads, UNROLL independent loads in flight per thread
//   bulk  : persistent CTAs, one producer thread issuing cp.async.bulk (1-D TMA) copies into an
//           mbarrier-tracked shared-memory ring, consumer warps summing the staged words
//   sparse: (`membench sparse`) the late-fetch data path of the fused scan: a 4-byte column streamed in full by the bulk
//           ring, and for each row that passes a uniform random test with probability p an 8-byte value of a second
//           column fetched with `cp.async` into the row's slot of the stage, issued `dist` tiles ahead of its use.
//           Per p: the time, the bytes touched under a 32 B and a 64 B sector model (counted exactly on the host)
//           and the rate each model implies.  A stage is held `dist` tiles, so the lead stream is bound by the ring depth
//           left for it (DESIGN.md section 4.1); compare the rows with each other, not with the streaming modes.
// Build: nvcc -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -o gpurun_out/membench tools/membench.cu
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#define CK(x) do { cudaError_t e = (x); if (e != cudaSuccess) { printf("%s: %s\n", #x, cudaGetErrorString(e)); exit(1); } } while (0)

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) { asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count)); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) { asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory"); }
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) { asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory"); }
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
  asm volatile("{\n.reg .pred P1;\nLAB_WAIT:\nmbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n@P1 bra DONE;\nbra LAB_WAIT;\nDONE:\n}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void bulk_g2s_hint(void *dst, const void *src, uint32_t bytes, uint64_t *bar, uint64_t pol) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)), "l"(pol) : "memory");
}

template <int UNROLL>
__global__ void __launch_bounds__(256) ldg_kernel(const int4 *__restrict__ in, size_t n16, unsigned long long *out) {
  size_t stride = (size_t)gridDim.x * blockDim.x;
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  long long acc = 0;
  for (; i + (UNROLL - 1) * stride < n16; i += UNROLL * stride) {
    int4 v[UNROLL];
#pragma unroll
    for (int u = 0; u < UNROLL; u++) v[u] = __ldcs(in + i + u * stride);
#pragma unroll
    for (int u = 0; u < UNROLL; u++) acc += v[u].x + v[u].y + v[u].z + v[u].w;
  }
  for (; i < n16; i += stride) { int4 v = in[i]; acc += v.x + v.y + v.z + v.w; }
  if (acc == 0x123456789LL) atomicAdd(out, 1ULL);
}

// ring of `stages` stages of `stage_bytes`, each filled by `ncopies` bulk copies (separate streams like columns)
__global__ void bulk_kernel(const char *__restrict__ in, size_t bytes, int stage_bytes, int stages, int ncopies, int hint, int consume,
                            unsigned long long *out) {
  extern __shared__ __align__(128) unsigned char smem[];
  uint64_t *full = (uint64_t *)(smem + (size_t)stages * stage_bytes);
  uint64_t *empty = full + stages;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int ncons = blockDim.x - 32;
  if (tid == 0) {
    for (int s = 0; s < stages; s++) { mbar_init(&full[s], 1); mbar_init(&empty[s], ncons / 32); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  size_t ntiles = bytes / stage_bytes;
  size_t stream_bytes = bytes / ncopies;           // stream c covers [c*stream_bytes, (c+1)*stream_bytes)
  int chunk = stage_bytes / ncopies;
  if (warp == 0) {
    if (lane == 0) {
      uint64_t pol;
      asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
      int st = 0; uint32_t ph = 0;
      for (size_t t = blockIdx.x; t < ntiles; t += gridDim.x) {
        mbar_wait(&empty[st], ph ^ 1);
        mbar_expect_tx(&full[st], (uint32_t)stage_bytes);
        for (int c = 0; c < ncopies; c++) {
          const char *src = in + (size_t)c * stream_bytes + t * chunk;
          if (hint) bulk_g2s_hint(smem + (size_t)st * stage_bytes + c * chunk, src, chunk, &full[st], pol);
          else bulk_g2s(smem + (size_t)st * stage_bytes + c * chunk, src, chunk, &full[st]);
        }
        if (++st == stages) { st = 0; ph ^= 1; }
      }
    }
    return;
  }
  const int ctid = tid - 32;
  long long acc = 0;
  int st = 0; uint32_t ph = 0;
  for (size_t t = blockIdx.x; t < ntiles; t += gridDim.x) {
    mbar_wait(&full[st], ph);
    if (consume) {
      const int4 *p = (const int4 *)(smem + (size_t)st * stage_bytes);
      for (int i = ctid; i < stage_bytes / 16; i += ncons) { int4 v = p[i]; acc += v.x + v.y + v.z + v.w; }
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(&empty[st]);
    if (++st == stages) { st = 0; ph ^= 1; }
  }
  if (acc == 0x123456789LL) atomicAdd(out, 1ULL);
}


// ---- sparse: stream a 4-byte column, late-fetch an 8-byte column for the rows that pass ----
__host__ __device__ __forceinline__ uint32_t row_hash(uint32_t x) {
  x ^= x >> 16; x *= 0x7feb352dU; x ^= x >> 15; x *= 0x846ca68bU; x ^= x >> 16;
  return x;
}
__device__ __forceinline__ void cp_async8(void *dst, const void *src) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(smem_u32(dst)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// Stage = [lead: tile_rows x 4 B][fetch slots: tile_rows x 8 B][pass masks: NC x 4 B].  Thread ctid owns rows
// ctid + k * NC of every tile: it fetches them, and DIST iterations later (cp.async.wait_group DIST) folds them.
template <int NC, int R, int DIST>
__global__ void __launch_bounds__(NC + 32, 1) sparse_kernel(const int32_t *__restrict__ a, const long long *__restrict__ b, size_t ntiles,
                                                           uint32_t thresh, int stages, unsigned long long *out) {
  extern __shared__ __align__(128) unsigned char smem[];
  constexpr int TR = NC * R, SB = TR * 12 + NC * 4;
  uint64_t *full = (uint64_t *)(smem + (size_t)stages * SB);
  uint64_t *empty = full + stages;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  if (tid == 0) {
    for (int s = 0; s < stages; s++) { mbar_init(&full[s], 1); mbar_init(&empty[s], NC / 32); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  if (warp == 0) {
    if (lane == 0) {
      uint64_t pol;
      asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
      int st = 0; uint32_t ph = 0;
      for (size_t t = blockIdx.x; t < ntiles; t += gridDim.x) {
        mbar_wait(&empty[st], ph ^ 1);
        mbar_expect_tx(&full[st], TR * 4);
        bulk_g2s_hint(smem + (size_t)st * SB, a + t * TR, TR * 4, &full[st], pol);
        if (++st == stages) { st = 0; ph ^= 1; }
      }
    }
    return;
  }
  const int ctid = tid - 32;
  long long acc = 0;
  int st = 0, it = 0;
  uint32_t ph = 0;
  auto fold = [&](int it_old) {
    const int s = it_old % stages;
    unsigned char *buf = smem + (size_t)s * SB;
    const unsigned m = ((const unsigned *)(buf + TR * 12))[ctid];
#pragma unroll
    for (int k = 0; k < R; k++)
      if ((m >> k) & 1) acc += ((const long long *)(buf + TR * 4))[ctid + k * NC];
    __syncwarp();
    if (lane == 0) mbar_arrive(&empty[s]);
  };
  for (size_t t = blockIdx.x; t < ntiles; t += gridDim.x, it++) {
    unsigned char *buf = smem + (size_t)st * SB;
    mbar_wait(&full[st], ph);
    unsigned m = 0;
#pragma unroll
    for (int k = 0; k < R; k++) {
      const int r = ctid + k * NC;
      const size_t row = t * TR + r;
      acc += ((const int32_t *)buf)[r];
      if (row_hash((uint32_t)row) < thresh) {
        m |= 1u << k;
        cp_async8(buf + TR * 4 + (size_t)r * 8, b + row);
      }
    }
    ((unsigned *)(buf + TR * 12))[ctid] = m;
    cp_async_commit();
    if (it >= DIST) {
      cp_async_wait<DIST>();
      fold(it - DIST);
    }
    if (++st == stages) { st = 0; ph ^= 1; }
  }
  cp_async_wait<0>();
  for (int i = it > DIST ? it - DIST : 0; i < it; i++) fold(i);
  if (acc == 0x123456789LL) atomicAdd(out, 1ULL);
}

template <int NC, int R, int DIST>
static void sparse_run(const int32_t *a, const long long *b, size_t rows, int stages, int sms, unsigned long long *out, cudaEvent_t e0,
                       cudaEvent_t e1) {
  constexpr int TR = NC * R, SB = TR * 12 + NC * 4;
  const size_t smem = (size_t)stages * SB + 16 * stages;
  CK(cudaFuncSetAttribute(sparse_kernel<NC, R, DIST>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const size_t ntiles = rows / TR;
  const double ps[] = {0.0, 1.0, 0.47, 0.27, 0.145, 0.04, 0.0185};
  double t0 = 0;
  for (double p : ps) {
    const uint32_t thresh = p >= 1.0 ? 0xffffffffu : (uint32_t)(p * 4294967296.0);
    // exact sector counts of the fetched column (8-byte rows) over the rows the kernel visits
    size_t n32 = 0, n64 = 0, nrow = 0;
    long long last32 = -1, last64 = -1;
    for (size_t r = 0; r < ntiles * TR; r++) {
      if (!(row_hash((uint32_t)r) < thresh)) continue;
      nrow++;
      if ((long long)(r / 4) != last32) { n32++; last32 = (long long)(r / 4); }
      if ((long long)(r / 8) != last64) { n64++; last64 = (long long)(r / 8); }
    }
    auto launch = [&] { sparse_kernel<NC, R, DIST><<<sms, NC + 32, smem>>>(a, b, ntiles, thresh, stages, out); };
    for (int w = 0; w < 2; w++) launch();
    CK(cudaDeviceSynchronize());
    float best = 1e9;
    for (int r = 0; r < 5; r++) {
      CK(cudaEventRecord(e0)); launch(); CK(cudaEventRecord(e1)); CK(cudaEventSynchronize(e1));
      float ms; CK(cudaEventElapsedTime(&ms, e0, e1)); best = ms < best ? ms : best;
    }
    CK(cudaGetLastError());
    const double lead = (double)ntiles * TR * 4, b32 = lead + n32 * 32.0, b64 = lead + n64 * 64.0;
    if (p == 0.0) t0 = best;
    printf("sparse tile=%d stages=%d dist=%d p=%.4f  %7.3f ms  fetch-only %6.3f ms  rows fetched %.4f  bytes/row 32B %5.2f 64B %5.2f  "
           "GB/s 32B %6.0f 64B %6.0f\n",
           TR, stages, DIST, p, best, best - t0, (double)nrow / (ntiles * TR), b32 / (ntiles * TR), b64 / (ntiles * TR), b32 / best / 1e6,
           b64 / best / 1e6);
  }
}

int main(int argc, char **argv) {
  if (argc > 1 && !strcmp(argv[1], "sparse")) {
    const size_t rows = (size_t)1 << 28;   // 1 GiB of 4-byte lead values, 2 GiB of 8-byte fetched values
    int32_t *a; long long *b; unsigned long long *out;
    CK(cudaMalloc(&a, rows * 4)); CK(cudaMalloc(&b, rows * 8)); CK(cudaMalloc(&out, 8));
    CK(cudaMemset(a, 1, rows * 4)); CK(cudaMemset(b, 1, rows * 8)); CK(cudaMemset(out, 0, 8));
    int sms; CK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, 0));
    cudaEvent_t e0, e1; CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1));
    sparse_run<256, 2, 12>(a, b, rows, 16, sms, out, e0, e1);
    sparse_run<256, 4, 6>(a, b, rows, 8, sms, out, e0, e1);
    sparse_run<256, 2, 20>(a, b, rows, 24, sms, out, e0, e1);
    return 0;
  }
  size_t bytes = (size_t)(argc > 1 ? atof(argv[1]) : 8.0) * (1ull << 30);
  char *buf; unsigned long long *out;
  CK(cudaMalloc(&buf, bytes)); CK(cudaMalloc(&out, 8));
  CK(cudaMemset(buf, 1, bytes)); CK(cudaMemset(out, 0, 8));
  int sms; CK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, 0));
  cudaEvent_t e0, e1; CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1));
  auto time_it = [&](const char *name, auto launch) {
    for (int w = 0; w < 2; w++) launch();
    CK(cudaDeviceSynchronize());
    float best = 1e9, sum = 0;
    for (int r = 0; r < 5; r++) {
      CK(cudaEventRecord(e0)); launch(); CK(cudaEventRecord(e1)); CK(cudaEventSynchronize(e1));
      float ms; CK(cudaEventElapsedTime(&ms, e0, e1)); best = ms < best ? ms : best; sum += ms;
    }
    CK(cudaGetLastError());
    printf("%-58s best %7.3f ms  %7.1f GB/s   mean %7.1f GB/s\n", name, best, bytes / best / 1e6, bytes / (sum / 5) / 1e6);
  };
  char name[128];
  size_t n16 = bytes / 16;
  for (int bps : {4, 8, 16}) {
    snprintf(name, sizeof name, "ldg128 unroll4 blocks/SM=%d", bps);
    time_it(name, [&] { ldg_kernel<4><<<sms * bps, 256>>>((const int4 *)buf, n16, out); });
    snprintf(name, sizeof name, "ldg128 unroll8 blocks/SM=%d", bps);
    time_it(name, [&] { ldg_kernel<8><<<sms * bps, 256>>>((const int4 *)buf, n16, out); });
  }
  CK(cudaFuncSetAttribute(bulk_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
  struct Cfg { int stage_kb, stages, ncopies, hint, consume, threads, ctas_per_sm; };
  Cfg cfgs[] = {
      {28, 7, 4, 1, 1, 544, 1}, {28, 7, 4, 0, 1, 544, 1}, {28, 7, 4, 0, 0, 544, 1}, {28, 7, 1, 0, 1, 544, 1},
      {32, 6, 1, 0, 1, 288, 1}, {32, 6, 4, 0, 1, 288, 1}, {16, 12, 4, 0, 1, 288, 1}, {8, 24, 4, 0, 1, 288, 1},
      {64, 3, 4, 0, 1, 288, 1}, {16, 6, 4, 0, 1, 160, 2}, {16, 6, 1, 0, 1, 160, 2}, {8, 6, 4, 0, 1, 160, 4},
      {16, 3, 4, 0, 1, 160, 4}, {32, 3, 4, 0, 1, 288, 2}, {28, 7, 4, 0, 1, 160, 1}, {28, 7, 4, 0, 1, 96, 1},
  };
  for (auto &c : cfgs) {
    int stage_bytes = c.stage_kb * 1024;
    size_t smem = (size_t)stage_bytes * c.stages + 16 * c.stages + 64;
    snprintf(name, sizeof name, "bulk stage=%dKB x%d copies/stage=%d hint=%d consume=%d thr=%d cta/SM=%d", c.stage_kb, c.stages, c.ncopies,
             c.hint, c.consume, c.threads, c.ctas_per_sm);
    time_it(name, [&] { bulk_kernel<<<sms * c.ctas_per_sm, c.threads, smem>>>(buf, bytes, stage_bytes, c.stages, c.ncopies, c.hint, c.consume, out); });
  }
  return 0;
}
