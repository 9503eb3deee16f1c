// Declarations shared by the device code of libvdl_cuda, written so that NVRTC can compile them too (the fused scan is
// specialised at run time: vdl_fused_jit.cu): no host headers, fixed-width types spelled out under __CUDACC_RTC__.
#pragma once

#ifdef __CUDACC_RTC__
typedef signed char int8_t;
typedef short int16_t;
typedef int int32_t;
typedef long long int64_t;
typedef unsigned char uint8_t;
typedef unsigned short uint16_t;
typedef unsigned int uint32_t;
typedef unsigned long long uint64_t;
typedef unsigned long size_t;
typedef unsigned long uintptr_t;
#define INT32_MAX 2147483647
#define INT32_MIN (-2147483647 - 1)
#define INT64_MAX 9223372036854775807LL
#define INT64_MIN (-9223372036854775807LL - 1)
#else
#include <stdint.h>
#endif

#include "vdl_cuda.h"

typedef int64_t i64;
typedef uint64_t u64;

// Peer-memory exchange of the partial tables (one buffer per rank, addressable by all ranks):
//   data  [2 (epoch parity)][world][stride] int64   rank r's table of the step lands in slot [parity][r] of EVERY buffer
//   flags [2][world] uint64                         epoch of the last step whose table rank r has fully stored
struct XDesc {
  int32_t rank, world;
  u64 epoch;                      // this step's number (1, 2, ...); parity double-buffers against a rank running ahead
  u64 timeout_ns;                 // give up waiting for a peer after this long: error flag, never a hang
  i64 stride;                     // int64 per table
  i64 *peer[VDL_MAX_RANKS];       // base of every rank's buffer as seen from this GPU
};

#define K_MAX_ACC 10              // table rows of SUM / MIN / MAX accumulators (the scan's, with count and first row)

// Merge of per-rank partial tables of [rows][domain] int64 into one dense vector per fold output (finalize_block).  A
// table holds accumulator rows (cnt_idx: row count, first_idx: smallest global row id of the key) and FoldChoose rows:
//   fused scan: [nacc accumulators][nchoose FoldChoose values]
//   probe:      [nfolds][count][first row] with nacc = 0, so that a FoldChoose output's row nacc + out_idx is its fold's
struct FinDesc {
  const i64 *parts;              // nranks tables back to back, each part_stride int64
  i64 part_stride, domain;
  int32_t nranks, nacc, nchoose, cnt_idx, first_idx, nout;
  int32_t acc_op[K_MAX_ACC];
  int32_t out_kind[VDL_MAX_AGGS], out_idx[VDL_MAX_AGGS];   // kind 0: accumulator row out_idx, 1: FoldChoose row nacc + out_idx
  i64 *out[VDL_MAX_AGGS];
  int32_t npost, pad;
  vdl_post_op post[VDL_MAX_POSTS];
  i64 *post_out[VDL_MAX_POSTS];
  i64 *ngroups;                  // [0] number of groups, [1] snapshot of the context's error counter, [2] (host mirror only) seq
  i64 seq;                       // number of this finalize: the last word the kernel publishes to the host mirror
  const int *errflag;
  i64 *hmirror;                  // mapped pinned host copy of the whole result buffer (same layout as out[0]...), or null
  i64 *reset_table;              // this rank's partial table, re-initialised for the next launch after the merge, or null
};


#ifdef __CUDACC__
// system-scope release / acquire and a wall clock for the peer-memory exchange (exchange_block)
__device__ __forceinline__ void st_release_sys(u64 *p, u64 v) { asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory"); }
__device__ __forceinline__ u64 ld_acquire_sys(const u64 *p) {
  u64 v;
  asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ u64 global_timer_ns() {
  u64 t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
// Elementwise op semantics (Vdl.hs:136-157, 209-231).  Comparisons / logicals give 0/1; BitShift: +k arithmetic right,
// -k left (Vlite.hs:205-208); Divide truncates, x/0 := 0, INT64_MIN/-1 wraps; Modulo is the C remainder, x%0 := 0.
__device__ __forceinline__ i64 binop_apply(int op, i64 a, i64 b) {
  switch (op) {
    case VDL_LOGICAL_AND: return (a != 0) && (b != 0);
    case VDL_LOGICAL_OR: return (a != 0) || (b != 0);
    case VDL_BITWISE_AND: return a & b;
    case VDL_BITWISE_OR: return a | b;
    case VDL_BITSHIFT:
      if (b >= 0) return b >= 64 ? (a < 0 ? -1 : 0) : (a >> b);
      return b <= -64 ? 0 : (i64)((u64)a << (-b));
    case VDL_EQUALS: return a == b;
    case VDL_ADD: return (i64)((u64)a + (u64)b);
    case VDL_SUBTRACT: return (i64)((u64)a - (u64)b);
    case VDL_GREATER: return a > b;
    case VDL_MULTIPLY: return (i64)((u64)a * (u64)b);
    case VDL_DIVIDE:
      if (b == 0) return 0;
      if (b == -1) return (i64)(0 - (u64)a);
      return a / b;
    case VDL_MODULO:
      if (b == 0 || b == -1) return 0;
      return a % b;
  }
  return 0;
}

// identity and combine of the SUM / MIN / MAX accumulators (op = VDL_FOLD_SUM / MIN / MAX)
__device__ __forceinline__ i64 acc_identity(int op) { return op == 0 ? 0 : (op == 1 ? INT64_MAX : INT64_MIN); }
__device__ __forceinline__ i64 acc_combine(int op, i64 a, i64 v) {
  return op == 0 ? (i64)((u64)a + (u64)v) : (op == 1 ? (v < a ? v : a) : (v > a ? v : a));
}

// Store this rank's table into every rank's exchange buffer, publish the epoch, wait for every rank's epoch.
// Returns the [world][stride] block of this rank's own buffer that now holds all tables of the step.  One thread block
// of NT threads (tid 0..NT-1; the barrier is the named barrier 2 so that the scan kernel's consumer warps can run it
// without the producer warp).
template <int NT>
__device__ __forceinline__ const i64 *exchange_block(const XDesc &x, const i64 *table, int *errflag, int tid) {
  auto bar = []() { asm volatile("bar.sync 2, %0;" ::"n"(NT) : "memory"); };
  const int par = (int)(x.epoch & 1);
  const size_t slot = ((size_t)par * x.world + x.rank) * x.stride, flags = (size_t)2 * x.world * x.stride;
  for (int p = 0; p < x.world; p++) {                // NVLink stores (plain st.global to the peer mapping)
    i64 *dst = x.peer[p] + slot;
    for (i64 i = tid; i < x.stride; i += NT) dst[i] = __ldcg(&table[i]);
  }
  __threadfence_system();
  bar();
  if (tid < x.world) {
    st_release_sys((u64 *)(x.peer[tid] + flags) + (size_t)par * x.world + x.rank, x.epoch);
    const u64 *mine = (const u64 *)(x.peer[x.rank] + flags) + (size_t)par * x.world + tid;
    const u64 t0 = global_timer_ns();
    while (ld_acquire_sys(mine) < x.epoch) {
      if (global_timer_ns() - t0 > x.timeout_ns) { atomicAdd(errflag, 1 << 20); break; }   // a peer never arrived: fail, do not hang
      __nanosleep(64);
    }
  }
  bar();
  return x.peer[x.rank] + (size_t)par * x.world * x.stride;
}

// FoldChoose value of output o at key k: the one the tables carry, from the rank `best` that holds the key's first row
// (global row id `first`)
struct ChooseFromTable {
  __device__ __forceinline__ i64 operator()(const FinDesc &f, const i64 *parts, int o, i64 k, int best, i64 first) const {
    return __ldcg(&parts[(size_t)best * f.part_stride + (size_t)(f.nacc + f.out_idx[o]) * f.domain + k]);
  }
};

// Merge the per-rank tables, drop empty keys, emit one dense vector per fold in ascending key order, run the post
// ops, optionally re-initialise this rank's table.  One thread block of NT threads, named barrier 2 (as exchange_block).
template <int NT, class Choose = ChooseFromTable>
__device__ __forceinline__ void finalize_block(const FinDesc &f, const i64 *parts, int nranks, int tid, int *warp_cnt, i64 *running,
                                               Choose choose = Choose()) {
  constexpr int NWF = NT / 32;
  auto bar = []() { asm volatile("bar.sync 2, %0;" ::"n"(NT) : "memory"); };
  const int lane = tid & 31, warp = tid >> 5;
  // out[] / post_out[] / ngroups live in one device buffer that starts at out[0]; hmirror has the same layout
  auto mirror = [&](i64 *dev) { return f.hmirror + (dev - f.out[0]); };
  if (tid == 0) *running = 0;
  bar();
  for (i64 base = 0; base < f.domain; base += NT) {
    i64 k = base + tid;
    i64 cnt = 0;
    if (k < f.domain)
      for (int r = 0; r < nranks; r++) cnt += __ldcg(&parts[(size_t)r * f.part_stride + (size_t)f.cnt_idx * f.domain + k]);
    bool exists = cnt > 0;
    unsigned m = __ballot_sync(0xffffffffu, exists);
    if (lane == 0) warp_cnt[warp] = __popc(m);
    bar();
    int before = 0, total = 0;
    for (int w = 0; w < NWF; w++) {
      if (w < warp) before += warp_cnt[w];
      total += warp_cnt[w];
    }
    if (exists) {
      i64 pos = *running + before + __popc(m & ((1u << lane) - 1));
      int best = 0;   // rank holding the first row of this key
      i64 bf = INT64_MAX;
      if (f.nchoose > 0) {
        for (int r = 0; r < nranks; r++) {
          i64 fr = __ldcg(&parts[(size_t)r * f.part_stride + (size_t)f.first_idx * f.domain + k]);
          if (fr < bf) { bf = fr; best = r; }
        }
      }
      i64 ov[VDL_MAX_AGGS], pv[VDL_MAX_POSTS];
      for (int o = 0; o < f.nout; o++) {
        i64 v;
        if (f.out_kind[o] == 1) {
          v = choose(f, parts, o, k, best, bf);
        } else {
          int j = f.out_idx[o], op = f.acc_op[j];
          v = acc_identity(op);
          for (int r = 0; r < nranks; r++) v = acc_combine(op, v, __ldcg(&parts[(size_t)r * f.part_stride + (size_t)j * f.domain + k]));
        }
        f.out[o][pos] = v;
        if (f.hmirror) mirror(f.out[o])[pos] = v;
        ov[o] = v;
      }
      // elementwise epilogue over the fold results (AVG's Divide, ...)
      for (int q = 0; q < f.npost; q++) {
        const vdl_post_op &P = f.post[q];
        i64 a = P.a_kind == VDL_POST_CONST ? P.a : (P.a_kind == VDL_POST_FOLD ? ov[P.a] : pv[P.a]);
        i64 b = P.b_kind == VDL_POST_CONST ? P.b : (P.b_kind == VDL_POST_FOLD ? ov[P.b] : pv[P.b]);
        pv[q] = binop_apply(P.op, a, b);
        f.post_out[q][pos] = pv[q];
        if (f.hmirror) mirror(f.post_out[q])[pos] = pv[q];
      }
    }
    bar();
    if (tid == 0) *running += total;
    bar();
  }
  if (tid == 0) {
    const i64 ng = *running, err = *f.errflag;
    f.ngroups[0] = ng; f.ngroups[1] = err;
    if (f.hmirror) {
      mirror(f.ngroups)[0] = ng; mirror(f.ngroups)[1] = err;
      __threadfence_system();                      // every result store of this block (barriers above) before the publication
      ((volatile i64 *)mirror(f.ngroups))[2] = f.seq;
    }
  }
  if (f.reset_table) {      // every thread has read what it needed (barriers above): identity-initialise for the next launch
    const i64 n = (i64)(f.nacc + f.nchoose) * f.domain;
    for (i64 i = tid; i < n; i += NT) {
      int j = (int)(i / f.domain);
      f.reset_table[i] = j < f.nacc ? acc_identity(f.acc_op[j]) : 0;
    }
  }
}
#endif
