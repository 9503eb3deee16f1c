// Device code of the fused FK-join probe (see vdl_probe.cu for what it replaces in the emitted graph and for the host
// side): the descriptor and probe_body, the tile loop of both probe kernels.  The precompiled interpreter probe_kernel
// (vdl_probe.cu) and the kernel specialised at run time to one descriptor (vdl_probe_jit, printed by probe_jit_source in
// vdl_probe.cu) instantiate probe_body with their own evaluator.  NVRTC compiles this header as well, so it must stay free
// of host headers.
#pragma once

#include "vdl_device.cuh"

#ifndef P_THREADS
#define P_THREADS 128
#endif
#define P_TILE (P_THREADS * 32)   // one bitmap word per thread (emit mode)
#ifndef P_BLOCKS
#define P_BLOCKS 12   // resident blocks per SM: 40 registers per thread, 12 x 17.9 KB of shared memory (measured: 8 blocks x 64 regs +15 %, 10 x 48 +3 %, 16 = 12 by shared memory)
#endif
#define P_MAX_DEPTH 6
#define P_SMEM_TABLE_BYTES (40 * 1024)

struct PLeaf { const void *ptr; i64 len; int32_t w4, parent; };
struct PTerm { int32_t leaf, shr; i64 a, b; };             // leaf -1: constant a; -2: global row id
struct PPred { int32_t kind, cmp; PTerm t, u; i64 lo; u64 span; int32_t nmore, pad; i64 lo_more[VDL_MAX_MORE_RANGES]; u64 span_more[VDL_MAX_MORE_RANGES]; };
struct PProd { int32_t nfac, pad; PTerm f[VDL_MAX_FACTORS]; };

struct PDesc {
  i64 rows, row_base, key_mask, domain, ntiles;
  int32_t nleaves, npreds, nkeys, nfolds, nemits, smem_table, pad0, pad1;
  PLeaf leaf[VDL_MAX_LEAVES];
  PPred pred[VDL_MAX_PROBE_PREDS];
  PTerm key[VDL_MAX_KEYS];
  int32_t key_shl[VDL_MAX_KEYS];
  int32_t fold_op[VDL_MAX_AGGS];
  PProd fold[VDL_MAX_AGGS];
  PProd emit[VDL_MAX_EMITS];
  int32_t nind, pad2;
  PPred ind[VDL_MAX_INDICATORS];
  // fact-table columns the predicate stages read for (nearly) every row: the tile's share of them (or that of the tile
  // `pf_dist` tickets ahead) is pulled into L2 at the start, so the later stages' dependent loads pay L2, not DRAM, latency
  int32_t npf, pf_dist;
  const unsigned char *pf_ptr[VDL_MAX_LEAVES];
  int32_t pf_shift[VDL_MAX_LEAVES];  // log2 bytes per value
  i64 *table;                       // fold mode: [nfolds + 2][domain]: fold accumulators, row count, first row
  i64 *emit_out[VDL_MAX_EMITS];     // emit mode: dense output vectors (capacity rows)
  unsigned long long *tile_state;   // emit mode look-back: (status << 62) | count; status 1 = tile aggregate, 2 = inclusive prefix
  unsigned int *ticket;
  i64 *total;                       // emit mode: number of surviving rows
  int *errflag;
};

// Identity of table_update's op on every fold op code: FoldChoose and COUNT rows start at 0.  (acc_identity, which the
// merge uses, is defined on SUM / MIN / MAX only.)
__device__ __forceinline__ i64 p_identity(int op) { return op == VDL_FOLD_MIN ? INT64_MAX : (op == VDL_FOLD_MAX ? INT64_MIN : 0); }

// Identity of row j of the [nfolds + 2][domain] table: the folds' rows, then the row count and the first row.
__device__ __forceinline__ i64 table_identity(const PDesc &d, int nfolds, int j) {
  return j < nfolds ? p_identity(d.fold_op[j]) : (j == nfolds ? 0 : INT64_MAX);
}

__device__ __forceinline__ void table_update(int op, i64 *p, i64 v) {
  if (op == VDL_FOLD_MIN) atomicMin((long long *)p, (long long)v);
  else if (op == VDL_FOLD_MAX) atomicMax((long long *)p, (long long)v);
  else atomicAdd((unsigned long long *)p, (unsigned long long)v);
}

// ---- staged evaluation: the tile loop of both probe kernels -----------------------------------------------------------
// A tile goes through the predicates one STAGE at a time; after every stage the surviving rows are compacted into a
// shared-memory queue, so the next stage runs with full warps on survivors only and its lookups are independent loads of
// different rows (memory-level parallelism instead of divergent lanes waiting on a long dependent chain).
//
// The evaluator Eval supplies what differs between the interpreter and a kernel specialised to one descriptor:
//   SUB                                 rows per thread and round of a stage
//   npreds(d), nfolds(d), nemits(d)     the counts (literals when specialised: fold-or-emit is static)
//   stages(d, n_in, run_stage)          calls run_stage(q) for the stages in order: the interpreter loops over d.npreds
//                                       and stops when no row survives; a specialised kernel calls run_stage(0),
//                                       run_stage(1), ..., so that each stage is compiled for its own q
//   stage(d, q)                         the set-up of stage q, once per tile
//   round(d, q, st, base, r, f, ok)     f[k]: does tile row r[k] pass stage q?  r[k] < 0: an empty slot, f[k] false
//   fold_row(d, row, tab, ok)           fold a surviving row into the table `tab`
//   emit_row(d, row, at, ok)            write a surviving row's emitted expressions to output row `at`
// ok is cleared where a lookup index or group key is out of range; a tile with such a row raises the error flag.  tid is
// the kernel's threadIdx.x, read there so that the compiler knows it from __launch_bounds__ to be below P_THREADS.
template <class Eval>
__device__ __forceinline__ void probe_body(const PDesc &d, const int tid) {
  constexpr int SUB = Eval::SUB;
  extern __shared__ __align__(16) unsigned char psm[];
  __shared__ uint16_t queue[2][P_TILE];
  __shared__ int s_cnt[3];                        // survivors appended by stage q: s_cnt[(q + 1) % 3]
  __shared__ unsigned int s_bits[P_TILE / 32];    // emit mode: the tile's survivors as a bitmap, to put them back in row order
  __shared__ int wsum[P_THREADS / 32];
  __shared__ i64 s_off;
  __shared__ unsigned int s_tile;
  const int lane = tid & 31, warp = tid >> 5;
  const int npreds = Eval::npreds(d), nfolds = Eval::nfolds(d);
  const bool folding = Eval::nemits(d) == 0;
  const int nacc = nfolds + 2;
  i64 *stab = (i64 *)psm;                         // [nacc][domain] when smem_table
  if (folding && d.smem_table) {
    for (i64 i = tid; i < (i64)nacc * d.domain; i += P_THREADS) stab[i] = table_identity(d, nfolds, (int)(i / d.domain));
  }
  __syncthreads();
  i64 *tab = (folding && d.smem_table) ? stab : d.table;

  for (;;) {
    if (tid == 0) { s_tile = atomicAdd(d.ticket, 1u); s_cnt[1] = 0; }
    __syncthreads();
    const i64 tile = s_tile;
    if (tile >= d.ntiles) break;
    const i64 base = tile * P_TILE;
    if (d.npf) {
      const i64 b2 = base + (i64)d.pf_dist * P_TILE;
      const i64 n2 = min((i64)P_TILE, d.rows - b2);
      for (int c = 0; c < d.npf && n2 > 0; c++) {
        const unsigned char *p0 = d.pf_ptr[c] + (b2 << d.pf_shift[c]);
        const i64 bytes = n2 << d.pf_shift[c];
        for (i64 o = (i64)tid * 128; o < bytes; o += P_THREADS * 128) asm volatile("prefetch.global.L2 [%0];" ::"l"(p0 + o));
      }
    }
    bool ok = true;
    int n_in = (int)min((i64)P_TILE, d.rows - base);      // stage input: all rows of the tile, then the previous stage's survivors
    int cur = 0;
    auto run_stage = [&](const int q) {
      const auto st = Eval::stage(d, q);
      for (int j0 = 0; j0 < n_in; j0 += SUB * P_THREADS) {
        bool f[SUB];
        int r[SUB];
#pragma unroll
        for (int k = 0; k < SUB; k++) {
          const int j = j0 + k * P_THREADS + tid;
          r[k] = j < n_in ? (q == 0 ? j : (int)queue[cur][j]) : -1;
        }
        Eval::round(d, q, st, base, r, f, ok);
        // append this round's survivors to the next stage's queue.  Queue order is irrelevant to a stage (and to a
        // fold); emit mode restores row order once, at the end.  One shared atomic per warp and round, no barrier.
        unsigned m[SUB];
        int wtotal = 0;
#pragma unroll
        for (int k = 0; k < SUB; k++) { m[k] = __ballot_sync(0xffffffffu, f[k]); wtotal += __popc(m[k]); }
        if (wtotal) {
          int at = 0;
          if (lane == 0) at = atomicAdd(&s_cnt[(q + 1) % 3], wtotal);
          at = __shfl_sync(0xffffffffu, at, 0);
#pragma unroll
          for (int k = 0; k < SUB; k++) {
            if (f[k]) queue[cur ^ 1][at + __popc(m[k] & ((1u << lane) - 1))] = (uint16_t)r[k];
            at += __popc(m[k]);
          }
        }
      }
      // the counter two stages ahead is idle: every thread read it (as its n_in) before the previous stage's barrier
      if (tid == 0) s_cnt[(q + 2) % 3] = 0;
      __syncthreads();
      n_in = s_cnt[(q + 1) % 3];
      cur ^= 1;
    };
    Eval::stages(d, n_in, run_stage);
    const bool implicit = npreds == 0;              // no predicate at all: every row of the tile survives
    // ---- survivors: fold into the table, or emit in order
    if (folding) {
      for (int j = tid; j < n_in; j += P_THREADS) Eval::fold_row(d, base + (implicit ? j : (int)queue[cur][j]), tab, ok);
    } else {
      if (!implicit) {
        // survivors back into row order: bitmap of the tile, one 32-row word per thread, block scan of the word counts
        static_assert(P_TILE / 32 == P_THREADS, "one bitmap word per thread");
        s_bits[tid] = 0;
        __syncthreads();
        for (int j = tid; j < n_in; j += P_THREADS) { const unsigned rr = queue[cur][j]; atomicOr(&s_bits[rr >> 5], 1u << (rr & 31)); }
        __syncthreads();
        unsigned w = s_bits[tid];
        const int c = __popc(w);
        int incl = c;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { int t = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += t; }
        if (lane == 31) wsum[warp] = incl;
        __syncthreads();
        int at = incl - c;
        for (int ww = 0; ww < warp; ww++) at += wsum[ww];
        while (w) { const int b = __ffs(w) - 1; w &= w - 1; queue[cur ^ 1][at++] = (uint16_t)(tid * 32 + b); }
        cur ^= 1;
        __syncthreads();
      }
      // tile offset by decoupled look-back over the tiles before this one
      if (tid == 0) {
        const unsigned long long T = (unsigned long long)n_in;
        i64 excl = 0;
        if (tile == 0) {
          atomicExch(d.tile_state, (2ull << 62) | T);
        } else {
          atomicExch(d.tile_state + tile, (1ull << 62) | T);
          for (i64 j = tile - 1;; j--) {
            unsigned long long st;
            do { st = *((volatile unsigned long long *)(d.tile_state + j)); } while ((st >> 62) == 0);
            excl += (i64)(st & ((1ull << 62) - 1));
            if ((st >> 62) == 2) break;
          }
          atomicExch(d.tile_state + tile, (2ull << 62) | (unsigned long long)(excl + (i64)T));
        }
        s_off = excl;
        if (tile == d.ntiles - 1) *d.total = excl + (i64)T;
      }
      __syncthreads();
      const i64 off = s_off;
      for (int j = tid; j < n_in; j += P_THREADS) Eval::emit_row(d, base + (implicit ? j : (int)queue[cur][j]), off + j, ok);
    }
    if (!ok) atomicAdd(d.errflag, 1);
    __syncthreads();
  }
  if (folding && d.smem_table) {
    __syncthreads();
    for (i64 i = tid; i < (i64)nacc * d.domain; i += P_THREADS) {
      int j = (int)(i / d.domain);
      const i64 v = stab[i];
      if (j < nfolds) { if (v != p_identity(d.fold_op[j])) table_update(d.fold_op[j], d.table + i, v); }
      else if (j == nfolds) { if (v) atomicAdd((unsigned long long *)(d.table + i), (unsigned long long)v); }
      else if (v != INT64_MAX) atomicMin((long long *)(d.table + i), (long long)v);
    }
  }
}
