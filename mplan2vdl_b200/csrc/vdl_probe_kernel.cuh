// Descriptor structures of the fused FK-join probe, shared by the precompiled interpreter kernel (vdl_probe.cu) and the
// kernels specialised at run time to one descriptor (vdl_probe.cu: probe_jit_source; compiled by NVRTC, so this header
// must stay free of host headers).
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

__device__ __forceinline__ void table_update(int op, i64 *p, i64 v) {
  if (op == VDL_FOLD_MIN) atomicMin((long long *)p, (long long)v);
  else if (op == VDL_FOLD_MAX) atomicMax((long long *)p, (long long)v);
  else atomicAdd((unsigned long long *)p, (unsigned long long)v);
}
