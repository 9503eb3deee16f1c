// Device code of the fused select -> map -> fold scan (see vdl_fused.cu for what it replaces in the emitted graph and for
// the host side).  Kept in a header that NVRTC can compile as well: vdl_fused.cu generates the shape-traits class of a
// prepared descriptor at run time and instantiates fused_scan_fold_body over it (compiled by vdl_jit.cu).
#pragma once

#include "vdl_device.cuh"

#define K_MAX_CHOOSE 6

// soff / w4 are derived by the host from col: byte offset of the column inside a staged tile, 4-byte flag.
struct KAffine { int32_t col, shr; i64 a, b; int32_t soff, w4; int32_t narrow, pad; };   // narrow: host-side, see FF_NARROW
struct KPred { int32_t col, shr; i64 lo; u64 span; int32_t soff, w4; int32_t lo32; uint32_t span32; };
struct KKey { KAffine e; int32_t shl, pad; };
// op: 0 sum, 1 min, 2 max.  chain: value = value of the previous accumulator x own factors (prefix sharing:
// ep, ep*(100-d), ep*(100-d)*(100+t) evaluate each factor once).
struct KAcc { int32_t op, nfac, chain, pad; KAffine fac[VDL_MAX_FACTORS]; };

struct KDesc {
  i64 rows, row_base, key_mask, domain, ntiles;
  const void *col[VDL_MAX_COLS];
  int32_t width[VDL_MAX_COLS], soff[VDL_MAX_COLS];
  int32_t ncols, npreds, nkeys, nacc, nchoose, cnt_idx, first_idx;
  int32_t tile_rows, stages, stage_bytes, stage_tx, gmax, pad0;
  KPred pred[VDL_MAX_PREDS];
  KKey key[VDL_MAX_KEYS];
  KAcc acc[K_MAX_ACC];
  KAcc choose[K_MAX_CHOOSE];
  i64 *table;                    // [nacc + nchoose][domain]
  int *errflag;
  // Epilogue run by the LAST CTA to finish (ticket counter `done`): 0 none, 1 FoldChoose values only (the partial
  // table is then complete for an external all-gather), 2 FoldChoose + finalize + table reset (single GPU: the scan
  // is the only launch of a step), 3 the same with the peer-memory exchange of the tables before the finalize.
  unsigned int *done;
  int32_t epilogue, pad1;
};

// ------------------------------------------------------------------------------ PTX helpers
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred P1;\n"
      "LAB_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
      "@P1 bra DONE;\n"
      "bra LAB_WAIT;\n"
      "DONE:\n"
      "}" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}
// 1-D TMA bulk copy global -> shared, completion counted in bytes on an mbarrier; L2 evict-first policy
// because every byte of a scan is touched exactly once.
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar, uint64_t policy) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(smem_u32(dst)),
      "l"(src), "r"(bytes), "r"(smem_u32(bar)), "l"(policy)
      : "memory");
}
__device__ __forceinline__ uint64_t policy_evict_first() {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
  return p;
}
template <int NC>
__device__ __forceinline__ void consumer_barrier() { asm volatile("bar.sync 1, %0;" ::"n"(NC) : "memory"); }

__device__ __forceinline__ void acc_global(int op, i64 *p, i64 v) {
  if (op == 0) atomicAdd((unsigned long long *)p, (unsigned long long)v);
  else if (op == 1) atomicMin((long long *)p, (long long)v);
  else atomicMax((long long *)p, (long long)v);
}
__device__ __forceinline__ i64 warp_reduce(int op, i64 v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = acc_combine(op, v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// ---- descriptor-driven evaluation over a staged tile -------------------------------------------
// Every loop over the descriptor (predicates, key parts, accumulators, factors) is unrolled as a chain of
// nested uniform `if (I < n)` tests, so each descriptor field is a constant-bank immediate operand of the
// instruction that uses it (no loads, no dependent latency) and unused slots cost one uniform branch.
//
// SHAPES.  The same code is instantiated over a shape-traits class S.  GenericShape answers every structural
// question (how many predicates / key parts / accumulators / factors, 4- or 8-byte column, shift or not, b == 1,
// a == 0, fits int32 ...) from the descriptor at run time, so one kernel runs any plan.  A static shape
// (vdl_shapes.cuh) answers them at compile time: the uniform tests fold away and arithmetic narrows to 32 bits
// where the column statistics allow (the executor's use of the reference's bound inference, Vlite.hs:417-467),
// leaving straight-line code -- while every constant (bounds, offsets, a, b, shifts, masks) stays a run-time
// descriptor field.  The host launches a static instantiation only when the prepared descriptor satisfies every
// assumption the shape makes (shape_matches), otherwise the generic one: identical results either way.

// factor flags (what the static code may assume about a KAffine)
#define FF_W4 1        // 4-byte column (else 8-byte)
#define FF_SHR0 2      // shr == 0
#define FF_B1 4        // b == 1
#define FF_BM1 8       // b == -1
#define FF_A0 16       // a == 0
#define FF_CONST 32    // col == -1
#define FF_ROWID 64    // col == -2
#define FF_NARROW 128  // leaf and a + b*leaf fit int32 (column statistics)
// how a register-slot kernel keeps an accumulator per thread (see vdl_shapes.cuh)
#define RK_WIDE 0
#define RK_N32 1
#define RK_FIRST 2
#define RK_MADW 3

struct GenericShape {
  static constexpr bool kStatic = false;
  static constexpr int NPREDS = 0, NKEYS = 0, NACC = 0, KEY32 = 0;
  static constexpr int PRED_MODE[VDL_MAX_PREDS] = {}, PRED_SHR0[VDL_MAX_PREDS] = {};
  static constexpr int KEY_FLAGS[VDL_MAX_KEYS] = {}, KEY_SHL0[VDL_MAX_KEYS] = {};
  static constexpr int ACC_OP[K_MAX_ACC] = {}, ACC_CHAIN[K_MAX_ACC] = {}, ACC_NFAC[K_MAX_ACC] = {};
  static constexpr int FAC[K_MAX_ACC][VDL_MAX_FACTORS] = {};
  static constexpr int RS_G = 0;
  static constexpr int ACC_RK[K_MAX_ACC] = {};
};

__device__ __forceinline__ i64 tile_leaf(const KAffine &A, const unsigned char *tile, int r, i64 grow) {
  if (A.col == -2) return grow;
  i64 v = A.w4 ? (i64)((const int32_t *)(tile + A.soff))[r] : ((const i64 *)(tile + A.soff))[r];
  if (A.shr) v >>= A.shr;
  return v;
}
// a + b * leaf; col -1: the constant a; col -2: leaf = global row id
__device__ __forceinline__ i64 tile_affine(const KAffine &A, const unsigned char *tile, int r, i64 grow) {
  if (A.col == -1) return A.a;
  i64 leaf = tile_leaf(A, tile, r, grow);
  if (A.b != 1) leaf = (i64)((u64)A.b * (u64)leaf);
  return (i64)((u64)A.a + (u64)leaf);
}
// the same with the structure known at compile time; 32-bit arithmetic when FF_NARROW
template <int FL>
__device__ __forceinline__ int32_t affine32(const KAffine &A, const unsigned char *tile, int r) {
  int32_t v = ((const int32_t *)(tile + A.soff))[(FL & FF_W4) ? r : 2 * r];   // low word of an 8-byte value
  if (!(FL & FF_SHR0)) v >>= A.shr;
  if (FL & FF_BM1) v = -v;
  else if (!(FL & FF_B1)) v *= (int32_t)A.b;
  if (!(FL & FF_A0)) v += (int32_t)A.a;
  return v;
}
template <int FL>
__device__ __forceinline__ i64 affine_static(const KAffine &A, const unsigned char *tile, int r, i64 grow) {
  if constexpr (FL & FF_CONST) return A.a;
  else if constexpr (FL & FF_NARROW) return (i64)affine32<FL>(A, tile, r);
  else {
    i64 v;
    if constexpr (FL & FF_ROWID) v = grow;
    else {
      v = (FL & FF_W4) ? (i64)((const int32_t *)(tile + A.soff))[r] : ((const i64 *)(tile + A.soff))[r];
      if (!(FL & FF_SHR0)) v >>= A.shr;
    }
    if (FL & FF_BM1) v = (i64)(0 - (u64)v);
    else if (!(FL & FF_B1)) v = (i64)((u64)A.b * (u64)v);
    if (!(FL & FF_A0)) v = (i64)((u64)A.a + (u64)v);
    return v;
  }
}

template <class S, int J, int F>
__device__ __forceinline__ i64 factor_chain(const KAcc &A, i64 v, const unsigned char *tile, int r, i64 grow) {
  if constexpr (F < VDL_MAX_FACTORS) {
    if constexpr (S::kStatic) {
      if constexpr (F < S::ACC_NFAC[J]) {
        i64 x = affine_static<S::FAC[J][F]>(A.fac[F], tile, r, grow);
        v = (F == 0 && !S::ACC_CHAIN[J]) ? x : (i64)((u64)v * (u64)x);
        return factor_chain<S, J, F + 1>(A, v, tile, r, grow);
      }
    } else {
      if (F < A.nfac) {
        i64 x = tile_affine(A.fac[F], tile, r, grow);
        v = (F == 0 && !A.chain) ? x : (i64)((u64)v * (u64)x);
        return factor_chain<S, J, F + 1>(A, v, tile, r, grow);
      }
    }
  }
  return v;
}
// generic (looping) form for the rare global-atomic path
__device__ __noinline__ i64 acc_value_slow(const KDesc &d, int j, const unsigned char *tile, int r, i64 grow) {
  i64 v = 1;
  int j0 = j;
  while (d.acc[j0].chain) j0--;
  for (int q = j0; q <= j; q++)
    for (int f = 0; f < d.acc[q].nfac; f++) v = (i64)((u64)v * (u64)tile_affine(d.acc[q].fac[f], tile, r, grow));
  return v;
}

template <class S, int I, int NC, int R>
__device__ __forceinline__ void pred_chain(const KDesc &d, const unsigned char *tile, int ctid, unsigned &pass) {
  if constexpr (I < VDL_MAX_PREDS && (!S::kStatic || I < S::NPREDS)) {
    if (S::kStatic || I < d.npreds) {
      const KPred &P = d.pred[I];
      const int mode = S::kStatic ? S::PRED_MODE[I] : P.w4;
      const bool shr0 = S::kStatic ? (bool)S::PRED_SHR0[I] : (P.shr == 0);
      if (mode) {      // 32-bit compare against bounds clamped to int32 by the host: a 4-byte column (mode 1), or
                       // the low words of an 8-byte column whose values all fit int32 per its statistics (mode 2)
        const int32_t *p = (const int32_t *)(tile + P.soff);
#pragma unroll
        for (int k = 0; k < R; k++) {
          int32_t v = p[(ctid + k * NC) * mode];
          if (!shr0) v >>= P.shr;
          if ((uint32_t)v - (uint32_t)P.lo32 > P.span32) pass &= ~(1u << k);
        }
      } else {
        const i64 *p = (const i64 *)(tile + P.soff);
#pragma unroll
        for (int k = 0; k < R; k++) {
          i64 v = p[ctid + k * NC];
          if (!shr0) v >>= P.shr;
          if ((u64)v - (u64)P.lo > P.span) pass &= ~(1u << k);
        }
      }
      pred_chain<S, I + 1, NC, R>(d, tile, ctid, pass);
    }
  }
}

template <class S, int Q>
__device__ __forceinline__ i64 key_chain(const KDesc &d, i64 key, const unsigned char *tile, int r, i64 grow) {
  if constexpr (Q < VDL_MAX_KEYS && (!S::kStatic || Q < S::NKEYS)) {
    if (S::kStatic || Q < d.nkeys) {
      i64 x;
      if constexpr (S::kStatic) x = affine_static<S::KEY_FLAGS[Q]>(d.key[Q].e, tile, r, grow);
      else x = tile_affine(d.key[Q].e, tile, r, grow);
      if (!(S::kStatic && S::KEY_SHL0[Q]) && d.key[Q].shl) x = (i64)((u64)x << d.key[Q].shl);
      return key_chain<S, Q + 1>(d, key | x, tile, r, grow);
    }
  }
  return key;
}
// all key parts narrow: the whole key in 32-bit arithmetic
template <class S, int Q>
__device__ __forceinline__ int32_t key_chain32(const KDesc &d, int32_t key, const unsigned char *tile, int r) {
  if constexpr (Q < S::NKEYS) {
    int32_t x = affine32<S::KEY_FLAGS[Q]>(d.key[Q].e, tile, r);
    if (!S::KEY_SHL0[Q]) x <<= d.key[Q].shl;
    return key_chain32<S, Q + 1>(d, key | x, tile, r);
  }
  return key;
}

// lane-private read-modify-write of accumulator J and all following ones
template <class S, int J, int NC>
__device__ __forceinline__ void acc_chain(const KDesc &d, i64 *t, i64 prev, const unsigned char *tile, int r, i64 grow) {
  if constexpr (J < K_MAX_ACC && (!S::kStatic || J < S::NACC)) {
    if (S::kStatic || J < d.nacc) {
      const bool chain = S::kStatic ? (bool)S::ACC_CHAIN[J] : (bool)d.acc[J].chain;
      const int op = S::kStatic ? S::ACC_OP[J] : d.acc[J].op;
      i64 v = factor_chain<S, J, 0>(d.acc[J], chain ? prev : 1, tile, r, grow);
      t[J * NC] = acc_combine(op, t[J * NC], v);
      acc_chain<S, J + 1, NC>(d, t, v, tile, r, grow);
    }
  }
}

// ---- register slots (G > 0): per-thread accumulators of the first G keys of the CTA live in registers ----------
// All indexing below is static after unrolling, so the arrays are plain registers and entries of the kind an
// accumulator does not use are never materialised.
template <class S, int G>
struct RegAcc {
  static constexpr int NA = (S::kStatic && S::NACC > 0) ? S::NACC : 1;
  static constexpr int NG = G > 0 ? G : 1;
  i64 w[NG][NA];
  int32_t n[NG][NA];
};
template <class S, int G, int J>
__device__ __forceinline__ void rs_init(RegAcc<S, G> &ra) {
  if constexpr (G > 0 && J < S::NACC) {
#pragma unroll
    for (int g = 0; g < G; g++) {
      constexpr int op = S::ACC_OP[J];
      if constexpr (S::ACC_RK[J] == RK_WIDE || S::ACC_RK[J] == RK_MADW) ra.w[g][J] = acc_identity(op);
      else if constexpr (S::ACC_RK[J] == RK_N32) ra.n[g][J] = 0;
      else ra.n[g][J] = INT32_MAX;
    }
    rs_init<S, G, J + 1>(ra);
  }
}
// product of own factors F0 .. F1-1 of accumulator J onto v
template <class S, int J, int F, int F1>
__device__ __forceinline__ i64 factor_range(const KAcc &A, i64 v, bool have, const unsigned char *tile, int r, i64 grow) {
  if constexpr (F < F1) {
    i64 x = affine_static<S::FAC[J][F]>(A.fac[F], tile, r, grow);
    return factor_range<S, J, F + 1, F1>(A, have ? (i64)((u64)v * (u64)x) : x, true, tile, r, grow);
  }
  return v;
}
// values of every accumulator for one row (prefix-shared exactly like acc_chain).  RK_MADW accumulators are kept as
// the pair (a, b) with value a * b, both int32 by the host's proof, so that the update is one `mad.wide.s32`.
template <class S, int J>
__device__ __forceinline__ void rs_values(const KDesc &d, i64 *v, int32_t *va, int32_t *vb, i64 prev, const unsigned char *tile, int r, i64 grow) {
  if constexpr (J < S::NACC) {
    constexpr bool chain = (bool)S::ACC_CHAIN[J];
    constexpr int nfac = S::ACC_NFAC[J];
    if constexpr (S::ACC_RK[J] == RK_FIRST) {
      v[J] = 0;   // the CTA-local row index is supplied by the caller
      rs_values<S, J + 1>(d, v, va, vb, prev, tile, r, grow);
    } else if constexpr (S::ACC_RK[J] == RK_MADW) {
      i64 a = factor_range<S, J, 0, nfac - 1>(d.acc[J], chain ? prev : 1, chain, tile, r, grow);
      va[J] = (int32_t)a;
      vb[J] = (int32_t)affine_static<S::FAC[J][nfac - 1]>(d.acc[J].fac[nfac - 1], tile, r, grow);
      v[J] = (i64)va[J] * (i64)vb[J];
      rs_values<S, J + 1>(d, v, va, vb, v[J], tile, r, grow);
    } else {
      v[J] = factor_chain<S, J, 0>(d.acc[J], chain ? prev : 1, tile, r, grow);
      rs_values<S, J + 1>(d, v, va, vb, v[J], tile, r, grow);
    }
  }
}
// Predicated updates (`@p add` / `@p min`): the slot test never branches, so a warp whose 32 rows hit 6 different
// slots runs ONE straight instruction stream instead of 6 divergent switch arms (the compiler turns an if-chain
// over `slot == g` into a jump table, which serialises the arms and stalls on every indirect branch).
__device__ __forceinline__ void pred_add64(i64 &acc, i64 v, int s, int g) {
  // split add with carry: ptxas keeps the low add predicated (a predicated add.s64 / mad.wide becomes add + 2 SEL)
  uint32_t lo = (uint32_t)acc, hi = (uint32_t)((u64)acc >> 32);
  asm("{\n .reg .pred p;\n setp.eq.s32 p, %4, %5;\n @p add.cc.u32 %0, %0, %2;\n @p addc.u32 %1, %1, %3;\n}"
      : "+r"(lo), "+r"(hi) : "r"((uint32_t)v), "r"((uint32_t)((u64)v >> 32)), "r"(s), "r"(g));
  acc = (i64)(((u64)hi << 32) | lo);
}
__device__ __forceinline__ void pred_min64(i64 &acc, i64 v, int s, int g) {
  asm("{\n .reg .pred p;\n setp.eq.s32 p, %2, %3;\n @p min.s64 %0, %0, %1;\n}" : "+l"(acc) : "l"(v), "r"(s), "r"(g));
}
__device__ __forceinline__ void pred_max64(i64 &acc, i64 v, int s, int g) {
  asm("{\n .reg .pred p;\n setp.eq.s32 p, %2, %3;\n @p max.s64 %0, %0, %1;\n}" : "+l"(acc) : "l"(v), "r"(s), "r"(g));
}
__device__ __forceinline__ void pred_madw(i64 &acc, int32_t a, int32_t b, int s, int g) {
  asm("{\n .reg .pred p;\n setp.eq.s32 p, %3, %4;\n @p mad.wide.s32 %0, %1, %2, %0;\n}" : "+l"(acc) : "r"(a), "r"(b), "r"(s), "r"(g));
}
__device__ __forceinline__ void pred_add32(int32_t &acc, int32_t v, int s, int g) {
  asm("{\n .reg .pred p;\n setp.eq.s32 p, %2, %3;\n @p add.s32 %0, %0, %1;\n}" : "+r"(acc) : "r"(v), "r"(s), "r"(g));
}
__device__ __forceinline__ void pred_min32(int32_t &acc, int32_t v, int s, int g) {
  asm("{\n .reg .pred p;\n setp.eq.s32 p, %2, %3;\n @p min.s32 %0, %0, %1;\n}" : "+r"(acc) : "r"(v), "r"(s), "r"(g));
}
// slot Q's accumulators take the row's values iff s == Q
template <class S, int G, int Q, int J>
__device__ __forceinline__ void rs_apply(RegAcc<S, G> &ra, int s, const i64 *v, const int32_t *va, const int32_t *vb, int lrow) {
  if constexpr (J < S::NACC) {
    constexpr int op = S::ACC_OP[J];
    if constexpr (S::ACC_RK[J] == RK_MADW) {
      // acc += (slot matches ? a : 0) * b as ONE 32x32+64 multiply-add (IMAD.WIDE.U32, fma pipe) after one select that
      // accumulators sharing `a` share; 0 <= a, b < 2^31 by the host's proof.  (A predicated 64-bit add costs 3.)
      const uint32_t am = (s == Q) ? (uint32_t)va[J] : 0u;
      ra.w[Q][J] = (i64)((u64)ra.w[Q][J] + (u64)am * (u64)(uint32_t)vb[J]);
    }
    else if constexpr (S::ACC_RK[J] == RK_WIDE) {
      if constexpr (op == 0) pred_add64(ra.w[Q][J], v[J], s, Q);
      else if constexpr (op == 1) pred_min64(ra.w[Q][J], v[J], s, Q);
      else pred_max64(ra.w[Q][J], v[J], s, Q);
    } else if constexpr (S::ACC_RK[J] == RK_N32) pred_add32(ra.n[Q][J], (int32_t)v[J], s, Q);
    else pred_min32(ra.n[Q][J], lrow, s, Q);
    rs_apply<S, G, Q, J + 1>(ra, s, v, va, vb, lrow);
  }
}
template <class S, int G, int GL, int Q>
__device__ __forceinline__ void rs_apply_slots(RegAcc<S, G> &ra, int s, const i64 *v, const int32_t *va, const int32_t *vb, int lrow) {
  if constexpr (Q < GL) {
    rs_apply<S, G, Q, 0>(ra, s, v, va, vb, lrow);
    rs_apply_slots<S, G, GL, Q + 1>(ra, s, v, va, vb, lrow);
  }
}

// end of kernel: warp-reduce every (slot, accumulator) and let lane 0 store it at out[g * NACC + J]
template <class S, int G, int J>
__device__ __forceinline__ void rs_flush(const KDesc &d, const RegAcc<S, G> &ra, i64 *out, int lane) {
  if constexpr (G > 0 && J < S::NACC) {
#pragma unroll
    for (int g = 0; g < G; g++) {
      i64 v;
      if constexpr (S::ACC_RK[J] == RK_WIDE || S::ACC_RK[J] == RK_MADW) v = ra.w[g][J];
      else if constexpr (S::ACC_RK[J] == RK_N32) v = (i64)ra.n[g][J];
      else {
        // CTA-local row index (iteration * tile_rows + row in tile) -> global row id; monotonic within the CTA
        const int idx = ra.n[g][J];
        v = INT64_MAX;
        if (idx != INT32_MAX) {
          const i64 tile = (i64)blockIdx.x + (i64)(idx / d.tile_rows) * gridDim.x;
          v = d.row_base + tile * d.tile_rows + idx % d.tile_rows;
        }
      }
      constexpr int op = S::ACC_OP[J];
      v = warp_reduce(op, v);
      if (lane == 0) out[g * S::NACC + J] = v;
    }
    rs_flush<S, G, J + 1>(d, ra, out, lane);
  }
}

// Per-CTA group state: key -> compact slot (lane-private accumulator tables are indexed by slot).
struct GroupState {
  int32_t *slotmap;   // [domain]  -1 unseen, -2 being claimed, -3 overflow (stays on the global-atomic path), >=0 slot
  int32_t *slotkey;   // [gmax]
  int32_t *nslots;
  i64 *tbl;           // [gmax][nacc][NC]
};

// Phase 2 (the Gathers + elementwise map + Fold of the plan): fold one selected row into the lane-private tables.
// GL (register slots only): the slot tests cover slots 0 .. GL-1 (= G today; a slot >= GL takes the global-atomic path).
template <class S, int NC, int G, int GL>
__device__ __forceinline__ void fold_row(const KDesc &d, const unsigned char *tile, int r, i64 grow, const GroupState &g, int ctid,
                                         RegAcc<S, G> &ra, int lrow) {
  i64 key;
  if constexpr (S::kStatic && S::KEY32) key = (i64)(key_chain32<S, 0>(d, 0, tile, r) & (int32_t)d.key_mask);
  else key = key_chain<S, 0>(d, 0, tile, r, grow) & d.key_mask;
  if ((u64)key >= (u64)d.domain) {   // the planner proves key < domain (mask); never expected
    atomicAdd(d.errflag, 1);
    return;
  }
  const int s = ((volatile int32_t *)g.slotmap)[key];
  if constexpr (G > 0) {
    i64 v[RegAcc<S, G>::NA];
    int32_t va[RegAcc<S, G>::NA], vb[RegAcc<S, G>::NA];
    rs_values<S, 0>(d, v, va, vb, 1, tile, r, grow);
    rs_apply_slots<S, G, GL, 0>(ra, s, v, va, vb, lrow);     // s < 0 (key without a slot yet) matches none
  }
  if (s >= 0 && (G == 0 || s < GL)) {
    if constexpr (G == 0) acc_chain<S, 0, NC>(d, g.tbl + (size_t)s * d.nacc * NC + ctid, 1, tile, r, grow);
  } else {
    // first rows of a key in this CTA: fold straight into the global table and claim a slot for the rest
#pragma unroll 1
    for (int j = 0; j < d.nacc; j++) acc_global(d.acc[j].op, d.table + (size_t)j * d.domain + key, acc_value_slow(d, j, tile, r, grow));
    if (s == -1 && atomicCAS(&g.slotmap[key], -1, -2) == -1) {
      int ns = atomicAdd(g.nslots, 1);
      if (ns < d.gmax) {
        g.slotkey[ns] = (int32_t)key;
        __threadfence_block();
        atomicExch(&g.slotmap[key], ns);
      } else {
        atomicExch(&g.slotmap[key], -3);
      }
    }
  }
}

// Dense tile, register slots: the R rows of a thread as ONE branch-free block so that their shared-memory loads and
// dependent chains overlap.  A row that did not pass the selection, or whose key has no register slot yet, gets
// slot -1 (matches no predicate); the latter rows are then redone by fold_row, which owns the claim / global path.
template <class S, int NC, int R, int G, int GL>
__device__ __forceinline__ void fold_dense(const KDesc &d, const unsigned char *tile, unsigned pass, int ctid, i64 grow0, const GroupState &g,
                                           RegAcc<S, G> &ra, int lrow0) {
  if constexpr (S::kStatic && S::KEY32) {
    int sl[R];
    unsigned redo = 0;
#pragma unroll
    for (int k = 0; k < R; k++) {
      // the host checked 0 <= key_mask < domain for a KEY32 shape: the masked key needs no range test
      const int key = key_chain32<S, 0>(d, 0, tile, ctid + k * NC) & (int32_t)d.key_mask;
      const int s = ((volatile int32_t *)g.slotmap)[key];
      const bool on = (pass >> k) & 1, have = (unsigned)s < (unsigned)GL;
      sl[k] = (on && have) ? s : -1;
      if (on && !have) redo |= 1u << k;
    }
#pragma unroll
    for (int k = 0; k < R; k++) {
      const int r = ctid + k * NC;
      i64 v[RegAcc<S, G>::NA];
      int32_t va[RegAcc<S, G>::NA], vb[RegAcc<S, G>::NA];
      rs_values<S, 0>(d, v, va, vb, 1, tile, r, grow0 + r);
      rs_apply_slots<S, G, GL, 0>(ra, sl[k], v, va, vb, lrow0 + r);
    }
    if (redo) {
#pragma unroll 1
      for (int k = 0; k < R; k++)
        if ((redo >> k) & 1) fold_row<S, NC, G, GL>(d, tile, ctid + k * NC, grow0 + ctid + k * NC, g, ctid, ra, lrow0 + ctid + k * NC);
    }
  } else {
#pragma unroll
    for (int k = 0; k < R; k++)
      if ((pass >> k) & 1) fold_row<S, NC, G, GL>(d, tile, ctid + k * NC, grow0 + ctid + k * NC, g, ctid, ra, lrow0 + ctid + k * NC);
  }
}
template <class S, int NC, int R, int G, int GL>
__device__ __forceinline__ void fold_queue(const KDesc &d, const unsigned char *buf, const uint16_t *queue, int e0, int nsel, i64 grow0,
                                           const GroupState &g, int ctid, RegAcc<S, G> &ra, int lrow0) {
  for (int e = e0; e < nsel; e += NC) {
    const int r = queue[e];
    fold_row<S, NC, G, GL>(d, buf, r, grow0 + r, g, ctid, ra, lrow0 + r);
  }
}

// Phase 1 of a tile (the plan's FoldSelect, Vlite.hs:721-730, done in shared memory): thread ctid evaluates the
// predicates of rows ctid + k*NC, k < R, together (R independent shared-memory loads in flight) and the rows
// that pass are compacted CTA-wide into `queue` with one warp-aggregated shared atomic per warp and k.
template <class S, int NC, int R, int G>
__device__ __forceinline__ void select_rows(const KDesc &d, const unsigned char *tile, int nvalid, int ctid, int *qcount, uint16_t *queue,
                                            i64 grow0, const GroupState &g, RegAcc<S, G> &ra, int lrow0) {
  unsigned pass = 0;
#pragma unroll
  for (int k = 0; k < R; k++)
    if (ctid + k * NC < nvalid) pass |= 1u << k;
  pred_chain<S, 0, NC, R>(d, tile, ctid, pass);
  const int lane = ctid & 31;
  const unsigned any = __ballot_sync(0xffffffffu, pass != 0);
  if (!any) return;
  if (__popc(any) >= 24) {
    // dense selection (most lanes own a selected row): compaction would buy nothing, fold the rows where they are
    if constexpr (G > 0) {   // straight-line predicated code: let the R rows of a thread overlap
      fold_dense<S, NC, R, G, G>(d, tile, pass, ctid, grow0, g, ra, lrow0);
    } else {
#pragma unroll 1
      for (int k = 0; k < R; k++)
        if ((pass >> k) & 1) fold_row<S, NC, G, 0>(d, tile, ctid + k * NC, grow0 + ctid + k * NC, g, ctid, ra, lrow0 + ctid + k * NC);
    }
    return;
  }
  if (__popc(any) <= 4) {
    // few selected rows in this warp (selective predicates): the owning lanes append on their own
    if (pass) {
      int base = atomicAdd(qcount, __popc(pass));
#pragma unroll
      for (int k = 0; k < R; k++)
        if ((pass >> k) & 1) queue[base++] = (uint16_t)(ctid + k * NC);
    }
    return;
  }
#pragma unroll
  for (int k = 0; k < R; k++) {
    const bool p = (pass >> k) & 1;
    const unsigned m = __ballot_sync(0xffffffffu, p);
    if (m) {
      int base = 0;
      if (lane == 0) base = atomicAdd(qcount, __popc(m));
      base = __shfl_sync(0xffffffffu, base, 0);
      if (p) queue[base + __popc(m & ((1u << lane) - 1))] = (uint16_t)(ctid + k * NC);
    }
  }
}

__device__ __forceinline__ void choose_keys(const KDesc &d, i64 k0, i64 kstride);

template <class S, int NC, int R, int G>
__device__ __forceinline__ void fused_scan_fold_body(const KDesc &d, const FinDesc &fd, const XDesc &xd) {
  extern __shared__ __align__(128) unsigned char smem[];
  // layout: [ring: stages * stage_bytes][full[stages]][empty[stages]][sel[stages]][qcount[stages]]
  //         [queue[stages][tile_rows]][nslots][slotkey[gmax]][slotmap[domain]][tables]
  constexpr int NW = NC / 32;                 // consumer warps
  unsigned char *ring = smem;
  uint64_t *full = (uint64_t *)(smem + (size_t)d.stages * d.stage_bytes);
  uint64_t *empty = full + d.stages;
  uint64_t *sel = empty + d.stages;
  int *qcount = (int *)(sel + d.stages);
  uint16_t *queue = (uint16_t *)(qcount + d.stages + (d.stages & 1));
  GroupState g;
  g.nslots = (int32_t *)(queue + (size_t)d.stages * (NC * R));
  g.slotkey = g.nslots + 2;
  g.slotmap = g.slotkey + d.gmax;
  size_t tbl_off = (size_t)((unsigned char *)(g.slotmap + d.domain) - smem);
  tbl_off = (tbl_off + 15) & ~(size_t)15;
  g.tbl = (i64 *)(smem + tbl_off);

  const int tid = threadIdx.x;
  const int warp = tid >> 5, lane = tid & 31;
  const bool dense = d.domain <= d.gmax;     // every key has its own slot from the start

  if (tid == 0) {
    for (int s = 0; s < d.stages; s++) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], NW);
      mbar_init(&sel[s], NW);
      qcount[s] = 0;
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    *g.nslots = dense ? (int)d.domain : 0;
  }
  for (i64 k = tid; k < d.domain; k += NC + 32) g.slotmap[k] = dense ? (int32_t)k : -1;
  if (dense && tid < d.gmax) g.slotkey[tid] = tid;
  if (G == 0 && tid >= 32) {
    const int ctid = tid - 32;
    for (int s = 0; s < d.gmax; s++)
      for (int j = 0; j < d.nacc; j++) g.tbl[((size_t)s * d.nacc + j) * NC + ctid] = acc_identity(d.acc[j].op);
  }
  __syncthreads();

  if (warp == 0) {
    // ------------------------------------------------------------------ producer
    if (lane == 0) {
      const uint64_t policy = policy_evict_first();
      int st = 0;
      uint32_t ph = 0;
      for (i64 tile = blockIdx.x; tile < d.ntiles; tile += gridDim.x) {
        mbar_wait(&empty[st], ph ^ 1);       // every consumer warp folded the stage's previous tile
        qcount[st] = 0;                      // (published to the consumers by the arrive below)
        mbar_expect_tx(&full[st], (uint32_t)d.stage_tx);
        unsigned char *dst = ring + (size_t)st * d.stage_bytes;
#pragma unroll 1
        for (int c = 0; c < d.ncols; c++) {
          uint32_t bytes = (uint32_t)(d.tile_rows * d.width[c]);
          bulk_g2s(dst + d.soff[c], (const char *)d.col[c] + (size_t)tile * bytes, bytes, &full[st], policy);
        }
        if (++st == d.stages) { st = 0; ph ^= 1; }
      }
    }
    return;
  }

  // -------------------------------------------------------------------- consumers
  // Software-pipelined by one tile and free of CTA-wide barriers in steady state: iteration `it` SELECTS tile it
  // (predicates -> the stage's compaction queue, then a non-blocking arrive on sel[stage]) and FOLDS tile it-1
  // (wait on its sel barrier -- normally long complete --, fold this warp's share of the queue, release the stage).
  const int ctid = tid - 32, cw = warp - 1;
  RegAcc<S, G> ra;
  rs_init<S, G, 0>(ra);
  // The rows past the last full tile form one more (partial) tile, owned by the CTA next in the round-robin; it
  // is staged with plain loads into the (by then idle) next ring stage and goes through the same code.
  const i64 ntiles_all = d.ntiles + (d.ntiles * d.tile_rows < d.rows ? 1 : 0);
  int st = 0, pst = 0, it = 0;
  uint32_t ph = 0, pph = 0;
  i64 ptile = -1;
  for (i64 tile = blockIdx.x;; tile += gridDim.x, it++) {
    const bool have = tile < ntiles_all;
    if (have) {
      unsigned char *buf = ring + (size_t)st * d.stage_bytes;
      int nvalid = d.tile_rows;
      if (tile < d.ntiles) {
        mbar_wait(&full[st], ph);
      } else {
        const i64 tail0 = d.ntiles * d.tile_rows;
        nvalid = (int)(d.rows - tail0);
        consumer_barrier<NC>();      // every warp is done with this stage's previous tile (folded >= 1 iteration ago)
        if (ctid == 0) qcount[st] = 0;
#pragma unroll 1
        for (int c = 0; c < d.ncols; c++) {
          if (d.width[c] == 4) {
            const int32_t *src = (const int32_t *)d.col[c] + tail0;
            for (int r = ctid; r < nvalid; r += NC) ((int32_t *)(buf + d.soff[c]))[r] = src[r];
          } else {
            const i64 *src = (const i64 *)d.col[c] + tail0;
            for (int r = ctid; r < nvalid; r += NC) ((i64 *)(buf + d.soff[c]))[r] = src[r];
          }
        }
        consumer_barrier<NC>();
      }
      select_rows<S, NC, R, G>(d, buf, nvalid, ctid, &qcount[st], queue + (size_t)st * (NC * R), d.row_base + tile * d.tile_rows, g, ra,
                               it * d.tile_rows);
      __syncwarp();
      if (lane == 0) mbar_arrive(&sel[st]);
    }
    if (ptile >= 0) {
      mbar_wait(&sel[pst], pph);
      const int nsel = ((volatile int *)qcount)[pst];
      const unsigned char *buf = ring + (size_t)pst * d.stage_bytes;
      const i64 grow0 = d.row_base + ptile * d.tile_rows;
      // queue entries in chunks of 32, dealt to the warps starting at a warp that rotates with the tile
      int chunk = cw - ((it - 1) % NW);
      if (chunk < 0) chunk += NW;
      const uint16_t *q = queue + (size_t)pst * (NC * R);
      const int e0 = chunk * 32 + lane, lrow0 = (it - 1) * d.tile_rows;
      fold_queue<S, NC, R, G, G>(d, buf, q, e0, nsel, grow0, g, ctid, ra, lrow0);
      __syncwarp();
      if (lane == 0 && ptile < d.ntiles) mbar_arrive(&empty[pst]);
    }
    if (!have) break;
    ptile = tile; pst = st; pph = ph;
    if (++st == d.stages) { st = 0; ph ^= 1; }
  }

  consumer_barrier<NC>();
  int ns = *((volatile int32_t *)g.nslots);
  if (ns > d.gmax) ns = d.gmax;
  if constexpr (G > 0) {
    // register slots -> warp shuffles -> one row per warp in the (now idle) ring -> one global atomic per (CTA, slot, accumulator)
    i64 *red = (i64 *)ring;                   // [NW][G * NACC]
    rs_flush<S, G, 0>(d, ra, red + (size_t)cw * (G * S::NACC), lane);
    consumer_barrier<NC>();
    for (int p = ctid; p < ns * S::NACC; p += NC) {
      const int j = p % S::NACC, op = d.acc[j].op;
      i64 v = acc_identity(op);
      for (int w = 0; w < NW; w++) v = acc_combine(op, v, red[(size_t)w * (G * S::NACC) + p]);
      if (v != acc_identity(op)) acc_global(op, d.table + (size_t)j * d.domain + g.slotkey[p / S::NACC], v);
    }
  } else {
    // lane-private tables -> one global atomic per (warp, slot, accumulator)
    for (int p = cw; p < ns * d.nacc; p += NW) {
      const int s = p / d.nacc, j = p % d.nacc, op = d.acc[j].op;
      i64 v = acc_identity(op);
      for (int t = lane; t < NC; t += 32) v = acc_combine(op, v, g.tbl[((size_t)s * d.nacc + j) * NC + t]);
      v = warp_reduce(op, v);
      if (lane == 0) acc_global(op, d.table + (size_t)j * d.domain + g.slotkey[s], v);
    }
  }

  // ---- epilogue by the last CTA to get here: the table is complete, finish the step without another launch
  if (d.epilogue) {
    __threadfence();                       // this CTA's atomics are ordered before its ticket
    consumer_barrier<NC>();
    if (ctid == 0) g.nslots[1] = atomicAdd(d.done, 1u) == gridDim.x - 1;
    consumer_barrier<NC>();
    if (g.nslots[1]) {
      __threadfence();
      if (d.nchoose) choose_keys(d, ctid, NC);
      if (d.epilogue >= 2) {
        __threadfence();
        consumer_barrier<NC>();
        const i64 *parts = fd.parts;
        int nranks = 1;
        if (d.epilogue == 3) {             // combine across GPUs through peer memory first
          parts = exchange_block<NC>(xd, d.table, d.errflag, ctid);
          nranks = xd.world;
        }
        // scratch in the idle ring: [running][warp counts]
        finalize_block<NC>(fd, parts, nranks, ctid, (int *)(ring + 16), (i64 *)ring);
      }
      if (ctid == 0) *d.done = 0;
    }
  }
}

// The precompiled instantiations (GenericShape and the static shapes of vdl_shapes.cuh); a shape generated at run time
// from a prepared descriptor gets its own `extern "C"` wrapper around fused_scan_fold_body (jit_scan_source, vdl_fused.cu).
template <class S, int NC, int R, int G>
__global__ void __launch_bounds__(NC + 32, 1) fused_scan_fold_kernel(const __grid_constant__ KDesc d, const __grid_constant__ FinDesc fd, const __grid_constant__ XDesc xd) {
  fused_scan_fold_body<S, NC, R, G>(d, fd, xd);
}

// identity-initialise the global table ([nacc][domain] by op, choose section zero)
#ifndef __CUDACC_RTC__
__global__ void fused_init_kernel(const __grid_constant__ KDesc d) {
  i64 n = (i64)(d.nacc + d.nchoose) * d.domain;
  for (i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (i64)gridDim.x * blockDim.x) {
    int j = (int)(i / d.domain);
    d.table[i] = j < d.nacc ? acc_identity(d.acc[j].op) : 0;
  }
}
#endif

// FoldChoose = first row of the run (App. G6) = the expression at the smallest selected row of the key.
// Reads the table with cache-global loads: other CTAs built it with atomics at L2.
__device__ __forceinline__ void choose_keys(const KDesc &d, i64 k0, i64 kstride) {
  for (i64 k = k0; k < d.domain; k += kstride) {
    if (__ldcg(&d.table[(size_t)d.cnt_idx * d.domain + k]) <= 0) continue;
    i64 grow = __ldcg(&d.table[(size_t)d.first_idx * d.domain + k]);
    i64 r = grow - d.row_base;
    for (int c = 0; c < d.nchoose; c++) {
      const KAcc &A = d.choose[c];
      i64 v = 1;
      for (int f = 0; f < A.nfac; f++) {
        const KAffine &F = A.fac[f];
        i64 x;
        if (F.col == -1) x = F.a;
        else {
          i64 leaf = F.col == -2 ? grow : ((d.width[F.col] == 4 ? (i64)((const int32_t *)d.col[F.col])[r] : ((const i64 *)d.col[F.col])[r]) >> F.shr);
          x = (i64)((u64)F.a + (u64)F.b * (u64)leaf);
        }
        v = (i64)((u64)v * (u64)x);
      }
      d.table[(size_t)(d.nacc + c) * d.domain + k] = v;
    }
  }
}
#ifndef __CUDACC_RTC__
__global__ void fused_choose_kernel(const __grid_constant__ KDesc d) {
  choose_keys(d, (i64)blockIdx.x * blockDim.x + threadIdx.x, (i64)gridDim.x * blockDim.x);
}
#endif
