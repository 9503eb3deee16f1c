// Fused FK-join probe: ONE pass over a fact-table shard that follows foreign-key index columns into
// dimension columns (replicated in HBM, mostly L2-resident), applies the selection predicates of the whole
// join chain, and either folds per group key (Q5-class plans) or emits the surviving rows' expressions as
// dense vectors in row order (Q3-class plans, whose high-cardinality group-by continues op-at-a-time on the
// few surviving rows).
//
// What it replaces in the emitted graph (reference Vlite.hs): handleGatherJoin / deduceMasks
// (Vlite.hs:1199-1232, 1248-1280; diagram 1420-1447) lower an FK join to
//     fk'      = Gather(Load fact.fk_idx, factmask)
//     valid    = Scatter(ones -> dimmask positions)         inv = Scatter(pos -> dimmask positions)
//     boolean  = Gather(valid, fk')                         gmask = Gather(inv, fk')
//     selmask  = FoldSelect(pos_ boolean, boolean)
//     fact cols, gmask <- Gather(., selmask)                dim cols <- Gather(Gather(col, dimmask), gmask)
// and chain that per join.  In the dense model (SURVEY.md App. G1) every vector of the joined row space is a
// function of the underlying fact row i:  dim column e -> e[fk(i)],  nested joins -> e[fk2[fk1(i)]], and the
// selection is the conjunction of the fact predicates and the dimension predicates evaluated at fk(i).  The
// planner (vdl_plan.cu, analyse) proves that normal form; this kernel evaluates it:
//   leaf      value(i) = column[ parent leaf's value(i) ]   (parent < 0: column[i] of the fact table)
//   term      a + b * (leaf >> shr), or a constant, or the row id
//   predicate lo <= term <= hi, or term == term; evaluated in chain order, first failure rejects the row
// No validity vector, inverse index, position vector or gathered copy is ever materialised.
//
// Kernel shape: persistent thread blocks take 4096-row tiles in order from a ticket counter and evaluate the
// predicates stage by stage, compacting the survivors after each (probe_body in vdl_probe_kernel.cuh; the
// fact-column loads of a stage are coalesced, and the lineitem->orders index is clustered, so the first dimension
// gather is nearly sequential too).  Fold mode accumulates into a shared-memory table per block (flushed with
// global atomics); emit mode places a tile's survivors with a decoupled look-back across tiles (one 64-bit
// status word per tile), so the output vectors are exactly the dense FoldSelect order.  Bound: HBM for the fact columns + L2 latency for the dimension gathers.
#include <stdio.h>
#include <string.h>

#include <algorithm>

#include "vdl_internal.h"

#include "vdl_probe_kernel.cuh"

// value of leaf l at fact row `row` (local to the shard): walk the parent chain, then load top-down
__device__ __forceinline__ i64 leaf_value(const PDesc &d, int l, i64 row, bool &ok) {
  int chain[P_MAX_DEPTH];
  int n = 0;
#pragma unroll
  for (int k = 0; k < P_MAX_DEPTH; k++)
    if (l >= 0) { chain[k] = l; n = k + 1; l = d.leaf[l].parent; }
  i64 idx = row;
#pragma unroll
  for (int k = P_MAX_DEPTH - 1; k >= 0; k--) {
    if (k < n) {
      const PLeaf &L = d.leaf[chain[k]];
      if ((u64)idx >= (u64)L.len) { ok = false; return 0; }
      idx = L.w4 ? (i64)__ldg((const int32_t *)L.ptr + idx) : __ldg((const i64 *)L.ptr + idx);
    }
  }
  return idx;
}
__device__ __forceinline__ i64 plain_term_value(const PDesc &d, const PTerm &t, i64 row, bool &ok) {
  if (t.leaf == -1) return t.a;
  i64 v = t.leaf == -2 ? d.row_base + row : leaf_value(d, t.leaf, row, ok);
  if (t.shr) v >>= t.shr;
  return (i64)((u64)t.a + (u64)t.b * (u64)v);
}
// does predicate P hold at the row?  (its terms are plain: no indicators inside predicates)
__device__ __forceinline__ bool pred_holds(const PDesc &d, const PPred &P, i64 row, bool &ok) {
  const i64 t = plain_term_value(d, P.t, row, ok);
  if (P.kind == 0) {
    if ((u64)t - (u64)P.lo <= P.span) return true;
    for (int k = 0; k < P.nmore; k++)
      if ((u64)t - (u64)P.lo_more[k] <= P.span_more[k]) return true;
    return false;
  }
  const i64 u = plain_term_value(d, P.u, row, ok);
  switch (P.cmp) {
    case VDL_CMP_EQ: return t == u;
    case VDL_CMP_NE: return t != u;
    case VDL_CMP_GT: return t > u;
    case VDL_CMP_GE: return t >= u;
    case VDL_CMP_LT: return t < u;
    default: return t <= u;
  }
}
__device__ __forceinline__ i64 term_value(const PDesc &d, const PTerm &t, i64 row, bool &ok) {
  if (t.leaf <= -3) {                       // indicator of a predicate as a 0/1 value
    const i64 v = pred_holds(d, d.ind[-3 - t.leaf], row, ok) ? 1 : 0;
    return (i64)((u64)t.a + (u64)t.b * (u64)v);
  }
  return plain_term_value(d, t, row, ok);
}
__device__ __forceinline__ i64 prod_value(const PDesc &d, const PProd &p, i64 row, bool &ok) {
  i64 v = 1;
  for (int f = 0; f < p.nfac; f++) v = (i64)((u64)v * (u64)term_value(d, p.f[f], row, ok));
  return v;
}

// ---- the interpreter's evaluator (probe_body: vdl_probe_kernel.cuh) -----------------------------------------------------
// A range predicate on a lookup chain of depth <= 4 -- every predicate the FK-join lowering produces -- runs as
// straight-line code: the chain (pointers, lengths, widths) is read from the descriptor once per tile and stage, not per row.
struct StageRegs { const void *ptr[4]; i64 len[4]; int w4mask, shr, depth; i64 a, b, lo; u64 span; };

// S.ptr[0] is the leaf's own column (the LAST load), S.ptr[D-1] the fact column (the first): all indexing static.
// The first hop is indexed by the fact row itself (in range: prepare checks the fact columns' lengths); PLAIN: the
// term is the bare leaf (a = 0, b = 1), as in every predicate the lowering emits.
template <int D, bool PLAIN>
__device__ __forceinline__ bool chain_test(const StageRegs &S, i64 row, i64 row_base, bool &ok) {
  i64 v = row;
  if (D == 0) v = row_base + row;
#pragma unroll
  for (int k = D - 1; k >= 0; k--) {
    if (k != D - 1 && (u64)v >= (u64)S.len[k]) { ok = false; return false; }
    v = ((S.w4mask >> k) & 1) ? (i64)__ldg((const int32_t *)S.ptr[k] + v) : __ldg((const i64 *)S.ptr[k] + v);
  }
  v >>= S.shr;
  if (!PLAIN) v = (i64)((u64)S.a + (u64)S.b * (u64)v);
  return (u64)v - (u64)S.lo <= S.span;
}

#ifndef P_SUB
#define P_SUB 4      // rows per thread and round of a stage (8 was best while every round ended in two barriers)
#endif

struct ProbeInterp {
  static constexpr int SUB = P_SUB;
  __device__ __forceinline__ static int npreds(const PDesc &d) { return d.npreds; }
  __device__ __forceinline__ static int nfolds(const PDesc &d) { return d.nfolds; }
  __device__ __forceinline__ static int nemits(const PDesc &d) { return d.nemits; }
  template <class F> __device__ __forceinline__ static void stages(const PDesc &d, const int &n_in, F &&run_stage) {
    for (int q = 0; q < d.npreds && n_in > 0; q++) run_stage(q);
  }
  // the chain of stage q's term, if it has the fast form
  __device__ __forceinline__ static StageRegs stage(const PDesc &d, int q) {
    const PPred &P = d.pred[q];
    StageRegs S;
    S.depth = -1;
    if (P.kind == 0 && P.nmore == 0 && P.t.leaf != -1) {
      int l = P.t.leaf, n = 0;
      S.w4mask = 0;
#pragma unroll
      for (int k = 0; k < 4; k++) {
        S.ptr[k] = nullptr; S.len[k] = 0;
        if (l >= 0) {
          const PLeaf &L = d.leaf[l];
          S.ptr[k] = L.ptr; S.len[k] = L.len; S.w4mask |= (L.w4 ? 1 : 0) << k;
          l = L.parent; n = k + 1;
        }
      }
      if (l < 0) { S.depth = n; S.shr = P.t.shr; S.a = P.t.a; S.b = P.t.b; S.lo = P.lo; S.span = P.span; if (P.t.a == 0 && P.t.b == 1) S.depth += 8; }   // +8: plain
    }
    return S;
  }
  __device__ __forceinline__ static void round(const PDesc &d, int q, const StageRegs &S, i64 base, const int (&r)[SUB], bool (&f)[SUB], bool &ok) {
#define STAGE_CASE(DEPTH, PL)                                                                                                   \
  _Pragma("unroll") for (int k = 0; k < SUB; k++) f[k] = r[k] >= 0 && chain_test<DEPTH, PL>(S, base + r[k], d.row_base, ok)
    if (S.depth == 8 + 2) { STAGE_CASE(2, true);
    } else if (S.depth == 8 + 1) { STAGE_CASE(1, true);
    } else if (S.depth == 8 + 3) { STAGE_CASE(3, true);
    } else if (S.depth == 8 + 4) { STAGE_CASE(4, true);
    } else if (S.depth == 1) { STAGE_CASE(1, false);
    } else if (S.depth == 2) { STAGE_CASE(2, false);
    } else if (S.depth == 3) { STAGE_CASE(3, false);
    } else if (S.depth == 4) { STAGE_CASE(4, false);
    } else if (S.depth == 0 || S.depth == 8) { STAGE_CASE(0, false);
    } else {      // generic: constants, column-vs-column comparisons, range sets, deeper chains
#pragma unroll 1
      for (int k = 0; k < SUB; k++) f[k] = r[k] >= 0 && pred_holds(d, d.pred[q], base + r[k], ok);
    }
  }
  __device__ __forceinline__ static void fold_row(const PDesc &d, i64 row, i64 *tab, bool &ok) {
    i64 key = 0;
    for (int q = 0; q < d.nkeys; q++) key |= (i64)((u64)term_value(d, d.key[q], row, ok) << d.key_shl[q]);
    key &= d.key_mask;
    if ((u64)key >= (u64)d.domain) { ok = false; return; }
    for (int j = 0; j < d.nfolds; j++) {
      const int op = d.fold_op[j];
      if (op == VDL_FOLD_CHOOSE || op == VDL_FOLD_COUNT) continue;     // from the first row / the row count
      table_update(op, tab + (size_t)j * d.domain + key, prod_value(d, d.fold[j], row, ok));
    }
    atomicAdd((unsigned long long *)(tab + (size_t)d.nfolds * d.domain + key), 1ull);
    atomicMin((long long *)(tab + (size_t)(d.nfolds + 1) * d.domain + key), (long long)(d.row_base + row));
  }
  __device__ __forceinline__ static void emit_row(const PDesc &d, i64 row, i64 at, bool &ok) {
    for (int e = 0; e < d.nemits; e++) d.emit_out[e][at] = prod_value(d, d.emit[e], row, ok);
  }
};

__global__ void __launch_bounds__(P_THREADS, P_BLOCKS) probe_kernel(const __grid_constant__ PDesc d) { probe_body<ProbeInterp>(d, threadIdx.x); }

__global__ void probe_init_kernel(const __grid_constant__ PDesc d) {
  const i64 n = (i64)(d.nfolds + 2) * d.domain;
  for (i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (i64)gridDim.x * blockDim.x) {
    d.table[i] = table_identity(d, d.nfolds, (int)(i / d.domain));
  }
}

// External combine (several ranks): every rank evaluates FoldChoose at ITS first row of each key and stores the value in
// the fold's (otherwise unused) table row, so the tables alone carry everything the merge needs.
__global__ void probe_choose_kernel(const __grid_constant__ PDesc d) {
  for (i64 k = (i64)blockIdx.x * blockDim.x + threadIdx.x; k < d.domain; k += (i64)gridDim.x * blockDim.x) {
    if (d.table[(size_t)d.nfolds * d.domain + k] <= 0) continue;
    const i64 first = d.table[(size_t)(d.nfolds + 1) * d.domain + k] - d.row_base;
    bool ok = true;
    for (int j = 0; j < d.nfolds; j++)
      if (d.fold_op[j] == VDL_FOLD_CHOOSE) d.table[(size_t)j * d.domain + k] = prod_value(d, d.fold[j], first, ok);
    if (!ok) atomicAdd(d.errflag, 1);
  }
}

// Single GPU: the finalize evaluates FoldChoose itself, at the key's first row (no choose launch).
struct ChooseAtFirstRow {
  const PDesc &d;
  __device__ __forceinline__ i64 operator()(const FinDesc &f, const i64 *, int o, i64, int, i64 first) const {
    bool ok = true;
    return prod_value(d, d.fold[o], first - d.row_base, ok);
  }
};
__global__ void __launch_bounds__(256, 1) probe_finalize_kernel(const __grid_constant__ PDesc d, const __grid_constant__ FinDesc f) {
  __shared__ int warp_cnt[8];
  __shared__ i64 running;
  finalize_block<256>(f, f.parts, 1, threadIdx.x, warp_cnt, &running, ChooseAtFirstRow{d});
}

#include <string>
#include "vdl_embedded.inc"

// ---- run-time specialisation of the probe (NVRTC) ---------------------------------------------------------------------
// probe_kernel above INTERPRETS the descriptor: per row and stage it walks parent chains through the leaf table, dispatches
// on predicate kinds and reads bounds from the constant bank -- 160 thread-instructions per lineitem row on Q5, a handful of
// them loads (profiles/r01e_q05_sf10_dominant_kernel.txt).  For tables of a few hundred thousand rows and up the descriptor
// is instead PRINTED as CUDA C: one straight-line function per predicate stage (typed loads along the lookup chain, bounds
// and constants as literals, out-of-range lookups turned into a flag and a clamped index so that no branch separates the
// loads), one each for the fold and the emit of a surviving row, and an evaluator struct that hands them to probe_body,
// the tile loop probe_kernel instantiates too.  The 8 rows a thread handles per round are independent straight-line
// chains, so their loads overlap (memory-level parallelism instead of one dependent chain per warp).  Same results as the
// interpreter (tests/test_gpu_probe.py and the fuzz plans run both).
struct ProbeGen {
  const PDesc &d;
  std::string body;                 // statements of the function being generated
  bool have[VDL_MAX_LEAVES];
  int tmp = 0;
  explicit ProbeGen(const PDesc &desc) : d(desc) { reset(); }
  void reset() { body.clear(); memset(have, 0, sizeof have); tmp = 0; }
  static std::string lit(i64 v) { char b[48]; snprintf(b, sizeof b, "((i64)0x%llxull)", (unsigned long long)v); return b; }
  static std::string ulit(u64 v) { char b[48]; snprintf(b, sizeof b, "0x%llxull", (unsigned long long)v); return b; }
  std::string leaf(int l) {
    char nm[16], b[320];
    snprintf(nm, sizeof nm, "L%d", l);
    if (have[l]) return nm;
    have[l] = true;
    const PLeaf &L = d.leaf[l];
    const char *ld = L.w4 ? "(i64)__ldg((const int *)d.leaf[%d].ptr + %s)" : "__ldg((const i64 *)d.leaf[%d].ptr + %s)";
    char load[200];
    if (L.parent < 0) {
      snprintf(load, sizeof load, ld, l, "row");
      snprintf(b, sizeof b, "  const i64 %s = %s;\n", nm, load);
    } else {
      const std::string p = leaf(L.parent);
      char idx[64];
      snprintf(idx, sizeof idx, "(in%d ? %s : 0)", l, p.c_str());
      snprintf(load, sizeof load, ld, l, idx);
      snprintf(b, sizeof b, "  const bool in%d = (u64)%s < (u64)d.leaf[%d].len; ok = ok && in%d;\n  const i64 %s = %s;\n", l, p.c_str(), l, l, nm, load);
    }
    body += b;
    return nm;
  }
  std::string term(const PTerm &t) {
    if (t.leaf == -1) return lit(t.a);
    std::string v;
    if (t.leaf == -2) v = "(d.row_base + row)";
    else if (t.leaf <= -3) v = "(i64)(" + pred(d.ind[-3 - t.leaf]) + " ? 1 : 0)";
    else {
      v = leaf(t.leaf);
      if (t.shr) v = "(" + v + " >> " + std::to_string(t.shr) + ")";
    }
    if (t.a == 0 && t.b == 1) return v;
    return "(i64)((u64)" + lit(t.a) + " + (u64)" + lit(t.b) + " * (u64)" + v + ")";
  }
  std::string pred(const PPred &P) {
    char nm[16];
    snprintf(nm, sizeof nm, "T%d", tmp++);
    body += std::string("  const i64 ") + nm + " = " + term(P.t) + ";\n";
    if (P.kind == 0) {
      std::string e = std::string("((u64)") + nm + " - (u64)" + lit(P.lo) + " <= " + ulit(P.span);
      for (int k = 0; k < P.nmore; k++) e += std::string(" || (u64)") + nm + " - (u64)" + lit(P.lo_more[k]) + " <= " + ulit(P.span_more[k]);
      return e + ")";
    }
    char un[16];
    snprintf(un, sizeof un, "T%d", tmp++);
    body += std::string("  const i64 ") + un + " = " + term(P.u) + ";\n";
    static const char *CMP[] = {"==", "!=", ">", ">=", "<", "<="};
    return std::string("(") + nm + " " + CMP[P.cmp] + " " + un + ")";
  }
  std::string product(const PProd &p) {
    if (p.nfac == 0) return lit(1);
    std::string e = "(i64)(";
    for (int f = 0; f < p.nfac; f++) e += std::string(f ? " * " : "") + "(u64)" + term(p.f[f]);
    return e + ")";
  }
};

static std::string probe_jit_source(const PDesc &d, int p_sub, int blocks) {
  ProbeGen g(d);
  char b[256];
  std::string s = "#include \"vdl_probe_kernel.cuh\"\n", stage_of_q, calls;
  for (int q = 0; q < d.npreds; q++) {
    g.reset();
    const std::string e = g.pred(d.pred[q]);
    snprintf(b, sizeof b, "__device__ __forceinline__ bool probe_stage_%d(const PDesc &d, const i64 row, bool &ok) {\n", q);
    s += b + g.body + "  return " + e + ";\n}\n";
    snprintf(b, sizeof b, "q == %d ? probe_stage_%d(d, row, okk) : ", q, q);
    stage_of_q += b;
    snprintf(b, sizeof b, " run_stage(%d);", q);
    calls += b;
  }
  // probe_body's evaluator.  Every stage is run, with a literal q, also when no row survived an earlier one.
  snprintf(b, sizeof b, "struct ProbeJit {\n  static constexpr int SUB = %d;\n", p_sub);
  s += b;
  snprintf(b, sizeof b, "  __device__ static int npreds(const PDesc &) { return %d; }\n  __device__ static int nfolds(const PDesc &) { return %d; }\n"
                        "  __device__ static int nemits(const PDesc &) { return %d; }\n", d.npreds, d.nfolds, d.nemits);
  s += b;
  s += "  template <class F> __device__ __forceinline__ static void stages(const PDesc &, const int &, F &&run_stage) {" + calls + " }\n"
       "  __device__ static int stage(const PDesc &, int) { return 0; }\n"
       "  __device__ __forceinline__ static void round(const PDesc &d, int q, int, i64 base, const int (&r)[SUB], bool (&f)[SUB], bool &ok) {\n"
       "#pragma unroll\n"
       "    for (int k = 0; k < SUB; k++) {   // every slot evaluates a row (its own, or the tile's row 0 as a stand-in): straight-line, loads overlap\n"
       "      bool okk = true;\n"
       "      const i64 row = base + (r[k] >= 0 ? r[k] : 0);\n"
       "      const bool pass = " + stage_of_q + "false;\n"
       "      f[k] = r[k] >= 0 && pass && okk;\n"
       "      if (r[k] >= 0 && !okk) ok = false;\n"
       "    }\n"
       "  }\n";
  // fold of one surviving row (fold mode) / its emitted expressions (emit mode)
  g.reset();
  s += "  __device__ __forceinline__ static void fold_row(const PDesc &d, const i64 row, i64 *tab, bool &ok) {\n";
  if (d.nemits == 0) {
    std::string keyexpr = "  i64 key = 0;\n";
    for (int q = 0; q < d.nkeys; q++) {
      const std::string t = g.term(d.key[q]);
      keyexpr += "  key |= (i64)((u64)" + t + " << " + std::to_string(d.key_shl[q]) + ");\n";
    }
    std::string vals;
    for (int j = 0; j < d.nfolds; j++) {
      if (d.fold_op[j] == VDL_FOLD_CHOOSE || d.fold_op[j] == VDL_FOLD_COUNT) continue;
      snprintf(b, sizeof b, "  table_update(%d, tab + (size_t)%d * d.domain + key, ", d.fold_op[j], j);
      vals += b + g.product(d.fold[j]) + ");\n";
    }
    s += g.body + keyexpr + "  key &= d.key_mask;\n  if ((u64)key >= (u64)d.domain) { ok = false; return; }\n" + vals;
    snprintf(b, sizeof b, "  atomicAdd((unsigned long long *)(tab + (size_t)%d * d.domain + key), 1ull);\n  atomicMin((long long *)(tab + (size_t)%d * d.domain + key), (long long)(d.row_base + row));\n",
             d.nfolds, d.nfolds + 1);
    s += b;
  }
  s += "  }\n";
  g.reset();
  s += "  __device__ __forceinline__ static void emit_row(const PDesc &d, const i64 row, const i64 at, bool &ok) {\n";
  {
    std::string st;
    for (int e = 0; e < d.nemits; e++) { snprintf(b, sizeof b, "  d.emit_out[%d][at] = ", e); st += b + g.product(d.emit[e]) + ";\n"; }
    s += g.body + st;
  }
  snprintf(b, sizeof b, "  }\n};\nextern \"C\" __global__ void __launch_bounds__(P_THREADS, %d) vdl_probe_jit(const __grid_constant__ PDesc d) { probe_body<ProbeJit>(d, threadIdx.x); }\n", blocks);
  return s + b;
}

static cudaKernel_t probe_jit_compile(vdl_ctx *ctx, const PDesc &d, size_t smem, int p_sub, int blocks, bool *ok, std::string *log) {
  const std::string src = probe_jit_source(d, p_sub, blocks);
  static const char *const headers[] = {EMB_vdl_cuda_h, EMB_vdl_device_cuh, EMB_vdl_probe_kernel_cuh};
  static const char *const names[] = {"vdl_cuda.h", "vdl_device.cuh", "vdl_probe_kernel.cuh"};
  if (getenv("VDL_DEBUG_JIT")) fprintf(stderr, "[vdl jit] probe:\n%s\n", src.c_str());
  cudaKernel_t kh = vdl_jit_kernel(ctx, "probe|" + src, src, "vdl_probe_jit", 3, headers, names, ok, log);
  if (kh && smem > 48 * 1024 && cudaFuncSetAttribute((const void *)kh, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) {
    cudaGetLastError();
    return nullptr;
  }
  return kh;
}

// Host-only check (no GPU): print a two-stage descriptor with a lookup chain, a range set, a column comparison, an
// indicator and two folds as CUDA C and compile it with NVRTC for sm_100a; then an emit-mode one.
extern "C" int vdl_probe_jit_selftest(char *log, int log_capacity) {
  if (log && log_capacity > 0) log[0] = 0;
  PDesc d;
  memset(&d, 0, sizeof d);
  d.nleaves = 4;
  d.leaf[0] = PLeaf{nullptr, 10, 0, -1}; d.leaf[1] = PLeaf{nullptr, 10, 1, 0}; d.leaf[2] = PLeaf{nullptr, 10, 0, 1}; d.leaf[3] = PLeaf{nullptr, 10, 1, -1};
  d.npreds = 2;
  d.pred[0].kind = 0; d.pred[0].t = PTerm{1, 0, 0, 1}; d.pred[0].lo = 5; d.pred[0].span = 7; d.pred[0].nmore = 1; d.pred[0].lo_more[0] = 40; d.pred[0].span_more[0] = 0;
  d.pred[1].kind = 1; d.pred[1].cmp = VDL_CMP_GE; d.pred[1].t = PTerm{2, 3, -1, 2}; d.pred[1].u = PTerm{3, 0, 0, 1};
  d.nind = 1; d.ind[0] = d.pred[0];
  d.nkeys = 1; d.key[0] = PTerm{2, 3, -2, 1}; d.key_shl[0] = 1; d.key_mask = 31; d.domain = 32;
  d.nfolds = 3; d.fold_op[0] = VDL_FOLD_SUM; d.fold[0].nfac = 2; d.fold[0].f[0] = PTerm{3, 0, 0, 1}; d.fold[0].f[1] = PTerm{-3, 0, 0, 1};
  d.fold_op[1] = VDL_FOLD_MIN; d.fold[1].nfac = 1; d.fold[1].f[0] = PTerm{-2, 0, 0, 1};
  d.fold_op[2] = VDL_FOLD_COUNT;
  std::string l;
  bool ok1 = false, ok2 = false;
  probe_jit_compile(nullptr, d, 0, 4, 12, &ok1, &l);
  if (l == "NVRTC is not installed") return VDL_ENOTFOUND;
  d.nfolds = 0; d.nkeys = 0; d.nemits = 2; d.emit[0] = d.fold[0]; d.emit[1].nfac = 1; d.emit[1].f[0] = PTerm{2, 0, 0, 1};
  if (ok1) probe_jit_compile(nullptr, d, 0, 4, 12, &ok2, &l);
  if (log && log_capacity > 1) snprintf(log, (size_t)log_capacity, "%s", l.c_str());
  return ok1 && ok2 ? VDL_OK : VDL_ECUDA;
}

struct vdl_probe {
  vdl_ctx *ctx = nullptr;
  PDesc pd;
  FoldCombine cb;                      // fold mode: the finalize's descriptor, the peer exchange, the results
  bool folding = true, ran = false, fetched = false;
  vdl_vec table = 0;
  i64 *h_out = nullptr;                // emit mode: host copy of the survivor count
  i64 *d_total = nullptr;              // [0] survivors (emit mode)
  unsigned int *d_ticket = nullptr;
  unsigned long long *d_state = nullptr;
  vdl_vec emit_vec[VDL_MAX_EMITS] = {0};
  i64 nselected = -1;
  int grid = 1;
  size_t smem = 0;
  KernelTimer timer;
  cudaKernel_t jit_kernel = nullptr;   // the descriptor printed as CUDA C and compiled at run time (probe_jit_source)
  // identity of the leaf columns at prepare time (device pointers and lengths are baked into the descriptor)
  int nleaves = 0;
  vdl_vec leaf_handle[VDL_MAX_LEAVES] = {0};
  u64 leaf_gen[VDL_MAX_LEAVES] = {0};
};

bool vdl_probe_current(vdl_probe *p) {
  for (int l = 0; l < p->nleaves; l++) {
    u64 g;
    if (!vec_identity(p->ctx, p->leaf_handle[l], &g) || g != p->leaf_gen[l]) return false;
  }
  return true;
}

static bool term_ok(const vdl_term &t, int nleaves, int nind = 0) { return t.leaf >= -2 - nind && t.leaf < nleaves && t.shr >= 0 && t.shr < 64; }
static PTerm to_p(const vdl_term &t) { return PTerm{t.leaf, t.shr, t.a, t.b}; }

extern "C" int vdl_abi_sizeof_probe_desc(void) { return (int)sizeof(vdl_probe_desc); }

extern "C" int vdl_probe_prepare(vdl_ctx *ctx, const vdl_probe_desc *desc, vdl_probe **out) {
  if (!ctx || !desc || !out) return VDL_EINVAL;
  *out = nullptr;
  if (desc->nleaves < 1 || desc->nleaves > VDL_MAX_LEAVES || desc->npreds < 0 || desc->npreds > VDL_MAX_PROBE_PREDS ||
      desc->nkeys < 0 || desc->nkeys > VDL_MAX_KEYS || desc->nfolds < 0 || desc->nfolds > VDL_MAX_AGGS || desc->nemits < 0 ||
      desc->nemits > VDL_MAX_EMITS || desc->nposts < 0 || desc->nposts > VDL_MAX_POSTS)
    return vdl_fail(ctx, VDL_EINVAL, "probe: descriptor counts out of range");
  if ((desc->nfolds > 0) == (desc->nemits > 0)) return vdl_fail(ctx, VDL_EINVAL, "probe: exactly one of folds / emits must be given");
  if (desc->rows < 0) return vdl_fail(ctx, VDL_EINVAL, "probe: negative row count");
  VDL_CUDA(ctx, cudaSetDevice(ctx->device));
  vdl_probe *p = new vdl_probe();
  p->ctx = ctx;
  PDesc &d = p->pd;
  memset(&d, 0, sizeof d);
  FinDesc &fd = p->cb.fd;
  memset(&fd, 0, sizeof fd);
  auto fail = [&](int rc) { vdl_probe_destroy(p); return rc; };
  d.rows = desc->rows;
  d.row_base = desc->row_base;
  d.nleaves = desc->nleaves;
  for (int l = 0; l < desc->nleaves; l++) {
    Vec *v = vec_get(ctx, desc->leaf[l].column);
    if (!v || v->is_range) return fail(vdl_fail(ctx, VDL_EINVAL, "probe: leaf %d is not a stored vector", l));
    int par = desc->leaf[l].parent;
    if (par >= l || par < -1) return fail(vdl_fail(ctx, VDL_EINVAL, "probe: leaf %d has parent %d (must precede it)", l, par));
    if (par < 0 && v->len < desc->rows) return fail(vdl_fail(ctx, VDL_EINVAL, "probe: fact column %s has %lld rows < %lld", v->name.c_str(), (long long)v->len, (long long)desc->rows));
    int depth = 1;
    for (int q = par; q >= 0; q = desc->leaf[q].parent) depth++;
    if (depth > P_MAX_DEPTH) return fail(vdl_fail(ctx, VDL_EUNSUPPORTED, "probe: lookup chain deeper than %d", P_MAX_DEPTH));
    d.leaf[l] = PLeaf{v->ptr, v->len, v->dtype == VDL_I32, par};
    p->leaf_handle[l] = desc->leaf[l].column;
    p->leaf_gen[l] = v->gen;
    p->nleaves = l + 1;
  }
  auto to_pred = [&](const vdl_probe_pred &s, PPred *o) -> bool {
    if ((s.kind != 0 && s.kind != 1) || !term_ok(s.t, desc->nleaves) || (s.kind == 1 && (!term_ok(s.u, desc->nleaves) || s.cmp < VDL_CMP_EQ || s.cmp > VDL_CMP_LE)) ||
        s.nmore < 0 || s.nmore > VDL_MAX_MORE_RANGES)
      return false;
    memset(o, 0, sizeof *o);
    o->kind = s.kind; o->cmp = s.cmp; o->t = to_p(s.t); o->u = to_p(s.u);
    if (s.kind == 0) {
      // empty ranges are dropped; no range left: never true (0 in [1, 1])
      i64 lo[1 + VDL_MAX_MORE_RANGES], hi[1 + VDL_MAX_MORE_RANGES];
      int n = 0;
      if (s.lo <= s.hi) { lo[n] = s.lo; hi[n++] = s.hi; }
      for (int k = 0; k < s.nmore; k++) if (s.lo_more[k] <= s.hi_more[k]) { lo[n] = s.lo_more[k]; hi[n++] = s.hi_more[k]; }
      if (n == 0) { o->t = PTerm{-1, 0, 0, 0}; o->lo = 1; o->span = 0; return true; }
      o->lo = lo[0]; o->span = (u64)hi[0] - (u64)lo[0];
      o->nmore = n - 1;
      for (int k = 1; k < n; k++) { o->lo_more[k - 1] = lo[k]; o->span_more[k - 1] = (u64)hi[k] - (u64)lo[k]; }
    }
    return true;
  };
  d.npreds = desc->npreds;
  for (int q = 0; q < desc->npreds; q++)
    if (!to_pred(desc->pred[q], &d.pred[q])) return fail(vdl_fail(ctx, VDL_EINVAL, "probe: bad predicate %d", q));
  if (desc->nindicators < 0 || desc->nindicators > VDL_MAX_INDICATORS) return fail(vdl_fail(ctx, VDL_EINVAL, "probe: %d indicators", desc->nindicators));
  d.nind = desc->nindicators;
  for (int q = 0; q < desc->nindicators; q++)
    if (!to_pred(desc->indicator[q], &d.ind[q])) return fail(vdl_fail(ctx, VDL_EINVAL, "probe: bad indicator %d", q));
  d.nkeys = desc->nkeys;
  for (int q = 0; q < desc->nkeys; q++) {
    if (!term_ok(desc->key[q], desc->nleaves, desc->nindicators) || desc->key_shl[q] < 0 || desc->key_shl[q] > 63) return fail(vdl_fail(ctx, VDL_EINVAL, "probe: bad key part %d", q));
    d.key[q] = to_p(desc->key[q]);
    d.key_shl[q] = desc->key_shl[q];
  }
  auto prod = [&](const vdl_product &s, PProd *o) {
    if (s.nfactors < 0 || s.nfactors > VDL_MAX_FACTORS) return false;
    o->nfac = s.nfactors;
    for (int t = 0; t < s.nfactors; t++) { if (!term_ok(s.factor[t], desc->nleaves, desc->nindicators)) return false; o->f[t] = to_p(s.factor[t]); }
    return true;
  };
  p->folding = desc->nfolds > 0;
  d.nfolds = desc->nfolds;
  d.nemits = desc->nemits;
  d.ntiles = (desc->rows + P_TILE - 1) / P_TILE;
  d.errflag = ctx->d_errflag;
  if (cudaMalloc(&p->d_ticket, sizeof(unsigned int)) != cudaSuccess || cudaMalloc(&p->d_total, 2 * sizeof(i64)) != cudaSuccess)
    return fail(vdl_fail(ctx, VDL_ENOMEM, "probe: counters"));
  d.ticket = p->d_ticket;
  d.total = p->d_total;
  if (p->folding) {
    if (desc->nkeys == 0 ? desc->domain != 1 : (desc->domain < 1 || desc->domain > (1 << 22)))
      return fail(vdl_fail(ctx, VDL_EUNSUPPORTED, "probe: key domain %lld not supported", (long long)desc->domain));
    d.key_mask = desc->key_mask;
    d.domain = desc->domain;
    for (int j = 0; j < desc->nfolds; j++) {
      int op = desc->fold[j].op;
      if (op < VDL_FOLD_SUM || op > VDL_FOLD_COUNT || !prod(desc->fold[j].value, &d.fold[j])) return fail(vdl_fail(ctx, VDL_EINVAL, "probe: bad fold %d", j));
      d.fold_op[j] = op;
    }
    int rc = vec_new(ctx, VDL_I64, (i64)(d.nfolds + 2) * d.domain, &p->table);
    if (rc) return fail(rc);
    d.table = (i64 *)ctx->vecs[p->table].ptr;
    size_t tb = (size_t)(d.nfolds + 2) * d.domain * 8;
    d.smem_table = tb <= P_SMEM_TABLE_BYTES;
    p->smem = d.smem_table ? tb : 0;
    for (int q = 0; q < desc->nposts; q++) {
      const vdl_post_op &P = desc->post[q];
      auto okk = [&](int kind, i64 v) { return kind == VDL_POST_CONST || (kind == VDL_POST_FOLD && v >= 0 && v < desc->nfolds) || (kind == VDL_POST_POST && v >= 0 && v < q); };
      if (P.op < 0 || P.op > VDL_MODULO || !okk(P.a_kind, P.a) || !okk(P.b_kind, P.b)) return fail(vdl_fail(ctx, VDL_EINVAL, "probe: bad post op %d", q));
      fd.post[q] = P;
    }
    // the table's layout for the merge: fold j in row j (a FoldChoose's value too: nacc = 0), count, first row
    fd.cnt_idx = d.nfolds;
    fd.first_idx = d.nfolds + 1;
    fd.acc_op[fd.cnt_idx] = VDL_FOLD_SUM;
    for (int j = 0; j < d.nfolds; j++) {
      fd.out_kind[j] = d.fold_op[j] == VDL_FOLD_CHOOSE;
      fd.out_idx[j] = d.fold_op[j] == VDL_FOLD_COUNT ? fd.cnt_idx : j;
      fd.acc_op[j] = d.fold_op[j];
      fd.nchoose += d.fold_op[j] == VDL_FOLD_CHOOSE;
    }
    static const FoldTexts texts = {"probe finalize: nranks %d without gathered partials",
                                    "probe: peer exchange requested before vdl_probe_set_peers",
                                    "probe ran for an external combine: call vdl_probe_finalize first",
                                    "probe: a peer GPU never delivered its partial table (exchange timed out)",
                                    "probe: %lld rows had a lookup index or group key out of range"};
    if (p->cb.allocate(ctx, &texts, d.table, (i64)(d.nfolds + 2) * d.domain, d.domain, d.nfolds, desc->nposts))
      return fail(vdl_fail(ctx, VDL_ENOMEM, "probe: result buffers"));
  } else {
    for (int e = 0; e < desc->nemits; e++)
      if (!prod(desc->emit[e], &d.emit[e])) return fail(vdl_fail(ctx, VDL_EINVAL, "probe: bad emit %d", e));
    if (cudaMalloc(&p->d_state, (size_t)std::max<i64>(1, d.ntiles) * 8) != cudaSuccess) return fail(vdl_fail(ctx, VDL_ENOMEM, "probe: tile states"));
    d.tile_state = p->d_state;
    if (cudaHostAlloc(&p->h_out, 2 * sizeof(i64), cudaHostAllocDefault) != cudaSuccess) return fail(vdl_fail(ctx, VDL_ENOMEM, "probe: host counter"));
  }
  // prefetch list: fact-table leaves (no parent) a predicate stage starts from.  Distance 0 = this tile's own columns,
  // pulled in while its first stage runs (measured best: Q12 -9 %, Q19 -10 %, Q3 -8 %, Q5 -4 % kernel time; a few tiles
  // ahead is as good, 256+ tiles ahead thrashes L2).  VDL_PROBE_PREFETCH=off disables it, =N looks N tiles ahead.
  d.npf = 0;
  d.pf_dist = 0;
  const char *pfenv = getenv("VDL_PROBE_PREFETCH");
  if (pfenv && *pfenv >= '0' && *pfenv <= '9') d.pf_dist = atoi(pfenv);
  if (!(pfenv && !strcmp(pfenv, "off"))) {
    std::vector<char> want(desc->nleaves, 0);
    auto root = [&](int l) { while (l >= 0 && desc->leaf[l].parent >= 0) l = desc->leaf[l].parent; return l; };
    for (int q = 0; q < desc->npreds; q++)
      for (int l : {desc->pred[q].t.leaf, desc->pred[q].kind == 1 ? desc->pred[q].u.leaf : -1}) { int r = root(l); if (r >= 0) want[r] = 1; }
    for (int l = 0; l < desc->nleaves; l++)
      if (want[l] && d.leaf[l].ptr) { d.pf_ptr[d.npf] = (const unsigned char *)d.leaf[l].ptr; d.pf_shift[d.npf] = d.leaf[l].w4 ? 2 : 3; d.npf++; }
  }
  p->timer.create();
  int per_sm = P_BLOCKS;
  p->grid = (int)std::max<i64>(1, std::min<i64>((i64)ctx->sm_count * per_sm, d.ntiles));
  if (p->smem > 48 * 1024) cudaFuncSetAttribute(probe_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p->smem);
  {   // load every kernel a step may launch now, not lazily behind a peer's spinning exchange (see FoldCombine::allocate)
    cudaFuncAttributes fa;
    cudaFuncGetAttributes(&fa, probe_kernel); cudaFuncGetAttributes(&fa, probe_init_kernel); cudaFuncGetAttributes(&fa, probe_choose_kernel);
    cudaFuncGetAttributes(&fa, probe_finalize_kernel);
    cudaGetLastError();
  }
  {   // run-time specialisation (VDL_PROBE_JIT=0 switches it off; VDL_PROBE_JIT_MIN_ROWS, default 262144)
    const char *e = getenv("VDL_PROBE_JIT");
    i64 min_rows = 1 << 18;
    if (const char *m = getenv("VDL_PROBE_JIT_MIN_ROWS")) min_rows = atoll(m);
    bool lens_ok = true;             // the generated code clamps a failed lookup to index 0: every looked-up column needs a row
    for (int l = 0; l < d.nleaves; l++) if (d.leaf[l].parent >= 0 && d.leaf[l].len < 1) lens_ok = false;
    int p_sub = 8, blocks = 8;       // measured on B200 (Q5 / Q3 / Q12 / Q19 SF10): 8 rows per thread and round, 8 blocks x 64 registers
    if (const char *s = getenv("VDL_PROBE_JIT_SUB")) p_sub = std::max(1, std::min(16, atoi(s)));
    if (const char *s = getenv("VDL_PROBE_JIT_BLOCKS")) blocks = std::max(1, std::min(16, atoi(s)));
    if (!(e && !strcmp(e, "0")) && d.rows >= min_rows && lens_ok) p->jit_kernel = probe_jit_compile(ctx, d, p->smem, p_sub, blocks, nullptr, nullptr);
  }
  *out = p;
  return VDL_OK;
}

extern "C" int vdl_probe_run(vdl_probe *p) { return vdl_probe_run_ex(p, 1); }

FoldCombine *vdl_probe_combine(vdl_probe *p) { return &p->cb; }

extern "C" int vdl_probe_exchange_bytes(vdl_probe *p, int world, int64_t *bytes) { return p && p->folding ? p->cb.exchange_bytes(world, bytes) : VDL_EINVAL; }

extern "C" int vdl_probe_set_peers(vdl_probe *p, int rank, int world, void *const *peer_buffers) {
  return p && p->folding ? p->cb.set_peers(rank, world, peer_buffers) : VDL_EINVAL;
}

extern "C" int vdl_probe_partials(vdl_probe *p, void **device_ptr, int64_t *n_int64) { return p && p->folding ? p->cb.partials(device_ptr, n_int64) : VDL_EINVAL; }

// Merge `nranks` partial tables laid out back to back (an all-gather result; NULL and 1: this rank's own) and finalize.
extern "C" int vdl_probe_finalize(vdl_probe *p, const void *all_partials, int nranks) {
  return p && p->folding ? p->cb.finalize(all_partials, nranks) : VDL_EINVAL;
}

// finalize != 0: single GPU, results on their way when this returns.  0 (fold mode): leave the complete partial
// table (FoldChoose values included) for an external combine, then vdl_probe_finalize().
extern "C" int vdl_probe_run_ex(vdl_probe *p, int finalize) {
  if (!p) return VDL_EINVAL;
  vdl_ctx *ctx = p->ctx;
  VDL_CUDA(ctx, cudaSetDevice(ctx->device));
  if (!vdl_probe_current(p))
    return vdl_fail(ctx, VDL_ESTALE, "probe: a column was rewritten or dropped after vdl_probe_prepare: prepare again");
  PDesc &d = p->pd;
  p->fetched = false;
  p->nselected = -1;
  p->cb.finalized = false;
  p->cb.ngroups = -1;
  VDL_CUDA(ctx, cudaMemsetAsync(p->d_ticket, 0, sizeof(unsigned int), ctx->stream));
  if (p->folding) {
    int nb = (int)std::min<i64>(ctx->sm_count, ((i64)(d.nfolds + 2) * d.domain + 255) / 256);
    probe_init_kernel<<<std::max(nb, 1), 256, 0, ctx->stream>>>(d);
    ctx->launches++;
  } else {
    VDL_CUDA(ctx, cudaMemsetAsync(p->d_state, 0, (size_t)std::max<i64>(1, d.ntiles) * 8, ctx->stream));
    VDL_CUDA(ctx, cudaMemsetAsync(p->d_total, 0, 2 * sizeof(i64), ctx->stream));
    // emit capacity: one vector of `rows` int64 per emitted expression (the survivors are usually far fewer; the
    // pool keeps the pages), released by the caller through the vector handles
    for (int e = 0; e < d.nemits; e++) {
      if (p->emit_vec[e]) { vdl_vec_free(ctx, p->emit_vec[e]); p->emit_vec[e] = 0; }
      VDL_TRY(vec_new(ctx, VDL_I64, d.rows, &p->emit_vec[e]));
      d.emit_out[e] = (i64 *)ctx->vecs[p->emit_vec[e]].ptr;
    }
  }
  VDL_TRY(p->timer.begin(ctx));
  if (d.rows > 0) {
    if (p->jit_kernel) {
      void *args[] = {(void *)&d};
      VDL_CUDA(ctx, cudaLaunchKernel((const void *)p->jit_kernel, dim3(p->grid), dim3(P_THREADS), args, p->smem, ctx->stream));
    } else {
      probe_kernel<<<p->grid, P_THREADS, p->smem, ctx->stream>>>(d);
    }
    ctx->launches++;
  }
  VDL_TRY(p->timer.end(ctx));
  if (p->folding && finalize == 2) {       // peer-memory combine: every rank ends with the global result, no host round trip
    VDL_TRY(p->cb.next_epoch());
    int nb = (int)std::min<i64>(ctx->sm_count, (d.domain + 255) / 256);
    probe_choose_kernel<<<std::max(nb, 1), 256, 0, ctx->stream>>>(d);
    ctx->launches++;
    VDL_TRY(p->cb.exchange());
  } else if (p->folding && finalize) {
    p->cb.fd.parts = d.table;
    p->cb.fd.seq++;
    probe_finalize_kernel<<<1, 256, 0, ctx->stream>>>(d, p->cb.fd);
    ctx->launches++;
  } else if (p->folding) {
    int nb = (int)std::min<i64>(ctx->sm_count, (d.domain + 255) / 256);
    probe_choose_kernel<<<std::max(nb, 1), 256, 0, ctx->stream>>>(d);
    ctx->launches++;
  } else {
    VDL_CUDA(ctx, cudaMemcpyAsync(p->h_out, p->d_total, sizeof(i64), cudaMemcpyDeviceToHost, ctx->stream));
  }
  VDL_CUDA(ctx, cudaGetLastError());
  p->cb.finalized = p->folding && finalize != 0;
  p->ran = true;
  return VDL_OK;
}

// Emit mode: the survivor count (the fold mode's results: FoldCombine::fetch).
static int probe_fetch(vdl_probe *p) {
  vdl_ctx *ctx = p->ctx;
  if (!p->ran) return vdl_fail(ctx, VDL_EINVAL, "probe has not run");
  if (p->fetched) return VDL_OK;
  VDL_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  p->nselected = p->h_out[0];
  for (int e = 0; e < p->pd.nemits; e++) {
    Vec &v = ctx->vecs[p->emit_vec[e]];
    v.len = p->nselected;
  }
  p->fetched = true;
  return VDL_OK;
}

extern "C" int vdl_probe_result_host(vdl_probe *p, int index, const int64_t **data, int64_t *len) {
  if (!p || !p->folding) return VDL_EINVAL;
  if (!p->ran) return vdl_fail(p->ctx, VDL_EINVAL, "probe has not run");
  return p->cb.result_host(index, data, len);
}

// Emit mode: the k-th emitted vector (length = number of surviving rows).  Ownership passes to the caller.
extern "C" int vdl_probe_emit_take(vdl_probe *p, int k, vdl_vec *out) {
  if (!p || !out || p->folding || k < 0 || k >= p->pd.nemits) return VDL_EINVAL;
  VDL_TRY(probe_fetch(p));
  if (!p->emit_vec[k]) return vdl_fail(p->ctx, VDL_EINVAL, "probe: emitted vector %d already taken", k);
  *out = p->emit_vec[k];
  p->emit_vec[k] = 0;
  return VDL_OK;
}

extern "C" int vdl_probe_last_kernel_ms(vdl_probe *p, float *ms) { return p && ms && p->ran ? p->timer.last_ms(p->ctx, ms) : VDL_EINVAL; }

extern "C" int vdl_probe_kernel_ms_stats(vdl_probe *p, int n, float *mean_ms, float *min_ms) {
  return p && n >= 1 && p->ran ? p->timer.stats(p->ctx, n, mean_ms, min_ms) : VDL_EINVAL;
}

extern "C" int vdl_probe_destroy(vdl_probe *p) {
  if (!p) return VDL_EINVAL;
  vdl_ctx *ctx = p->ctx;
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  if (p->table) vdl_vec_free(ctx, p->table);
  for (int e = 0; e < VDL_MAX_EMITS; e++)
    if (p->emit_vec[e]) vdl_vec_free(ctx, p->emit_vec[e]);
  p->cb.release();
  if (p->h_out) cudaFreeHost(p->h_out);
  if (p->d_total) cudaFree(p->d_total);
  if (p->d_ticket) cudaFree(p->d_ticket);
  if (p->d_state) cudaFree(p->d_state);
  p->timer.destroy();
  delete p;
  return VDL_OK;
}
