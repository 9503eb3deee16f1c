// Fused select -> map -> fold: ONE launch that streams the columns of a table shard through shared
// memory with TMA bulk copies and folds products of affine column terms per group key.
//
// What it replaces in the emitted graph (reference Vlite.hs):
//   idx = FoldSelect(pos_ p, p); c_i @@ idx          solve' Select          Vlite.hs:721-730
//   key = ((c >> tz) - min) << bits | ... & hint     makeCompositeKey       Vlite.hs:1123-1170, 1111-1115
//   Partition(key) -> Scatter(x, .) -> Fold(op, ., .) solveAgg / getScatterMask Vlite.hs:1048-1098
// In the dense model (SURVEY.md App. G1) elementwise ops commute with the Gather by the selection, the
// stable Partition+Scatter only orders rows by key, and Fold emits one row per existing key in ascending
// order -- so the whole chain is "for every row that passes p: acc[key][j] op= value_j(row)", followed
// by dropping the keys that saw no row.  No intermediate vector ever reaches HBM.
//
// Kernel shape (B200, sm_100a): persistent, one CTA per SM.  Warp 0 is the producer: one elected lane
// issues `cp.async.bulk` (TMA, 1-D) copies of TILE rows of every column into a ring of shared-memory
// stages, completion tracked by mbarriers (expect_tx).  The other 8 warps are consumers: they wait on
// the stage's "full" barrier, evaluate predicate / key / products straight from shared memory (column
// chosen by runtime index = just an address, so ONE kernel serves every plan), and release the stage
// through its "empty" barrier.  Ungrouped folds accumulate in registers; grouped folds accumulate in
// lane-private shared-memory tables (plain LDS/STS read-modify-write, no atomics, no bank conflicts)
// over a per-CTA compacted slot map so that sparse key domains (Q1: 6 of 32 slots) stay small.
// HBM traffic = the columns, once.  Roofline: HBM (DESIGN.md section 4).
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <map>
#include <vector>

#include "vdl_internal.h"

#include "vdl_fused_kernel.cuh"

// ------------------------------------------------------------------------------ host side
typedef void (*scan_kernel_fn)(const KDesc, const FinDesc, const XDesc);
struct vdl_fused {
  vdl_ctx *ctx = nullptr;
  KDesc kd;
  FoldCombine cb;                 // the finalize's descriptor, the peer exchange, the results (views: out[])
  vdl_vec table = 0;
  vdl_vec out[VDL_MAX_AGGS] = {0};
  int nout = 0;
  bool always_false = false, rs = false;
  unsigned int *d_done = nullptr; // ticket counter of the scan kernel's last-CTA epilogue
  // register slots: kernels by slot count; the launch picks the smallest count that covers the groups the previous
  // run of this scan produced (more slots = more predicated work per row; too few = keys on the slow global path)
  scan_kernel_fn rs_kernel[9] = {nullptr};
  int rs_gmax = 0;
  i64 groups_seen = -1;
  size_t smem_bytes = 0;
  int grid = 1, nc = 256, r = 4;
  scan_kernel_fn kernel = nullptr;
  const char *shape = "generic";
  KernelTimer timer;
  // run-time specialised kernels (vdl_jit_kernel): the shape-traits class generated from THIS descriptor
  bool jit = false;
  std::string jit_struct, jit_name;     // the generated `struct ShapeJit {...}` text; "jit:<hash>"
  cudaKernel_t jit_kernel = nullptr;    // shared-memory tables (G = 0)
  cudaKernel_t jit_rs_kernel[9] = {nullptr};
  bool jit_rs_tried[9] = {false};
  // identity of the columns at prepare time (the proofs above hold for exactly this data)
  int ncols = 0;
  vdl_vec col_handle[VDL_MAX_COLS] = {0};
  u64 col_gen[VDL_MAX_COLS] = {0};
};

bool vdl_fused_current(vdl_fused *f) {
  for (int c = 0; c < f->ncols; c++) {
    u64 g;
    if (!vec_identity(f->ctx, f->col_handle[c], &g) || g != f->col_gen[c]) return false;
  }
  return true;
}

#include "vdl_shapes.cuh"

template <class S>
static scan_kernel_fn scan_kernel_for(int nc, int r) {
  if (nc == 512) return r == 4 ? fused_scan_fold_kernel<S, 512, 4, 0> : (r == 2 ? fused_scan_fold_kernel<S, 512, 2, 0> : fused_scan_fold_kernel<S, 512, 1, 0>);
  return r == 4 ? fused_scan_fold_kernel<S, 256, 4, 0> : (r == 2 ? fused_scan_fold_kernel<S, 256, 2, 0> : fused_scan_fold_kernel<S, 256, 1, 0>);
}
// register-slot instantiations (geometries: rs_geometries) for g of the shape's RS_G slots in registers
template <class S, int G>
static scan_kernel_fn rs_kernel_for_g(int nc, int r) {
  // consumer warps + the producer warp are dealt round-robin to the 4 SM sub-partitions (16 K registers each):
  // 11 + 1 warps -> 3 per sub-partition -> 168 registers per thread; 15 + 1 -> 4 -> 128; 7 + 1 -> 2 -> 255
  if (nc == 352 && r == 4) return fused_scan_fold_kernel<S, 352, 4, G>;
  if (nc == 352 && r == 2) return fused_scan_fold_kernel<S, 352, 2, G>;
  if (nc == 480 && r == 2) return fused_scan_fold_kernel<S, 480, 2, G>;
  return nullptr;
}
template <class S>
static scan_kernel_fn rs_kernel_for(int nc, int r, int g) {
  if constexpr (S::RS_G > 0) {
    static_assert(S::RS_G == 8, "instantiate the slot counts this shape allows");
    if (g == 8) return rs_kernel_for_g<S, 8>(nc, r);
    if (g == 6) return rs_kernel_for_g<S, 6>(nc, r);
    if (g == 4) return rs_kernel_for_g<S, 4>(nc, r);
  }
  return nullptr;
}
static const int rs_slot_counts[] = {4, 6, 8};
static const int rs_geometries[][2] = {{352, 4}, {352, 2}, {480, 2}};

// does the prepared descriptor satisfy every assumption static shape S compiles in?
static bool flags_ok(int fl, const KAffine &a) {
  if (((fl & FF_CONST) != 0) != (a.col == -1) || ((fl & FF_ROWID) != 0) != (a.col == -2)) return false;
  if (a.col >= 0 && ((fl & FF_W4) != 0) != (a.w4 != 0)) return false;
  if ((fl & FF_SHR0) && a.shr != 0) return false;
  if ((fl & FF_B1) && a.b != 1) return false;
  if ((fl & FF_BM1) && a.b != -1) return false;
  if ((fl & FF_A0) && a.a != 0) return false;
  if ((fl & FF_NARROW) && !a.narrow) return false;
  return true;
}
template <class S>
static bool shape_matches(const KDesc &k) {
  if (k.npreds != S::NPREDS || k.nkeys != S::NKEYS || k.nacc != S::NACC) return false;
  for (int i = 0; i < k.npreds; i++)
    if (k.pred[i].w4 != S::PRED_MODE[i] || (S::PRED_SHR0[i] && k.pred[i].shr != 0)) return false;
  for (int i = 0; i < k.nkeys; i++) {
    if (!flags_ok(S::KEY_FLAGS[i], k.key[i].e) || (S::KEY_SHL0[i] && k.key[i].shl != 0)) return false;
    if (S::KEY32 && !k.key[i].e.narrow) return false;
  }
  if (S::KEY32 && (k.key_mask < 0 || k.key_mask > INT32_MAX || k.key_mask >= k.domain)) return false;
  for (int j = 0; j < k.nacc; j++) {
    if (k.acc[j].op != S::ACC_OP[j] || k.acc[j].chain != S::ACC_CHAIN[j] || k.acc[j].nfac != S::ACC_NFAC[j]) return false;
    for (int t = 0; t < k.acc[j].nfac; t++)
      if (!flags_ok(S::FAC[j][t], k.acc[j].fac[t])) return false;
  }
  return true;
}


// ---- run-time specialisation of the scan (NVRTC) ---------------------------------------------------------------------
// What the two hand-written shapes of vdl_shapes.cuh do for Q6 and Q1, done for ANY descriptor: the structure of the
// prepared descriptor (counts, widths, trivial shr / a / b, what the column statistics prove to fit 32 bits, which
// accumulators may live in registers and how) is printed as a shape-traits class, fused_scan_fold_body is instantiated
// over it by NVRTC for sm_100a and cached per context.  Every constant stays a run-time descriptor field, exactly as with
// the static shapes, so one compiled kernel serves every plan of that structure.
#include "vdl_embedded.inc"      // the three headers the generated source includes, as strings (written by build.py)

static int flags_of(const KAffine &a) {
  if (a.col == -1) return FF_CONST;
  int fl = 0;
  if (a.col == -2) fl |= FF_ROWID;
  else if (a.w4) fl |= FF_W4;
  if (a.shr == 0) fl |= FF_SHR0;
  if (a.b == 1) fl |= FF_B1;
  else if (a.b == -1) fl |= FF_BM1;
  if (a.a == 0) fl |= FF_A0;
  if (a.col >= 0 && a.narrow) fl |= FF_NARROW;
  return fl;
}

static bool jit_key32(const KDesc &k) {
  if (k.nkeys == 0 || k.key_mask < 0 || k.key_mask > INT32_MAX || k.key_mask >= k.domain) return false;
  for (int i = 0; i < k.nkeys; i++)
    if (!(k.key[i].e.col >= 0 && k.key[i].e.narrow)) return false;     // low 32 bits of every part are exact; OR / AND / << are bitwise
  return true;
}

static std::string jit_shape_struct(const KDesc &k, int key32, int rs_g, const int *rk) {
  std::string s = "struct ShapeJit {\n  static constexpr bool kStatic = true;\n";
  char b[256];
  auto list = [&](const char *name, const char *dim, int n, auto get) {
    s += std::string("  static constexpr int ") + name + "[" + dim + "] = {";
    for (int i = 0; i < n; i++) { snprintf(b, sizeof b, "%s%d", i ? ", " : "", (int)get(i)); s += b; }
    s += "};\n";
  };
  snprintf(b, sizeof b, "  static constexpr int NPREDS = %d, NKEYS = %d, NACC = %d, KEY32 = %d, RS_G = %d;\n", k.npreds, k.nkeys, k.nacc, key32, rs_g);
  s += b;
  list("PRED_MODE", "VDL_MAX_PREDS", k.npreds, [&](int i) { return k.pred[i].w4; });
  list("PRED_SHR0", "VDL_MAX_PREDS", k.npreds, [&](int i) { return k.pred[i].shr == 0; });
  list("KEY_FLAGS", "VDL_MAX_KEYS", k.nkeys, [&](int i) { return flags_of(k.key[i].e); });
  list("KEY_SHL0", "VDL_MAX_KEYS", k.nkeys, [&](int i) { return k.key[i].shl == 0; });
  list("ACC_OP", "K_MAX_ACC", k.nacc, [&](int j) { return k.acc[j].op; });
  list("ACC_CHAIN", "K_MAX_ACC", k.nacc, [&](int j) { return k.acc[j].chain; });
  list("ACC_NFAC", "K_MAX_ACC", k.nacc, [&](int j) { return k.acc[j].nfac; });
  list("ACC_RK", "K_MAX_ACC", k.nacc, [&](int j) { return rs_g > 0 ? rk[j] : 0; });
  s += "  static constexpr int FAC[K_MAX_ACC][VDL_MAX_FACTORS] = {";
  for (int j = 0; j < k.nacc; j++) {
    s += j ? ", {" : "{";
    for (int t = 0; t < k.acc[j].nfac; t++) { snprintf(b, sizeof b, "%s%d", t ? ", " : "", flags_of(k.acc[j].fac[t])); s += b; }
    s += "}";
  }
  s += "};\n};\n";
  return s;
}

static cudaKernel_t jit_scan_compile(vdl_ctx *ctx, const std::string &shape_struct, int nc, int r, int g, int smem_max, bool *ok, std::string *log) {
  char b[512];
  snprintf(b, sizeof b,
           "extern \"C\" __global__ void __launch_bounds__(%d, 1) vdl_scan_jit(const __grid_constant__ KDesc d, const __grid_constant__ FinDesc fd, "
           "const __grid_constant__ XDesc xd) {\n  fused_scan_fold_body<ShapeJit, %d, %d, %d>(d, fd, xd);\n}\n", nc + 32, nc, r, g);
  const std::string src = std::string("#include \"vdl_fused_kernel.cuh\"\n") + shape_struct + b;
  static const char *const headers[] = {EMB_vdl_cuda_h, EMB_vdl_device_cuh, EMB_vdl_fused_kernel_cuh};
  static const char *const names[] = {"vdl_cuda.h", "vdl_device.cuh", "vdl_fused_kernel.cuh"};
  if (getenv("VDL_DEBUG_JIT")) fprintf(stderr, "[vdl jit] fused scan nc=%d r=%d g=%d:\n%s\n", nc, r, g, shape_struct.c_str());
  cudaKernel_t kh = vdl_jit_kernel(ctx, "scan|" + src, src, "vdl_scan_jit", 3, headers, names, ok, log);
  if (kh && cudaFuncSetAttribute((const void *)kh, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_max) != cudaSuccess) {
    cudaGetLastError();
    if (ok) *ok = false;
    return nullptr;
  }
  return kh;
}

// Host-only check (no GPU): generate the shape of a Q1-like descriptor and compile it with NVRTC for sm_100a.
extern "C" int vdl_scan_jit_selftest(char *log, int log_capacity) {
  if (log && log_capacity > 0) log[0] = 0;
  KDesc k;
  memset(&k, 0, sizeof k);
  k.npreds = 2; k.nkeys = 2; k.nacc = 4; k.domain = 32; k.key_mask = 31;
  k.pred[0].w4 = 1; k.pred[1].w4 = 2; k.pred[1].shr = 3;
  for (int i = 0; i < 2; i++) { k.key[i].e = KAffine{i, 3, -2, 1, 0, 0, 1, 0}; k.key[i].shl = i ? 0 : 2; }
  k.acc[0].nfac = 1; k.acc[0].fac[0] = KAffine{2, 0, 0, 1, 0, 0, 1, 0};
  k.acc[1].nfac = 2; k.acc[1].fac[0] = KAffine{3, 0, 0, 1, 0, 1, 0, 0}; k.acc[1].fac[1] = KAffine{2, 0, 100, -1, 0, 0, 1, 0};
  k.acc[2].nfac = 0;
  k.acc[3].op = 1; k.acc[3].nfac = 1; k.acc[3].fac[0] = KAffine{-2, 0, 0, 1, 0, 0, 0, 0};
  const int rk[K_MAX_ACC] = {RK_N32, RK_MADW, RK_N32, RK_FIRST};
  std::string l;
  bool ok1 = false, ok2 = false;
  jit_scan_compile(nullptr, jit_shape_struct(k, 1, 8, rk), 352, 4, 6, 0, &ok1, &l);
  if (l == "NVRTC is not installed") return VDL_ENOTFOUND;
  if (ok1) jit_scan_compile(nullptr, jit_shape_struct(k, 0, 0, rk), 512, 4, 0, 0, &ok2, &l);
  if (log && log_capacity > 1) snprintf(log, (size_t)log_capacity, "%s", l.c_str());
  return ok1 && ok2 ? VDL_OK : VDL_ECUDA;
}

static bool affine_ok(const vdl_affine &a, int ncols) { return a.column >= -2 && a.column < ncols && a.shr >= 0 && a.shr < 64; }
static KAffine to_k(const vdl_affine &a) { return KAffine{a.column, a.shr, a.a, a.b, 0, 0, 0, 0}; }

extern "C" int vdl_fused_prepare(vdl_ctx *ctx, const vdl_fused_desc *desc, vdl_fused **out) {
  if (!ctx || !desc || !out) return VDL_EINVAL;
  *out = nullptr;
  if (desc->ncolumns < 1 || desc->ncolumns > VDL_MAX_COLS) return vdl_fail(ctx, VDL_EINVAL, "fused scan: %d columns (1..%d)", desc->ncolumns, VDL_MAX_COLS);
  if (desc->npreds < 0 || desc->npreds > VDL_MAX_PREDS || desc->nkeys < 0 || desc->nkeys > VDL_MAX_KEYS || desc->nfolds < 1 || desc->nfolds > VDL_MAX_AGGS)
    return vdl_fail(ctx, VDL_EINVAL, "fused scan: preds/keys/folds out of range");
  if (desc->domain < 1 || desc->domain > (1 << 20)) return vdl_fail(ctx, VDL_EUNSUPPORTED, "fused scan: key domain %lld not in [1, 2^20]", (long long)desc->domain);
  if (desc->nkeys == 0 && desc->domain != 1) return vdl_fail(ctx, VDL_EINVAL, "fused scan: no key parts but domain %lld", (long long)desc->domain);
  if (desc->nposts < 0 || desc->nposts > VDL_MAX_POSTS) return vdl_fail(ctx, VDL_EINVAL, "fused scan: %d post ops (0..%d)", desc->nposts, VDL_MAX_POSTS);
  for (int q = 0; q < desc->nposts; q++) {
    const vdl_post_op &P = desc->post[q];
    auto ok = [&](int kind, i64 v) { return kind == VDL_POST_CONST || (kind == VDL_POST_FOLD && v >= 0 && v < desc->nfolds) || (kind == VDL_POST_POST && v >= 0 && v < q); };
    if (P.op < 0 || P.op > VDL_MODULO || !ok(P.a_kind, P.a) || !ok(P.b_kind, P.b)) return vdl_fail(ctx, VDL_EINVAL, "fused scan: bad post op %d", q);
  }
  VDL_CUDA(ctx, cudaSetDevice(ctx->device));

  vdl_fused *f = new vdl_fused();
  f->ctx = ctx;
  KDesc &k = f->kd;
  memset(&k, 0, sizeof k);
  FinDesc &fd = f->cb.fd;
  memset(&fd, 0, sizeof fd);
  k.rows = desc->rows;
  k.row_base = desc->row_base;
  k.key_mask = desc->key_mask;
  k.domain = desc->domain;
  k.ncols = desc->ncolumns;
  k.errflag = ctx->d_errflag;
  int rowbytes = 0;
  for (int c = 0; c < desc->ncolumns; c++) {
    Vec *v = vec_get(ctx, desc->column[c]);
    if (!v || v->is_range) { delete f; return vdl_fail(ctx, VDL_EINVAL, "fused scan: column %d is not a stored column", c); }
    if (v->len < desc->rows) { delete f; return vdl_fail(ctx, VDL_EINVAL, "fused scan: column %s has %lld rows < %lld", v->name.c_str(), (long long)v->len, (long long)desc->rows); }
    k.col[c] = v->ptr;
    k.width[c] = v->dtype;
    rowbytes += v->dtype;
    f->col_handle[c] = desc->column[c];
    f->col_gen[c] = v->gen;
  }
  f->ncols = desc->ncolumns;
  for (int i = 0; i < desc->npreds; i++) {
    const vdl_range_pred &p = desc->pred[i];
    if (p.column < 0 || p.column >= desc->ncolumns || p.shr < 0 || p.shr > 63) { delete f; return vdl_fail(ctx, VDL_EINVAL, "fused scan: bad predicate %d", i); }
    if (p.lo > p.hi) f->always_false = true;
    k.pred[k.npreds++] = KPred{p.column, p.shr, p.lo, (u64)p.hi - (u64)p.lo, 0, 0, 0, 0};
  }
  for (int i = 0; i < desc->nkeys; i++) {
    if (!affine_ok(desc->key[i].e, desc->ncolumns) || desc->key[i].shl < 0 || desc->key[i].shl > 63) { delete f; return vdl_fail(ctx, VDL_EINVAL, "fused scan: bad key part %d", i); }
    k.key[k.nkeys++] = KKey{to_k(desc->key[i].e), desc->key[i].shl, 0};
  }
  // folds -> scan-time accumulators (+ count, + first row when a FoldChoose is present)
  f->nout = desc->nfolds;
  for (int i = 0; i < desc->nfolds; i++) {
    const vdl_fold_spec &s = desc->fold[i];
    if (s.nfactors < 0 || s.nfactors > VDL_MAX_FACTORS) { delete f; return vdl_fail(ctx, VDL_EINVAL, "fused scan: fold %d has %d factors", i, s.nfactors); }
    for (int t = 0; t < s.nfactors; t++)
      if (!affine_ok(s.factor[t], desc->ncolumns)) { delete f; return vdl_fail(ctx, VDL_EINVAL, "fused scan: fold %d factor %d invalid", i, t); }
    KAcc a;
    memset(&a, 0, sizeof a);
    a.nfac = s.nfactors;
    for (int t = 0; t < s.nfactors; t++) a.fac[t] = to_k(s.factor[t]);
    if (s.op == VDL_FOLD_SUM || s.op == VDL_FOLD_MIN || s.op == VDL_FOLD_MAX) {
      a.op = s.op == VDL_FOLD_SUM ? 0 : (s.op == VDL_FOLD_MIN ? 1 : 2);
      fd.out_kind[i] = 0;
      fd.out_idx[i] = k.nacc;
      k.acc[k.nacc++] = a;
    } else if (s.op == VDL_FOLD_CHOOSE) {
      if (k.nchoose == K_MAX_CHOOSE) { delete f; return vdl_fail(ctx, VDL_EUNSUPPORTED, "fused scan: more than %d FoldChoose", K_MAX_CHOOSE); }
      fd.out_kind[i] = 1;
      fd.out_idx[i] = k.nchoose;
      k.choose[k.nchoose++] = a;
    } else if (s.op == VDL_FOLD_COUNT) {
      fd.out_kind[i] = 0;
      fd.out_idx[i] = -1;   // patched to cnt_idx below
    } else { delete f; return vdl_fail(ctx, VDL_EINVAL, "fused scan: fold op %d", s.op); }
  }
  KAcc cnt;
  memset(&cnt, 0, sizeof cnt);
  k.cnt_idx = k.nacc;
  k.acc[k.nacc++] = cnt;                  // SUM of the empty product = row count per key
  k.first_idx = -1;
  if (k.nchoose) {
    KAcc first;
    memset(&first, 0, sizeof first);
    first.op = 1;
    first.nfac = 1;
    first.fac[0] = KAffine{-2, 0, 0, 1, 0, 0, 0, 0};  // MIN over the global row id
    k.first_idx = k.nacc;
    k.acc[k.nacc++] = first;
  }
  for (int i = 0; i < desc->nfolds; i++)
    if (fd.out_kind[i] == 0 && fd.out_idx[i] < 0) fd.out_idx[i] = k.cnt_idx;

  // geometry: consumer threads NC, rows per thread and tile R, ring depth, lane-private tables (or none: register slots)
  const int smem_max = ctx->smem_optin > 0 ? ctx->smem_optin : 232448;
  if ((size_t)desc->domain * 4 > 64 * 1024) { delete f; return vdl_fail(ctx, VDL_EUNSUPPORTED, "fused scan: key domain %lld too large for the shared-memory slot map", (long long)desc->domain); }
  auto set_geometry = [&](int nc, int r, int gmax, bool tables, int min_stages) -> bool {
    int tile_rows = nc * r, off = 0;
    size_t fixed = (tables ? (size_t)gmax * k.nacc * nc * 8 : 0) + (size_t)desc->domain * 4 + (size_t)gmax * 4 + 16 + 256;
    size_t per_stage = 3 * 8 + 4 + 4 + 2 * (size_t)tile_rows;   // barriers, queue count, queue
    for (int c = 0; c < k.ncols; c++) { k.soff[c] = off; off += ((tile_rows * k.width[c] + 127) / 128) * 128; }
    int stages = (int)(((long)smem_max - (long)fixed) / (long)(off + per_stage));
    if (stages < min_stages) return false;
    k.tile_rows = tile_rows; k.stage_bytes = off; k.stage_tx = tile_rows * rowbytes; k.stages = std::min(stages, 12);
    k.gmax = gmax; f->nc = nc; f->r = r;
    f->smem_bytes = (size_t)k.stages * (k.stage_bytes + per_stage) + fixed;
    k.ntiles = desc->rows / k.tile_rows;
    f->grid = (int)std::max<i64>(1, std::min<i64>(ctx->sm_count, k.ntiles));
    return true;
  };
  auto default_geometry = [&]() -> bool {
    for (int nc = 512; nc >= 256; nc /= 2) {
      // slots with lane-private tables: as many as the domain needs, up to what ~100 KB holds
      int gmax = 1;
      while (gmax < desc->domain && gmax < 64 && (size_t)(gmax * 2) * k.nacc * nc * 8 <= 120 * 1024) gmax *= 2;
      if (nc == 512 && gmax < desc->domain && gmax < 8) continue;     // too few slots: halve the consumers instead
      for (int r = 2048 / nc; r >= 1; r /= 2) {
        if (r > 4) continue;
        if (set_geometry(nc, r, gmax, true, (r == 1 && nc == 256) ? 2 : 3)) return true;
      }
    }
    return false;
  };
  if (!default_geometry()) { delete f; return vdl_fail(ctx, VDL_EUNSUPPORTED, "fused scan: %d columns x %d accumulators do not fit shared memory", k.ncols, k.nacc); }

  // prefix sharing between consecutive accumulators (ep, ep*(100-d), ep*(100-d)*(100+t) evaluate each factor once)
  for (int j = 1; j < k.nacc; j++) {
    KAcc &a = k.acc[j];
    if (j == k.cnt_idx || j == k.first_idx || j - 1 == k.cnt_idx) continue;
    // full factor list of the previous accumulator (its own chain expanded) a prefix of this one?
    std::vector<KAffine> prev;
    int q = j - 1;
    std::vector<int> chain_members;
    while (true) { chain_members.push_back(q); if (!k.acc[q].chain) break; q--; }
    for (int m = (int)chain_members.size() - 1; m >= 0; m--)
      for (int t = 0; t < k.acc[chain_members[m]].nfac; t++) prev.push_back(k.acc[chain_members[m]].fac[t]);
    bool prefix = !prev.empty() && (int)prev.size() < a.nfac;
    for (size_t t = 0; prefix && t < prev.size(); t++)
      prefix = prev[t].col == a.fac[t].col && prev[t].shr == a.fac[t].shr && prev[t].a == a.fac[t].a && prev[t].b == a.fac[t].b;
    if (prefix) {
      int np = (int)prev.size();
      for (int t = np; t < a.nfac; t++) a.fac[t - np] = a.fac[t];
      a.nfac -= np;
      a.chain = 1;
    }
  }

  // derived descriptor fields (depend on the geometry): staged offsets / width flags, 32-bit bounds for 4-byte
  // predicate columns, value bounds of every affine term from the column statistics
  struct Bound { __int128 lo, hi; };
  std::map<const KAffine *, Bound> bound;
  int place_rc = VDL_OK;
  auto place = [&](KAffine &a) {
    if (a.col == -1) { bound[&a] = Bound{a.a, a.a}; return; }
    if (a.col == -2) {
      __int128 v0 = (__int128)a.a + (__int128)a.b * k.row_base, v1 = (__int128)a.a + (__int128)a.b * (k.row_base + k.rows);
      bound[&a] = Bound{std::min(v0, v1), std::max(v0, v1)};
      return;
    }
    a.soff = k.soff[a.col];
    a.w4 = k.width[a.col] == 4;
    // narrow: leaf and a + b*leaf provably fit int32 given the column's exact min/max (cf. inferBounds, Vlite.hs:417-467).
    // The narrow device code (affine32) shifts the LOW WORD of an 8-byte value, so the raw values must fit int32 as well:
    // (x >> shr) fitting is not enough when x itself does not.
    i64 cmin, cmax;
    int rc2 = vdl_column_analyze(ctx, desc->column[a.col], &cmin, &cmax);
    if (rc2) { place_rc = rc2; return; }
    __int128 l0 = cmin >> a.shr, l1 = cmax >> a.shr;
    __int128 v0 = (__int128)a.a + (__int128)a.b * l0, v1 = (__int128)a.a + (__int128)a.b * l1;
    auto fits = [](__int128 x) { return x >= INT32_MIN && x <= INT32_MAX; };
    a.narrow = cmin <= cmax && fits(cmin) && fits(cmax) && fits(l0) && fits(l1) && fits(v0) && fits(v1) && fits(a.a) && fits(a.b);
    bound[&a] = Bound{std::min(v0, v1), std::max(v0, v1)};
  };
  auto derive = [&]() -> int {
    for (int i = 0; i < k.npreds; i++) {
      KPred &p = k.pred[i];
      p.soff = k.soff[p.col];
      p.w4 = k.width[p.col] == 4;
      if (!p.w4) {   // 8-byte column: when the column statistics say every raw value fits int32, read low words only
        i64 cmin, cmax;  // (the device shifts the low word: a raw value beyond int32 whose shifted value fits still needs all 8 bytes)
        int rc2 = vdl_column_analyze(ctx, desc->column[p.col], &cmin, &cmax);
        if (rc2) return rc2;
        if (cmin >= INT32_MIN && cmax <= INT32_MAX) p.w4 = 2;
      }
      if (p.w4) {   // values of a 4-byte column (shifted or not) lie in int32: clamp the bounds, compare in 32 bits
        i64 lo = std::max<i64>(p.lo, INT32_MIN), hi = std::min<i64>((i64)((u64)p.lo + p.span), INT32_MAX);
        if (lo > hi) f->always_false = true;
        p.lo32 = (int32_t)lo;
        p.span32 = (uint32_t)(hi - lo);
      }
    }
    for (int i = 0; i < k.nkeys; i++) place(k.key[i].e);
    for (int j = 0; j < k.nacc; j++)
      for (int t = 0; t < k.acc[j].nfac; t++) place(k.acc[j].fac[t]);
    return place_rc;
  };
  { int rc2 = derive(); if (rc2) { vdl_fused_destroy(f); return rc2; } }

  // largest |value| accumulator j can take on one row (chain expanded), saturating
  auto acc_maxabs = [&](int j) -> __int128 {
    __int128 m = 1;
    const __int128 cap = (__int128)1 << 100;
    for (int q = j;; q--) {
      for (int t = 0; t < k.acc[q].nfac; t++) {
        const Bound &b = bound[&k.acc[q].fac[t]];
        __int128 x = std::max(b.lo < 0 ? -b.lo : b.lo, b.hi < 0 ? -b.hi : b.hi);
        m = m * x;
        if (m > cap) m = cap;
      }
      if (!k.acc[q].chain) break;
    }
    return m;
  };
  // the proof accumulator j needs to be kept as `rk` by a register-slot kernel under the CURRENT geometry (vdl_shapes.cuh)
  auto rs_proof = [&](int j, int rk) -> bool {
    const i64 ntiles_all = k.ntiles + (k.ntiles * k.tile_rows < k.rows ? 1 : 0);
    const i64 tiles_per_cta = (ntiles_all + f->grid - 1) / f->grid;
    const __int128 rows_per_thread = (__int128)tiles_per_cta * 2 * f->r;   // own rows of a dense tile + a share of the queue
    if (rk == RK_N32 && (k.acc[j].op != 0 || rows_per_thread * acc_maxabs(j) > INT32_MAX)) return false;
    if (rk == RK_MADW) {          // value = a * b with a = everything but the last own factor, b = that factor
      if (k.acc[j].op != 0 || k.acc[j].nfac < 1) return false;
      const Bound &bb = bound[&k.acc[j].fac[k.acc[j].nfac - 1]];
      __int128 bmax = std::max(bb.lo < 0 ? -bb.lo : bb.lo, bb.hi < 0 ? -bb.hi : bb.hi);
      if (bmax > INT32_MAX || (bmax > 0 && acc_maxabs(j) / bmax > INT32_MAX) || acc_maxabs(j) >= ((__int128)1 << 100)) return false;
      for (int q = j;; q--) {        // every factor nonnegative: the multiply-add is unsigned
        for (int t = 0; t < k.acc[q].nfac; t++)
          if (bound[&k.acc[q].fac[t]].lo < 0) return false;
        if (!k.acc[q].chain) break;
      }
    }
    if (rk == RK_FIRST && (k.acc[j].op != 1 || j != k.first_idx || (__int128)tiles_per_cta * k.tile_rows >= INT32_MAX)) return false;
    return true;
  };
  auto rs_proofs_hold = [&](const int *rk) -> bool {
    for (int j = 0; j < k.nacc; j++) if (!rs_proof(j, rk[j])) return false;
    return true;
  };

  // Run-time specialisation first: the shape of THIS descriptor, compiled by NVRTC (cached per context).  Worth it for
  // tables of a few million rows and up (VDL_SCAN_JIT_MIN_ROWS; VDL_SCAN_JIT=0 switches it off); without NVRTC, or for
  // small tables, the precompiled instantiations below run: a static shape of vdl_shapes.cuh when one matches, else the
  // generic kernel.  Identical results whichever runs (tests/test_gpu_fuzz.py runs every random plan through both).
  auto try_jit = [&]() -> int {
    const char *e = getenv("VDL_SCAN_JIT");
    if (e && !strcmp(e, "0")) return 0;
    i64 min_rows = 4 << 20;
    if (const char *m = getenv("VDL_SCAN_JIT_MIN_ROWS")) min_rows = atoll(m);
    if (k.rows < min_rows || f->always_false) return 0;
    const int key32 = jit_key32(k);
    int rk[K_MAX_ACC] = {0};
    bool ok = false;
    std::string log;
    if (key32 && k.nacc <= 8 && k.domain <= 64 && !getenv("VDL_NO_REGISTER_SLOTS")) {
      int want_nc = 0, want_r = 0;
      if (const char *g = getenv("VDL_RS_GEOMETRY")) sscanf(g, "%d,%d", &want_nc, &want_r);
      for (auto &geo : rs_geometries) {
        if (want_nc && (geo[0] != want_nc || geo[1] != want_r)) continue;
        if (!set_geometry(geo[0], geo[1], 8, false, 3)) continue;
        int rc2 = derive();
        if (rc2) return -rc2;
        for (int j = 0; j < k.nacc; j++)      // cheapest representation whose proof holds
          rk[j] = rs_proof(j, RK_FIRST) ? RK_FIRST : (rs_proof(j, RK_N32) ? RK_N32 : (rs_proof(j, RK_MADW) ? RK_MADW : RK_WIDE));
        f->jit_struct = jit_shape_struct(k, key32, 8, rk);
        cudaKernel_t kh = jit_scan_compile(ctx, f->jit_struct, geo[0], geo[1], 8, smem_max, &ok, &log);
        if (kh) {
          f->jit_rs_kernel[8] = kh; f->jit_rs_tried[8] = true;
          f->rs = true; f->rs_gmax = 8; f->jit = true;
          return 1;
        }
        break;
      }
      default_geometry();
      int rc2 = derive();
      if (rc2) return -rc2;
    }
    f->jit_struct = jit_shape_struct(k, key32, 0, rk);
    f->jit_kernel = jit_scan_compile(ctx, f->jit_struct, f->nc, f->r, 0, smem_max, &ok, &log);
    if (!f->jit_kernel) return 0;
    f->jit = true;
    return 1;
  };

  // pick the kernel: a static shape whose assumptions all hold, else the generic one; a shape with register slots
  // runs in that mode when the key domain's slots and the 32-bit proofs allow it
  f->kernel = scan_kernel_for<GenericShape>(f->nc, f->r);
  auto try_shape = [&](auto shape_tag) -> int {
    using S = decltype(shape_tag);
    if (!shape_matches<S>(k)) return 0;
    f->kernel = scan_kernel_for<S>(f->nc, f->r);
    f->shape = S::kName;
    if constexpr (S::RS_G > 0) {
      if (getenv("VDL_NO_REGISTER_SLOTS")) return 1;
      int want_nc = 0, want_r = 0;
      if (const char *e = getenv("VDL_RS_GEOMETRY")) sscanf(e, "%d,%d", &want_nc, &want_r);
      for (auto &geo : rs_geometries) {
        if (want_nc && (geo[0] != want_nc || geo[1] != want_r)) continue;
        if (!rs_kernel_for<S>(geo[0], geo[1], S::RS_G) || !set_geometry(geo[0], geo[1], S::RS_G, false, 3)) continue;
        int rc2 = derive();
        if (rc2) return -rc2;
        if (shape_matches<S>(k) && rs_proofs_hold(S::ACC_RK)) {
          for (int g : rs_slot_counts) f->rs_kernel[g] = rs_kernel_for<S>(geo[0], geo[1], g);
          f->kernel = f->rs_kernel[S::RS_G];
          f->rs = true;
          f->rs_gmax = S::RS_G;
          return 1;
        }
      }
      default_geometry();               // no register-slot geometry qualified: back to the shared-memory tables
      int rc2 = derive();
      if (rc2) return -rc2;
    }
    return 1;
  };
  if (!getenv("VDL_GENERIC_ONLY")) {
    int m = try_jit();
    if (m > 0) {
      u64 h = 0xCBF29CE484222325ull;
      for (unsigned char c : f->jit_struct) h = (h ^ c) * 0x100000001B3ull;
      char nm[32];
      snprintf(nm, sizeof nm, "jit:%08x", (unsigned)(h ^ (h >> 32)));
      f->jit_name = nm;
      f->shape = f->jit_name.c_str();
    }
    if (m == 0) m = try_shape(ShapeSel3Sum2{});
    if (m == 0) m = try_shape(ShapeSel1Key2Sum5{});
    if (m < 0) { vdl_fused_destroy(f); return -m; }
  }
  if (getenv("VDL_DEBUG_SHAPE")) {
    fprintf(stderr, "[vdl] fused scan: shape=%s%s nc=%d r=%d stages=%d gmax=%d npreds=%d nkeys=%d nacc=%d smem=%zu\n", f->shape, f->rs ? " (register slots)" : "", f->nc, f->r, k.stages, k.gmax, k.npreds, k.nkeys, k.nacc, f->smem_bytes);
    for (int i = 0; i < k.npreds; i++) fprintf(stderr, "[vdl]   pred %d: mode=%d shr=%d\n", i, k.pred[i].w4, k.pred[i].shr);
    for (int i = 0; i < k.nkeys; i++) fprintf(stderr, "[vdl]   key %d: col=%d w4=%d shr=%d a=%lld b=%lld shl=%d narrow=%d\n", i, k.key[i].e.col, k.key[i].e.w4, k.key[i].e.shr, (long long)k.key[i].e.a, (long long)k.key[i].e.b, k.key[i].shl, k.key[i].e.narrow);
    for (int j = 0; j < k.nacc; j++) {
      fprintf(stderr, "[vdl]   acc %d: op=%d chain=%d nfac=%d", j, k.acc[j].op, k.acc[j].chain, k.acc[j].nfac);
      for (int t = 0; t < k.acc[j].nfac; t++) fprintf(stderr, " [col=%d w4=%d shr=%d a=%lld b=%lld narrow=%d]", k.acc[j].fac[t].col, k.acc[j].fac[t].w4, k.acc[j].fac[t].shr, (long long)k.acc[j].fac[t].a, (long long)k.acc[j].fac[t].b, k.acc[j].fac[t].narrow);
      fprintf(stderr, "\n");
    }
  }

  // device buffers
  int rc = vec_new(ctx, VDL_I64, (i64)(k.nacc + k.nchoose) * k.domain, &f->table);
  if (rc) { delete f; return rc; }
  k.table = (i64 *)ctx->vecs[f->table].ptr;
  fd.nacc = k.nacc;
  fd.nchoose = k.nchoose;
  fd.cnt_idx = k.cnt_idx;
  fd.first_idx = k.first_idx;
  for (int j = 0; j < k.nacc; j++) fd.acc_op[j] = k.acc[j].op;
  for (int q = 0; q < desc->nposts; q++) fd.post[q] = desc->post[q];
  fd.reset_table = k.table;      // a finalize is the last reader of the table: it leaves the identities for the next launch
  static const FoldTexts texts = {"finalize: nranks %d without gathered partials",
                                  "fused scan: peer exchange requested before vdl_fused_set_peers", "fused scan not finalized",
                                  "fused scan: a peer GPU never delivered its partial table (exchange timed out)",
                                  "fused scan: %lld rows produced a group key outside the key domain"};
  if (f->cb.allocate(ctx, &texts, k.table, (i64)(k.nacc + k.nchoose) * k.domain, k.domain, f->nout, desc->nposts) ||
      cudaMalloc(&f->d_done, sizeof(unsigned int)) != cudaSuccess || cudaMemsetAsync(f->d_done, 0, sizeof(unsigned int), ctx->stream) != cudaSuccess) {
    vdl_fused_destroy(f);
    return vdl_fail(ctx, VDL_ENOMEM, "fused scan: result buffers");
  }
  k.done = f->d_done;
  for (int i = 0; i < f->nout; i++) {   // the fold results are views into the one result buffer
    rc = vec_new_range(ctx, 0, 0, 0, &f->out[i]);
    if (rc) { vdl_fused_destroy(f); return rc; }
    Vec &v = ctx->vecs[f->out[i]];
    v.is_range = false;
    v.ptr = fd.out[i];
    v.dtype = VDL_I64;
    v.cap_rows = k.domain;
    v.domain = -1;
  }
  f->timer.create();

  {   // load every kernel a step may launch now, not lazily behind a peer's spinning exchange (see FoldCombine::allocate)
    cudaFuncAttributes fa;
    cudaFuncGetAttributes(&fa, fused_init_kernel); cudaFuncGetAttributes(&fa, fused_choose_kernel);
    cudaGetLastError();
  }
  cudaError_t e = cudaFuncSetAttribute(f->kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_max);
  if (e != cudaSuccess) { vdl_fused_destroy(f); return vdl_cuda_fail(ctx, e, "cudaFuncSetAttribute(fused_scan_fold_kernel)"); }
  for (int g : rs_slot_counts)
    if (f->rs && f->rs_kernel[g] && (e = cudaFuncSetAttribute(f->rs_kernel[g], cudaFuncAttributeMaxDynamicSharedMemorySize, smem_max)) != cudaSuccess) {
      vdl_fused_destroy(f);
      return vdl_cuda_fail(ctx, e, "cudaFuncSetAttribute(fused_scan_fold_kernel, register slots)");
    }
  *out = f;
  return VDL_OK;
}

// self_finalize != 0: single-GPU step -- the scan kernel's last CTA also runs FoldChoose, the finalize and the table
// reset, so a step is ONE launch and the results are on the host (mapped pinned memory) when the stream drains.
// self_finalize == 0: the scan leaves the complete partial table (FoldChoose values included) for an external
// combine across ranks; vdl_fused_finalize() then merges the gathered tables.
extern "C" int vdl_fused_launch_ex(vdl_fused *f, int self_finalize) {
  if (!f) return VDL_EINVAL;
  vdl_ctx *ctx = f->ctx;
  VDL_CUDA(ctx, cudaSetDevice(ctx->device));
  if (!vdl_fused_current(f))
    return vdl_fail(ctx, VDL_ESTALE, "fused scan: a column was rewritten or dropped after vdl_fused_prepare (its statistics proofs no longer hold): prepare again");
  f->cb.finalized = false;
  f->cb.ngroups = -1;
  if (!f->cb.table_clean) {
    int nb = (int)std::min<i64>(ctx->sm_count, ((i64)(f->kd.nacc + f->kd.nchoose) * f->kd.domain + 255) / 256);
    fused_init_kernel<<<std::max(nb, 1), 256, 0, ctx->stream>>>(f->kd);
    ctx->launches++;
    f->cb.table_clean = true;
  }
  VDL_TRY(f->timer.begin(ctx));
  cudaKernel_t jit_launch = f->jit ? f->jit_kernel : nullptr;
  if (f->rs) {
    int g = f->rs_gmax;
    if (f->groups_seen >= 0 && !getenv("VDL_RS_ALL_SLOTS"))
      for (int c : rs_slot_counts)
        if (c >= f->groups_seen && c < g) {
          if (f->jit && !f->jit_rs_tried[c]) {        // the variant with fewer register slots: compiled on first use
            f->jit_rs_tried[c] = true;
            const int smem_max = ctx->smem_optin > 0 ? ctx->smem_optin : 232448;
            f->jit_rs_kernel[c] = jit_scan_compile(ctx, f->jit_struct, f->nc, f->r, c, smem_max, nullptr, nullptr);
          }
          if (f->jit ? f->jit_rs_kernel[c] != nullptr : f->rs_kernel[c] != nullptr) g = c;
        }
    if (f->jit) jit_launch = f->jit_rs_kernel[g];
    else f->kernel = f->rs_kernel[g];
    f->kd.gmax = g;
  }
  const bool scan = f->kd.rows > 0 && !f->always_false;
  FoldCombine &cb = f->cb;
  if (self_finalize == 2) VDL_TRY(cb.next_epoch());
  if (scan) {
    cb.fd.parts = f->kd.table;           // the epilogue's single-rank finalize
    if (self_finalize) cb.fd.seq++;
    f->kd.epilogue = self_finalize == 2 ? 3 : (self_finalize ? 2 : 1);
    if (jit_launch) {
      void *args[] = {(void *)&f->kd, (void *)&cb.fd, (void *)&cb.xd};
      VDL_CUDA(ctx, cudaLaunchKernel((const void *)jit_launch, dim3(f->grid), dim3(f->nc + 32), args, f->smem_bytes, ctx->stream));
    } else {
      f->kernel<<<f->grid, f->nc + 32, f->smem_bytes, ctx->stream>>>(f->kd, cb.fd, cb.xd);
    }
    ctx->launches++;
    f->cb.table_clean = self_finalize != 0;
  } else if (self_finalize == 2) {       // nothing to scan here, but the other ranks wait for this rank's table
    VDL_TRY(cb.exchange());
  } else if (self_finalize) {            // nothing to scan: the (identity) table finalizes to zero groups
    VDL_TRY(cb.finalize(nullptr, 1));
  }
  VDL_TRY(f->timer.end(ctx));
  VDL_CUDA(ctx, cudaGetLastError());
  if (self_finalize) cb.finalized = true;
  return VDL_OK;
}

FoldCombine *vdl_fused_combine(vdl_fused *f) { return &f->cb; }

extern "C" int vdl_fused_exchange_bytes(vdl_fused *f, int world, int64_t *bytes) { return f ? f->cb.exchange_bytes(world, bytes) : VDL_EINVAL; }

extern "C" int vdl_fused_set_peers(vdl_fused *f, int rank, int world, void *const *peer_buffers) { return f ? f->cb.set_peers(rank, world, peer_buffers) : VDL_EINVAL; }

extern "C" int vdl_fused_launch(vdl_fused *f) { return vdl_fused_launch_ex(f, 0); }

extern "C" int vdl_fused_partials(vdl_fused *f, void **device_ptr, int64_t *n_int64) { return f ? f->cb.partials(device_ptr, n_int64) : VDL_EINVAL; }

extern "C" int vdl_fused_finalize(vdl_fused *f, const void *all_partials, int nranks) { return f ? f->cb.finalize(all_partials, nranks) : VDL_EINVAL; }

// The group count, the error counter and every result, published by the finalize into mapped pinned memory.
static int fused_fetch(vdl_fused *f) {
  VDL_TRY(f->cb.fetch());
  f->groups_seen = f->cb.ngroups;
  for (int i = 0; i < f->nout; i++) f->ctx->vecs[f->out[i]].len = f->cb.ngroups;
  return VDL_OK;
}

extern "C" int vdl_fused_num_groups(vdl_fused *f, int64_t *ngroups) {
  if (!f || !ngroups) return VDL_EINVAL;
  VDL_TRY(fused_fetch(f));
  *ngroups = f->cb.ngroups;
  return VDL_OK;
}

// Host copy of fold `fold_index`'s result (valid until the next launch); no device work beyond the one fetch.
extern "C" int vdl_fused_result_host(vdl_fused *f, int fold_index, const int64_t **data, int64_t *len) {
  if (!f || fold_index < 0 || fold_index >= f->nout) return VDL_EINVAL;
  VDL_TRY(fused_fetch(f));
  return f->cb.result_host(fold_index, data, len);
}

extern "C" int vdl_fused_post_host(vdl_fused *f, int post_index, const int64_t **data, int64_t *len) {
  if (!f || post_index < 0 || post_index >= f->cb.fd.npost) return VDL_EINVAL;
  VDL_TRY(fused_fetch(f));
  return f->cb.result_host(f->nout + post_index, data, len);
}

extern "C" int vdl_fused_result(vdl_fused *f, int fold_index, vdl_vec *out) {
  if (!f || !out || fold_index < 0 || fold_index >= f->nout) return VDL_EINVAL;
  int64_t n;
  VDL_TRY(vdl_fused_num_groups(f, &n));
  *out = f->out[fold_index];
  return VDL_OK;
}

extern "C" int vdl_fused_last_kernel_ms(vdl_fused *f, float *ms) {
  if (!f || !ms) return VDL_EINVAL;
  if (!f->timer.n) return vdl_fail(f->ctx, VDL_EINVAL, "fused scan not launched yet");
  return f->timer.last_ms(f->ctx, ms);
}

// Mean / minimum duration of the scan kernel over the last `n` launches (n <= VDL_EVENT_RING), from event pairs recorded
// around each launch: a timed loop reads them afterwards instead of synchronising on an event every step.
extern "C" int vdl_fused_kernel_ms_stats(vdl_fused *f, int n, float *mean_ms, float *min_ms) {
  if (!f || n < 1) return VDL_EINVAL;
  if (!f->timer.n) return vdl_fail(f->ctx, VDL_EINVAL, "fused scan not launched yet");
  return f->timer.stats(f->ctx, n, mean_ms, min_ms);
}

extern "C" const char *vdl_fused_shape_name(vdl_fused *f) { return f ? f->shape : ""; }

extern "C" int vdl_fused_destroy(vdl_fused *f) {
  if (!f) return VDL_EINVAL;
  vdl_ctx *ctx = f->ctx;
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  if (f->table) vdl_vec_free(ctx, f->table);
  for (int i = 0; i < f->nout; i++)
    if (f->out[i]) vdl_vec_free(ctx, f->out[i]);
  f->cb.release();
  if (f->d_done) cudaFree(f->d_done);
  f->timer.destroy();
  delete f;
  return VDL_OK;
}
