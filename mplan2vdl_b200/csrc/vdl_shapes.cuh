// Static shapes of the fused scan: compile-time answers to the structural questions of a descriptor
// (see "SHAPES" in vdl_fused_kernel.cuh).  A shape only fixes STRUCTURE -- counts, column widths, which of
// shr / a / b are trivial, what fits 32 bits; every constant stays a run-time descriptor field, so a shape
// serves any plan of that structure (other columns, other bounds, other scale factors).  The host checks all
// of a shape's assumptions against the prepared descriptor (shape_matches, vdl_fused.cu) before launching it and
// otherwise uses GenericShape; results are identical.  To see the struct a plan needs, run it with VDL_DEBUG_JIT=1
// and VDL_SCAN_JIT_MIN_ROWS=0: the scan prints the `ShapeJit` it generates for the prepared descriptor, in these
// fields (needs a GPU: narrowing depends on the column statistics).
#pragma once

#define FF_COLN (FF_SHR0 | FF_B1 | FF_A0 | FF_NARROW)      /* a plain 8-byte column whose values fit int32 */

// REGISTER SLOTS.  A grouped shape may declare RS_G > 0: the first RS_G keys a CTA meets get their accumulators in
// the REGISTERS of every consumer thread (updated under `slot == g` predicates: no shared-memory read-modify-write
// at all), reduced once at the end of the kernel.  ACC_RK says how accumulator J is kept per thread:
//   RK_WIDE  64-bit;  RK_MADW  64-bit SUM of a product a x b with 0 <= a, b < 2^31 proved from the statistics (the
//   update is one select + one 32x32+64 multiply-add);  RK_N32  32-bit SUM -- the host proves from the column statistics and the launch geometry that
//   rows-per-thread x max|value| < 2^31;  RK_FIRST  MIN(row id) kept as a 32-bit CTA-local row index.
// The host falls back to the shared-memory tables (same shape, G = 0) when a proof fails.

// select(3 ranges: int32 col, 2 x narrow 8-byte col) -> SUM(col * col), COUNT          [TPC-H Q6, Vlite.hs:721-730]
struct ShapeSel3Sum2 {
  static constexpr bool kStatic = true;
  static constexpr const char *kName = "sel3_sum2";
  static constexpr int NPREDS = 3, NKEYS = 0, NACC = 2, KEY32 = 0;
  static constexpr int PRED_MODE[VDL_MAX_PREDS] = {1, 2, 2}, PRED_SHR0[VDL_MAX_PREDS] = {1, 1, 1};
  static constexpr int KEY_FLAGS[VDL_MAX_KEYS] = {}, KEY_SHL0[VDL_MAX_KEYS] = {};
  static constexpr int ACC_OP[K_MAX_ACC] = {0, 0}, ACC_CHAIN[K_MAX_ACC] = {0, 0}, ACC_NFAC[K_MAX_ACC] = {2, 0};
  static constexpr int FAC[K_MAX_ACC][VDL_MAX_FACTORS] = {{FF_COLN, FF_COLN}, {}};
  static constexpr int RS_G = 0;
  static constexpr int ACC_RK[K_MAX_ACC] = {};
};

// select(1 range on an int32 col) -> group by a 2-part narrow key -> SUM c, SUM c, SUM c*(k-c), chain*(k+c), SUM c,
// COUNT, first row                                                                         [TPC-H Q1, Vlite.hs:1048-1098]
struct ShapeSel1Key2Sum5 {
  static constexpr bool kStatic = true;
  static constexpr const char *kName = "sel1_key2_sum5";
  static constexpr int NPREDS = 1, NKEYS = 2, NACC = 7, KEY32 = 1;
  static constexpr int PRED_MODE[VDL_MAX_PREDS] = {1}, PRED_SHR0[VDL_MAX_PREDS] = {1};
  static constexpr int KEY_FLAGS[VDL_MAX_KEYS] = {FF_NARROW, FF_NARROW}, KEY_SHL0[VDL_MAX_KEYS] = {1, 1};
  static constexpr int ACC_OP[K_MAX_ACC] = {0, 0, 0, 0, 0, 0, 1};
  static constexpr int ACC_CHAIN[K_MAX_ACC] = {0, 0, 1, 1, 0, 0, 0};
  static constexpr int ACC_NFAC[K_MAX_ACC] = {1, 1, 1, 1, 1, 0, 1};
  static constexpr int FAC[K_MAX_ACC][VDL_MAX_FACTORS] = {
      {FF_COLN}, {FF_COLN}, {FF_SHR0 | FF_BM1 | FF_NARROW}, {FF_SHR0 | FF_B1 | FF_NARROW}, {FF_COLN}, {},
      {FF_ROWID | FF_SHR0 | FF_B1 | FF_A0}};
  static constexpr int RS_G = 8;
  static constexpr int ACC_RK[K_MAX_ACC] = {RK_N32, RK_MADW, RK_MADW, RK_MADW, RK_N32, RK_N32, RK_FIRST};
};
