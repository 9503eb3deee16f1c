// Per-op kernels: one entry point per Voodoo op (reference op set Vdl.hs:32-44, 110-131), so that any
// emitted graph runs op-at-a-time when the fusion pass does not apply, and for the per-op sweep.
// Semantics: SURVEY.md section 2.3 / Appendix G (dense vectors, int64 wraparound).
#include <stdio.h>
#include <string.h>

#include <algorithm>
#include <memory>

#include "vdl_internal.h"
#include <type_traits>

// ---------------------------------------------------------------------------------- RangeV / RangeC
extern "C" int vdl_op_range(vdl_ctx *ctx, int64_t from, int64_t step, int64_t len, vdl_vec *out) {
  if (!ctx || !out) return VDL_EINVAL;
  return vec_new_range(ctx, from, step, len, out);   // virtual: consumers read from + i*step
}

// ---------------------------------------------------------------------------------- elementwise
// op semantics: binop_apply in vdl_device.cuh
template <int OP>
__global__ void __launch_bounds__(256) binary_kernel(Operand a, Operand b, i64 *__restrict__ out, i64 n) {
  // two elements per thread and step: 16-byte stores, 2 x (8 or 4)-byte loads per operand in flight
  i64 stride = (i64)gridDim.x * blockDim.x * 2;
  for (i64 i = ((i64)blockIdx.x * blockDim.x + threadIdx.x) * 2; i < n; i += stride) {
    if (i + 1 < n) {
      longlong2 r;
      r.x = binop_apply(OP, op_ld(a, i), op_ld(b, i));
      r.y = binop_apply(OP, op_ld(a, i + 1), op_ld(b, i + 1));
      *(longlong2 *)(out + i) = r;
    } else {
      out[i] = binop_apply(OP, op_ld(a, i), op_ld(b, i));
    }
  }
}

typedef void (*binary_fn)(Operand, Operand, i64 *, i64);
static binary_fn binary_table[12] = {
    binary_kernel<0>, binary_kernel<1>, binary_kernel<2>, binary_kernel<3>, binary_kernel<4>,  binary_kernel<5>,
    binary_kernel<6>, binary_kernel<7>, binary_kernel<8>, binary_kernel<9>, binary_kernel<10>, binary_kernel<11>};

extern "C" int vdl_op_binary(vdl_ctx *ctx, int op, vdl_vec a, vdl_vec b, vdl_vec *out) {
  if (!ctx || !out) return VDL_EINVAL;
  if (op < 0 || op > VDL_MODULO) return vdl_fail(ctx, VDL_EINVAL, "binary op %d unknown", op);
  Vec *va = vec_get(ctx, a), *vb = vec_get(ctx, b);
  if (!va || !vb) return VDL_EINVAL;
  if (va->len != vb->len) return vdl_fail(ctx, VDL_EINVAL, "elementwise op on lengths %lld vs %lld", (long long)va->len, (long long)vb->len);
  i64 n = va->len;
  Operand oa = operand_of(*va), ob = operand_of(*vb);
  // positions `p % k` with a constant k > 0 -- the scatter size hint of addScatterSizeHint (Vlite.hs:1117-1120) -- index
  // a space of k slots (App. G2 / G9)
  i64 dom = -1;
  if (op == VDL_MODULO && vb->is_range && vb->step == 0 && vb->from > 0) dom = vb->from;
  VDL_TRY(vec_new(ctx, VDL_I64, n, out));
  ctx->vecs[*out].domain = dom;
  if (n == 0) return VDL_OK;
  VDL_CUDA(ctx, cudaSetDevice(ctx->device));
  i64 want = (n / 2 + 255) / 256;
  int blocks = (int)std::max<i64>(1, std::min<i64>(want, (i64)ctx->sm_count * 16));
  binary_table[op]<<<blocks, 256, 0, ctx->stream>>>(oa, ob, (i64 *)ctx->vecs[*out].ptr, n);
  ctx->launches++;
  VDL_CUDA(ctx, cudaGetLastError());
  return VDL_OK;
}

// ---------------------------------------------------------------------------------- Like over a string heap
// Vlite.hs:1010-1014 -> Vdl.hs:244-247: the data vector holds byte offsets into the column's string heap.  One thread per
// row reads its (NUL-terminated) string and runs the glob match with one backtrack point (the last `%`): sequential byte
// reads of a string that is 8-byte aligned and a few tens of bytes long, so a row costs its 8-byte offset plus one or two
// 32-byte sectors of the heap (L2-resident for dictionary-like columns such as p_type).  Bound: HBM / L2 bandwidth.
struct LikeArgs { char pat[VDL_LIKE_MAX_PATTERN]; };
__global__ void __launch_bounds__(256) like_kernel(Operand data, const unsigned char *__restrict__ heap, i64 heap_len, const __grid_constant__ LikeArgs a,
                                                   i64 *__restrict__ out, i64 n, int *errflag) {
  for (i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (i64)gridDim.x * blockDim.x) {
    const i64 off = op_ld(data, i);
    if ((u64)off >= (u64)heap_len) { atomicAdd(errflag, 1); out[i] = 0; continue; }
    const unsigned char *s = heap + off, *end = heap + heap_len, *star_s = nullptr;
    int p = 0, star_p = -1;
    bool ok = true;
    while (s < end && *s) {
      const char c = a.pat[p];
      if (c == '%') { star_p = ++p; star_s = s; }
      else if (c && (c == '_' || (unsigned char)c == *s)) { p++; s++; }
      else if (star_p >= 0) { p = star_p; s = ++star_s; }
      else { ok = false; break; }
    }
    if (ok) {
      while (a.pat[p] == '%') p++;
      ok = a.pat[p] == 0;
    }
    out[i] = ok ? 1 : 0;
  }
}

extern "C" int vdl_op_like(vdl_ctx *ctx, vdl_vec data, vdl_vec heap, const char *pattern, vdl_vec *out) {
  if (!ctx || !out || !pattern) return VDL_EINVAL;
  Vec *vd = vec_get(ctx, data), *vh = vec_get_any(ctx, heap);
  if (!vd || !vh) return VDL_EINVAL;
  if (vh->dtype != VDL_U8) return vdl_fail(ctx, VDL_EINVAL, "Like: the dictionary must be a string heap (a VDL_U8 vector; Load,<table>.<col>.heap)");
  if (strlen(pattern) >= VDL_LIKE_MAX_PATTERN) return vdl_fail(ctx, VDL_EUNSUPPORTED, "Like: pattern longer than %d bytes", VDL_LIKE_MAX_PATTERN - 1);
  const i64 n = vd->len;
  const Operand od = operand_of(*vd);
  const unsigned char *hp = (const unsigned char *)vh->ptr;
  const i64 hl = vh->len;
  VDL_TRY(vec_new(ctx, VDL_I64, n, out));
  if (n == 0) return VDL_OK;
  VDL_CUDA(ctx, cudaSetDevice(ctx->device));
  LikeArgs a;
  memset(&a, 0, sizeof a);
  strcpy(a.pat, pattern);
  int blocks = (int)std::max<i64>(1, std::min<i64>((n + 255) / 256, (i64)ctx->sm_count * 16));
  like_kernel<<<blocks, 256, 0, ctx->stream>>>(od, hp, hl, a, (i64 *)ctx->vecs[*out].ptr, n, ctx->d_errflag);
  ctx->launches++;
  VDL_CUDA(ctx, cudaGetLastError());
  return VDL_OK;
}

// ---------------------------------------------------------------------------------- map (expression tree in one launch)
// The op-at-a-time remainder of a plan is mostly long chains of elementwise ops over short vectors (Q19's OR of ANDs over
// the join's survivors: ~150 launches of a few microseconds each).  One launch interprets the whole tree per row: the
// program is the same for every thread (no divergence), the register file lives in local memory (L1), and each input is
// read from HBM once instead of once per consumer.
#define VDL_MAP_JIT_MIN_ROWS (1 << 16)
__global__ void __launch_bounds__(256) map_kernel(const __grid_constant__ MapArgs m, i64 *__restrict__ out, i64 n, int *errflag) {
  const i64 stride = (i64)gridDim.x * blockDim.x;
  const int nt = m.d.ninstrs;
  for (i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    i64 r[VDL_MAP_MAX_REGS];
    int last = 0;
    for (int t = 0; t < nt; t++) {
      const vdl_map_instr ins = m.d.instr[t];
      i64 v;
      if (ins.op == VDL_MAP_LOAD) {
        v = op_ld(m.in[ins.b], i);
      } else if (ins.op == VDL_MAP_RANGE) {
        v = (i64)((u64)m.d.imm[ins.a] + (u64)i * (u64)m.d.imm[ins.b]);
      } else if (ins.op == VDL_MAP_GATHER) {
        const i64 a = r[ins.a];
        if ((u64)a >= (u64)m.tab_len[ins.b]) { atomicAdd(errflag, 1); v = 0; }
        else v = op_ld(m.tab[ins.b], a);
      } else {
        v = binop_apply(ins.op, r[ins.a], r[ins.b]);
      }
      r[ins.dst] = v;
      last = ins.dst;
    }
    out[i] = r[last];
  }
}

extern "C" int vdl_abi_sizeof_map_desc(void) { return (int)sizeof(vdl_map_desc); }

extern "C" int vdl_op_map(vdl_ctx *ctx, const vdl_map_desc *d, const vdl_vec *inputs, const vdl_vec *tables, vdl_vec *out) {
  if (!ctx || !d || !out || !inputs || (d->ntables > 0 && !tables)) return VDL_EINVAL;
  if (d->ninputs < 1 || d->ninputs > VDL_MAP_MAX_INPUTS || d->ntables < 0 || d->ntables > VDL_MAP_MAX_TABLES || d->ninstrs < 1 ||
      d->ninstrs > VDL_MAP_MAX_INSTRS || d->nimms < 0 || d->nimms > VDL_MAP_MAX_IMMS)
    return vdl_fail(ctx, VDL_EINVAL, "map: %d inputs, %d tables, %d instructions, %d immediates out of range", d->ninputs, d->ntables, d->ninstrs, d->nimms);
  MapArgs *mp = new MapArgs();          // ~3 KB: off the stack
  std::unique_ptr<MapArgs> hold(mp);
  MapArgs &m = *mp;
  m.d = *d;
  i64 n = -1;
  for (int k = 0; k < d->ninputs; k++) {
    Vec *v = vec_get(ctx, inputs[k]);
    if (!v) return VDL_EINVAL;
    if (n >= 0 && v->len != n) return vdl_fail(ctx, VDL_EINVAL, "elementwise op on lengths %lld vs %lld", (long long)n, (long long)v->len);
    n = v->len;
    m.in[k] = operand_of(*v);
  }
  for (int k = 0; k < d->ntables; k++) {
    Vec *v = vec_get(ctx, tables[k]);
    if (!v) return VDL_EINVAL;
    m.tab[k] = operand_of(*v);
    m.tab_len[k] = v->len;
  }
  i64 domain = -1;
  i64 regconst[VDL_MAP_MAX_REGS];      // constant value of a register, when isconst
  bool isconst[VDL_MAP_MAX_REGS] = {false};
  unsigned written = 0;
  auto reg_ok = [&](int r, bool read) { return r >= 0 && r < VDL_MAP_MAX_REGS && (!read || (written >> r & 1)); };
  for (int t = 0; t < d->ninstrs; t++) {
    const vdl_map_instr &ins = d->instr[t];
    bool ok = reg_ok(ins.dst, false);
    if (ins.op == VDL_MAP_LOAD) ok = ok && ins.b >= 0 && ins.b < d->ninputs;
    else if (ins.op == VDL_MAP_RANGE) ok = ok && ins.a >= 0 && ins.a < d->nimms && ins.b >= 0 && ins.b < d->nimms;
    else if (ins.op == VDL_MAP_GATHER) ok = ok && reg_ok(ins.a, true) && ins.b >= 0 && ins.b < d->ntables;
    else ok = ok && ins.op >= 0 && ins.op <= VDL_MODULO && reg_ok(ins.a, true) && reg_ok(ins.b, true);
    if (!ok) return vdl_fail(ctx, VDL_EINVAL, "map: instruction %d (op %d dst %d a %d b %d) is malformed or reads a register nothing wrote", t, ins.op, ins.dst, ins.a, ins.b);
    written |= 1u << ins.dst;
    // index space of the result (App. G2): gathering positions keeps their space; `p % k` is the scatter size hint
    i64 dm = -1, cv = 0;
    bool ic = false;
    if (ins.op == VDL_MAP_GATHER) dm = ctx->vecs[tables[ins.b]].domain;
    else if (ins.op == VDL_MAP_LOAD) dm = ctx->vecs[inputs[ins.b]].domain;
    else if (ins.op == VDL_MAP_RANGE) { ic = d->imm[ins.b] == 0; cv = d->imm[ins.a]; }
    else if (ins.op == VDL_MODULO && isconst[ins.b] && regconst[ins.b] > 0) dm = regconst[ins.b];
    regconst[ins.dst] = cv; isconst[ins.dst] = ic;
    if (t == d->ninstrs - 1) domain = dm;
  }
  VDL_TRY(vec_new(ctx, VDL_I64, n, out));
  ctx->vecs[*out].domain = domain;
  if (n == 0) return VDL_OK;
  VDL_CUDA(ctx, cudaSetDevice(ctx->device));
  int blocks = (int)std::max<i64>(1, std::min<i64>((n + 255) / 256, (i64)ctx->sm_count * 8));
  // long vectors: a kernel specialised to this program (vdl_jit.cu); short ones are launch-bound either way
  int jitted = n >= VDL_MAP_JIT_MIN_ROWS ? vdl_jit_map_launch(ctx, m, (i64 *)ctx->vecs[*out].ptr, n, blocks) : 0;
  if (jitted < 0) return VDL_ECUDA;
  if (!jitted) map_kernel<<<blocks, 256, 0, ctx->stream>>>(m, (i64 *)ctx->vecs[*out].ptr, n, ctx->d_errflag);
  ctx->launches++;
  VDL_CUDA(ctx, cudaGetLastError());
  return VDL_OK;
}

// ---------------------------------------------------------------------------------- scan helpers
// Exclusive scan of `n` int64 counters in place by ONE block (n is #blocks or 256 * #blocks: small next to
// the data), total written to *total.  Warp-shuffle scan, 1024 elements per step, running carry.
__global__ void __launch_bounds__(1024, 1) exclusive_scan_kernel(i64 *data, i64 n, i64 *total) {
  __shared__ i64 warp_sum[32];
  __shared__ i64 carry;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0) carry = 0;
  __syncthreads();
  for (i64 base = 0; base < n; base += 1024) {
    i64 i = base + tid;
    i64 v = i < n ? data[i] : 0, x = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      i64 y = __shfl_up_sync(0xffffffffu, x, o);
      if (lane >= o) x += y;
    }
    if (lane == 31) warp_sum[warp] = x;
    __syncthreads();
    if (warp == 0) {
      i64 w = warp_sum[lane], s = w;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        i64 y = __shfl_up_sync(0xffffffffu, s, o);
        if (lane >= o) s += y;
      }
      warp_sum[lane] = s - w;   // exclusive prefix of the warp sums
    }
    __syncthreads();
    i64 c = carry;
    if (i < n) data[i] = c + warp_sum[warp] + x - v;
    __syncthreads();
    if (tid == 1023) carry = c + warp_sum[31] + x;
    __syncthreads();
  }
  if (tid == 0) *total = carry;
}

// Large inputs (radix histograms: 256 counters per 4096 rows; a billion-row FoldSelect: 244 K block counts): scan
// 4096-element chunks in parallel, scan the chunk totals with the one-block kernel, add the chunk offsets back.
#define SCAN_CHUNK 4096
__global__ void __launch_bounds__(1024) scan_chunks_kernel(i64 *data, i64 n, i64 *chunk_sum) {
  __shared__ i64 warp_sum[32];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const i64 base = (i64)blockIdx.x * SCAN_CHUNK + tid * 4;
  i64 v[4], t = 0;
#pragma unroll
  for (int k = 0; k < 4; k++) { v[k] = base + k < n ? data[base + k] : 0; t += v[k]; }
  i64 x = t;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) { i64 y = __shfl_up_sync(0xffffffffu, x, o); if (lane >= o) x += y; }
  if (lane == 31) warp_sum[warp] = x;
  __syncthreads();
  if (warp == 0) {
    i64 w = warp_sum[lane], q = w;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { i64 y = __shfl_up_sync(0xffffffffu, q, o); if (lane >= o) q += y; }
    warp_sum[lane] = q - w;
    if (lane == 31) chunk_sum[blockIdx.x] = q;
  }
  __syncthreads();
  i64 run = warp_sum[warp] + x - t;
#pragma unroll
  for (int k = 0; k < 4; k++) { if (base + k < n) data[base + k] = run; run += v[k]; }
}
__global__ void __launch_bounds__(1024) add_chunk_offsets_kernel(i64 *data, i64 n, const i64 *chunk_off) {
  const i64 off = chunk_off[blockIdx.x], base = (i64)blockIdx.x * SCAN_CHUNK + threadIdx.x * 4;
#pragma unroll
  for (int k = 0; k < 4; k++) if (base + k < n) data[base + k] += off;
}
// elements of scratch a scan of n counters needs, counters included: [n counters][total][chunk sums][their total]
static size_t scan_elems(i64 n) { return (size_t)n + 1 + 2 * (size_t)((n + SCAN_CHUNK - 1) / SCAN_CHUNK) + 64; }
// exclusive scan of data[0..n) in place, total to data[n]; data must have scan_elems(n) elements
static void device_exclusive_scan(vdl_ctx *ctx, i64 *data, i64 n) {
  if (n <= 4 * SCAN_CHUNK) {
    exclusive_scan_kernel<<<1, 1024, 0, ctx->stream>>>(data, n, data + n);
    ctx->launches++;
    return;
  }
  const i64 nc = (n + SCAN_CHUNK - 1) / SCAN_CHUNK;
  i64 *sums = data + n + 1;
  scan_chunks_kernel<<<(unsigned)nc, 1024, 0, ctx->stream>>>(data, n, sums);
  device_exclusive_scan(ctx, sums, nc);                        // recursion depth <= 2 for any realistic n
  add_chunk_offsets_kernel<<<(unsigned)nc, 1024, 0, ctx->stream>>>(data, n, sums);
  cudaMemcpyAsync(data + n, sums + nc, 8, cudaMemcpyDeviceToDevice, ctx->stream);
  ctx->launches += 2;
}

#define SEL_TILE 4096   // rows per tile of the compaction kernel (16 steps of 256)

// ---------------------------------------------------------------------------------- FoldSelect
// Vlite.hs:721-730: idx = Fold FSel (pos_ p) p.  Dense model: global stable compaction of positions.
// Single pass: a block takes 4096-element tiles in ticket order, reads its predicates ONCE (16 flags per thread kept
// as a bit mask), gets the tile's output offset by a decoupled look-back over one 64-bit status word per tile
// ((status << 62) | count; 1 = tile aggregate, 2 = inclusive prefix) and writes the positions in order.
__global__ void __launch_bounds__(256) select_lookback_kernel(Operand o, i64 n, i64 ntiles, unsigned long long *state, unsigned int *ticket,
                                                              i64 *__restrict__ out, i64 *total) {
  __shared__ int wcnt[8];
  __shared__ i64 s_off;
  __shared__ unsigned int s_tile;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (;;) {
    if (tid == 0) s_tile = atomicAdd(ticket, 1u);
    __syncthreads();
    const i64 tile = s_tile;
    if (tile >= ntiles) break;
    const i64 base = tile * SEL_TILE;
    unsigned flags = 0;
#pragma unroll
    for (int s = 0; s < SEL_TILE / 256; s++) {
      const i64 i = base + s * 256 + tid;
      if (i < n && op_ld(o, i) != 0) flags |= 1u << s;
    }
    int c = __popc(flags);
#pragma unroll
    for (int k = 16; k > 0; k >>= 1) c += __shfl_xor_sync(0xffffffffu, c, k);
    if (lane == 0) wcnt[warp] = c;
    __syncthreads();
    if (tid == 0) {
      unsigned long long T = 0;
      for (int w = 0; w < 8; w++) T += (unsigned long long)wcnt[w];
      i64 excl = 0;
      if (tile == 0) atomicExch(state, (2ull << 62) | T);
      else {
        atomicExch(state + tile, (1ull << 62) | T);
        for (i64 j = tile - 1;; j--) {
          unsigned long long st;
          do { st = *((volatile unsigned long long *)(state + j)); } while ((st >> 62) == 0);
          excl += (i64)(st & ((1ull << 62) - 1));
          if ((st >> 62) == 2) break;
        }
        atomicExch(state + tile, (2ull << 62) | (unsigned long long)(excl + (i64)T));
      }
      s_off = excl;
      if (tile == ntiles - 1) *total = excl + (i64)T;
    }
    __syncthreads();
    i64 off = s_off;
    // order inside the tile: step-major, then thread: rank by ballots per step
#pragma unroll 1
    for (int s = 0; s < SEL_TILE / 256; s++) {
      const bool f = (flags >> s) & 1;
      const unsigned m = __ballot_sync(0xffffffffu, f);
      if (lane == 0) wcnt[warp] = __popc(m);
      __syncthreads();
      int before = 0, tot = 0;
#pragma unroll
      for (int w = 0; w < 8; w++) { const int cw = wcnt[w]; if (w < warp) before += cw; tot += cw; }
      if (f) out[off + before + __popc(m & ((1u << lane) - 1))] = base + s * 256 + tid;
      off += tot;
      __syncthreads();
    }
  }
}

extern "C" int vdl_op_fold_select(vdl_ctx *ctx, vdl_vec pred, vdl_vec *out) {
  if (!ctx || !out) return VDL_EINVAL;
  Vec *vp = vec_get(ctx, pred);
  if (!vp) return VDL_EINVAL;
  VDL_CUDA(ctx, cudaSetDevice(ctx->device));
  i64 n = vp->len;
  Operand o = operand_of(*vp);
  if (n == 0) {
    VDL_TRY(vec_new(ctx, VDL_I64, 0, out));
    ctx->vecs[*out].domain = 0;
    return VDL_OK;
  }
  const i64 ntiles = (n + SEL_TILE - 1) / SEL_TILE;
  VDL_TRY(scratch_reserve(ctx, (size_t)(ntiles + 4) * 8));
  unsigned long long *state = (unsigned long long *)ctx->scratch;          // [ntiles] status words, then total, ticket
  i64 *d_total = (i64 *)(state + ntiles);
  unsigned int *ticket = (unsigned int *)(state + ntiles + 1);
  VDL_CUDA(ctx, cudaMemsetAsync(state, 0, (size_t)(ntiles + 2) * 8, ctx->stream));
  VDL_TRY(vec_new(ctx, VDL_I64, n, out));                                   // capacity n; the length is known after the pass
  const int grid = (int)std::min<i64>(ntiles, (i64)ctx->sm_count * 8);
  select_lookback_kernel<<<grid, 256, 0, ctx->stream>>>(o, n, ntiles, state, ticket, (i64 *)ctx->vecs[*out].ptr, d_total);
  ctx->launches++;
  i64 total = 0;
  VDL_TRY(read_scalar(ctx, d_total, &total, 8));
  Vec &v = ctx->vecs[*out];
  v.len = total;
  v.domain = n;   // these positions index the predicate's row space (App. G2)
  return VDL_OK;
}

// ---------------------------------------------------------------------------------- Gather / Scatter
// Gather (Vlite.hs:86-87 `@@`, FK fetch 1264, 1276-1277): out[i] = src[pos[i]].
__global__ void __launch_bounds__(256) gather_kernel(Operand src, i64 src_len, Operand pos, i64 n, i64 *__restrict__ out, int *errflag) {
  i64 stride = (i64)gridDim.x * blockDim.x;
  for (i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    i64 p = op_ld(pos, i);
    if ((u64)p >= (u64)src_len) { atomicAdd(errflag, 1); out[i] = 0; }
    else out[i] = op_ld(src, p);
  }
}

extern "C" int vdl_op_gather(vdl_ctx *ctx, vdl_vec src, vdl_vec pos, vdl_vec *out) {
  if (!ctx || !out) return VDL_EINVAL;
  Vec *vs = vec_get(ctx, src), *vp = vec_get(ctx, pos);
  if (!vs || !vp) return VDL_EINVAL;
  i64 n = vp->len, m = vs->len, dom = vs->domain;
  const bool narrow = vec_is_narrow(*vs);
  Operand os = operand_of(*vs), op = operand_of(*vp);
  VDL_TRY(vec_new(ctx, VDL_I64, n, out));
  ctx->vecs[*out].domain = dom;   // gathering positions keeps their index space
  ctx->vecs[*out].narrow32 = narrow;
  if (n == 0) return VDL_OK;
  VDL_CUDA(ctx, cudaSetDevice(ctx->device));
  int blocks = (int)std::max<i64>(1, std::min<i64>((n + 255) / 256, (i64)ctx->sm_count * 16));
  gather_kernel<<<blocks, 256, 0, ctx->stream>>>(os, m, op, n, (i64 *)ctx->vecs[*out].ptr, ctx->d_errflag);
  ctx->launches++;
  VDL_CUDA(ctx, cudaGetLastError());
  return VDL_OK;
}

// Scatter (Vlite.hs:1057-1059 group sort, 1268-1275 dim validity / inverse index): out[pos[i]] = src[i],
// unwritten slots 0.  Positions are unique in every use the translator emits (permutations, Unique masks).
__global__ void __launch_bounds__(256) scatter_kernel(Operand src, Operand pos, i64 n, i64 *__restrict__ out, i64 out_len, int *errflag) {
  // 4 independent (position, value) pairs per thread and step: the stores are fire-and-forget, the loads are what waits
  const i64 stride = (i64)gridDim.x * blockDim.x;
  i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x;
  for (; i + 3 * stride < n; i += 4 * stride) {
    i64 p[4], v[4];
#pragma unroll
    for (int k = 0; k < 4; k++) { p[k] = op_ld(pos, i + k * stride); v[k] = op_ld(src, i + k * stride); }
#pragma unroll
    for (int k = 0; k < 4; k++) {
      if ((u64)p[k] >= (u64)out_len) atomicAdd(errflag, 1);
      else out[p[k]] = v[k];
    }
  }
  for (; i < n; i += stride) {
    i64 p = op_ld(pos, i);
    if ((u64)p >= (u64)out_len) atomicAdd(errflag, 1);
    else out[p] = op_ld(src, i);
  }
}

extern "C" int vdl_op_scatter(vdl_ctx *ctx, vdl_vec src, vdl_vec pos, int64_t out_len, vdl_vec *out) {
  if (!ctx || !out) return VDL_EINVAL;
  Vec *vs = vec_get(ctx, src), *vp = vec_get(ctx, pos);
  if (!vs || !vp) return VDL_EINVAL;
  if (vs->len != vp->len) return vdl_fail(ctx, VDL_EINVAL, "Scatter: source length %lld != positions length %lld", (long long)vs->len, (long long)vp->len);
  if (out_len < 0) return vdl_fail(ctx, VDL_EINVAL, "Scatter: negative output length");
  i64 n = vs->len, dom = vs->domain;
  const bool covers = vp->is_perm && out_len == n;      // a permutation of 0..n-1 leaves no slot unwritten: nothing to zero
  const bool narrow = vec_is_narrow(*vs);
  Operand os = operand_of(*vs), op = operand_of(*vp);
  VDL_TRY(vec_new(ctx, VDL_I64, out_len, out));
  ctx->vecs[*out].domain = dom;
  ctx->vecs[*out].narrow32 = narrow;
  VDL_CUDA(ctx, cudaSetDevice(ctx->device));
  if (out_len > 0 && !covers) VDL_CUDA(ctx, cudaMemsetAsync(ctx->vecs[*out].ptr, 0, (size_t)out_len * 8, ctx->stream));
  if (n == 0) return VDL_OK;
  int blocks = (int)std::max<i64>(1, std::min<i64>((n + 1023) / 1024, (i64)ctx->sm_count * 16));
  scatter_kernel<<<blocks, 256, 0, ctx->stream>>>(os, op, n, (i64 *)ctx->vecs[*out].ptr, out_len, ctx->d_errflag);
  ctx->launches++;
  VDL_CUDA(ctx, cudaGetLastError());
  return VDL_OK;
}

// ---------------------------------------------------------------------------------- int64 -> int32 (typed result columns)
__global__ void __launch_bounds__(256) narrow_kernel(const i64 *__restrict__ in, i64 n, int *__restrict__ out) {
  const i64 stride = (i64)gridDim.x * blockDim.x * 2;
  for (i64 i = ((i64)blockIdx.x * blockDim.x + threadIdx.x) * 2; i < n; i += stride) {
    if (i + 1 < n) { const longlong2 v = *(const longlong2 *)(in + i); *(int2 *)(out + i) = make_int2((int)v.x, (int)v.y); }
    else out[i] = (int)in[i];
  }
}
// the low words of an int64 vector as a new VDL_I32 vector (the caller knows that every value fits)
int vec_narrow_copy(vdl_ctx *ctx, vdl_vec src, vdl_vec *out) {
  Vec *vs = vec_get(ctx, src);
  if (!vs || vs->is_range || vs->dtype != VDL_I64) return vdl_fail(ctx, VDL_EINVAL, "narrow copy of a vector that is not a stored int64 vector");
  const i64 n = vs->len;
  const i64 *in = (const i64 *)vs->ptr;
  VDL_TRY(vec_new(ctx, VDL_I32, n, out));
  if (n == 0) return VDL_OK;
  VDL_CUDA(ctx, cudaSetDevice(ctx->device));
  const int blocks = (int)std::max<i64>(1, std::min<i64>((n + 511) / 512, (i64)ctx->sm_count * 16));
  narrow_kernel<<<blocks, 256, 0, ctx->stream>>>(in, n, (int *)ctx->vecs[*out].ptr);
  ctx->launches++;
  VDL_CUDA(ctx, cudaGetLastError());
  return VDL_OK;
}

// ---------------------------------------------------------------------------------- CrossProduct
// Vlite.hs:89-93, 283-292: "0,1,2,3 X 0,1 = 0,0,1,1,2,2,3,3 (outer), 0,1,0,1,0,1,0,1 (inner)".
__global__ void __launch_bounds__(256) cross_kernel(i64 n, i64 nr, int inner, i64 *__restrict__ out) {
  const i64 stride = (i64)gridDim.x * blockDim.x;
  for (i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) out[i] = inner ? i % nr : i / nr;
}

extern "C" int vdl_op_cross_product(vdl_ctx *ctx, vdl_vec left, vdl_vec right, int inner, vdl_vec *out) {
  if (!ctx || !out) return VDL_EINVAL;
  Vec *vl = vec_get(ctx, left), *vr = vec_get(ctx, right);
  if (!vl || !vr) return VDL_EINVAL;
  const i64 nl = vl->len, nr = vr->len;
  if (nr > 0 && nl > ((i64)1 << 33) / nr) return vdl_fail(ctx, VDL_EUNSUPPORTED, "CrossProduct of %lld x %lld rows", (long long)nl, (long long)nr);
  const i64 n = nl * nr;
  VDL_TRY(vec_new(ctx, VDL_I64, n, out));
  ctx->vecs[*out].domain = inner ? nr : nl;          // positions into that side (App. G2)
  if (n == 0) return VDL_OK;
  VDL_CUDA(ctx, cudaSetDevice(ctx->device));
  const int blocks = (int)std::max<i64>(1, std::min<i64>((n + 255) / 256, (i64)ctx->sm_count * 16));
  cross_kernel<<<blocks, 256, 0, ctx->stream>>>(n, nr, inner, (i64 *)ctx->vecs[*out].ptr);
  ctx->launches++;
  VDL_CUDA(ctx, cudaGetLastError());
  return VDL_OK;
}

// ---------------------------------------------------------------------------------- stable LSD radix sort (Partition, Order)
// 8 bits per pass over tiles of RDX_TILE rows: a digit histogram per tile, one exclusive scan over all of them (digit-major:
// the global stable order), a stable scatter of key and row id.
#define RDX_TILE 4096

// digit histogram per block, stored digit-major: hist[d * nblocks + block]
__global__ void __launch_bounds__(256) radix_hist_kernel(const u64 *__restrict__ key, i64 n, int shift, i64 nblocks, i64 *__restrict__ hist) {
  __shared__ int h[256];
  h[threadIdx.x] = 0;
  __syncthreads();
  i64 base = (i64)blockIdx.x * RDX_TILE;
  for (int s = 0; s < RDX_TILE / 256; s++) {
    i64 i = base + s * 256 + threadIdx.x;
    if (i < n) atomicAdd(&h[(key[i] >> shift) & 255], 1);
  }
  __syncthreads();
  hist[(i64)threadIdx.x * nblocks + blockIdx.x] = h[threadIdx.x];
}

// stable scatter: rank inside the block = elements with the same digit earlier in the block.  No idx_in: the row ids are
// the positions themselves (the first pass of a sort)
__global__ void __launch_bounds__(256) radix_scatter_kernel(const u64 *__restrict__ key_in, const i64 *__restrict__ idx_in, i64 n, int shift,
                                                            i64 nblocks, const i64 *__restrict__ offs, u64 *__restrict__ key_out,
                                                            i64 *__restrict__ idx_out) {
  __shared__ int wcount[8][256];   // per-warp count of each digit in the current step
  __shared__ int wbase[8][256];    // per-warp base of each digit in the current step
  __shared__ int run[256];         // elements of each digit in earlier steps of this block
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (int w = 0; w < 8; w++) wcount[w][tid] = 0;
  run[tid] = 0;
  __syncthreads();
  i64 base = (i64)blockIdx.x * RDX_TILE;
  for (int s = 0; s < RDX_TILE / 256; s++) {
    i64 i = base + s * 256 + tid;
    bool valid = i < n;
    u64 k = valid ? key_in[i] : 0;
    int d = valid ? (int)((k >> shift) & 255) : 256 + lane;   // invalid lanes never match anybody
    unsigned peers = __match_any_sync(0xffffffffu, d);
    int rank_in_warp = __popc(peers & ((1u << lane) - 1));
    if (valid && rank_in_warp == 0) wcount[warp][d] = __popc(peers);
    __syncthreads();
    {   // thread `tid` owns digit `tid`: per-warp counts -> per-warp bases; counts are cleared for the next step
      int off = run[tid];
#pragma unroll
      for (int w = 0; w < 8; w++) {
        int c = wcount[w][tid];
        wcount[w][tid] = 0;
        wbase[w][tid] = off;
        off += c;
      }
      run[tid] = off;
    }
    __syncthreads();
    if (valid) {
      i64 dst = offs[(i64)d * nblocks + blockIdx.x] + wbase[warp][d] + rank_in_warp;
      key_out[dst] = k;
      idx_out[dst] = idx_in ? idx_in[i] : i;
    }
  }
}

__global__ void __launch_bounds__(256) order_gather_kernel(const u64 *__restrict__ src, const i64 *__restrict__ pos, i64 n, u64 *__restrict__ dst) {
  for (i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (i64)gridDim.x * blockDim.x) dst[i] = src[pos[i]];
}

namespace {
struct VecScope {      // temporaries of one op, released (stream-ordered) when it returns
  vdl_ctx *ctx;
  std::vector<vdl_vec> v;
  ~VecScope() { for (vdl_vec h : v) vdl_vec_free(ctx, h); }
};
}  // namespace

// Stable sort of positions 0..n-1 (n >= 1) by packed words: word w of position i at words[w * n + i], word 0 the least
// significant, wbits[w] >= 1 bits of it in use (Order packs only the keys that are not constant, Partition has at least one
// pivot).  *out = the positions in sorted order, a new vector of length n.  Words are sorted least significant first, each
// gathered into the order reached so far.
static int lsd_sort(vdl_ctx *ctx, const u64 *words, int nwords, const int *wbits, i64 n, vdl_vec *out) {
  const i64 nb = (n + RDX_TILE - 1) / RDX_TILE;
  vdl_vec tk[2], ti[2];
  VecScope tmp{ctx, {}};
  for (int k = 0; k < 2; k++) {
    VDL_TRY(vec_new(ctx, VDL_I64, n, &tk[k])); tmp.v.push_back(tk[k]);
    VDL_TRY(vec_new(ctx, VDL_I64, n, &ti[k])); tmp.v.push_back(ti[k]);
  }
  int cur = 0;
  VDL_TRY(scratch_reserve(ctx, scan_elems(256 * nb) * 8));
  i64 *hist = (i64 *)ctx->scratch;
  u64 *key[2] = {(u64 *)ctx->vecs[tk[0]].ptr, (u64 *)ctx->vecs[tk[1]].ptr};
  i64 *idx[2] = {(i64 *)ctx->vecs[ti[0]].ptr, (i64 *)ctx->vecs[ti[1]].ptr};
  const i64 *ids = nullptr;       // the positions in the order reached so far; none before the first pass
  const int grid = (int)std::max<i64>(1, std::min<i64>((n + 255) / 256, (i64)ctx->sm_count * 16));
  for (int w = 0; w < nwords; w++) {
    const u64 *kin = words + (i64)w * n;
    if (w > 0) {          // the next more significant word, in the order reached so far
      order_gather_kernel<<<grid, 256, 0, ctx->stream>>>(kin, ids, n, key[cur]);
      ctx->launches++;
      kin = key[cur];
    }
    for (int shift = 0; shift < wbits[w]; shift += 8) {
      radix_hist_kernel<<<(unsigned)nb, 256, 0, ctx->stream>>>(kin, n, shift, nb, hist);
      device_exclusive_scan(ctx, hist, 256 * nb);
      radix_scatter_kernel<<<(unsigned)nb, 256, 0, ctx->stream>>>(kin, ids, n, shift, nb, hist, key[cur ^ 1], idx[cur ^ 1]);
      ctx->launches += 2;
      cur ^= 1;
      kin = key[cur];
      ids = idx[cur];
    }
  }
  VDL_CUDA(ctx, cudaGetLastError());
  tmp.v.erase(std::find(tmp.v.begin(), tmp.v.end(), ti[cur]));
  *out = ti[cur];
  return VDL_OK;
}

// ---------------------------------------------------------------------------------- Partition
// Vlite.hs:1082-1098 emits Partition(key, RangeC(min,1,max-min+1)); its result is the scatter position that
// sorts rows stably by key (1057-1060, 1172).  bucket(v) = number of pivots below v (App. G3).  Up to 256 buckets of
// unit-step pivots the permutation comes from a counting partition; otherwise it is lsd_sort of the rows by bucket (one
// word of the bits the pivot count needs: Q3's 38-bit composite key = 5 passes), inverted.
__device__ __forceinline__ u64 bucket_of(i64 v, i64 pfrom, i64 pstep, i64 pcount) {
  if (v <= pfrom) return 0;
  u64 d = (u64)v - (u64)pfrom;
  u64 b = pstep == 1 ? d : (d + (u64)pstep - 1) / (u64)pstep;     // every emitted Partition has unit-step pivots (Vlite.hs:1088-1091)
  return b > (u64)pcount ? (u64)pcount : b;
}

__global__ void __launch_bounds__(256) bucket_kernel(Operand data, i64 n, i64 pfrom, i64 pstep, i64 pcount, u64 *__restrict__ key) {
  i64 stride = (i64)gridDim.x * blockDim.x;
  for (i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) key[i] = bucket_of(op_ld(data, i), pfrom, pstep, pcount);
}

// Counting partition for <= 256 buckets (every low-cardinality group-by: Q1's 32, Q5's 128): two passes over the keys, no
// key / index ping-pong, no inversion.  The unit of work is a WARP: warp gw owns the contiguous rows [gw*chunk, (gw+1)*chunk)
// and a private table in shared memory, so neither pass has a block barrier or an atomic (a shared-memory atomic costs
// 32-64 cycles per warp instruction -- more than the whole per-row budget at HBM speed).  Per 32 rows the lanes that share
// a bucket are found with one ballot per bucket-index bit; the first of them updates the warp's table with a plain
// read-modify-write.
//   pass 1 (bucket_count_kernel): hist[d * nwarps + gw] = rows of bucket d in warp gw's chunk; the same pass counts the
//          descents, so keys that are already in bucket order cost ONE read (the Partition then stays an identity range);
//   scan over hist (bucket-major = the global stable order);
//   pass 2 (bucket_place_kernel): out[i] = running position of row i's bucket in its warp's table + rank among the 32.
#define CP_UNROLL 8
// bucket index of row i for unit-step pivots (every emitted Partition: Vlite.hs:1088-1091), operand kind fixed at compile time
template <int KIND>
__device__ __forceinline__ int bucket_at(const Operand &o, i64 i, i64 pfrom, i64 pcount) {
  const i64 v = KIND == 0 ? __ldg((const i64 *)o.p + i) : (KIND == 1 ? (i64)__ldg((const int *)o.p + i) : (i64)((u64)o.from + (u64)i * (u64)o.step));
  return (int)bucket_of(v, pfrom, 1, pcount);
}
// lanes whose bucket index has bit K set.  Written in PTX so that the test stays "and, compare with zero" (one LOP3 with a
// predicate result): the compiler's own canonical form is shift, mask, compare -- three instructions of the pipe that bounds
// these kernels, per bit and row.
template <int K>
__device__ __forceinline__ unsigned ballot_bit(int d) {
  unsigned b;
  asm volatile("{\n\t.reg .pred p;\n\t.reg .b32 t;\n\tand.b32 t, %1, %2;\n\tsetp.ne.u32 p, t, 0;\n\tvote.sync.ballot.b32 %0, p, 0xffffffff;\n\t}"
               : "=r"(b) : "r"(d), "n"(1 << K));
  return b;
}
template <int NBITS, int K = 0>
struct BucketBits {
  static __device__ __forceinline__ unsigned same(int d, unsigned peers) {          // lanes that agree with mine on bits K..NBITS-1
    const unsigned b = ballot_bit<K>(d);
    return BucketBits<NBITS, K + 1>::same(d, peers & ((d & (1 << K)) ? b : ~b));
  }
  static __device__ __forceinline__ unsigned owned(int d, unsigned a, const unsigned (&inv)[5]) {   // bits K..min(NBITS,5)-1 against the lane's own id
    return BucketBits<NBITS, K + 1>::owned(d, a & (ballot_bit<K>(d) ^ inv[K]), inv);
  }
};
template <int NBITS>
struct BucketBits<NBITS, NBITS> {
  static __device__ __forceinline__ unsigned same(int, unsigned peers) { return peers; }
  static __device__ __forceinline__ unsigned owned(int, unsigned a, const unsigned (&)[5]) { return a; }
};
template <int NBITS>
__device__ __forceinline__ unsigned same_bucket_lanes(int d, unsigned valid_lanes) { return BucketBits<NBITS>::same(d, valid_lanes); }
// Up to 64 buckets: lane l OWNS buckets l and l + 32.  m0 / m1 = the rows (lanes) of this step that fall into them: one
// ballot per bucket-index bit, combined with masks that depend on the lane id only -- the kernels are bound by the integer
// pipe, and this costs a third of the selects and compares of asking "who shares MY row's bucket" in every lane.
template <int NBITS, bool FULL>
__device__ __forceinline__ void owned_bucket_rows(int d, bool valid, const unsigned (&inv)[5], unsigned *m0, unsigned *m1) {
  const unsigned a = BucketBits<(NBITS < 5 ? NBITS : 5)>::owned(d, FULL ? 0xffffffffu : __ballot_sync(0xffffffffu, valid), inv);
  if (NBITS > 5) {
    const unsigned b5 = ballot_bit<5>(d);
    *m0 = a & ~b5; *m1 = a & b5;
  } else {
    *m0 = a; *m1 = 0;
  }
}

template <int NBITS, int KIND>
__global__ void __launch_bounds__(256, 5) bucket_count_kernel(Operand data, i64 n, i64 pfrom, i64 pcount, i64 chunk, i64 nwarps,
                                                              i64 *__restrict__ hist, int *descents) {
  __shared__ unsigned wh[8][NBITS > 6 ? 1 << NBITS : 1];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const i64 gw = (i64)blockIdx.x * 8 + w;
  if (gw >= nwarps) return;
  unsigned *h = wh[w];
  if (NBITS > 6) {
    for (int d = lane; d < (1 << NBITS); d += 32) h[d] = 0;
    __syncwarp();
  }
  unsigned inv[5];
#pragma unroll
  for (int k = 0; k < 5; k++) inv[k] = (lane >> k & 1) ? 0u : ~0u;
  unsigned cnt0 = 0, cnt1 = 0;
  const i64 r0 = gw * chunk, r1 = r0 + chunk < n ? r0 + chunk : n;
  const unsigned lt = (1u << lane) - 1;
  int bad = 0;
  int prev = r0 > 0 && r0 < n ? bucket_at<KIND>(data, r0 - 1, pfrom, pcount) : 0;
  auto step = [&](const i64 base, auto full_tag) {
    constexpr bool FULL = decltype(full_tag)::value;          // all 32 * CP_UNROLL rows exist: no bounds tests, no validity ballot
    int d[CP_UNROLL];
#pragma unroll
    for (int u = 0; u < CP_UNROLL; u++) {
      const i64 i = base + u * 32 + lane;
      d[u] = FULL || i < r1 ? bucket_at<KIND>(data, i, pfrom, pcount) : -1;
    }
#pragma unroll
    for (int u = 0; u < CP_UNROLL; u++) {
      const bool valid = FULL || d[u] >= 0;
      int left = __shfl_up_sync(0xffffffffu, d[u], 1);
      if (lane == 0) left = prev;
      bad |= valid && left > d[u];
      prev = __shfl_sync(0xffffffffu, d[u], 31);
      if (NBITS <= 6) {
        unsigned m0, m1;
        owned_bucket_rows<NBITS, FULL>(valid ? d[u] : 0, valid, inv, &m0, &m1);
        cnt0 += __popc(m0);
        if (NBITS > 5) cnt1 += __popc(m1);
      } else {
        const unsigned peers = same_bucket_lanes<NBITS>(d[u], FULL ? 0xffffffffu : __ballot_sync(0xffffffffu, valid));
        if (valid && (peers & lt) == 0) h[d[u]] += __popc(peers);
        __syncwarp();
      }
    }
  };
  i64 base = r0;
  for (; base + 32 * CP_UNROLL <= r1; base += 32 * CP_UNROLL) step(base, std::true_type());
  if (base < r1) step(base, std::false_type());
  if (NBITS <= 6) {
    if (lane <= pcount) hist[(i64)lane * nwarps + gw] = cnt0;
    if (NBITS > 5 && lane + 32 <= pcount) hist[(i64)(lane + 32) * nwarps + gw] = cnt1;
  } else {
    for (int d = lane; d <= pcount; d += 32) hist[(i64)d * nwarps + gw] = h[d];
  }
  if (__any_sync(0xffffffffu, bad) && lane == 0) atomicAdd(descents, 1);
}

template <int NBITS, int KIND>
__global__ void __launch_bounds__(256, 5) bucket_place_kernel(Operand data, i64 n, i64 pfrom, i64 pcount, i64 chunk, i64 nwarps,
                                                              const i64 *__restrict__ offs, i64 *__restrict__ out) {
  __shared__ i64 wpos[8][1 << NBITS];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const i64 gw = (i64)blockIdx.x * 8 + w;
  if (gw >= nwarps) return;
  i64 *pos = wpos[w];
  for (int d = lane; d <= pcount; d += 32) pos[d] = offs[(i64)d * nwarps + gw];
  __syncwarp();
  unsigned inv[5];
#pragma unroll
  for (int k = 0; k < 5; k++) inv[k] = (lane >> k & 1) ? 0u : ~0u;
  unsigned cnt0 = 0, cnt1 = 0;            // rows of this warp's chunk so far in the buckets this lane owns
  const i64 r0 = gw * chunk, r1 = r0 + chunk < n ? r0 + chunk : n;
  const unsigned lt = (1u << lane) - 1;
  auto step = [&](const i64 base, auto full_tag) {
    constexpr bool FULL = decltype(full_tag)::value;
    int d[CP_UNROLL];
#pragma unroll
    for (int u = 0; u < CP_UNROLL; u++) {
      const i64 i = base + u * 32 + lane;
      d[u] = FULL || i < r1 ? bucket_at<KIND>(data, i, pfrom, pcount) : -1;
    }
#pragma unroll
    for (int u = 0; u < CP_UNROLL; u++) {
      const bool valid = FULL || d[u] >= 0;
      if (NBITS <= 6) {
        const int dd = valid ? d[u] : 0;
        unsigned m0, m1;
        owned_bucket_rows<NBITS, FULL>(dd, valid, inv, &m0, &m1);
        // what the owner of my row's bucket knows: the rows of this step in it, and the rows before this step
        unsigned peers = __shfl_sync(0xffffffffu, m0, dd & 31), before = __shfl_sync(0xffffffffu, cnt0, dd & 31);
        if (NBITS > 5) {
          const unsigned peers1 = __shfl_sync(0xffffffffu, m1, dd & 31), before1 = __shfl_sync(0xffffffffu, cnt1, dd & 31);
          if (dd & 32) { peers = peers1; before = before1; }
        }
        if (valid) out[base + u * 32 + lane] = pos[dd] + (i64)(before + __popc(peers & lt));
        cnt0 += __popc(m0);
        if (NBITS > 5) cnt1 += __popc(m1);
      } else {
        const unsigned peers = same_bucket_lanes<NBITS>(d[u], FULL ? 0xffffffffu : __ballot_sync(0xffffffffu, valid));
        const int rank = __popc(peers & lt);
        const i64 at = valid ? pos[d[u]] : 0;
        if (valid) out[base + u * 32 + lane] = at + rank;
        __syncwarp();
        if (valid && rank == 0) pos[d[u]] = at + __popc(peers);
        __syncwarp();
      }
    }
  };
  i64 base = r0;
  for (; base + 32 * CP_UNROLL <= r1; base += 32 * CP_UNROLL) step(base, std::true_type());
  if (base < r1) step(base, std::false_type());
}

__global__ void __launch_bounds__(256) invert_perm_kernel(const i64 *__restrict__ order, i64 n, i64 *__restrict__ out) {
  i64 stride = (i64)gridDim.x * blockDim.x;
  for (i64 j = (i64)blockIdx.x * blockDim.x + threadIdx.x; j < n; j += stride) out[order[j]] = j;
}

// rows already ordered by bucket (e.g. lineitem clustered on l_orderkey, storage.csv `sorted`)?  counts the descents
__global__ void __launch_bounds__(256) descents_kernel(Operand data, i64 n, i64 pfrom, i64 pstep, i64 pcount, int *descents) {
  // 4 consecutive elements per thread (+ the next one): independent loads in flight, every element read ~1.25 times
  const i64 stride = (i64)gridDim.x * blockDim.x * 4;
  int bad = 0;
  for (i64 i0 = ((i64)blockIdx.x * blockDim.x + threadIdx.x) * 4; i0 < n; i0 += stride) {
    u64 b[5];
#pragma unroll
    for (int k = 0; k < 5; k++) b[k] = i0 + k < n ? bucket_of(op_ld(data, i0 + k), pfrom, pstep, pcount) : ~0ull;
#pragma unroll
    for (int k = 0; k < 4; k++) bad |= b[k] > b[k + 1] && i0 + k + 1 < n;
  }
  if (__any_sync(0xffffffffu, bad) && (threadIdx.x & 31) == 0) atomicAdd(descents, 1);
}

extern "C" int vdl_op_partition(vdl_ctx *ctx, vdl_vec data, int64_t pfrom, int64_t pstep, int64_t pcount, vdl_vec *out) {
  if (!ctx || !out) return VDL_EINVAL;
  Vec *vd = vec_get(ctx, data);
  if (!vd) return VDL_EINVAL;
  if (pcount < 1 || pstep < 1) return vdl_fail(ctx, VDL_EINVAL, "Partition: pivots must be an ascending range (count %lld step %lld)", (long long)pcount, (long long)pstep);
  i64 n = vd->len;
  Operand od = operand_of(*vd);
  VDL_CUDA(ctx, cudaSetDevice(ctx->device));
  int bits = 0;
  while (bits < 63 && ((u64)pcount >> bits)) bits++;
  if (n > 0 && pcount < 256 && pstep == 1) {   // buckets 0..pcount fit one digit: counting partition, sortedness checked by its first pass
    const int nbits = bits <= 2 ? 2 : (bits <= 4 ? 4 : (bits <= 5 ? 5 : (bits <= 6 ? 6 : 8)));
    const i64 step = 32 * CP_UNROLL;
    i64 nwarps = std::min<i64>((n + step - 1) / step, (i64)ctx->sm_count * 5 * 8);      // one wave: 5 blocks of 8 warps per SM (48 registers)
    const i64 chunk = ((n + nwarps - 1) / nwarps + step - 1) / step * step;
    nwarps = (n + chunk - 1) / chunk;
    const unsigned grid = (unsigned)((nwarps + 7) / 8);
    const i64 nh = (pcount + 1) * nwarps;
    VDL_TRY(scratch_reserve(ctx, (scan_elems(nh) + 8) * 8));
    i64 *h = (i64 *)ctx->scratch;
    int *d_desc = (int *)(h + scan_elems(nh)), h_desc = 1;
    VDL_CUDA(ctx, cudaMemsetAsync(d_desc, 0, sizeof(int), ctx->stream));
#define CP_LAUNCH_K(KERNEL, NB, ...)                                                                                  \
    switch (od.kind) {                                                                                                \
      case 0: KERNEL<NB, 0><<<grid, 256, 0, ctx->stream>>>(__VA_ARGS__); break;                                       \
      case 1: KERNEL<NB, 1><<<grid, 256, 0, ctx->stream>>>(__VA_ARGS__); break;                                       \
      default: KERNEL<NB, 2><<<grid, 256, 0, ctx->stream>>>(__VA_ARGS__); break;                                      \
    }
#define CP_LAUNCH(KERNEL, ...)                                                                                        \
    switch (nbits) {                                                                                                  \
      case 2: CP_LAUNCH_K(KERNEL, 2, __VA_ARGS__) break;                                                              \
      case 4: CP_LAUNCH_K(KERNEL, 4, __VA_ARGS__) break;                                                              \
      case 5: CP_LAUNCH_K(KERNEL, 5, __VA_ARGS__) break;                                                              \
      case 6: CP_LAUNCH_K(KERNEL, 6, __VA_ARGS__) break;                                                              \
      default: CP_LAUNCH_K(KERNEL, 8, __VA_ARGS__) break;                                                             \
    }
    CP_LAUNCH(bucket_count_kernel, od, n, pfrom, pcount, chunk, nwarps, h, d_desc)
    ctx->launches++;
    VDL_TRY(read_scalar(ctx, d_desc, &h_desc, sizeof(int)));
    // keys already in bucket order sort to the identity permutation, which stays a virtual range -- a Scatter by it is the
    // source vector itself (its domain is n: positions 0..n-1)
    if (h_desc == 0) return vec_new_range(ctx, 0, 1, n, out);
    VDL_TRY(vec_new(ctx, VDL_I64, n, out));
    ctx->vecs[*out].domain = n;
    ctx->vecs[*out].is_perm = true;
    device_exclusive_scan(ctx, h, nh);
    CP_LAUNCH(bucket_place_kernel, od, n, pfrom, pcount, chunk, nwarps, h, (i64 *)ctx->vecs[*out].ptr)
#undef CP_LAUNCH
#undef CP_LAUNCH_K
    ctx->launches++;
    VDL_CUDA(ctx, cudaGetLastError());
    return VDL_OK;
  }
  VecScope tmp{ctx, {}};
  vdl_vec sorted = -1;
  const int grid = (int)std::max<i64>(1, std::min<i64>((n + 255) / 256, (i64)ctx->sm_count * 16));
  if (n > 0) {
    // one cheap pass first: keys that are already in bucket order sort to the identity permutation, which stays a
    // virtual range -- no radix passes, and a Scatter by it is the source vector itself
    VDL_TRY(scratch_reserve(ctx, 64));
    int *d_desc = (int *)ctx->scratch, h_desc = 1;
    VDL_CUDA(ctx, cudaMemsetAsync(d_desc, 0, sizeof(int), ctx->stream));
    int g0 = (int)std::max<i64>(1, std::min<i64>((n + 1023) / 1024, (i64)ctx->sm_count * 16));
    descents_kernel<<<g0, 256, 0, ctx->stream>>>(od, n, pfrom, pstep, pcount, d_desc);
    ctx->launches++;
    VDL_TRY(read_scalar(ctx, d_desc, &h_desc, sizeof(int)));
    if (h_desc == 0) return vec_new_range(ctx, 0, 1, n, out);      // (its domain is n: positions 0..n-1)
    // the rows in stable bucket order: one word of `bits` bits per row
    vdl_vec kv;
    VDL_TRY(vec_new(ctx, VDL_I64, n, &kv));
    tmp.v.push_back(kv);
    bucket_kernel<<<grid, 256, 0, ctx->stream>>>(od, n, pfrom, pstep, pcount, (u64 *)ctx->vecs[kv].ptr);
    ctx->launches++;
    VDL_TRY(lsd_sort(ctx, (const u64 *)ctx->vecs[kv].ptr, 1, &bits, n, &sorted));
    tmp.v.push_back(sorted);
  }
  // allocated after the sort, whose temporaries are released by then: the peak stays at five n-row vectors
  VDL_TRY(vec_new(ctx, VDL_I64, n, out));
  ctx->vecs[*out].domain = n;
  ctx->vecs[*out].is_perm = true;
  if (n == 0) return VDL_OK;
  invert_perm_kernel<<<grid, 256, 0, ctx->stream>>>((const i64 *)ctx->vecs[sorted].ptr, n, (i64 *)ctx->vecs[*out].ptr);
  ctx->launches++;
  VDL_CUDA(ctx, cudaGetLastError());
  return VDL_OK;
}

// ---------------------------------------------------------------------------------- Order (ORDER BY / LIMIT)
// Every key becomes its distance from its minimum (ascending) or from its maximum (descending) in uint64 -- exact at
// INT64_MIN / INT64_MAX, where -x is not -- and the distances are bit-packed: the last key in the least significant bits,
// each key in the bits its range needs, a constant key in none.  Keys that do not fit one 64-bit word spill into further
// words (word 0 least significant).  A full order is lsd_sort over the packed words, the one Partition uses.  With a LIMIT a
// radix select comes first: the pack kernel also counts the top 8-bit digit, the host finds the digit at which the count
// reaches the limit, the rows at or below it are compacted in row order by FoldSelect (so ties stay stable) -- refined digit
// by digit while there are many more of them than the limit -- and only those candidates are sorted.
struct OrderArgs {
  Operand key[VDL_MAX_ORDER_KEYS];
  u64 base[VDL_MAX_ORDER_KEYS];     // minimum (ascending) or maximum (descending)
  int desc[VDL_MAX_ORDER_KEYS];
  int word[VDL_MAX_ORDER_KEYS];     // packed word of the key; -1: constant key (or no key)
  int shift[VDL_MAX_ORDER_KEYS];    // its lowest bit in that word
  int nkeys, nwords, top_shift;     // top_shift: lowest bit of the most significant word's top digit
};

__global__ void __launch_bounds__(256) order_minmax_kernel(const __grid_constant__ OrderArgs a, i64 n, i64 *mm /* [min, max] per key */) {
  const i64 stride = (i64)gridDim.x * blockDim.x;
  for (int k = 0; k < a.nkeys; k++) {
    i64 lo = INT64_MAX, hi = INT64_MIN;
    for (i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
      const i64 v = op_ld(a.key[k], i);
      lo = v < lo ? v : lo;
      hi = v > hi ? v : hi;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const i64 x = __shfl_xor_sync(0xffffffffu, lo, o), y = __shfl_xor_sync(0xffffffffu, hi, o);
      lo = x < lo ? x : lo;
      hi = y > hi ? y : hi;
    }
    if ((threadIdx.x & 31) == 0) {
      atomicMin((long long *)&mm[2 * k], (long long)lo);
      atomicMax((long long *)&mm[2 * k + 1], (long long)hi);
    }
  }
}

// words[w * n + i] = packed word w of row i; HIST: hist[d] += rows whose most significant word has top digit d (shared
// counters, one global atomic per digit and block)
template <bool HIST>
__global__ void __launch_bounds__(256) order_pack_kernel(const __grid_constant__ OrderArgs a, i64 n, u64 *__restrict__ words,
                                                         unsigned long long *__restrict__ hist) {
  __shared__ unsigned h[256];
  if (HIST) {
    h[threadIdx.x] = 0;
    __syncthreads();
  }
  const i64 stride = (i64)gridDim.x * blockDim.x;
  for (i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    u64 v[VDL_MAX_ORDER_KEYS];
#pragma unroll
    for (int k = 0; k < VDL_MAX_ORDER_KEYS; k++) {
      v[k] = 0;
      if (a.word[k] >= 0) {
        const u64 x = (u64)op_ld(a.key[k], i);
        v[k] = (a.desc[k] ? a.base[k] - x : x - a.base[k]) << a.shift[k];
      }
    }
#pragma unroll
    for (int w = 0; w < VDL_MAX_ORDER_KEYS; w++) {
      if (w >= a.nwords) break;
      u64 acc = 0;
#pragma unroll
      for (int k = 0; k < VDL_MAX_ORDER_KEYS; k++) acc |= a.word[k] == w ? v[k] : 0;
      words[(i64)w * n + i] = acc;
      if (HIST && w == a.nwords - 1) atomicAdd(&h[(acc >> a.top_shift) & 255], 1u);
    }
  }
  if (HIST) {
    __syncthreads();
    if (h[threadIdx.x]) atomicAdd(&hist[threadIdx.x], (unsigned long long)h[threadIdx.x]);
  }
}

// the next digit, bits [s_new, s_old), of the rows whose bits from s_old up equal `prefix`
__global__ void __launch_bounds__(256) order_refine_hist_kernel(const u64 *__restrict__ top, i64 n, int s_old, u64 prefix, int s_new,
                                                                unsigned long long *__restrict__ hist) {
  __shared__ unsigned h[256];
  h[threadIdx.x] = 0;
  __syncthreads();
  const u64 mask = (1ull << (s_old - s_new)) - 1;
  for (i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (i64)gridDim.x * blockDim.x) {
    const u64 x = top[i];
    if ((x >> s_old) == prefix) atomicAdd(&h[(x >> s_new) & mask], 1u);
  }
  __syncthreads();
  if (h[threadIdx.x]) atomicAdd(&hist[threadIdx.x], (unsigned long long)h[threadIdx.x]);
}

__global__ void __launch_bounds__(256) order_candidate_kernel(const u64 *__restrict__ top, i64 n, int s, u64 prefix, int *__restrict__ flag) {
  for (i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (i64)gridDim.x * blockDim.x) flag[i] = (top[i] >> s) <= prefix;
}

extern "C" int vdl_op_order(vdl_ctx *ctx, int nkeys, const vdl_vec *keys, const int *descending, int64_t limit, vdl_vec *out) {
  if (!ctx || !out || (nkeys > 0 && !keys)) return VDL_EINVAL;
  if (nkeys < 0 || nkeys > VDL_MAX_ORDER_KEYS) return vdl_fail(ctx, VDL_EINVAL, "Order: %d keys (at most %d)", nkeys, VDL_MAX_ORDER_KEYS);
  if (nkeys == 0) {
    if (limit < 0) return vdl_fail(ctx, VDL_EINVAL, "Order: neither keys nor a limit");
    return vec_new_range(ctx, 0, 1, limit, out);
  }
  OrderArgs a;
  memset(&a, 0, sizeof a);
  i64 n = -1;
  for (int k = 0; k < VDL_MAX_ORDER_KEYS; k++) a.word[k] = -1;
  for (int k = 0; k < nkeys; k++) {
    Vec *v = vec_get(ctx, keys[k]);
    if (!v) return VDL_EINVAL;
    if (n >= 0 && v->len != n) return vdl_fail(ctx, VDL_EINVAL, "Order: key %d has %lld rows, key 0 has %lld", k, (long long)v->len, (long long)n);
    n = v->len;
    a.key[k] = operand_of(*v);
    a.desc[k] = descending && descending[k] ? 1 : 0;
  }
  a.nkeys = nkeys;
  const i64 m = limit < 0 || limit > n ? n : limit;
  if (m == 0) {
    VDL_TRY(vec_new(ctx, VDL_I64, 0, out));
    ctx->vecs[*out].domain = n;
    return VDL_OK;
  }
  VDL_CUDA(ctx, cudaSetDevice(ctx->device));
  VecScope tmp{ctx, {}};
  // minimum and maximum of every key in one pass ([min, max] per key, then the 256 top-digit counters of the select)
  vdl_vec mmv;
  VDL_TRY(vec_new(ctx, VDL_I64, 2 * VDL_MAX_ORDER_KEYS + 256, &mmv));
  tmp.v.push_back(mmv);
  i64 *mm = (i64 *)ctx->vecs[mmv].ptr;
  unsigned long long *hist = (unsigned long long *)(mm + 2 * VDL_MAX_ORDER_KEYS);
  i64 hmm[2 * VDL_MAX_ORDER_KEYS];
  for (int k = 0; k < VDL_MAX_ORDER_KEYS; k++) { hmm[2 * k] = INT64_MAX; hmm[2 * k + 1] = INT64_MIN; }
  VDL_CUDA(ctx, cudaMemcpyAsync(mm, hmm, sizeof hmm, cudaMemcpyHostToDevice, ctx->stream));
  VDL_CUDA(ctx, cudaMemsetAsync(hist, 0, 256 * sizeof(unsigned long long), ctx->stream));
  const int grid = (int)std::max<i64>(1, std::min<i64>((n + 255) / 256, (i64)ctx->sm_count * 8));
  order_minmax_kernel<<<grid, 256, 0, ctx->stream>>>(a, n, mm);
  ctx->launches++;
  VDL_TRY(read_scalar(ctx, mm, hmm, 64));
  if (nkeys > 4) VDL_TRY(read_scalar(ctx, mm + 8, hmm + 8, 64));
  // packing, least significant key first: a key takes bits(max - min) bits, a word holds what fits in 64
  int wbits[VDL_MAX_ORDER_KEYS] = {0}, nwords = 0;
  for (int k = nkeys - 1; k >= 0; k--) {
    const u64 span = (u64)hmm[2 * k + 1] - (u64)hmm[2 * k];
    const int width = span ? 64 - __builtin_clzll(span) : 0;
    a.base[k] = (u64)hmm[2 * k + a.desc[k]];
    if (!width) continue;
    if (nwords == 0 || wbits[nwords - 1] + width > 64) nwords++;
    a.word[k] = nwords - 1;
    a.shift[k] = wbits[nwords - 1];
    wbits[nwords - 1] += width;
  }
  a.nwords = nwords;
  if (nwords == 0) {       // every key constant: row order
    VDL_TRY(vec_new_range(ctx, 0, 1, m, out));
    ctx->vecs[*out].domain = n;
    return VDL_OK;
  }
  const int W = nwords - 1;
  a.top_shift = wbits[W] > 8 ? wbits[W] - 8 : 0;
  const bool select = m < n;
  vdl_vec wv;
  VDL_TRY(vec_new(ctx, VDL_I64, (i64)nwords * n, &wv));
  tmp.v.push_back(wv);
  u64 *words = (u64 *)ctx->vecs[wv].ptr;
  const int pgrid = (int)std::max<i64>(1, std::min<i64>((n + 255) / 256, (i64)ctx->sm_count * 16));
  if (select) order_pack_kernel<true><<<pgrid, 256, 0, ctx->stream>>>(a, n, words, hist);
  else order_pack_kernel<false><<<pgrid, 256, 0, ctx->stream>>>(a, n, words, hist);
  ctx->launches++;
  VDL_CUDA(ctx, cudaGetLastError());
  if (!select) {
    VDL_TRY(lsd_sort(ctx, words, nwords, wbits, n, out));
    ctx->vecs[*out].domain = n;
    ctx->vecs[*out].is_perm = true;
    return VDL_OK;
  }
  // radix select on the most significant word: `prefix` (its bits from s up) such that the first m rows in order are among
  // the rows whose bits from s up are <= prefix
  const u64 *top = words + (i64)W * n;
  int s_hi = wbits[W], s = a.top_shift;
  u64 hi = 0, prefix = 0;
  i64 cands = 0;
  i64 below = 0;                                   // rows whose bits from s_hi up are < hi: all of them come first
  const i64 enough = std::max<i64>(2 * m, 4096);
  unsigned long long hh[256];
  for (;;) {
    VDL_CUDA(ctx, cudaMemcpyAsync(hh, hist, sizeof hh, cudaMemcpyDeviceToHost, ctx->stream));
    VDL_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    int t = 0;
    i64 run = below;
    while (t < 255 && run + (i64)hh[t] < m) run += (i64)hh[t++];
    prefix = (hi << (s_hi - s)) | (u64)t;
    below = run;
    cands = run + (i64)hh[t];
    if (cands <= enough || s == 0) break;
    hi = prefix;
    s_hi = s;
    s = s > 8 ? s - 8 : 0;
    VDL_CUDA(ctx, cudaMemsetAsync(hist, 0, 256 * sizeof(unsigned long long), ctx->stream));
    order_refine_hist_kernel<<<pgrid, 256, 0, ctx->stream>>>(top, n, s_hi, hi, s, hist);
    ctx->launches++;
  }
  vdl_vec fv, cand, cw, sorted;
  VDL_TRY(vec_new(ctx, VDL_I32, n, &fv));
  tmp.v.push_back(fv);
  order_candidate_kernel<<<pgrid, 256, 0, ctx->stream>>>(top, n, s, prefix, (int *)ctx->vecs[fv].ptr);
  ctx->launches++;
  VDL_TRY(vdl_op_fold_select(ctx, fv, &cand));      // candidate positions in row order
  tmp.v.push_back(cand);
  const i64 c = ctx->vecs[cand].len;
  if (c != cands) return vdl_fail(ctx, VDL_ECUDA, "Order: %lld candidates compacted, %lld counted", (long long)c, (long long)cands);
  VDL_TRY(vec_new(ctx, VDL_I64, (i64)nwords * c, &cw));
  tmp.v.push_back(cw);
  u64 *cwords = (u64 *)ctx->vecs[cw].ptr;
  const i64 *cpos = (const i64 *)ctx->vecs[cand].ptr;
  const int cgrid = (int)std::max<i64>(1, std::min<i64>((c + 255) / 256, (i64)ctx->sm_count * 16));
  for (int w = 0; w < nwords; w++) order_gather_kernel<<<cgrid, 256, 0, ctx->stream>>>(words + (i64)w * n, cpos, c, cwords + (i64)w * c);
  ctx->launches += nwords;
  VDL_TRY(lsd_sort(ctx, cwords, nwords, wbits, c, &sorted));
  tmp.v.push_back(sorted);
  ctx->vecs[sorted].len = m;                        // the first m candidates in order, mapped back to row positions
  return vdl_op_gather(ctx, cand, sorted, out);
}

// ---------------------------------------------------------------------------------- Collate (string ranks)
// A char / varchar value is a heap offset (or a dictionary code, origin != 0), and offset order is not string order.
// vdl_op_collate turns the offsets into dense collation ranks, which vdl_op_order then sorts like any integer key:
//  - scan: min, max and OR of the in-range values v = data - origin in one pass; a = trailing zeros of the OR, so every
//    value is a multiple of 2^a and (v >> a) - (min >> a) indexes a slot table over [min, max] (8-aligned heaps: a = 3);
//  - the slots that occur are flagged and compacted in ascending offset order by FoldSelect: m distinct strings;
//  - their lengths, then their bytes as big-endian 8-byte words (zero after the NUL, sign bit flipped, so signed int64
//    order is unsigned byte order and a proper prefix sorts first), 8 words at a time: the last chunk is sorted first
//    by vdl_op_order (stable), each earlier chunk is written in the order reached so far and sorted again -- no length
//    cap and no sort code of its own; a word equal across all strings takes no radix pass (a constant key);
//  - neighbours in the final order are compared over their full bytes, the "differs" flags scanned to dense ranks,
//    the ranks scattered into the slot table and gathered per row.
// The m strings are the heap's distinct entries that occur, not the rows: at TPC-H's result sizes a handful to a few
// hundred thousand.  The rows are read three times (scan, flag, gather) and written once.  The host waits on the device
// at least four times: for the scan's min / max, FoldSelect's count, the longest string, and once per chunk inside
// vdl_op_order (twice when a chunk has more than 4 words), which is why small inputs are expected to cost launches and
// round trips rather than bytes.
#define COLLATE_CHUNK 8

__device__ __forceinline__ bool collate_in_range(const Operand &data, i64 i, i64 origin, i64 heap_len, i64 *v) {
  *v = (i64)((u64)op_ld(data, i) - (u64)origin);
  return (u64)*v < (u64)heap_len;
}

__global__ void __launch_bounds__(256) collate_scan_kernel(Operand data, i64 n, i64 origin, i64 heap_len, i64 *mm /* min, max, or */,
                                                           int *errflag) {
  i64 lo = INT64_MAX, hi = INT64_MIN;
  unsigned long long bits = 0;
  int bad = 0;
  for (i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (i64)gridDim.x * blockDim.x) {
    i64 v;
    if (!collate_in_range(data, i, origin, heap_len, &v)) { bad++; continue; }
    lo = v < lo ? v : lo;
    hi = v > hi ? v : hi;
    bits |= (unsigned long long)v;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const i64 x = __shfl_xor_sync(0xffffffffu, lo, o), y = __shfl_xor_sync(0xffffffffu, hi, o);
    lo = x < lo ? x : lo;
    hi = y > hi ? y : hi;
    bits |= __shfl_xor_sync(0xffffffffu, bits, o);
    bad += __shfl_xor_sync(0xffffffffu, bad, o);
  }
  if ((threadIdx.x & 31) == 0) {
    if (lo <= hi) {
      atomicMin((long long *)&mm[0], (long long)lo);
      atomicMax((long long *)&mm[1], (long long)hi);
      atomicOr((unsigned long long *)&mm[2], bits);
    }
    if (bad) atomicAdd(errflag, bad);
  }
}

__global__ void __launch_bounds__(256) collate_flag_kernel(Operand data, i64 n, i64 origin, i64 heap_len, int a, i64 slot0, int *__restrict__ flag) {
  for (i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (i64)gridDim.x * blockDim.x) {
    i64 v;
    if (collate_in_range(data, i, origin, heap_len, &v)) flag[(v >> a) - slot0] = 1;
  }
}

// len[j] of distinct string j (slot sel[j]); a string the heap ends inside counts as ending there, and as a range error
__global__ void __launch_bounds__(256) collate_len_kernel(const unsigned char *__restrict__ heap, i64 heap_len, const i64 *__restrict__ sel, i64 m,
                                                          int a, i64 slot0, i64 *__restrict__ len, i64 *maxlen, int *errflag) {
  i64 mx = 0;
  for (i64 j = (i64)blockIdx.x * blockDim.x + threadIdx.x; j < m; j += (i64)gridDim.x * blockDim.x) {
    const i64 off = (slot0 + sel[j]) << a;
    i64 k = off;
    while (k < heap_len && heap[k]) k++;
    if (k == heap_len) atomicAdd(errflag, 1);
    len[j] = k - off;
    mx = k - off > mx ? k - off : mx;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const i64 x = __shfl_xor_sync(0xffffffffu, mx, o);
    mx = x > mx ? x : mx;
  }
  if ((threadIdx.x & 31) == 0 && mx) atomicMax((long long *)maxlen, (long long)mx);
}

// words w0 .. w0 + nw - 1 of the string at position i of the order reached so far (perm; none: ascending offset order)
struct CollateWords { i64 *w[COLLATE_CHUNK]; };
__global__ void __launch_bounds__(256) collate_words_kernel(const unsigned char *__restrict__ heap, const i64 *__restrict__ sel, const i64 *__restrict__ len,
                                                            Operand perm, bool has_perm, i64 m, int a, i64 slot0, int w0, int nw,
                                                            const __grid_constant__ CollateWords out) {
  for (i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x; i < m; i += (i64)gridDim.x * blockDim.x) {
    const i64 j = has_perm ? op_ld(perm, i) : i;
    const unsigned char *s = heap + ((slot0 + sel[j]) << a);
    const i64 l = len[j];
#pragma unroll
    for (int w = 0; w < COLLATE_CHUNK; w++) {
      if (w >= nw) break;
      u64 x = 0;
      const i64 b0 = (i64)(w0 + w) * 8;
#pragma unroll
      for (int b = 0; b < 8; b++) x |= (b0 + b < l ? (u64)s[b0 + b] : 0ull) << (56 - 8 * b);
      out.w[w][i] = (i64)(x ^ (1ull << 63));
    }
  }
}

// diff[k] = 1 when the k-th and (k+1)-th strings of the final order differ (the exclusive scan of it is the dense rank)
__global__ void __launch_bounds__(256) collate_diff_kernel(const unsigned char *__restrict__ heap, const i64 *__restrict__ sel, const i64 *__restrict__ len,
                                                           Operand perm, i64 m, int a, i64 slot0, i64 *__restrict__ diff) {
  for (i64 k = (i64)blockIdx.x * blockDim.x + threadIdx.x; k < m; k += (i64)gridDim.x * blockDim.x) {
    i64 d = 0;
    if (k + 1 < m) {
      const i64 x = op_ld(perm, k), y = op_ld(perm, k + 1);
      const i64 l = len[x];
      d = l != len[y];
      const unsigned char *s = heap + ((slot0 + sel[x]) << a), *t = heap + ((slot0 + sel[y]) << a);
      for (i64 b = 0; !d && b < l; b++) d = s[b] != t[b];
    }
    diff[k] = d;
  }
}

__global__ void __launch_bounds__(256) collate_scatter_kernel(const i64 *__restrict__ rank, const i64 *__restrict__ sel, Operand perm, i64 m,
                                                              int *__restrict__ table) {
  for (i64 k = (i64)blockIdx.x * blockDim.x + threadIdx.x; k < m; k += (i64)gridDim.x * blockDim.x) table[sel[op_ld(perm, k)]] = (int)rank[k];
}

__global__ void __launch_bounds__(256) collate_gather_kernel(Operand data, i64 n, i64 origin, i64 heap_len, int a, i64 slot0, const int *__restrict__ table,
                                                             i64 *__restrict__ out) {
  for (i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (i64)gridDim.x * blockDim.x) {
    i64 v;
    out[i] = collate_in_range(data, i, origin, heap_len, &v) ? (i64)table[(v >> a) - slot0] : 0;
  }
}

extern "C" int vdl_op_collate(vdl_ctx *ctx, vdl_vec data, vdl_vec heap, int64_t origin, vdl_vec *out) {
  if (!ctx || !out) return VDL_EINVAL;
  Vec *vd = vec_get(ctx, data), *vh = vec_get_any(ctx, heap);
  if (!vd || !vh) return VDL_EINVAL;
  if (vh->dtype != VDL_U8) return vdl_fail(ctx, VDL_EINVAL, "Collate: the heap must be a string heap (a VDL_U8 vector; Load,<table>.<col>.heap)");
  const i64 n = vd->len, hl = vh->len;
  const Operand od = operand_of(*vd);
  const unsigned char *hp = (const unsigned char *)vh->ptr;
  VDL_TRY(vec_new(ctx, VDL_I64, n, out));
  ctx->vecs[*out].narrow32 = true;                  // ranks < m < 2^31
  if (n == 0) return VDL_OK;
  VDL_CUDA(ctx, cudaSetDevice(ctx->device));
  i64 *res = (i64 *)ctx->vecs[*out].ptr;
  VecScope tmp{ctx, {}};
  const int grid = (int)std::max<i64>(1, std::min<i64>((n + 255) / 256, (i64)ctx->sm_count * 16));
  // scan: [min, max, or] of the in-range values, then the longest string
  vdl_vec mmv;
  VDL_TRY(vec_new(ctx, VDL_I64, 4, &mmv));
  tmp.v.push_back(mmv);
  i64 *mm = (i64 *)ctx->vecs[mmv].ptr;
  i64 hmm[4] = {INT64_MAX, INT64_MIN, 0, 0};
  VDL_CUDA(ctx, cudaMemcpyAsync(mm, hmm, sizeof hmm, cudaMemcpyHostToDevice, ctx->stream));
  collate_scan_kernel<<<grid, 256, 0, ctx->stream>>>(od, n, origin, hl, mm, ctx->d_errflag);
  ctx->launches++;
  VDL_TRY(read_scalar(ctx, mm, hmm, 24));
  if (hmm[0] > hmm[1]) {                            // no offset inside the heap: every row is a range error, rank 0
    VDL_CUDA(ctx, cudaMemsetAsync(res, 0, (size_t)n * 8, ctx->stream));
    return VDL_OK;
  }
  const int a = hmm[2] ? __builtin_ctzll((u64)hmm[2]) : 0;
  const i64 slot0 = hmm[0] >> a, slots = (hmm[1] >> a) - slot0 + 1;
  if (slots > INT32_MAX) return vdl_fail(ctx, VDL_EUNSUPPORTED, "Collate: %lld string slots (at most %d)", (long long)slots, INT32_MAX);
  // distinct strings: the slots that occur, in ascending offset order
  vdl_vec tv, sv;
  VDL_TRY(vec_new(ctx, VDL_I32, slots, &tv));
  tmp.v.push_back(tv);
  int *table = (int *)ctx->vecs[tv].ptr;
  VDL_CUDA(ctx, cudaMemsetAsync(table, 0, (size_t)slots * 4, ctx->stream));
  collate_flag_kernel<<<grid, 256, 0, ctx->stream>>>(od, n, origin, hl, a, slot0, table);
  ctx->launches++;
  VDL_TRY(vdl_op_fold_select(ctx, tv, &sv));
  tmp.v.push_back(sv);
  const i64 m = ctx->vecs[sv].len;
  const i64 *sel = (const i64 *)ctx->vecs[sv].ptr;
  const int mgrid = (int)std::max<i64>(1, std::min<i64>((m + 255) / 256, (i64)ctx->sm_count * 16));
  vdl_vec lv;
  VDL_TRY(vec_new(ctx, VDL_I64, m, &lv));
  tmp.v.push_back(lv);
  const i64 *len = (const i64 *)ctx->vecs[lv].ptr;
  collate_len_kernel<<<mgrid, 256, 0, ctx->stream>>>(hp, hl, sel, m, a, slot0, (i64 *)len, mm + 3, ctx->d_errflag);
  ctx->launches++;
  i64 maxlen = 0;
  VDL_TRY(read_scalar(ctx, mm + 3, &maxlen, 8));
  if (maxlen == 0) {                                // every string empty: one rank
    VDL_CUDA(ctx, cudaMemsetAsync(res, 0, (size_t)n * 8, ctx->stream));
    return VDL_OK;
  }
  // sort the m strings, the last chunk of 8 words first
  const int nwords = (int)((maxlen + 7) / 8), nchunks = (nwords + COLLATE_CHUNK - 1) / COLLATE_CHUNK;
  CollateWords cw;
  vdl_vec wv[COLLATE_CHUNK];
  const int wk = std::min(nwords, COLLATE_CHUNK);
  for (int w = 0; w < wk; w++) {
    VDL_TRY(vec_new(ctx, VDL_I64, m, &wv[w]));
    tmp.v.push_back(wv[w]);
    cw.w[w] = (i64 *)ctx->vecs[wv[w]].ptr;
  }
  vdl_vec perm = 0;
  for (int c = nchunks - 1; c >= 0; c--) {
    const int w0 = c * COLLATE_CHUNK, nw = std::min(COLLATE_CHUNK, nwords - w0);
    const Operand op = perm ? operand_of(ctx->vecs[perm]) : Operand{nullptr, 0, 0, 0};
    collate_words_kernel<<<mgrid, 256, 0, ctx->stream>>>(hp, sel, len, op, perm != 0, m, a, slot0, w0, nw, cw);
    ctx->launches++;
    VDL_CUDA(ctx, cudaGetLastError());
    vdl_vec p;
    VDL_TRY(vdl_op_order(ctx, nw, wv, nullptr, -1, &p));
    tmp.v.push_back(p);
    if (perm) {                                     // positions of this pass index the order reached so far
      vdl_vec q;
      VDL_TRY(vdl_op_gather(ctx, perm, p, &q));
      tmp.v.push_back(q);
      for (vdl_vec done : {perm, p}) {              // only the composed order lives on: O(m) however many chunks
        tmp.v.erase(std::find(tmp.v.begin(), tmp.v.end(), done));
        vdl_vec_free(ctx, done);
      }
      p = q;
    }
    perm = p;
  }
  // dense ranks: neighbours compared over their full bytes, the "differs" flags scanned
  vdl_vec dv;
  VDL_TRY(vec_new(ctx, VDL_I64, (i64)scan_elems(m), &dv));
  tmp.v.push_back(dv);
  i64 *diff = (i64 *)ctx->vecs[dv].ptr;
  const Operand op = operand_of(ctx->vecs[perm]);
  collate_diff_kernel<<<mgrid, 256, 0, ctx->stream>>>(hp, sel, len, op, m, a, slot0, diff);
  ctx->launches++;
  device_exclusive_scan(ctx, diff, m);
  collate_scatter_kernel<<<mgrid, 256, 0, ctx->stream>>>(diff, sel, op, m, table);
  collate_gather_kernel<<<grid, 256, 0, ctx->stream>>>(od, n, origin, hl, a, slot0, table, res);
  ctx->launches += 2;
  VDL_CUDA(ctx, cudaGetLastError());
  return VDL_OK;
}

// ---------------------------------------------------------------------------------- Fold by runs
#include "vdl_fold_kernel.cuh"

extern "C" int vdl_op_fold(vdl_ctx *ctx, int fold_op, vdl_vec groups, vdl_vec data, vdl_vec *out) {
  if (!ctx || !out) return VDL_EINVAL;
  if (fold_op < VDL_FOLD_SUM || fold_op > VDL_FOLD_COUNT) return vdl_fail(ctx, VDL_EINVAL, "fold op %d unknown", fold_op);
  Vec *vg = vec_get(ctx, groups), *vd = vec_get(ctx, data);
  if (!vg || !vd) return VDL_EINVAL;
  if (vg->len != vd->len) {
    // Level 2 of a hierarchical fold (make2LevelFold, Vlite.hs:1181-1192): `data` holds one result per level-1 run and
    // `groups` is still row-aligned.  Dense model: result k belongs to the group value at the first row of level-1 run k,
    // i.e. FoldChoose(level-1 groups, groups).  Anything else of unequal lengths is an error.
    const vdl_vec g1 = vd->fold_groups;
    Vec *v1 = g1 > 0 && (size_t)g1 < ctx->vecs.size() && ctx->vecs[g1].live ? &ctx->vecs[g1] : nullptr;
    if (!v1 || v1->gen != vd->fold_groups_gen || v1->len != vg->len)
      return vdl_fail(ctx, VDL_EINVAL, "Fold: groups length %lld != data length %lld", (long long)vg->len, (long long)vd->len);
    vdl_vec heads = 0;
    VDL_TRY(vdl_op_fold(ctx, VDL_FOLD_CHOOSE, g1, groups, &heads));
    int rc = vdl_op_fold(ctx, fold_op, heads, data, out);
    vdl_vec_free(ctx, heads);
    return rc;
  }
  VDL_CUDA(ctx, cudaSetDevice(ctx->device));
  const u64 groups_gen = vg->gen;
  const bool narrow = (fold_op == VDL_FOLD_CHOOSE || fold_op == VDL_FOLD_MIN || fold_op == VDL_FOLD_MAX) && vec_is_narrow(*vd);
  i64 n = vd->len;
  Operand og = operand_of(*vg), od = operand_of(*vd);
  if (n == 0) {
    VDL_TRY(vec_new(ctx, VDL_I64, 0, out));
    ctx->vecs[*out].fold_groups = groups;
    ctx->vecs[*out].fold_groups_gen = groups_gen;
    return VDL_OK;
  }
  if (vg->is_range && vg->step == 0) {           // constant groups: one run
    VDL_TRY(vec_new(ctx, VDL_I64, 1, out));
    i64 *o = (i64 *)ctx->vecs[*out].ptr;
    ctx->vecs[*out].fold_groups = groups;
    ctx->vecs[*out].fold_groups_gen = groups_gen;
    ctx->vecs[*out].narrow32 = narrow;
    fold_all_init_kernel<<<1, 1, 0, ctx->stream>>>(fold_op, od, n, o);
    ctx->launches++;
    const int grid = (int)std::max<i64>(1, std::min<i64>((n + 2047) / 2048, (i64)ctx->sm_count * 8));
    if (fold_op == VDL_FOLD_SUM) fold_all_kernel<VDL_FOLD_SUM><<<grid, 256, 0, ctx->stream>>>(od, n, o);
    else if (fold_op == VDL_FOLD_MIN) fold_all_kernel<VDL_FOLD_MIN><<<grid, 256, 0, ctx->stream>>>(od, n, o);
    else if (fold_op == VDL_FOLD_MAX) fold_all_kernel<VDL_FOLD_MAX><<<grid, 256, 0, ctx->stream>>>(od, n, o);
    if (fold_op == VDL_FOLD_SUM || fold_op == VDL_FOLD_MIN || fold_op == VDL_FOLD_MAX) ctx->launches++;
    VDL_CUDA(ctx, cudaGetLastError());
    return VDL_OK;
  }
  const i64 ntiles = (n + FL_TILE - 1) / FL_TILE;
  VDL_TRY(scratch_reserve(ctx, (size_t)ntiles * sizeof(FoldTileState) + 64));
  FoldTileState *state = (FoldTileState *)ctx->scratch;
  i64 *d_total = (i64 *)(state + ntiles);
  unsigned int *ticket = (unsigned int *)(d_total + 1);
  VDL_CUDA(ctx, cudaMemsetAsync(state, 0, (size_t)ntiles * sizeof(FoldTileState) + 16, ctx->stream));
  VDL_TRY(vec_new(ctx, VDL_I64, n, out));                                   // capacity n; the run count is known after the pass
  i64 *o = (i64 *)ctx->vecs[*out].ptr;
  const int grid = (int)std::min<i64>(ntiles, (i64)ctx->sm_count * (1024 / FL_THREADS));
  switch (fold_op) {
    case VDL_FOLD_SUM: fold_lookback_kernel<VDL_FOLD_SUM><<<grid, FL_THREADS, 0, ctx->stream>>>(og, od, n, ntiles, state, ticket, o, d_total); break;
    case VDL_FOLD_MIN: fold_lookback_kernel<VDL_FOLD_MIN><<<grid, FL_THREADS, 0, ctx->stream>>>(og, od, n, ntiles, state, ticket, o, d_total); break;
    case VDL_FOLD_MAX: fold_lookback_kernel<VDL_FOLD_MAX><<<grid, FL_THREADS, 0, ctx->stream>>>(og, od, n, ntiles, state, ticket, o, d_total); break;
    case VDL_FOLD_CHOOSE: fold_lookback_kernel<VDL_FOLD_CHOOSE><<<grid, FL_THREADS, 0, ctx->stream>>>(og, od, n, ntiles, state, ticket, o, d_total); break;
    default: fold_lookback_kernel<VDL_FOLD_COUNT><<<grid, FL_THREADS, 0, ctx->stream>>>(og, od, n, ntiles, state, ticket, o, d_total); break;
  }
  ctx->launches++;
  VDL_CUDA(ctx, cudaGetLastError());
  i64 total = 0;
  VDL_TRY(read_scalar(ctx, d_total, &total, 8));
  Vec &v = ctx->vecs[*out];
  v.len = total;
  v.fold_groups = groups;
  v.fold_groups_gen = groups_gen;
  v.narrow32 = narrow;
  return VDL_OK;
}
