// Plan front end of libvdl_cuda: parses the Voodoo program text mplan2vdl prints (VdlFormat,
// reference Vdl.hs:410-453 toVoodooList / 455-477 printLine), hash-conses it (the emitter's own
// CSE is keyed on (node, metadata) and can print duplicates: SURVEY.md App. F caveat, G10), runs the
// select->map->fold fusion peephole, and executes what is left op-at-a-time.
//
// The fusion pass is the executor-side twin of the Vlite peepholes (Vlite.hs:1295-1340,
// `Vx -> Maybe Vexp`, applied bottom-up with memoisation 1351-1417): every node is given a small
// symbolic normal form (constant / product of affine column terms / conjunction of column ranges /
// bit-packed key / selection / partition / sorted-by-partition) and a Fold whose operands normalise
// is replaced by one `vdl_fused_scan_fold` launch.  Anything that does not normalise is simply not
// fused and runs through the per-op kernels with identical results.
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <functional>
#include <map>
#include <set>
#include <string>
#include <vector>

#include "vdl_internal.h"

#include <chrono>
static double now_ms() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); }

namespace {

enum NodeOp { N_LOAD, N_RANGEV, N_RANGEC, N_BINARY, N_FSELECT, N_GATHER, N_SCATTER, N_PARTITION, N_FOLD, N_LIKE, N_CROSS };

struct Node {
  int op = 0, sub = 0;         // sub: binary op / fold op
  int a = -1, b = -1, c = -1;  // argument node indices
  i64 k0 = 0, k1 = 0, k2 = 0;  // RangeV: from, step; RangeC: from, count, step
  std::string name;            // Load: "table.column"; Like: the pattern
};

// data points at the result's host copy: the fused scan's / probe's mapped result buffer, or this output's own pinned buffer
// dtype 4: the values travelled as int32 (typed outputs: vdl_plan_set_typed_outputs); data then points at int32 values
struct Output { std::string name; int node; const i64 *data = nullptr; i64 len = 0; i64 *pinned = nullptr; size_t cap = 0; int dtype = 8; };
inline i64 out_get(const Output &o, i64 i) { return o.dtype == 4 ? (i64)((const int *)o.data)[i] : o.data[i]; }

// ---- symbolic normal forms ------------------------------------------------------------------
struct Aff { int col = -1; int shr = 0; i64 a = 0, b = 0; };   // a + b*(col >> shr); col = Load node, -1: constant a
struct RangeTerm { int col, shr; i64 lo, hi; };
enum SymKind { S_NONE, S_VALUE, S_PRED, S_KEY, S_POS, S_SELECTION, S_PARTITION, S_SORTED };
struct Sym {
  int kind = S_NONE;
  int table = -1;              // table id of the row space (-1: a constant, fits any space)
  int sel = -1;                // node index of the predicate whose selection this lives in (-1: base rows)
  int ref = -1;                // S_VALUE const / S_POS: node whose length it copies
  std::vector<Aff> fac;        // S_VALUE: product of factors; S_KEY: OR of parts
  std::vector<RangeTerm> ranges;  // S_PRED
  bool never = false;          // S_PRED that no row satisfies
  i64 mask = -1;               // S_KEY
  bool masked = false;
  int n0 = -1, n1 = -1;        // S_SELECTION: pred node; S_PARTITION: key node; S_SORTED: partition node, inner node
  i64 lo = 0, cnt = 0;         // S_PARTITION pivots RangeC(lo, cnt, 1)
};

// Elementwise / Gather / Range nodes of the op-at-a-time remainder that run as ONE vdl_op_map launch (build_clusters).
struct MapCluster {
  int root = -1;
  std::vector<int> members;             // ascending node index = evaluation order; the root is last
  std::vector<int> inputs, tables;      // leaf nodes: row-aligned inputs / Gather sources
  vdl_map_desc desc;
};

struct FusedFold { int node; vdl_fold_spec spec; };
// peer-memory combine of a fused scan or a probe fold group (vdl_plan_set_peers): re-applied whenever its scan or probe is
// re-prepared, with the step counter carried over
struct PeerState {
  int rank = -1, world = 0;
  std::vector<void *> buffers;
  u64 epoch = 0;
};
struct FusedGroup {
  int table, sel, keynode;
  std::vector<int> cols;                // Load node of each column slot
  std::vector<FusedFold> folds;         // deduplicated specs
  std::map<int, int> fold_of_node;      // Fold node -> index into folds
  std::vector<vdl_post_op> posts;       // elementwise epilogue over the fold results, run by the finalize kernel
  std::map<int, int> post_of_node;      // Binary node -> index into posts
  vdl_fused_desc desc;
  vdl_fused *fused = nullptr;
  std::vector<vdl_vec> bound;           // column handles the prepared scan was built for
  i64 bound_rows = -1, bound_base = -1;
  PeerState peer;
};

}  // namespace

namespace {
struct JoinAnalysis;
struct ProbeFoldGroup;
struct EmitGroup;
}  // namespace

struct vdl_plan {
  vdl_ctx *ctx = nullptr;
  int flags = 0;
  int statements = 0;
  std::vector<Node> nodes;
  std::vector<Output> outputs;
  std::vector<std::string> tables;
  std::vector<Sym> sym;
  std::vector<char> sym_done;
  std::vector<FusedGroup> groups;
  std::vector<int> group_of_node;       // Fold node (or Binary node computed as a post op) -> group index or -1
  // FK-join plans (vdl_plan_join.inc): join-aware normal forms, Folds run by the probe kernel, vectors it emits
  JoinAnalysis *join = nullptr;
  std::vector<ProbeFoldGroup *> pgroups;
  std::vector<int> pgroup_of_node;      // Fold node -> probe fold group or -1
  std::vector<EmitGroup *> egroups;
  std::vector<int> egroup_of_node, eslot_of_node;   // node materialised by a probe in emit mode -> group, slot
  std::vector<MapCluster> clusters;
  std::vector<int> cluster_of_root;     // node -> index into clusters when it is the root of one, else -1
  i64 row_base = 0;
  // Sharded tail (vdl_plan_tail_*): every output is a Fold by runs of ONE groups vector, so a row-range shard's result is a
  // slice of the global one up to the groups that straddle shard boundaries
  bool typed_outputs = false;                    // result columns whose values provably fit travel as int32
  bool tail_ok = false, tail_on = false;
  int tail_groups = -1, tail_partition = -1;     // groups node; its Partition (-1: constant groups)
  i64 tail_rec[4] = {0, 0, 0, 0};                // of the last run: sorted, runs, first key, last key
  // ORDER BY / LIMIT (vdl_plan_set_order): output indices of the keys, their DESC flags; limit < 0: none
  std::vector<int> order_key, order_desc;
  i64 order_limit = -1;
  // per key: the string heap its output's values point into (vdl_plan_set_order_heap; 0: compared as integers), origin
  std::vector<vdl_vec> order_heap;
  std::vector<i64> order_origin;
  // run state
  std::vector<vdl_vec> val;
  std::vector<vdl_vec> temps;
  i64 launches_last = 0;
  bool local_done = false, self_finalized = false;
  bool trace = false;
  double trace_t0 = 0, trace_last = 0;
};

namespace {

// ---------------------------------------------------------------------------------- parsing
bool parse_ref(const std::string &s, int *out) {
  if (s.compare(0, 3, "Id ") != 0) return false;
  char *end;
  long v = strtol(s.c_str() + 3, &end, 10);
  if (*end || v <= 0) return false;
  *out = (int)v;
  return true;
}
bool parse_i64(const std::string &s, i64 *out) {
  if (s.empty()) return false;
  char *end;
  long long v = strtoll(s.c_str(), &end, 10);
  if (*end) return false;
  *out = (i64)v;
  return true;
}

const char *BINOPS[] = {"LogicalAnd", "LogicalOr", "BitwiseAnd", "BitwiseOr", "BitShift", "Equals",
                        "Add", "Subtract", "Greater", "Multiply", "Divide", "Modulo"};
const char *FOLDS[] = {"FoldSum", "FoldMin", "FoldMax", "FoldChoose", "FoldCount"};

// ---- two-level folds (--agghierarchical: make2LevelFold, Vlite.hs:1181-1192) -------------------------------------
// Fold(op, G, Fold(op, G1, D)) equals Fold(op, G, D) for Sum / Min / Max / Choose whenever equal G1 values imply equal G
// values (the level-1 runs then refine G's runs).  That is proven structurally, on the shapes composeKeys prints
// (Vlite.hs:1162-1170): G1 = ((G [- c]) << k) | x with 0 <= x < 2^k, or anything at all over constant groups.  Unproven
// pairs stay two Folds and vdl_op_fold evaluates level 2 literally (see there).
bool const_value(const std::vector<Node> &nd, int ni, i64 *k) {
  const Node &n = nd[ni];
  if (n.op == N_RANGEV && n.k1 == 0) { *k = n.k0; return true; }
  if (n.op == N_BINARY && (n.sub == VDL_ADD || n.sub == VDL_SUBTRACT)) {
    i64 x, y;
    if (!const_value(nd, n.a, &x) || !const_value(nd, n.b, &y)) return false;
    *k = n.sub == VDL_ADD ? (i64)((u64)x + (u64)y) : (i64)((u64)x - (u64)y);
    return true;
  }
  return false;
}
// the node a vector copies its length from, followed through the elementwise ops
int length_class(const std::vector<Node> &nd, int ni) {
  const Node &n = nd[ni];
  if (n.op == N_RANGEV || n.op == N_BINARY) return length_class(nd, n.a);
  if (n.op == N_GATHER) return length_class(nd, n.b);
  return ni;
}
bool below_pow2(const std::vector<Node> &nd, int ni, i64 bits) {      // 0 <= value < 2^bits, structurally
  const Node &n = nd[ni];
  i64 k;
  if (const_value(nd, ni, &k)) return k >= 0 && (bits >= 63 || k < ((i64)1 << bits));
  if (n.op == N_BINARY && n.sub == VDL_BITWISE_AND) {
    for (int side : {n.a, n.b})
      if (const_value(nd, side, &k) && k >= 0 && (bits >= 63 || k < ((i64)1 << bits))) return true;
  }
  return false;
}
bool determines(const std::vector<Node> &nd, int x, int g, int depth = 0) {   // the value of x determines the value of g
  if (x == g) return true;
  if (depth > 16) return false;
  const Node &n = nd[x];
  if (n.op != N_BINARY) return false;
  i64 k;
  switch (n.sub) {
    case VDL_ADD: case VDL_SUBTRACT:
      return const_value(nd, n.b, &k) && determines(nd, n.a, g, depth + 1);
    case VDL_BITSHIFT:                       // left shifts keep every bit while the key fits (composeKeys asserts < 65 bits)
      return const_value(nd, n.b, &k) && k <= 0 && k > -63 && determines(nd, n.a, g, depth + 1);
    case VDL_BITWISE_OR: {
      for (int t = 0; t < 2; t++) {
        const int hi = t ? n.b : n.a, lo = t ? n.a : n.b;
        const Node &h = nd[hi];
        if (h.op == N_BINARY && h.sub == VDL_BITSHIFT && const_value(nd, h.b, &k) && k <= 0 && k > -63 && below_pow2(nd, lo, -k) &&
            determines(nd, h.a, g, depth + 1))
          return true;
      }
      return false;
    }
    default: return false;
  }
}
void collapse_two_level_fold(const std::vector<Node> &nd, Node *f) {
  if (f->op != N_FOLD || f->sub == VDL_FOLD_COUNT || f->b < 0) return;
  const Node &inner = nd[f->b];
  if (inner.op != N_FOLD || inner.sub != f->sub) return;
  if (length_class(nd, inner.a) != length_class(nd, f->a)) return;
  i64 k;
  if (const_value(nd, f->a, &k) || determines(nd, inner.a, f->a)) f->b = inner.b;
}

int parse_plan(vdl_plan *p, const char *text) {
  vdl_ctx *ctx = p->ctx;
  std::vector<int> canon;          // statement id -> node index (aliases resolved)
  std::vector<std::string> outname;  // statement id -> Project out name ("" if none)
  canon.push_back(-1);
  outname.push_back("");
  std::map<std::string, int> cse;
  const char *q = text;
  int lineno = 0;
  while (*q) {
    const char *eol = strchr(q, '\n');
    std::string line = eol ? std::string(q, eol - q) : std::string(q);
    q = eol ? eol + 1 : q + line.size();
    lineno++;
    size_t m = line.find(" ;; ");               // --metadata suffix (Vdl.hs:463-466)
    if (m != std::string::npos) line.resize(m);
    while (!line.empty() && (line.back() == '\r' || line.back() == ' ')) line.pop_back();
    if (line.empty()) continue;
    std::vector<std::string> f;
    size_t pos = 0;
    for (;;) {
      size_t c = line.find(',', pos);
      if (c == std::string::npos) { f.push_back(line.substr(pos)); break; }
      f.push_back(line.substr(pos, c - pos));
      pos = c + 1;
    }
    i64 id;
    if (f.size() < 2 || !parse_i64(f[0], &id) || id != (i64)canon.size())
      return vdl_fail(ctx, VDL_EINVAL, "plan line %d: statement ids must run 1,2,3,... (Vdl.hs:297-311)", lineno);
    const std::string &op = f[1];
    auto bad = [&]() { return vdl_fail(ctx, VDL_EINVAL, "plan line %d: malformed %s statement", lineno, op.c_str()); };
    auto arg = [&](const std::string &s, int *out) {
      int r;
      if (!parse_ref(s, &r) || r >= (int)canon.size()) return false;
      *out = canon[r];
      return *out >= 0;
    };
    Node n;
    std::string oname;
    int alias = -1;
    bool is_output = false;
    if (op == "Load") {
      if (f.size() != 3) return bad();
      n.op = N_LOAD; n.name = f[2];
    } else if (op == "Project") {           // Project,<out>,Id n,<in>: rename only
      int r;
      if (f.size() != 5 || !parse_ref(f[3], &r) || r >= (int)canon.size()) return bad();
      alias = canon[r];
      if (f[2] != "val") oname = f[2];
    } else if (op == "Shuffle") {
      int r;
      if (f.size() != 3 || !parse_ref(f[2], &r) || r >= (int)canon.size()) return bad();
      alias = canon[r];
    } else if (op == "MaterializeCompact") {
      int r;
      if (f.size() != 3 || !parse_ref(f[2], &r) || r >= (int)canon.size()) return bad();
      alias = canon[r];
      oname = outname[r].empty() ? "val" : outname[r];
      is_output = true;
    } else if (op == "RangeV") {
      if (f.size() != 6 || f[2] != "val" || !parse_i64(f[3], &n.k0) || !arg(f[4], &n.a) || !parse_i64(f[5], &n.k1)) return bad();
      n.op = N_RANGEV;
    } else if (op == "RangeC") {
      if (f.size() != 6 || f[2] != "val" || !parse_i64(f[3], &n.k0) || !parse_i64(f[4], &n.k1) || !parse_i64(f[5], &n.k2)) return bad();
      n.op = N_RANGEC;
    } else if (op == "Gather") {
      if (f.size() != 5 || f[4] != "val" || !arg(f[2], &n.a) || !arg(f[3], &n.b)) return bad();
      n.op = N_GATHER;
    } else if (op == "Scatter") {
      if (f.size() != 7 || f[4] != "val" || f[6] != "val" || !arg(f[2], &n.a) || !arg(f[3], &n.b) || !arg(f[5], &n.c)) return bad();
      n.op = N_SCATTER;
    } else if (op == "Like") {              // id,Like,val,Id data,val,Id heap,val,pattern (Vdl.hs:444-447); the pattern may contain commas
      if (f.size() < 8 || f[2] != "val" || f[4] != "val" || f[6] != "val" || !arg(f[3], &n.a) || !arg(f[5], &n.b)) return bad();
      n.op = N_LIKE;
      n.name = f[7];
      for (size_t k = 8; k < f.size(); k++) n.name += "," + f[k];
    } else if (op == "CrossProductOuter" || op == "CrossProductInner") {   // id,CrossProductOuter,Id left,Id right (Vdl.hs:412-416)
      if (f.size() != 4 || !arg(f[2], &n.a) || !arg(f[3], &n.b)) return bad();
      n.op = N_CROSS;
      n.sub = op == "CrossProductInner";
    } else if (op == "Semisort") {
      return vdl_fail(ctx, VDL_EUNSUPPORTED, "plan line %d: op %s is outside the supported vocabulary", lineno, op.c_str());
    } else {
      if (f.size() != 7 || f[2] != "val" || f[4] != "val" || f[6] != "val" || !arg(f[3], &n.a) || !arg(f[5], &n.b)) return bad();
      n.op = -1;
      for (int k = 0; k < 12; k++) if (op == BINOPS[k]) { n.op = N_BINARY; n.sub = k; }
      for (int k = 0; k < 5; k++) if (op == FOLDS[k]) { n.op = N_FOLD; n.sub = k; }
      if (op == "FoldSelect") n.op = N_FSELECT;
      if (op == "Partition") n.op = N_PARTITION;
      if (n.op < 0) return vdl_fail(ctx, VDL_EINVAL, "plan line %d: unknown op %s", lineno, op.c_str());
    }
    if (alias == -1 && (op == "Project" || op == "Shuffle" || op == "MaterializeCompact")) return bad();
    int idx;
    if (alias >= 0) {
      idx = alias;
    } else {
      if (p->flags & VDL_PLAN_FUSE) collapse_two_level_fold(p->nodes, &n);
      char key[512];
      snprintf(key, sizeof key, "%d|%d|%d|%d|%d|%lld|%lld|%lld|%s", n.op, n.sub, n.a, n.b, n.c, (long long)n.k0, (long long)n.k1,
               (long long)n.k2, n.name.c_str());
      auto it = cse.find(key);
      if (it != cse.end()) idx = it->second;
      else {
        idx = (int)p->nodes.size();
        p->nodes.push_back(n);
        cse[key] = idx;
      }
    }
    canon.push_back(idx);
    outname.push_back(oname);
    if (is_output) { Output o; o.name = oname; o.node = idx; p->outputs.push_back(o); }
  }
  p->statements = (int)canon.size() - 1;
  if (p->outputs.empty()) return vdl_fail(ctx, VDL_EINVAL, "plan has no MaterializeCompact output");
  return VDL_OK;
}

// ---------------------------------------------------------------------------------- symbolic analysis
int table_id(vdl_plan *p, const std::string &col) {
  std::string t = col.substr(0, col.find('.'));
  for (size_t i = 0; i < p->tables.size(); i++) if (p->tables[i] == t) return (int)i;
  p->tables.push_back(t);
  return (int)p->tables.size() - 1;
}

bool is_const(const Sym &s) { return s.kind == S_VALUE && s.fac.size() == 1 && s.fac[0].col < 0; }
bool is_single(const Sym &s) { return s.kind == S_VALUE && s.fac.size() == 1; }
bool is_leaf(const Sym &s) { return is_single(s) && s.fac[0].col >= 0 && s.fac[0].a == 0 && s.fac[0].b == 1; }

// space of a binary result: constants fit anywhere; otherwise (table, sel) must agree
bool join_space(const Sym &x, const Sym &y, Sym *r) {
  if (x.table < 0) { r->table = y.table; r->sel = y.sel; r->ref = y.table < 0 ? x.ref : -1; return true; }
  if (y.table < 0) { r->table = x.table; r->sel = x.sel; return true; }
  if (x.table != y.table || x.sel != y.sel) return false;
  r->table = x.table; r->sel = x.sel;
  return true;
}

Sym value_const(i64 k) { Sym s; s.kind = S_VALUE; Aff a; a.a = k; s.fac.push_back(a); return s; }

void add_range(Sym *s, int col, int shr, i64 lo, i64 hi) {
  for (auto &r : s->ranges)
    if (r.col == col && r.shr == shr) {
      r.lo = std::max(r.lo, lo);
      r.hi = std::min(r.hi, hi);
      if (r.lo > r.hi) s->never = true;
      return;
    }
  s->ranges.push_back(RangeTerm{col, shr, lo, hi});
  if (lo > hi) s->never = true;
}

i64 wadd(i64 a, i64 b) { return (i64)((u64)a + (u64)b); }
i64 wsub(i64 a, i64 b) { return (i64)((u64)a - (u64)b); }
i64 wmul(i64 a, i64 b) { return (i64)((u64)a * (u64)b); }

const Sym &analyse(vdl_plan *p, int ni);

Sym analyse_binary(vdl_plan *p, const Node &n) {
  const Sym x = analyse(p, n.a), y = analyse(p, n.b);
  Sym r;
  if (x.kind == S_NONE || y.kind == S_NONE) return r;
  if (!join_space(x, y, &r)) return Sym();
  auto none = [&]() { Sym z; z.table = r.table; z.sel = r.sel; return z; };
  switch (n.sub) {
    case VDL_ADD:
    case VDL_SUBTRACT: {
      if (!is_single(x) || !is_single(y)) return none();
      const Aff &fx = x.fac[0], &fy = y.fac[0];
      bool sub = n.sub == VDL_SUBTRACT;
      Aff o;
      if (fx.col >= 0 && fy.col >= 0) {
        if (fx.col != fy.col || fx.shr != fy.shr) return none();
        o = fx;
        o.a = sub ? wsub(fx.a, fy.a) : wadd(fx.a, fy.a);
        o.b = sub ? wsub(fx.b, fy.b) : wadd(fx.b, fy.b);
      } else if (fx.col >= 0) {
        o = fx;
        o.a = sub ? wsub(fx.a, fy.a) : wadd(fx.a, fy.a);
      } else if (fy.col >= 0) {
        o = fy;
        o.a = sub ? wsub(fx.a, fy.a) : wadd(fx.a, fy.a);
        o.b = sub ? wsub(0, fy.b) : fy.b;
      } else {
        o.a = sub ? wsub(fx.a, fy.a) : wadd(fx.a, fy.a);
      }
      r.kind = S_VALUE;
      r.fac.push_back(o);
      return r;
    }
    case VDL_MULTIPLY: {
      if (x.kind != S_VALUE || y.kind != S_VALUE) return none();
      // constants fold into the first factor of the other operand (exact in Z/2^64)
      const Sym *cs = is_const(x) ? &x : (is_const(y) ? &y : nullptr);
      r.kind = S_VALUE;
      if (cs) {
        const Sym &o = cs == &x ? y : x;
        r.fac = o.fac;
        i64 k = cs->fac[0].a;
        r.fac[0].a = wmul(r.fac[0].a, k);
        r.fac[0].b = wmul(r.fac[0].b, k);
        return r;
      }
      if (x.fac.size() + y.fac.size() > VDL_MAX_FACTORS) return none();
      r.fac = x.fac;
      r.fac.insert(r.fac.end(), y.fac.begin(), y.fac.end());
      return r;
    }
    case VDL_BITSHIFT: {
      if (!is_const(y) || !is_single(x)) return none();
      i64 k = y.fac[0].a;
      Aff o = x.fac[0];
      if (o.col < 0) {                      // constant folding, same rule as the kernels
        if (k >= 0) o.a = k >= 64 ? (o.a < 0 ? -1 : 0) : (o.a >> k);
        else o.a = k <= -64 ? 0 : (i64)((u64)o.a << (-k));
      } else if (k >= 0) {                  // (col >> s) >> k == col >> (s + k) for arithmetic shifts
        if (o.a != 0 || o.b != 1 || o.shr + k > 63) return none();
        o.shr += (int)k;
      } else {                              // left shift = multiply by 2^-k, exact in Z/2^64
        if (k <= -64) return none();
        o.a = (i64)((u64)o.a << (-k));
        o.b = (i64)((u64)o.b << (-k));
      }
      r.kind = S_VALUE;
      r.fac.push_back(o);
      return r;
    }
    case VDL_BITWISE_OR: {
      auto parts = [](const Sym &s, std::vector<Aff> *out) {
        if (s.kind == S_KEY && !s.masked) { out->insert(out->end(), s.fac.begin(), s.fac.end()); return true; }
        if (is_single(s)) { out->push_back(s.fac[0]); return true; }
        return false;
      };
      r.kind = S_KEY;
      if (!parts(x, &r.fac) || !parts(y, &r.fac) || r.fac.size() > VDL_MAX_KEYS) return none();
      return r;
    }
    case VDL_BITWISE_AND: {
      const Sym *cs = is_const(y) ? &y : (is_const(x) ? &x : nullptr);
      if (!cs) return none();
      const Sym &o = cs == &y ? x : y;
      i64 mk = cs->fac[0].a;
      if (mk < 0) return none();
      r.kind = S_KEY;
      if (o.kind == S_KEY) { r.fac = o.fac; r.mask = o.masked ? (o.mask & mk) : mk; }
      else if (is_single(o)) { r.fac.push_back(o.fac[0]); r.mask = mk; }
      else return none();
      r.masked = true;
      return r;
    }
    case VDL_GREATER: {                     // column > k  or  k > column
      r.kind = S_PRED;
      if (is_leaf(x) && is_const(y)) {
        i64 k = y.fac[0].a;
        if (k == INT64_MAX) r.never = true; else add_range(&r, x.fac[0].col, x.fac[0].shr, k + 1, INT64_MAX);
        return r;
      }
      if (is_const(x) && is_leaf(y)) {
        i64 k = x.fac[0].a;
        if (k == INT64_MIN) r.never = true; else add_range(&r, y.fac[0].col, y.fac[0].shr, INT64_MIN, k - 1);
        return r;
      }
      return none();
    }
    case VDL_EQUALS: {
      const Sym *cs = is_const(y) ? &y : (is_const(x) ? &x : nullptr);
      const Sym &o = cs == &y ? x : y;
      if (!cs || !is_leaf(o)) return none();
      r.kind = S_PRED;
      add_range(&r, o.fac[0].col, o.fac[0].shr, cs->fac[0].a, cs->fac[0].a);
      return r;
    }
    case VDL_LOGICAL_AND: {
      if (x.kind != S_PRED || y.kind != S_PRED) return none();
      r.kind = S_PRED;
      r.ranges = x.ranges;
      r.never = x.never || y.never;
      for (auto &t : y.ranges) add_range(&r, t.col, t.shr, t.lo, t.hi);
      if (r.ranges.size() > VDL_MAX_PREDS) return none();
      return r;
    }
    case VDL_LOGICAL_OR: {                  // union of two ranges of one column, when it is again a range
      if (x.kind != S_PRED || y.kind != S_PRED) return none();
      if (x.never) { Sym z = y; z.table = r.table; z.sel = r.sel; return z; }
      if (y.never) { Sym z = x; z.table = r.table; z.sel = r.sel; return z; }
      if (x.ranges.size() != 1 || y.ranges.size() != 1) return none();
      const RangeTerm &s = x.ranges[0], &t = y.ranges[0];
      if (s.col != t.col || s.shr != t.shr) return none();
      bool touch = (s.hi == INT64_MAX || t.lo <= s.hi + 1) && (t.hi == INT64_MAX || s.lo <= t.hi + 1);
      if (!touch) return none();
      r.kind = S_PRED;
      r.ranges.push_back(RangeTerm{s.col, s.shr, std::min(s.lo, t.lo), std::max(s.hi, t.hi)});
      return r;
    }
  }
  return none();
}

const Sym &analyse(vdl_plan *p, int ni) {
  if (p->sym_done[ni]) return p->sym[ni];
  p->sym_done[ni] = 1;
  const Node &n = p->nodes[ni];
  Sym r;
  switch (n.op) {
    case N_LOAD: {
      r.kind = S_VALUE;
      r.table = table_id(p, n.name);
      Aff a; a.col = ni; a.b = 1;
      r.fac.push_back(a);
      break;
    }
    case N_RANGEV: {
      const Sym s = analyse(p, n.a);
      if (n.k1 == 0) { r = value_const(n.k0); }
      else if (n.k0 == 0 && n.k1 == 1) r.kind = S_POS;
      // constants/positions live in the row space of the vector whose length they copy
      if (s.kind == S_SELECTION) { r.table = s.table; r.sel = s.n0; }
      else { r.table = s.table; r.sel = s.sel; }
      r.ref = n.a;
      if (s.kind == S_NONE || s.kind == S_PARTITION) r.table = -2;   // unknown space: never joins
      break;
    }
    case N_BINARY: r = analyse_binary(p, n); break;
    case N_FSELECT: {
      const Sym f = analyse(p, n.a), q = analyse(p, n.b);
      if (f.kind == S_POS && q.kind == S_PRED && q.table >= 0 && q.sel < 0 && f.table == q.table && f.sel < 0) {
        r.kind = S_SELECTION; r.table = q.table; r.n0 = n.b;
      }
      break;
    }
    case N_GATHER: {
      const Sym x = analyse(p, n.a), s = analyse(p, n.b);
      if (s.kind == S_SELECTION && (x.kind == S_VALUE || x.kind == S_KEY || x.kind == S_PRED) && x.table == s.table && x.sel < 0) {
        r = x; r.sel = s.n0;
      }
      break;
    }
    case N_PARTITION: {
      const Sym k = analyse(p, n.a);
      const Node &pv = p->nodes[n.b];
      if (pv.op == N_RANGEC && pv.k2 == 1 && (k.kind == S_KEY || is_single(k)) && k.table >= 0) {
        r.kind = S_PARTITION; r.table = k.table; r.sel = k.sel; r.n0 = n.a; r.lo = pv.k0; r.cnt = pv.k1;
      }
      break;
    }
    case N_SCATTER: {
      const Sym x = analyse(p, n.a), pt = analyse(p, n.c);
      if (pt.kind == S_PARTITION && (x.kind == S_VALUE || x.kind == S_KEY)) {
        bool same = x.table == pt.table && x.sel == pt.sel;
        if (x.table == -1 && x.ref >= 0) {   // a constant: accept when it copies the length of a vector in the key's space
          const Sym rs = analyse(p, x.ref);
          same = rs.table == pt.table && rs.sel == pt.sel;
        }
        if (same) { r.kind = S_SORTED; r.table = pt.table; r.sel = pt.sel; r.n0 = n.c; r.n1 = n.a; }
      }
      break;
    }
    default: break;   // RangeC, Fold: opaque
  }
  p->sym[ni] = r;
  return p->sym[ni];
}

// ---------------------------------------------------------------------------------- fusion
int column_slot(FusedGroup *g, int loadnode) {
  for (size_t i = 0; i < g->cols.size(); i++) if (g->cols[i] == loadnode) return (int)i;
  g->cols.push_back(loadnode);
  return (int)g->cols.size() - 1;
}

bool to_affine(FusedGroup *g, const Aff &a, vdl_affine *out) {
  out->a = a.a; out->b = a.b; out->shr = a.shr; out->column = -1;
  if (a.col >= 0) { out->column = column_slot(g, a.col); if (g->cols.size() > VDL_MAX_COLS) return false; }
  return true;
}

// Try to express Fold node `ni` as a member of a fused scan.  Returns false when it does not normalise.
bool try_fuse_fold(vdl_plan *p, int ni) {
  const Node &n = p->nodes[ni];
  const Sym G = analyse(p, n.a), D = analyse(p, n.b);
  int table, sel, keynode = -1;
  const Sym *value = nullptr;
  Sym inner;
  if (G.kind == S_VALUE && is_const(G) && (D.kind == S_VALUE) && D.table >= 0) {
    // Fold over constant groups: one run (Vlite.hs:636-638 zeros_ refv for an empty group-by)
    if (G.table != D.table || G.sel != D.sel) return false;
    table = D.table; sel = D.sel; value = &D;
  } else if (G.kind == S_SORTED && D.kind == S_SORTED && G.n0 == D.n0) {
    // groups = keys sorted by Partition(keys), data = x sorted by the same partition (Vlite.hs:1057-1060)
    const Sym P = analyse(p, G.n0);
    if (P.kind != S_PARTITION || G.n1 != P.n0) return false;
    inner = analyse(p, D.n1);
    if (inner.kind != S_VALUE) return false;
    table = P.table; sel = P.sel; keynode = P.n0; value = &inner;
    const Sym K = analyse(p, keynode);
    // bucket(key) = clamp(key - lo, 0, cnt); it is the key itself only when 0 <= key < cnt is proven
    if (!(K.kind == S_KEY && K.masked && K.mask >= 0 && P.lo == 0 && P.cnt >= K.mask + 1)) return false;
    if (K.mask + 1 > (1 << 14)) return false;
  } else {
    return false;
  }
  if (sel >= 0) {
    const Sym Q = analyse(p, sel);
    if (Q.kind != S_PRED || Q.table != table || Q.sel >= 0) return false;
  }
  if (value->fac.size() > VDL_MAX_FACTORS) return false;

  int gi = -1;
  for (size_t i = 0; i < p->groups.size(); i++)
    if (p->groups[i].table == table && p->groups[i].sel == sel && p->groups[i].keynode == keynode) gi = (int)i;
  if (gi < 0) {
    FusedGroup g;
    g.table = table; g.sel = sel; g.keynode = keynode;
    memset(&g.desc, 0, sizeof g.desc);
    p->groups.push_back(g);
    gi = (int)p->groups.size() - 1;
  }
  FusedGroup saved = p->groups[gi];
  FusedGroup &g = p->groups[gi];
  vdl_fold_spec spec;
  memset(&spec, 0, sizeof spec);
  spec.op = n.sub;
  if (n.sub != VDL_FOLD_COUNT) {
    bool all_const_one = value->fac.size() == 1 && value->fac[0].col < 0 && value->fac[0].a == 1;
    if (n.sub == VDL_FOLD_SUM && all_const_one) spec.op = VDL_FOLD_COUNT;     // COUNT(*) = FoldSum of ones (Vlite.hs:1043-1046)
    else {
      spec.nfactors = (int)value->fac.size();
      for (size_t t = 0; t < value->fac.size(); t++)
        if (!to_affine(&g, value->fac[t], &spec.factor[t])) { g = saved; return false; }
    }
  }
  int fi = -1;
  for (size_t i = 0; i < g.folds.size(); i++)
    if (!memcmp(&g.folds[i].spec, &spec, sizeof spec)) fi = (int)i;
  if (fi < 0) {
    if (g.folds.size() == VDL_MAX_AGGS) { g = saved; return false; }
    g.folds.push_back(FusedFold{ni, spec});
    fi = (int)g.folds.size() - 1;
  }
  g.fold_of_node[ni] = fi;
  p->group_of_node[ni] = gi;
  return true;
}

// Fill the ABI descriptor of a group (predicates, key, folds); column handles are bound at run time.
bool build_desc(vdl_plan *p, FusedGroup *g) {
  vdl_fused_desc &d = g->desc;
  memset(&d, 0, sizeof d);
  d.key_mask = -1;
  d.domain = 1;
  if (g->sel >= 0) {
    const Sym Q = analyse(p, g->sel);
    if (Q.never) { d.npreds = 1; d.pred[0].column = 0; d.pred[0].lo = 1; d.pred[0].hi = 0; if (g->cols.empty()) return false; }
    else {
      for (auto &t : Q.ranges) {
        if (t.lo == INT64_MIN && t.hi == INT64_MAX) continue;
        vdl_range_pred &o = d.pred[d.npreds++];
        o.column = column_slot(g, t.col); o.shr = t.shr; o.lo = t.lo; o.hi = t.hi;
      }
    }
  }
  if (g->keynode >= 0) {
    const Sym K = analyse(p, g->keynode);
    for (auto &a : K.fac) {
      vdl_key_part &kp = d.key[d.nkeys++];
      if (!to_affine(g, a, &kp.e)) return false;
    }
    d.key_mask = K.mask;
    d.domain = K.mask + 1;
  }
  d.nfolds = (int)g->folds.size();
  for (int i = 0; i < d.nfolds; i++) d.fold[i] = g->folds[i].spec;
  d.nposts = (int)g->posts.size();
  for (int i = 0; i < d.nposts; i++) d.post[i] = g->posts[i];
  if (g->cols.empty() || g->cols.size() > VDL_MAX_COLS) return false;
  d.ncolumns = (int)g->cols.size();
  return true;
}

#include "vdl_plan_join.inc"

struct ProbeFoldGroup {
  int space = -1, keynode = -1;
  ProbeBuild b;
  std::map<int, int> fold_of_node;
  std::map<int, int> post_of_node;      // Binary output node -> post op (evaluated by the probe's finalize kernel)
  vdl_probe *probe = nullptr;
  std::vector<vdl_vec> bound;
  i64 bound_rows = -1, bound_base = -1;
  PeerState peer;
};
struct EmitGroup {
  int space = -1;
  std::vector<int> nodes;
  ProbeBuild b;
  vdl_probe *probe = nullptr;
  std::vector<vdl_vec> bound;
  i64 bound_rows = -1, bound_base = -1;
  bool ran = false;
};

// Fold node `ni` over a joined space with a small key domain -> member of a probe fold group (Q5-class).
bool try_probe_fold(vdl_plan *p, int ni) {
  JoinAnalysis &J = *p->join;
  const Node &n = p->nodes[ni];
  const JSym G = janalyse(p, J, n.a), D = janalyse(p, J, n.b);
  int space, keynode = -1;
  JSym value;
  if (G.kind == Z_SORTED && D.kind == Z_SORTED && G.n0 == D.n0) {
    const JSym P = janalyse(p, J, G.n0);
    if (P.kind != Z_PART || G.n1 != P.n0) return false;
    value = janalyse(p, J, D.n1);
    if (value.kind != Z_VALUE) return false;
    space = P.space; keynode = P.n0;
    const JSym K = janalyse(p, J, keynode);
    if (!(K.kind == Z_KEY && K.masked && K.mask >= 0 && P.lo == 0 && P.cnt >= K.mask + 1) || K.mask + 1 > (1 << 20)) return false;
  } else if (j_is_const(G) && D.kind == Z_VALUE && D.space >= 0 && (G.space == D.space || G.space < 0)) {
    space = D.space; value = D;                        // one group (empty group-by, Vlite.hs:636-638)
  } else {
    return false;
  }
  if (space < 0) return false;   // (single-table Folds reach this point only when the TMA-staged fused scan could not express them)
  ProbeFoldGroup *g = nullptr;
  for (auto *q : p->pgroups) if (q->space == space && q->keynode == keynode) g = q;
  bool fresh = !g;
  if (fresh) {
    g = new ProbeFoldGroup();
    g->space = space; g->keynode = keynode;
    if (!pb_init(p, J, space, &g->b)) { delete g; return false; }
    if (keynode >= 0) {
      const JSym K = janalyse(p, J, keynode);
      g->b.desc.nkeys = (int)K.fac.size();
      for (size_t i = 0; i < K.fac.size(); i++)
        if (!pb_term(p, J, &g->b, K.fac[i], J.spaces[space].table, &g->b.desc.key[i])) { delete g; return false; }
      g->b.desc.key_mask = K.mask;
      g->b.desc.domain = K.mask + 1;
    }
  }
  ProbeBuild saved = g->b;
  vdl_probe_fold spec;
  memset(&spec, 0, sizeof spec);
  spec.op = n.sub;
  bool ok = true;
  if (n.sub != VDL_FOLD_COUNT) {
    bool ones = value.fac.size() == 1 && value.fac[0].leaf == -1 && value.fac[0].a == 1;
    if (n.sub == VDL_FOLD_SUM && ones) spec.op = VDL_FOLD_COUNT;
    else {
      ok = pb_product(p, J, &g->b, value.fac, J.spaces[space].table, &spec.value);
    }
  }
  int fi = -1;
  if (ok) {
    for (int i = 0; i < g->b.desc.nfolds; i++) if (!memcmp(&g->b.desc.fold[i], &spec, sizeof spec)) fi = i;
    if (fi < 0) {
      if (g->b.desc.nfolds == VDL_MAX_AGGS) ok = false;
      else { fi = g->b.desc.nfolds; g->b.desc.fold[g->b.desc.nfolds++] = spec; }
    }
  }
  if (ok) {     // the pass walks the fact table's rows: it needs at least one column of it (a bare COUNT(*), or a selection
                // that folded to "never", reads none -- those stay op-at-a-time)
    bool fact_leaf = false;
    for (int l = 0; l < g->b.desc.nleaves; l++) if (g->b.desc.leaf[l].parent < 0) fact_leaf = true;
    ok = fact_leaf;
  }
  if (!ok) {
    g->b = saved;
    if (fresh) delete g;
    return false;
  }
  if (fresh) p->pgroups.push_back(g);
  g->fold_of_node[ni] = fi;
  for (size_t i = 0; i < p->pgroups.size(); i++) if (p->pgroups[i] == g) p->pgroup_of_node[ni] = (int)i;
  return true;
}

// Which nodes does an op-at-a-time evaluation of the outputs touch?  A Gather / elementwise node whose normal form is
// a product of leaf terms over a joined space is cut off there and materialised by a probe in emit mode.
void mark_emits(vdl_plan *p, int ni, std::vector<char> &seen) {
  if (seen[ni]) return;
  seen[ni] = 1;
  JoinAnalysis &J = *p->join;
  const Node &n = p->nodes[ni];
  if (n.op == N_FOLD && (p->group_of_node[ni] >= 0 || p->pgroup_of_node[ni] >= 0)) return;
  if (n.op == N_BINARY && (p->group_of_node[ni] >= 0 || p->pgroup_of_node[ni] >= 0)) return;
  const JSym &z = janalyse(p, J, ni);
  if ((n.op == N_GATHER || n.op == N_BINARY) && z.kind == Z_VALUE && z.space >= 0 && !j_is_base(J, z.space) && !j_is_const(z)) {
    bool rooted = true;
    for (auto &t : z.fac) if (t.leaf >= 0 && !pb_rooted(p, J, t.leaf, J.spaces[z.space].table)) rooted = false;
    if (rooted) {
      EmitGroup *g = nullptr;
      for (auto *q : p->egroups) if (q->space == z.space && q->b.desc.nemits < VDL_MAX_EMITS) g = q;
      bool fresh = !g;
      if (fresh) { g = new EmitGroup(); g->space = z.space; if (!pb_init(p, J, z.space, &g->b)) { delete g; g = nullptr; } }
      if (g) {
        ProbeBuild saved = g->b;
        bool fact_leaf = false;
        if (pb_product(p, J, &g->b, z.fac, J.spaces[z.space].table, &g->b.desc.emit[g->b.desc.nemits]))
          for (int l = 0; l < g->b.desc.nleaves; l++) if (g->b.desc.leaf[l].parent < 0) fact_leaf = true;
        if (fact_leaf) {         // (a pass needs a column of the fact table to walk: see try_probe_fold)
          if (fresh) p->egroups.push_back(g);
          for (size_t i = 0; i < p->egroups.size(); i++) if (p->egroups[i] == g) p->egroup_of_node[ni] = (int)i;
          p->eslot_of_node[ni] = g->b.desc.nemits++;
          g->nodes.push_back(ni);
          return;
        }
        g->b = saved;
        if (fresh) delete g;
      }
    }
  }
  switch (n.op) {
    case N_RANGEV: mark_emits(p, n.a, seen); break;
    case N_BINARY: case N_GATHER: case N_FOLD: mark_emits(p, n.a, seen); mark_emits(p, n.b, seen); break;
    case N_FSELECT: mark_emits(p, n.b, seen); break;
    case N_LIKE: mark_emits(p, n.a, seen); break;
    case N_CROSS: mark_emits(p, n.a, seen); mark_emits(p, n.b, seen); break;
    case N_SCATTER: mark_emits(p, n.a, seen); mark_emits(p, n.c, seen); break;
    case N_PARTITION: mark_emits(p, n.a, seen); break;
    default: break;
  }
}

// An output that is an elementwise expression over the Folds of ONE fused scan (AVG = Divide(FoldSum x, FoldSum 1),
// Vlite.hs:1038-1041) becomes a post op of that scan: evaluated per group inside the finalize kernel and returned by
// the scan's single result copy, instead of op-at-a-time launches over a handful of elements.
// Returns the operand kind (VDL_POST_*) or -1 when `ni` is not such an expression.
int post_operand(vdl_plan *p, int ni, int *gi, i64 *val) {
  const Node &n = p->nodes[ni];
  if (n.op == N_FOLD) {
    int g = p->group_of_node[ni];
    if (g < 0 || (*gi >= 0 && *gi != g)) return -1;
    *gi = g;
    *val = p->groups[g].fold_of_node[ni];
    return VDL_POST_FOLD;
  }
  if (n.op == N_RANGEV && n.k1 == 0) {             // a constant as long as a vector of the same scan's results
    i64 dummy;
    if (post_operand(p, n.a, gi, &dummy) < 0) return -1;
    *val = n.k0;
    return VDL_POST_CONST;
  }
  if (n.op == N_BINARY) {
    int g0 = *gi;
    if (g0 >= 0) {
      auto it = p->groups[g0].post_of_node.find(ni);
      if (it != p->groups[g0].post_of_node.end()) { *val = it->second; return VDL_POST_POST; }
    }
    vdl_post_op op;
    memset(&op, 0, sizeof op);
    op.op = n.sub;
    int ka = post_operand(p, n.a, gi, &op.a);
    if (ka < 0) return -1;
    int kb = post_operand(p, n.b, gi, &op.b);
    if (kb < 0 || *gi < 0) return -1;
    op.a_kind = ka; op.b_kind = kb;
    FusedGroup &g = p->groups[*gi];
    auto it = g.post_of_node.find(ni);           // the group may only have become known through the operands
    if (it != g.post_of_node.end()) { *val = it->second; return VDL_POST_POST; }
    if (g.posts.size() == VDL_MAX_POSTS) return -1;
    g.posts.push_back(op);
    g.post_of_node[ni] = (int)g.posts.size() - 1;
    *val = (i64)g.posts.size() - 1;
    return VDL_POST_POST;
  }
  return -1;
}

// ---- map clusters ------------------------------------------------------------------------------------------------
// What is left for op-at-a-time evaluation after the scans and probe passes is dominated by chains of elementwise ops
// (Q19: the OR of three AND groups over the join's survivors, ~150 nodes).  A cluster is a root node plus every
// Binary / Gather / RangeV descendant ALL of whose consumers are inside the cluster, so nothing outside ever needs an
// interior value and the leaves cannot depend on members; it compiles to one register program (vdl_op_map).
// `cons` counts consumer edges of the demand-driven evaluation only (nodes inside fused scans / probe passes are dead here).
void live_walk(vdl_plan *p, int ni, std::vector<char> &live, std::vector<int> &cons) {
  if (live[ni]) return;
  live[ni] = 1;
  if (p->egroup_of_node[ni] >= 0) return;
  const Node &n = p->nodes[ni];
  auto use = [&](int a) { cons[a]++; live_walk(p, a, live, cons); };
  const bool fused = p->group_of_node[ni] >= 0 || p->pgroup_of_node[ni] >= 0;
  switch (n.op) {
    case N_RANGEV: use(n.a); break;
    case N_BINARY: if (!fused) { use(n.a); use(n.b); } break;
    case N_FSELECT: use(n.b); break;
    case N_LIKE: use(n.a); use(n.b); break;
    case N_CROSS: use(n.a); use(n.b); break;
    case N_GATHER: use(n.a); use(n.b); break;
    case N_SCATTER: use(n.a); use(n.c); break;
    case N_PARTITION: use(n.a); break;
    case N_FOLD: if (!fused) { use(n.a); use(n.b); } break;
    default: break;
  }
}

// Register program of a cluster; false when it exceeds vdl_op_map's limits.
bool compile_cluster(vdl_plan *p, MapCluster *c) {
  std::vector<int> mem = c->members;
  std::sort(mem.begin(), mem.end());
  std::set<int> in_cluster(mem.begin(), mem.end());
  c->inputs.clear(); c->tables.clear();
  memset(&c->desc, 0, sizeof c->desc);
  vdl_map_desc &d = c->desc;
  auto slot = [](std::vector<int> &v, int x) { for (size_t i = 0; i < v.size(); i++) if (v[i] == x) return (int)i; v.push_back(x); return (int)v.size() - 1; };
  // values: members and loaded inputs; last use position (in member order) for register release
  std::map<int, int> last_use;
  for (size_t t = 0; t < mem.size(); t++) {
    const Node &n = p->nodes[mem[t]];
    if (n.op == N_BINARY) { last_use[n.a] = (int)t; last_use[n.b] = (int)t; }
    else if (n.op == N_GATHER) last_use[n.b] = (int)t;
  }
  std::map<int, int> reg_of;
  unsigned busy = 0;
  auto alloc = [&]() { for (int r = 0; r < VDL_MAP_MAX_REGS; r++) if (!(busy >> r & 1)) { busy |= 1u << r; return r; } return -1; };
  auto emit = [&](int op, int dst, int a, int b) {
    if (d.ninstrs == VDL_MAP_MAX_INSTRS) return false;
    d.instr[d.ninstrs++] = vdl_map_instr{(int16_t)op, (int16_t)dst, (int16_t)a, (int16_t)b};
    return true;
  };
  auto imm = [&](i64 v) { for (int i = 0; i < d.nimms; i++) if (d.imm[i] == v) return i; if (d.nimms == VDL_MAP_MAX_IMMS) return -1; d.imm[d.nimms] = v; return d.nimms++; };
  auto operand = [&](int node) -> int {       // register holding `node`'s value at this point (loads a leaf on first use)
    auto it = reg_of.find(node);
    if (it != reg_of.end()) return it->second;
    if (in_cluster.count(node)) return -1;    // members are defined before use (ascending order); cannot happen
    int r = alloc();
    if (r < 0) return -1;
    int k = slot(c->inputs, node);
    if (k >= VDL_MAP_MAX_INPUTS || !emit(VDL_MAP_LOAD, r, 0, k)) return -1;
    reg_of[node] = r;
    return r;
  };
  for (size_t t = 0; t < mem.size(); t++) {
    const int ni = mem[t];
    const Node &n = p->nodes[ni];
    int ra = -1, rb = -1, tab = -1;
    if (n.op == N_BINARY) { ra = operand(n.a); rb = operand(n.b); if (ra < 0 || rb < 0) return false; }
    else if (n.op == N_GATHER) { ra = operand(n.b); tab = slot(c->tables, n.a); if (ra < 0 || tab >= VDL_MAP_MAX_TABLES) return false; }
    else if (n.op == N_RANGEV) { if (!in_cluster.count(n.a)) { if (slot(c->inputs, n.a) >= VDL_MAP_MAX_INPUTS) return false; } }   // length witness
    // operands dying here free their registers before the destination is chosen (the kernel reads before it writes)
    for (int o : {n.op == N_BINARY ? n.a : -1, n.op == N_BINARY || n.op == N_GATHER ? n.b : -1})
      if (o >= 0 && last_use[o] == (int)t) { auto it = reg_of.find(o); if (it != reg_of.end()) { busy &= ~(1u << it->second); reg_of.erase(it); } }
    int rd = alloc();
    if (rd < 0) return false;
    bool ok;
    if (n.op == N_BINARY) ok = emit(n.sub, rd, ra, rb);
    else if (n.op == N_GATHER) ok = emit(VDL_MAP_GATHER, rd, ra, tab);
    else { int i0 = imm(n.k0), i1 = imm(n.k1); ok = i0 >= 0 && i1 >= 0 && emit(VDL_MAP_RANGE, rd, i0, i1); }
    if (!ok) return false;
    reg_of[ni] = rd;
    if (!last_use.count(ni) && ni != c->root) { busy &= ~(1u << rd); reg_of.erase(ni); }    // only a length witness for a member RangeV
  }
  d.ninputs = (int)c->inputs.size();
  d.ntables = (int)c->tables.size();
  return d.ninputs >= 1 && mem.back() == c->root;
}

void build_clusters(vdl_plan *p) {
  const int nn = (int)p->nodes.size();
  p->cluster_of_root.assign(nn, -1);
  if (getenv("VDL_NO_MAP")) return;
  for (int i = 0; i < nn; i++) for (int a : {p->nodes[i].a, p->nodes[i].b, p->nodes[i].c}) if (a >= i) return;   // not in definition order: leave the plan alone
  std::vector<char> live(nn, 0);
  std::vector<int> cons(nn, 0);
  for (auto &o : p->outputs) {
    if (p->group_of_node[o.node] >= 0 || p->pgroup_of_node[o.node] >= 0) continue;
    cons[o.node]++;
    live_walk(p, o.node, live, cons);
  }
  auto eligible = [&](int ni) {
    const Node &n = p->nodes[ni];
    if (!live[ni] || p->egroup_of_node[ni] >= 0 || p->group_of_node[ni] >= 0 || p->pgroup_of_node[ni] >= 0) return false;
    return n.op == N_BINARY || n.op == N_GATHER || n.op == N_RANGEV;
  };
  std::vector<int> member_of(nn, -1);
  for (int ni = nn - 1; ni >= 0; ni--) {
    if (member_of[ni] >= 0 || !eligible(ni) || p->nodes[ni].op == N_RANGEV) continue;
    MapCluster c;
    c.root = ni;
    c.members.push_back(ni);
    member_of[ni] = ni;
    std::set<int> refused;
    for (bool changed = true; changed;) {
      changed = false;
      for (size_t k = 0; k < c.members.size(); k++) {
        const Node &m = p->nodes[c.members[k]];
        for (int dnode : {m.op == N_BINARY ? m.a : -1, m.op == N_RANGEV ? m.a : m.b}) {     // row-aligned operands (a Gather's source is a table)
          if (dnode < 0 || member_of[dnode] >= 0 || refused.count(dnode) || !eligible(dnode)) continue;
          int inside = 0;
          for (int q : c.members) {
            const Node &mq = p->nodes[q];
            if (mq.op == N_BINARY) inside += (mq.a == dnode) + (mq.b == dnode);
            else if (mq.op == N_GATHER) inside += (mq.b == dnode);
            else inside += (mq.a == dnode);
          }
          if (inside != cons[dnode]) continue;
          MapCluster trial = c;
          trial.members.push_back(dnode);
          if (!compile_cluster(p, &trial)) { refused.insert(dnode); continue; }
          c.members.push_back(dnode);
          member_of[dnode] = ni;
          changed = true;
        }
      }
    }
    int real = 0;
    for (int q : c.members) if (p->nodes[q].op != N_RANGEV) real++;
    if (real < 2 || !compile_cluster(p, &c)) {       // a lone op: the per-op kernel is as good
      for (int q : c.members) member_of[q] = -1;
      continue;
    }
    std::sort(c.members.begin(), c.members.end());
    p->cluster_of_root[ni] = (int)p->clusters.size();
    p->clusters.push_back(c);
  }
}

int fuse(vdl_plan *p) {
  size_t nn = p->nodes.size();
  p->sym.assign(nn, Sym());
  p->sym_done.assign(nn, 0);
  p->group_of_node.assign(nn, -1);
  p->pgroup_of_node.assign(nn, -1);
  p->egroup_of_node.assign(nn, -1);
  p->eslot_of_node.assign(nn, -1);
  p->cluster_of_root.assign(nn, -1);
  if (!(p->flags & VDL_PLAN_FUSE)) return VDL_OK;
  for (size_t i = 0; i < nn; i++)
    if (p->nodes[i].op == N_FOLD) try_fuse_fold(p, (int)i);
  for (auto &o : p->outputs) {
    if (p->nodes[o.node].op != N_BINARY) continue;
    std::vector<size_t> mark;
    for (auto &g : p->groups) mark.push_back(g.posts.size());
    int gi = -1;
    i64 v;
    if (post_operand(p, o.node, &gi, &v) != VDL_POST_POST)      // roll back partial registrations
      for (size_t g = 0; g < p->groups.size(); g++) {
        FusedGroup &G = p->groups[g];
        for (auto it = G.post_of_node.begin(); it != G.post_of_node.end();)
          it = it->second >= (int)mark[g] ? G.post_of_node.erase(it) : std::next(it);
        G.posts.resize(mark[g]);
      }
  }
  for (size_t gi = 0; gi < p->groups.size(); gi++) {
    if (!build_desc(p, &p->groups[gi])) {      // cannot be expressed after all: un-fuse its folds
      for (auto &kv : p->groups[gi].fold_of_node) p->group_of_node[kv.first] = -1;
      p->groups[gi].folds.clear();
      p->groups[gi].fold_of_node.clear();
      p->groups[gi].post_of_node.clear();
    }
  }
  p->groups.erase(std::remove_if(p->groups.begin(), p->groups.end(), [](const FusedGroup &g) { return g.folds.empty(); }), p->groups.end());
  // group indices may have shifted
  std::fill(p->group_of_node.begin(), p->group_of_node.end(), -1);
  for (size_t gi = 0; gi < p->groups.size(); gi++) {
    for (auto &kv : p->groups[gi].fold_of_node) p->group_of_node[kv.first] = (int)gi;
    for (auto &kv : p->groups[gi].post_of_node) p->group_of_node[kv.first] = (int)gi;
  }
  // FK-join plans: Folds over a joined space -> probe fold groups; vectors of joined spaces that op-at-a-time
  // consumers need -> probe emit groups
  if (!getenv("VDL_NO_PROBE")) {
    p->join = new JoinAnalysis();
    p->join->sym.assign(nn, JSym());
    p->join->done.assign(nn, 0);
    std::vector<int> uses(nn, 0);
    for (auto &n : p->nodes) for (int a : {n.a, n.b, n.c}) if (a >= 0) uses[a]++;
    // Folds may be consumed by OUTPUT expressions made of elementwise ops over Folds and constants (AVG's Divide):
    // those become post ops of the probe's finalize kernel.  A Fold with any other consumer is not fused.
    std::vector<int> post_refs(nn, 0), bin_refs(nn, 0);
    std::vector<char> in_out_expr(nn, 0);
    {
      std::vector<int> stack;
      for (auto &o : p->outputs) if (p->nodes[o.node].op == N_BINARY) stack.push_back(o.node);
      while (!stack.empty()) {
        int ni = stack.back(); stack.pop_back();
        if (in_out_expr[ni]) continue;
        in_out_expr[ni] = 1;
        const Node &n = p->nodes[ni];
        for (int a : {n.a, n.b}) {
          if (a < 0) continue;
          const Node &c = p->nodes[a];
          if (c.op == N_FOLD) post_refs[a]++;
          else if (c.op == N_BINARY) { stack.push_back(a); bin_refs[a]++; }
          else if (c.op == N_RANGEV && c.k1 == 0 && c.a >= 0 && p->nodes[c.a].op == N_FOLD) post_refs[c.a]++;   // a constant as long as a Fold result
        }
      }
    }
    for (size_t i = 0; i < nn; i++)        // an inner node of an output expression that something else consumes too: no post ops in this plan
      if (in_out_expr[i] && uses[i] != bin_refs[i]) { std::fill(post_refs.begin(), post_refs.end(), 0); break; }
    for (size_t i = 0; i < nn; i++)
      if (p->nodes[i].op == N_FOLD && p->group_of_node[i] < 0 && uses[i] == post_refs[i]) try_probe_fold(p, (int)i);
    // outputs over probe Folds -> post ops; if one cannot be expressed, the Folds it needs fall back to op-at-a-time
    std::function<int(int, int *, i64 *)> ppost = [&](int ni, int *gi, i64 *val) -> int {
      const Node &n = p->nodes[ni];
      if (n.op == N_FOLD) {
        int g = p->pgroup_of_node[ni];
        if (g < 0 || (*gi >= 0 && *gi != g)) return -1;
        *gi = g; *val = p->pgroups[g]->fold_of_node[ni];
        return VDL_POST_FOLD;
      }
      if (n.op == N_RANGEV && n.k1 == 0) { i64 d; if (ppost(n.a, gi, &d) < 0) return -1; *val = n.k0; return VDL_POST_CONST; }
      if (n.op == N_BINARY) {
        vdl_post_op op; memset(&op, 0, sizeof op);
        op.op = n.sub;
        int ka = ppost(n.a, gi, &op.a); if (ka < 0) return -1;
        int kb = ppost(n.b, gi, &op.b); if (kb < 0 || *gi < 0) return -1;
        op.a_kind = ka; op.b_kind = kb;
        ProbeFoldGroup &g = *p->pgroups[*gi];
        auto it = g.post_of_node.find(ni);
        if (it != g.post_of_node.end()) { *val = it->second; return VDL_POST_POST; }
        if (g.b.desc.nposts == VDL_MAX_POSTS) return -1;
        g.b.desc.post[g.b.desc.nposts] = op;
        g.post_of_node[ni] = g.b.desc.nposts;
        *val = g.b.desc.nposts++;
        return VDL_POST_POST;
      }
      return -1;
    };
    bool unfuse = false;
    for (auto &o : p->outputs) {
      if (p->nodes[o.node].op != N_BINARY) continue;
      int gi = -1; i64 v;
      if (ppost(o.node, &gi, &v) == VDL_POST_POST) p->pgroup_of_node[o.node] = gi;
      else unfuse = true;       // some consumer of a fused Fold is not a post op: be safe, un-fuse every probe fold group
    }
    if (unfuse) {
      bool any_needed = false;
      for (size_t i = 0; i < nn; i++) if (p->nodes[i].op == N_FOLD && p->pgroup_of_node[i] >= 0 && post_refs[i] > 0) any_needed = true;
      if (any_needed) {
        for (auto *g : p->pgroups) delete g;
        p->pgroups.clear();
        std::fill(p->pgroup_of_node.begin(), p->pgroup_of_node.end(), -1);
        for (size_t i = 0; i < nn; i++)            // keep the Folds nobody consumes
          if (p->nodes[i].op == N_FOLD && p->group_of_node[i] < 0 && uses[i] == 0) try_probe_fold(p, (int)i);
      }
    }
    std::vector<char> seen(nn, 0);
    for (auto &o : p->outputs) mark_emits(p, o.node, seen);
  }
  build_clusters(p);
  return VDL_OK;
}

// ---------------------------------------------------------------------------------- execution
void free_temps(vdl_plan *p) {
  for (vdl_vec v : p->temps) vdl_vec_free(p->ctx, v);
  p->temps.clear();
  for (auto *g : p->egroups) g->ran = false;
  std::fill(p->val.begin(), p->val.end(), 0);
}

// Bind a probe descriptor's leaves to the registered columns and (re)prepare it when the binding changed.
int bind_probe(vdl_plan *p, ProbeBuild *b, vdl_probe **probe, std::vector<vdl_vec> *bound, i64 *bound_rows, i64 *bound_base) {
  vdl_ctx *ctx = p->ctx;
  std::vector<vdl_vec> h(b->loadnode.size());
  i64 rows = -1;
  for (size_t l = 0; l < h.size(); l++) {
    VDL_TRY(vdl_column_lookup(ctx, p->nodes[b->loadnode[l]].name.c_str(), &h[l]));
    if (b->desc.leaf[l].parent < 0) {
      i64 len; VDL_TRY(vdl_vec_len(ctx, h[l], &len));
      if (rows >= 0 && len != rows) return vdl_fail(ctx, VDL_EINVAL, "probe: fact columns differ in length (%lld vs %lld)", (long long)len, (long long)rows);
      rows = len;
    }
  }
  if (rows < 0) return vdl_fail(ctx, VDL_EUNSUPPORTED, "probe: no fact column among the leaves");
  if (!*probe || !vdl_probe_current(*probe) || h != *bound || rows != *bound_rows || p->row_base != *bound_base) {
    if (*probe) { vdl_probe_destroy(*probe); *probe = nullptr; }
    b->desc.rows = rows;
    b->desc.row_base = p->row_base;
    for (size_t l = 0; l < h.size(); l++) b->desc.leaf[l].column = h[l];
    VDL_TRY(vdl_probe_prepare(ctx, &b->desc, probe));
    *bound = h; *bound_rows = rows; *bound_base = p->row_base;
  }
  return VDL_OK;
}

int run_emit_group(vdl_plan *p, EmitGroup &g) {
  if (g.ran) return VDL_OK;
  VDL_TRY(bind_probe(p, &g.b, &g.probe, &g.bound, &g.bound_rows, &g.bound_base));
  VDL_TRY(vdl_probe_run(g.probe));
  for (size_t k = 0; k < g.nodes.size(); k++) {
    vdl_vec v;
    VDL_TRY(vdl_probe_emit_take(g.probe, (int)k, &v));
    p->val[g.nodes[k]] = v;
    p->temps.push_back(v);
    // a plain leaf of a 4-byte column: every emitted value fits int32 (typed result columns, vdl_plan_set_typed_outputs)
    const vdl_product &e = g.b.desc.emit[k];
    if (e.nfactors == 1 && e.factor[0].leaf >= 0 && e.factor[0].shr == 0 && e.factor[0].a == 0 && e.factor[0].b == 1) {
      Vec *col = vec_get(p->ctx, g.b.desc.leaf[e.factor[0].leaf].column), *ev = vec_get(p->ctx, v);
      if (col && ev && col->dtype == VDL_I32) ev->narrow32 = true;
    }
  }
  g.ran = true;
  return VDL_OK;
}

int eval(vdl_plan *p, int ni, vdl_vec *out) {
  vdl_ctx *ctx = p->ctx;
  if (p->val[ni]) { *out = p->val[ni]; return VDL_OK; }
  if (p->egroup_of_node[ni] >= 0) {        // materialised by one probe pass together with its siblings of the same space
    VDL_TRY(run_emit_group(p, *p->egroups[p->egroup_of_node[ni]]));
    *out = p->val[ni];
    return VDL_OK;
  }
  const Node &n = p->nodes[ni];
  vdl_vec r = 0, a = 0, b = 0, c = 0;
  bool temp = true;
  if (p->cluster_of_root[ni] >= 0) {        // this node and its private elementwise / Gather subtree: one launch
    const MapCluster &mc = p->clusters[p->cluster_of_root[ni]];
    std::vector<vdl_vec> in(mc.inputs.size()), tab(mc.tables.size());
    for (size_t k = 0; k < in.size(); k++) VDL_TRY(eval(p, mc.inputs[k], &in[k]));
    for (size_t k = 0; k < tab.size(); k++) VDL_TRY(eval(p, mc.tables[k], &tab[k]));
    VDL_TRY(vdl_op_map(ctx, &mc.desc, in.data(), tab.data(), &r));
  } else
  switch (n.op) {
    case N_LOAD: VDL_TRY(vdl_column_lookup(ctx, n.name.c_str(), &r)); temp = false; break;
    case N_RANGEV: {
      VDL_TRY(eval(p, n.a, &a));
      i64 len; VDL_TRY(vdl_vec_len(ctx, a, &len));
      VDL_TRY(vdl_op_range(ctx, n.k0, n.k1, len, &r));
      break;
    }
    case N_RANGEC: VDL_TRY(vdl_op_range(ctx, n.k0, n.k2, n.k1, &r)); break;
    case N_BINARY: VDL_TRY(eval(p, n.a, &a)); VDL_TRY(eval(p, n.b, &b)); VDL_TRY(vdl_op_binary(ctx, n.sub, a, b, &r)); break;
    case N_FSELECT: {
      const Node &fn = p->nodes[n.a];
      if (!(fn.op == N_RANGEV && fn.k0 == 0 && fn.k1 == 1))
        return vdl_fail(ctx, VDL_EUNSUPPORTED, "FoldSelect: fold argument must be pos_ of the predicate (Vlite.hs:726-727)");
      VDL_TRY(eval(p, n.b, &b));
      VDL_TRY(vdl_op_fold_select(ctx, b, &r));
      break;
    }
    case N_GATHER: VDL_TRY(eval(p, n.a, &a)); VDL_TRY(eval(p, n.b, &b)); VDL_TRY(vdl_op_gather(ctx, a, b, &r)); break;
    case N_LIKE: VDL_TRY(eval(p, n.a, &a)); VDL_TRY(eval(p, n.b, &b)); VDL_TRY(vdl_op_like(ctx, a, b, n.name.c_str(), &r)); break;
    case N_CROSS: VDL_TRY(eval(p, n.a, &a)); VDL_TRY(eval(p, n.b, &b)); VDL_TRY(vdl_op_cross_product(ctx, a, b, n.sub, &r)); break;
    case N_SCATTER: {
      VDL_TRY(eval(p, n.a, &a)); VDL_TRY(eval(p, n.c, &c));
      Vec *pv = vec_get(ctx, c), *sv = vec_get(ctx, a);
      if (!pv || !sv) return VDL_EINVAL;
      i64 out_len = pv->domain;
      if (out_len < 0 && p->join) {
        // positions materialised by a probe pass carry no index space of their own; when the join analysis knows them to
        // be row ids of a table (the dimension selection of deduceMasks, Vlite.hs:1268-1275), the output has that table's
        // length -- the reference's `dimref` (Vlite.hs:782; App. G2)
        const JSym &pt = janalyse(p, *p->join, n.c);
        if (j_is_rowid(pt) && pt.space >= 0) {
          const std::string prefix = p->tables[p->join->spaces[pt.space].table] + ".";
          for (const Node &ld : p->nodes)
            if (ld.op == N_LOAD && ld.name.compare(0, prefix.size(), prefix) == 0 && !(ld.name.size() > 5 && ld.name.compare(ld.name.size() - 5, 5, ".heap") == 0)) {
              vdl_vec h; VDL_TRY(vdl_column_lookup(ctx, ld.name.c_str(), &h));
              VDL_TRY(vdl_vec_len(ctx, h, &out_len));
              break;
            }
          pv = vec_get(ctx, c); sv = vec_get(ctx, a);
        }
      }
      if (out_len < 0) return vdl_fail(ctx, VDL_EUNSUPPORTED, "Scatter: output length unknown (positions carry no index space; App. G2)");
      if (pv->is_range && pv->from == 0 && pv->step == 1 && pv->len == out_len && sv->len == pv->len && !sv->is_range && sv->dtype == VDL_I64) {
        r = a; temp = false;       // scattering by the identity permutation (Partition of keys already in order): the source itself
        break;
      }
      VDL_TRY(vdl_op_scatter(ctx, a, c, out_len, &r));
      break;
    }
    case N_PARTITION: {
      const Node &pv = p->nodes[n.b];
      if (pv.op != N_RANGEC || pv.k2 <= 0) return vdl_fail(ctx, VDL_EUNSUPPORTED, "Partition: pivots must be an ascending RangeC (Vlite.hs:1088-1091)");
      VDL_TRY(eval(p, n.a, &a));
      VDL_TRY(vdl_op_partition(ctx, a, pv.k0, pv.k2, pv.k1, &r));
      break;
    }
    case N_FOLD: {
      int gi = p->group_of_node[ni];
      if (p->pgroup_of_node[ni] >= 0) return vdl_fail(ctx, VDL_EUNSUPPORTED, "a Fold run by the probe kernel has no device vector (it is only fused when nothing consumes it)");
      if (gi >= 0) {
        FusedGroup &g = p->groups[gi];
        VDL_TRY(vdl_fused_result(g.fused, g.fold_of_node[ni], &r));
        temp = false;
      } else {
        VDL_TRY(eval(p, n.a, &a)); VDL_TRY(eval(p, n.b, &b));
        VDL_TRY(vdl_op_fold(ctx, n.sub, a, b, &r));
      }
      break;
    }
  }
  p->val[ni] = r;
  if (temp) p->temps.push_back(r);
  *out = r;
  if (p->trace) {      // VDL_TRACE: host wall time per node, synchronised (debugging aid: serialises the plan)
    cudaStreamSynchronize(ctx->stream);
    double t1 = now_ms();
    i64 len = 0;
    vdl_vec_len(ctx, r, &len);
    static const char *OPN[] = {"Load", "RangeV", "RangeC", "Binary", "FoldSelect", "Gather", "Scatter", "Partition", "Fold", "Like"};
    fprintf(stderr, "[vdl trace] node %3d %-10s sub %2d len %10lld  %8.3f ms (cumulative since plan start %8.3f)\n", ni, OPN[n.op], n.sub, (long long)len,
            t1 - p->trace_last, t1 - p->trace_t0);
    p->trace_last = now_ms();
  }
  return VDL_OK;
}

// A plan whose outputs are ALL op-at-a-time Folds (Sum / Min / Max / Choose / Count) by runs of one groups vector -- a
// constant (one run: Q19's single SUM over the join's survivors) or keys sorted by their own Partition (Vlite.hs:1057-1060:
// Q3's group-by on the 38-bit composite key) -- can run its whole tail on a row-range shard: rank r's result is the slice of
// the global result for its rows, except that the last group of rank r and the first of rank r+1 may be the same group.
void detect_mergeable_tail(vdl_plan *p) {
  int G = -1;
  for (auto &o : p->outputs) {
    const Node &n = p->nodes[o.node];
    if (n.op != N_FOLD || p->group_of_node[o.node] >= 0 || p->pgroup_of_node[o.node] >= 0) return;
    if (G >= 0 && n.a != G) return;
    G = n.a;
  }
  if (G < 0) return;
  const Node &g = p->nodes[G];
  int P = -1;
  if (g.op == N_RANGEV && g.k1 == 0) P = -1;
  else if (g.op == N_SCATTER && p->nodes[g.c].op == N_PARTITION && p->nodes[g.c].a == g.a) P = g.c;
  else return;
  for (auto &o : p->outputs) {              // the data of every Fold rides the same sort
    const Node &d = p->nodes[p->nodes[o.node].b];
    if (P >= 0 && !(d.op == N_SCATTER && d.c == P)) return;
    if (p->nodes[d.op == N_SCATTER ? d.a : p->nodes[o.node].b].op == N_FOLD) return;    // no second level
  }
  p->tail_ok = true; p->tail_groups = G; p->tail_partition = P;
}

int capture_tail_boundary(vdl_plan *p) {
  vdl_ctx *ctx = p->ctx;
  i64 *r = p->tail_rec;
  r[0] = r[1] = r[2] = r[3] = 0;
  r[1] = p->outputs.empty() ? 0 : p->outputs[0].len;
  const vdl_vec gh = p->val[p->tail_groups];
  Vec *g = gh ? vec_get(ctx, gh) : nullptr;
  if (!g) return vdl_fail(ctx, VDL_EINVAL, "sharded tail: the groups vector was not evaluated");
  bool sorted = true;
  if (p->tail_partition >= 0) {
    Vec *pv = p->val[p->tail_partition] ? vec_get(ctx, p->val[p->tail_partition]) : nullptr;
    sorted = pv && pv->is_range && pv->from == 0 && pv->step == 1;     // the local keys were already in order
  }
  r[0] = sorted;
  const i64 n = g->len;
  if (n > 0) {
    if (g->is_range) { r[2] = g->from; r[3] = (i64)((u64)g->from + (u64)(n - 1) * (u64)g->step); }
    else if (g->dtype == VDL_I64) {
      VDL_TRY(read_scalar(ctx, (const i64 *)g->ptr, &r[2], 8));
      VDL_TRY(read_scalar(ctx, (const i64 *)g->ptr + (n - 1), &r[3], 8));
    } else {
      int a = 0, b = 0;
      VDL_TRY(read_scalar(ctx, (const int *)g->ptr, &a, 4));
      VDL_TRY(read_scalar(ctx, (const int *)g->ptr + (n - 1), &b, 4));
      r[2] = a; r[3] = b;
    }
  }
  return VDL_OK;
}

// the output's own pinned host buffer, grown to hold len values (pinned, so a copy into it is one DMA at PCIe rate)
int reserve_pinned(vdl_ctx *ctx, Output &o, i64 len) {
  if (o.pinned) cudaFreeHost(o.pinned);
  o.pinned = nullptr; o.cap = 0;
  size_t want = (size_t)len + (size_t)len / 4 + 16;
  if (cudaHostAlloc(&o.pinned, want * sizeof(i64), cudaHostAllocDefault) != cudaSuccess) return vdl_fail(ctx, VDL_ENOMEM, "output buffer of %lld values", (long long)len);
  o.cap = want;
  return VDL_OK;
}

}  // namespace

// ---------------------------------------------------------------------------------- ABI
extern "C" int vdl_plan_load(vdl_ctx *ctx, const char *vdl_text, int flags, vdl_plan **out) {
  if (!ctx || !vdl_text || !out) return VDL_EINVAL;
  *out = nullptr;
  vdl_plan *p = new vdl_plan();
  p->ctx = ctx;
  p->flags = flags;
  int rc = parse_plan(p, vdl_text);
  if (!rc) rc = fuse(p);
  if (rc) { delete p; return rc; }
  p->val.assign(p->nodes.size(), 0);
  detect_mergeable_tail(p);
  if (getenv("VDL_DEBUG_PLAN")) {
    fprintf(stderr, "[vdl plan] %d statements, %zu nodes: %zu fused scans, %zu probe fold groups, %zu probe emit groups\n", p->statements, p->nodes.size(),
            p->groups.size(), p->pgroups.size(), p->egroups.size());
    for (auto *g : p->pgroups)
      fprintf(stderr, "[vdl plan]   probe fold: table %s, %d leaves, %d predicates, %d key parts (domain %lld), %d folds\n", p->tables[p->join->spaces[g->space].table].c_str(),
              g->b.desc.nleaves, g->b.desc.npreds, g->b.desc.nkeys, (long long)g->b.desc.domain, g->b.desc.nfolds);
    for (auto *g : p->pgroups) {
      const vdl_probe_desc &d = g->b.desc;
      for (int l = 0; l < d.nleaves; l++) fprintf(stderr, "[vdl plan]     leaf %d: %s parent %d\n", l, p->nodes[g->b.loadnode[l]].name.c_str(), d.leaf[l].parent);
      for (int q = 0; q < d.npreds; q++) fprintf(stderr, "[vdl plan]     pred %d: kind %d t(leaf %d shr %d a %lld b %lld) u(leaf %d) [%lld, %lld]\n", q, d.pred[q].kind, d.pred[q].t.leaf, d.pred[q].t.shr, (long long)d.pred[q].t.a, (long long)d.pred[q].t.b, d.pred[q].u.leaf, (long long)d.pred[q].lo, (long long)d.pred[q].hi);
      for (int j = 0; j < d.nfolds; j++) {
        fprintf(stderr, "[vdl plan]     fold %d: op %d nfactors %d", j, d.fold[j].op, d.fold[j].value.nfactors);
        for (int t = 0; t < d.fold[j].value.nfactors; t++) fprintf(stderr, " (leaf %d shr %d a %lld b %lld)", d.fold[j].value.factor[t].leaf, d.fold[j].value.factor[t].shr, (long long)d.fold[j].value.factor[t].a, (long long)d.fold[j].value.factor[t].b);
        fprintf(stderr, "\n");
      }
    }
    for (auto &c : p->clusters)
      fprintf(stderr, "[vdl plan]   map cluster: root %d, %zu nodes, %d inputs, %d tables, %d instructions\n", c.root, c.members.size(), c.desc.ninputs, c.desc.ntables, c.desc.ninstrs);
    for (auto *g : p->egroups) {
      fprintf(stderr, "[vdl plan]   probe emit: table %s, %d leaves, %d predicates, nodes", p->tables[p->join->spaces[g->space].table].c_str(), g->b.desc.nleaves, g->b.desc.npreds);
      for (int n : g->nodes) fprintf(stderr, " %d", n);
      fprintf(stderr, "\n");
    }
  }
  *out = p;
  return VDL_OK;
}

// What the planner makes of a program, without a device: parse, CSE, both fusion passes, map clusters, the tail check -- as
// JSON.  No column is looked up and nothing is compiled or launched (binding happens at run time), so this runs on a host
// without a GPU: the planner's decisions are testable where the kernels are not.
extern "C" int vdl_plan_explain(const char *vdl_text, int flags, char *out, int capacity) {
  if (!vdl_text || !out || capacity < 2) return VDL_EINVAL;
  vdl_ctx *ctx = new vdl_ctx();          // a message sink only: never touches CUDA, never passed to anything that does
  ctx->device = -1;
  vdl_plan *p = new vdl_plan();
  p->ctx = ctx;
  p->flags = flags;
  int rc = parse_plan(p, vdl_text);
  if (!rc) rc = fuse(p);
  std::string js;
  char b[512];
  auto add = [&](const char *fmt, auto... a) { snprintf(b, sizeof b, fmt, a...); js += b; };
  if (rc) {
    std::string msg = ctx->err;
    for (auto &c : msg) if (c == '"' || c == '\\' || (unsigned char)c < 32) c = ' ';
    add("{\"error\": %d, \"message\": \"%s\"}", rc, msg.c_str());
  } else {
    detect_mergeable_tail(p);
    add("{\"statements\": %d, \"nodes\": %d, \"outputs\": %d, \"fused_scans\": [", p->statements, (int)p->nodes.size(), (int)p->outputs.size());
    for (size_t i = 0; i < p->groups.size(); i++) {
      const FusedGroup &g = p->groups[i];
      add("%s{\"table\": \"%s\", \"columns\": %d, \"predicates\": %d, \"key_parts\": %d, \"domain\": %lld, \"folds\": %d, \"posts\": %d}", i ? ", " : "",
          p->tables[g.table].c_str(), g.desc.ncolumns, g.desc.npreds, g.desc.nkeys, (long long)g.desc.domain, g.desc.nfolds, g.desc.nposts);
    }
    js += "], \"probe_folds\": [";
    for (size_t i = 0; i < p->pgroups.size(); i++) {
      const vdl_probe_desc &d = p->pgroups[i]->b.desc;
      add("%s{\"table\": \"%s\", \"leaves\": %d, \"predicates\": %d, \"key_parts\": %d, \"domain\": %lld, \"folds\": %d, \"posts\": %d}", i ? ", " : "",
          p->tables[p->join->spaces[p->pgroups[i]->space].table].c_str(), d.nleaves, d.npreds, d.nkeys, (long long)d.domain, d.nfolds, d.nposts);
    }
    js += "], \"probe_emits\": [";
    for (size_t i = 0; i < p->egroups.size(); i++) {
      const vdl_probe_desc &d = p->egroups[i]->b.desc;
      add("%s{\"table\": \"%s\", \"leaves\": %d, \"predicates\": %d, \"vectors\": %d}", i ? ", " : "",
          p->tables[p->join->spaces[p->egroups[i]->space].table].c_str(), d.nleaves, d.npreds, d.nemits);
    }
    js += "], \"map_clusters\": [";
    for (size_t i = 0; i < p->clusters.size(); i++) {
      const MapCluster &c = p->clusters[i];
      add("%s{\"nodes\": %d, \"inputs\": %d, \"tables\": %d, \"instructions\": %d}", i ? ", " : "", (int)c.members.size(), c.desc.ninputs, c.desc.ntables, c.desc.ninstrs);
    }
    int folds_left = 0;
    for (size_t i = 0; i < p->nodes.size(); i++)
      if (p->nodes[i].op == N_FOLD && p->group_of_node[i] < 0 && p->pgroup_of_node[i] < 0) folds_left++;
    add("], \"folds_op_at_a_time\": %d, \"mergeable_tail\": %s}", folds_left, p->tail_ok ? "true" : "false");
  }
  vdl_plan_destroy(p);
  delete ctx;
  if ((int)js.size() + 1 > capacity) return VDL_ENOMEM;
  memcpy(out, js.c_str(), js.size() + 1);
  return rc;
}

extern "C" int vdl_plan_stats(vdl_plan *p, int *statements, int *nodes, int *fused_scans, int64_t *launches) {
  if (!p) return VDL_EINVAL;
  if (statements) *statements = p->statements;
  if (nodes) *nodes = (int)p->nodes.size();
  if (fused_scans) *fused_scans = (int)p->groups.size();
  if (launches) *launches = p->launches_last;
  return VDL_OK;
}

extern "C" int vdl_plan_probe_stats(vdl_plan *p, int *fold_groups, int *emit_groups, int *emitted_vectors) {
  if (!p) return VDL_EINVAL;
  if (fold_groups) *fold_groups = (int)p->pgroups.size();
  if (emit_groups) *emit_groups = (int)p->egroups.size();
  int n = 0;
  for (auto *g : p->egroups) n += (int)g->nodes.size();
  if (emitted_vectors) *emitted_vectors = n;
  return VDL_OK;
}

// The table whose rows probe emit group `group` walks (its fact side).  A row-range sharded run is only meaningful when that
// is the sharded table: a pass over a replicated dimension table would emit the same survivors on every rank.
extern "C" int vdl_plan_emit_group_table(vdl_plan *p, int group, const char **table) {
  if (!p || !table || group < 0 || group >= (int)p->egroups.size() || !p->join) return VDL_EINVAL;
  const int space = p->egroups[group]->space;
  if (space < 0 || space >= (int)p->join->spaces.size()) return VDL_EINVAL;
  const int t = p->join->spaces[space].table;
  if (t < 0 || t >= (int)p->tables.size()) return VDL_EINVAL;
  *table = p->tables[t].c_str();
  return VDL_OK;
}

extern "C" int vdl_plan_map_stats(vdl_plan *p, int *clusters, int *nodes_covered) {
  if (!p) return VDL_EINVAL;
  if (clusters) *clusters = (int)p->clusters.size();
  int n = 0;
  for (auto &c : p->clusters) n += (int)c.members.size();
  if (nodes_covered) *nodes_covered = n;
  return VDL_OK;
}

// Sum of the probe kernels' durations in the last run (CUDA events on the context stream); synchronises.
extern "C" int vdl_plan_probe_kernel_ms(vdl_plan *p, float *ms) {
  if (!p || !ms) return VDL_EINVAL;
  *ms = 0;
  for (auto *g : p->pgroups) if (g->probe) { float t = 0; VDL_TRY(vdl_probe_last_kernel_ms(g->probe, &t)); *ms += t; }
  for (auto *g : p->egroups) if (g->probe) { float t = 0; VDL_TRY(vdl_probe_last_kernel_ms(g->probe, &t)); *ms += t; }
  return VDL_OK;
}

// Mean and minimum, over the last n runs, of the plan's dominant-kernel time: the first fused scan's kernel, or else the
// sum over the probe passes -- from event pairs the library records around every launch, read after a timed loop.
extern "C" int vdl_plan_kernel_ms_stats(vdl_plan *p, int n, float *mean_ms, float *min_ms) {
  if (!p || n < 1) return VDL_EINVAL;
  if (!p->groups.empty()) {
    if (!p->groups[0].fused) return vdl_fail(p->ctx, VDL_EINVAL, "plan has not run yet");
    return vdl_fused_kernel_ms_stats(p->groups[0].fused, n, mean_ms, min_ms);
  }
  float mean = 0, mn = 0;
  for (auto *g : p->pgroups) if (g->probe) { float a = 0, b = 0; VDL_TRY(vdl_probe_kernel_ms_stats(g->probe, n, &a, &b)); mean += a; mn += b; }
  for (auto *g : p->egroups) if (g->probe) { float a = 0, b = 0; VDL_TRY(vdl_probe_kernel_ms_stats(g->probe, n, &a, &b)); mean += a; mn += b; }
  if (mean_ms) *mean_ms = mean;
  if (min_ms) *min_ms = mn;
  return VDL_OK;
}

extern "C" int vdl_plan_set_row_base(vdl_plan *p, int64_t row_base) {
  if (!p) return VDL_EINVAL;
  p->row_base = row_base;
  return VDL_OK;
}

// A freshly prepared scan or probe takes the peers set on the plan and continues its predecessor's step count.
static int reapply_peers(PeerState &ps, FoldCombine *cb) {
  if (ps.world < 1) return VDL_OK;
  VDL_TRY(cb->set_peers(ps.rank, ps.world, ps.buffers.data()));
  cb->xd.epoch = ps.epoch;
  return VDL_OK;
}

static int plan_run_local(vdl_plan *p, int self_finalize) {
  if (!p) return VDL_EINVAL;
  vdl_ctx *ctx = p->ctx;
  free_temps(p);
  i64 l0 = ctx->launches;
  for (auto &g : p->groups) {
    std::vector<vdl_vec> h(g.cols.size());
    i64 rows = -1;
    for (size_t c = 0; c < g.cols.size(); c++) {
      VDL_TRY(vdl_column_lookup(ctx, p->nodes[g.cols[c]].name.c_str(), &h[c]));
      i64 len; VDL_TRY(vdl_vec_len(ctx, h[c], &len));
      if (rows >= 0 && len != rows)
        return vdl_fail(ctx, VDL_EINVAL, "columns of table %s differ in length (%lld vs %lld)", p->tables[g.table].c_str(), (long long)len, (long long)rows);
      rows = len;
    }
    // (re)prepare when the binding changed OR a bound column was written since (new write generation): the scan's
    // int32-narrowing / 32-bit-accumulator / static-shape proofs come from statistics of the data it was prepared on
    if (!g.fused || !vdl_fused_current(g.fused) || h != g.bound || rows != g.bound_rows || p->row_base != g.bound_base) {
      if (g.fused) { g.peer.epoch = vdl_fused_combine(g.fused)->xd.epoch; vdl_fused_destroy(g.fused); g.fused = nullptr; }
      g.desc.rows = rows;
      g.desc.row_base = p->row_base;
      for (size_t c = 0; c < h.size(); c++) g.desc.column[c] = h[c];
      VDL_TRY(vdl_fused_prepare(ctx, &g.desc, &g.fused));
      g.bound = h; g.bound_rows = rows; g.bound_base = p->row_base;
      VDL_TRY(reapply_peers(g.peer, vdl_fused_combine(g.fused)));
    }
    VDL_TRY(vdl_fused_launch_ex(g.fused, self_finalize && g.peer.world > 0 ? 2 : self_finalize));
  }
  for (auto *g : p->pgroups) {
    vdl_probe *before = g->probe;
    if (before) g->peer.epoch = vdl_probe_combine(before)->xd.epoch;   // (read before a re-prepare destroys the probe)
    VDL_TRY(bind_probe(p, &g->b, &g->probe, &g->bound, &g->bound_rows, &g->bound_base));
    if (g->probe != before) VDL_TRY(reapply_peers(g->peer, vdl_probe_combine(g->probe)));
    VDL_TRY(vdl_probe_run_ex(g->probe, self_finalize && g->peer.world > 0 ? 2 : self_finalize));
  }
  if (!self_finalize)        // sharded run: the survivors' vectors are exchanged between ranks before the tail is evaluated
    for (auto *g : p->egroups) VDL_TRY(run_emit_group(p, *g));
  p->launches_last = ctx->launches - l0;
  p->local_done = true;
  p->self_finalized = self_finalize != 0;
  return VDL_OK;
}

extern "C" int vdl_plan_run_local(vdl_plan *p) { return plan_run_local(p, 0); }
// The launches of vdl_plan_run without the wait: asynchronous on the context's stream; vdl_plan_finish(p, NULL, 1) awaits
// the results.  With peers set (vdl_plan_set_peers) every rank's launches must be issued before any rank is awaited.
extern "C" int vdl_plan_launch(vdl_plan *p) { return plan_run_local(p, 1); }

extern "C" int vdl_plan_num_fused(vdl_plan *p) { return p ? (int)p->groups.size() : 0; }
extern "C" int vdl_plan_fused(vdl_plan *p, int i, vdl_fused **out) {
  if (!p || !out || i < 0 || i >= (int)p->groups.size()) return VDL_EINVAL;
  *out = p->groups[i].fused;
  return *out ? VDL_OK : vdl_fail(p->ctx, VDL_EINVAL, "plan has not run yet");
}

// Partial table i of the plan, in the order of vdl_plan_partials: fused scans first, then probe fold groups.  *cb is the
// combine of its prepared scan or probe, null before the plan has run.
static PeerState *plan_partial(vdl_plan *p, int i, FoldCombine **cb) {
  if (i < (int)p->groups.size()) {
    FusedGroup &g = p->groups[i];
    *cb = g.fused ? vdl_fused_combine(g.fused) : nullptr;
    return &g.peer;
  }
  ProbeFoldGroup *g = p->pgroups[i - p->groups.size()];
  *cb = g->probe ? vdl_probe_combine(g->probe) : nullptr;
  return &g->peer;
}

extern "C" int vdl_plan_exchange_bytes(vdl_plan *p, int index, int world, int64_t *bytes) {
  if (!p || index < 0 || index >= vdl_plan_num_partials(p)) return VDL_EINVAL;
  FoldCombine *cb;
  plan_partial(p, index, &cb);
  if (!cb) return vdl_fail(p->ctx, VDL_EINVAL, "plan has not run yet");
  return cb->exchange_bytes(world, bytes);
}

extern "C" int vdl_plan_set_peers(vdl_plan *p, int index, int rank, int world, void *const *peer_buffers) {
  if (!p || index < 0 || index >= vdl_plan_num_partials(p) || !peer_buffers || world < 1 || world > VDL_MAX_RANKS) return VDL_EINVAL;
  FoldCombine *cb;
  PeerState &ps = *plan_partial(p, index, &cb);
  ps.rank = rank; ps.world = world;
  ps.buffers.assign(peer_buffers, peer_buffers + world);
  ps.epoch = 0;
  return cb ? cb->set_peers(rank, world, ps.buffers.data()) : VDL_OK;
}

// ---- vectors emitted by probe passes, for the exchange of survivors in a sharded run --------------------------------
static bool emit_slot(vdl_plan *p, int i, EmitGroup **g, int *k) {
  for (auto *q : p->egroups) {
    if (i < (int)q->nodes.size()) { *g = q; *k = i; return true; }
    i -= (int)q->nodes.size();
  }
  return false;
}
extern "C" int vdl_plan_num_emits(vdl_plan *p) {
  int n = 0;
  if (p) for (auto *g : p->egroups) n += (int)g->nodes.size();
  return n;
}
extern "C" int vdl_plan_emit(vdl_plan *p, int i, void **device_ptr, int64_t *len) {
  EmitGroup *g; int k;
  if (!p || !device_ptr || !len || !emit_slot(p, i, &g, &k)) return VDL_EINVAL;
  if (!g->ran) return vdl_fail(p->ctx, VDL_EINVAL, "emitted vectors exist after vdl_plan_run_local");
  Vec *v = vec_get(p->ctx, p->val[g->nodes[k]]);
  if (!v) return VDL_EINVAL;
  *device_ptr = v->ptr;
  *len = v->len;
  return VDL_OK;
}
// Substitute emitted vector i by caller-owned device memory (the concatenation of all ranks' survivors, in rank order
// = global row order); it must stay valid until vdl_plan_finish returns.
extern "C" int vdl_plan_emit_replace(vdl_plan *p, int i, void *device_ptr, int64_t len) {
  EmitGroup *g; int k;
  if (!p || len < 0 || (len > 0 && !device_ptr) || !emit_slot(p, i, &g, &k)) return VDL_EINVAL;
  if (!g->ran) return vdl_fail(p->ctx, VDL_EINVAL, "emitted vectors exist after vdl_plan_run_local");
  vdl_vec h;
  VDL_TRY(vec_new_range(p->ctx, 0, 0, 0, &h));
  Vec &v = p->ctx->vecs[h];
  v.is_range = false; v.ptr = device_ptr; v.dtype = VDL_I64; v.len = len; v.cap_rows = len; v.owned = false; v.domain = -1;
  p->val[g->nodes[k]] = h;          // the local vector stays in temps and is released with them
  p->temps.push_back(h);
  return VDL_OK;
}

extern "C" int vdl_plan_num_partials(vdl_plan *p) { return p ? (int)(p->groups.size() + p->pgroups.size()) : 0; }
extern "C" int vdl_plan_partials(vdl_plan *p, int i, void **device_ptr, int64_t *n_int64) {
  if (!p || i < 0 || i >= vdl_plan_num_partials(p)) return VDL_EINVAL;
  FoldCombine *cb;
  plan_partial(p, i, &cb);
  if (!cb) return vdl_fail(p->ctx, VDL_EINVAL, "plan has not run yet");
  return cb->partials(device_ptr, n_int64);
}

extern "C" int vdl_plan_finish(vdl_plan *p, const void *const *all_partials, int nranks) {
  if (!p) return VDL_EINVAL;
  vdl_ctx *ctx = p->ctx;
  if (!p->local_done) return vdl_fail(ctx, VDL_EINVAL, "vdl_plan_finish before vdl_plan_run_local");
  p->trace = getenv("VDL_TRACE") != nullptr;
  if (p->trace) p->trace_t0 = p->trace_last = now_ms();
  if (nranks > 1 && p->groups.empty() && p->pgroups.empty() && p->egroups.empty())
    return vdl_fail(ctx, VDL_EUNSUPPORTED, "a plan without a fused scan or a probe pass cannot be row-sharded");
  i64 l0 = ctx->launches;
  if (!(p->self_finalized && nranks == 1 && !all_partials)) {
    for (int i = 0; i < vdl_plan_num_partials(p); i++) {
      FoldCombine *cb;
      plan_partial(p, i, &cb);
      if (!cb) return vdl_fail(ctx, VDL_EINVAL, "plan has not run yet");
      VDL_TRY(cb->finalize(all_partials ? all_partials[i] : nullptr, nranks));
    }
  }
  bool ran_ops = false, copies_pending = false, collated = false;
  const bool ordered = !p->order_key.empty() || p->order_limit >= 0;
  std::vector<vdl_vec> dev(p->outputs.size(), 0);    // ordered: the device value of every op-at-a-time output
  // the device -> host copy of op-at-a-time output o, whose value is v
  auto deliver = [&](Output &o, vdl_vec v) -> int {
    i64 len;
    VDL_TRY(vdl_vec_len(ctx, v, &len));
    if ((size_t)len > o.cap) {              // pinned, so the copy is one DMA at PCIe rate
      int rc = reserve_pinned(ctx, o, len);
      if (rc) { free_temps(p); return rc; }
    }
    Vec *vv = vec_get(ctx, v);
    o.dtype = 8;
    if (p->typed_outputs && vv && !vv->is_range && vv->dtype == VDL_I64 && vv->narrow32 && len > 0) {
      // every value is a value of a 4-byte column: half the bytes over PCIe (a narrowing kernel, then the same async copy)
      vdl_vec nv;
      int rc = vec_narrow_copy(ctx, v, &nv);
      if (rc) { if (copies_pending) cudaStreamSynchronize(ctx->copy_stream); free_temps(p); return rc; }
      p->temps.push_back(nv);
      VDL_CUDA(ctx, cudaEventRecord(ctx->copy_event, ctx->stream));
      VDL_CUDA(ctx, cudaStreamWaitEvent(ctx->copy_stream, ctx->copy_event, 0));
      VDL_CUDA(ctx, cudaMemcpyAsync(o.pinned, vec_get(ctx, nv)->ptr, (size_t)len * 4, cudaMemcpyDeviceToHost, ctx->copy_stream));
      copies_pending = true;
      o.dtype = 4;
    } else if (vv && !vv->is_range && vv->dtype == VDL_I64 && len > 0) {
      // the copy runs on its own stream behind an event, so the next output's kernels overlap it; one wait at the end
      VDL_CUDA(ctx, cudaEventRecord(ctx->copy_event, ctx->stream));
      VDL_CUDA(ctx, cudaStreamWaitEvent(ctx->copy_stream, ctx->copy_event, 0));
      VDL_CUDA(ctx, cudaMemcpyAsync(o.pinned, vv->ptr, (size_t)len * 8, cudaMemcpyDeviceToHost, ctx->copy_stream));
      copies_pending = true;
    } else {
      int rc = vdl_vec_download(ctx, v, o.pinned, len);
      if (rc) { if (copies_pending) cudaStreamSynchronize(ctx->copy_stream); free_temps(p); return rc; }
    }
    o.data = o.pinned; o.len = len;
    return VDL_OK;
  };
  for (size_t oi = 0; oi < p->outputs.size(); oi++) {
    Output &o = p->outputs[oi];
    int gi = p->group_of_node[o.node];
    if (p->pgroup_of_node[o.node] >= 0) {   // a Fold over a joined space: the probe's result buffer is already on its way
      ProbeFoldGroup &g = *p->pgroups[p->pgroup_of_node[o.node]];
      const int64_t *data; int64_t len;
      const int idx = p->nodes[o.node].op == N_FOLD ? g.fold_of_node[o.node] : g.b.desc.nfolds + g.post_of_node[o.node];
      VDL_TRY(vdl_probe_result_host(g.probe, idx, &data, &len));
      o.data = data; o.len = len; o.dtype = 8;
      continue;
    }
    if (gi >= 0) {   // the output IS a fused fold or a post op of one: it arrived with the scan's single result copy
      const int64_t *data; int64_t len;
      if (p->nodes[o.node].op == N_FOLD) VDL_TRY(vdl_fused_result_host(p->groups[gi].fused, p->groups[gi].fold_of_node[o.node], &data, &len));
      else VDL_TRY(vdl_fused_post_host(p->groups[gi].fused, p->groups[gi].post_of_node[o.node], &data, &len));
      o.data = data; o.len = len; o.dtype = 8;
      continue;
    }
    ran_ops = true;
    vdl_vec v;
    int rc = eval(p, o.node, &v);
    if (rc) { if (copies_pending) cudaStreamSynchronize(ctx->copy_stream); free_temps(p); return rc; }
    if (ordered) { dev[oi] = v; continue; }
    VDL_TRY(deliver(o, v));
  }
  if (ordered) {
    // ORDER BY / LIMIT: one permutation of the rows, computed over the key outputs, applied to every output before its copy
    int rc = VDL_OK;
    const size_t no = p->outputs.size();
    std::vector<i64> len(no, 0);
    for (size_t i = 0; i < no && !rc; i++) {
      if (dev[i]) rc = vdl_vec_len(ctx, dev[i], &len[i]);
      else len[i] = p->outputs[i].len;
      if (!rc && len[i] != len[0])
        rc = vdl_fail(ctx, VDL_EINVAL, "ORDER BY / LIMIT needs outputs of one length: %s has %lld rows, %s has %lld", p->outputs[0].name.c_str(),
                      (long long)len[0], p->outputs[i].name.c_str(), (long long)len[i]);
    }
    const i64 n = no ? len[0] : 0;
    std::vector<vdl_vec> keys(p->order_key.size(), 0);
    for (size_t k = 0; k < keys.size() && !rc; k++) {
      const int i = p->order_key[k];
      if (dev[i]) { keys[k] = dev[i]; continue; }
      // a host-resident result (fused scan, probe fold): its key values go back to the device for the order; the result
      // buffer itself is shared by the scan's / probe's outputs and stays as it is
      rc = vec_new(ctx, VDL_I64, n, &keys[k]);
      if (rc) break;
      p->temps.push_back(keys[k]);
      if (n > 0) {
        const cudaError_t e = cudaMemcpyAsync(ctx->vecs[keys[k]].ptr, p->outputs[i].data, (size_t)n * 8, cudaMemcpyHostToDevice, ctx->stream);
        if (e != cudaSuccess) rc = vdl_cuda_fail(ctx, e, "ORDER BY key upload");
      }
    }
    for (size_t k = 0; k < keys.size() && !rc; k++) {
      if (!p->order_heap[k]) continue;
      // a string key: its values (heap offsets or dictionary codes) are replaced by their collation ranks for the order
      // only; the output itself keeps them
      vdl_vec r;
      rc = vdl_op_collate(ctx, keys[k], p->order_heap[k], p->order_origin[k], &r);
      if (rc) break;
      p->temps.push_back(r);
      keys[k] = r;
      collated = true;
    }
    vdl_vec perm = 0;
    if (!rc) {
      const i64 limit = keys.empty() ? std::min<i64>(p->order_limit, n) : p->order_limit;
      rc = vdl_op_order(ctx, (int)keys.size(), keys.data(), p->order_desc.data(), limit, &perm);
      if (!rc) p->temps.push_back(perm);
    }
    i64 m = 0;
    if (!rc) rc = vdl_vec_len(ctx, perm, &m);
    std::vector<i64> hperm;                 // the permutation on the host, for host-resident results
    for (size_t i = 0; i < no && !rc; i++) {
      Output &o = p->outputs[i];
      if (dev[i]) {
        vdl_vec g;
        rc = vdl_op_gather(ctx, dev[i], perm, &g);     // (keeps narrow32: typed outputs still travel as int32)
        if (rc) break;
        p->temps.push_back(g);
        rc = deliver(o, g);
        if (rc) return rc;
        continue;
      }
      if (keys.empty()) { o.len = m; continue; }          // LIMIT alone: the first m rows, in place
      if (hperm.empty() && m > 0) {
        hperm.resize((size_t)m);
        rc = vdl_vec_download(ctx, perm, hperm.data(), m);
        if (rc) break;
      }
      if ((size_t)m > o.cap && (rc = reserve_pinned(ctx, o, m))) break;
      for (i64 j = 0; j < m; j++) o.pinned[j] = o.data[hperm[j]];
      o.data = o.pinned; o.len = m; o.dtype = 8;
    }
    if (rc) { if (copies_pending) cudaStreamSynchronize(ctx->copy_stream); free_temps(p); return rc; }
  }
  if (copies_pending) VDL_CUDA(ctx, cudaStreamSynchronize(ctx->copy_stream));     // before the temporaries are released
  int rc = ran_ops || collated ? check_errflag(ctx, "plan") : VDL_OK;
  if (!rc && p->tail_on && p->tail_ok) rc = capture_tail_boundary(p);
  p->launches_last += ctx->launches - l0;
  free_temps(p);
  p->local_done = false;
  return rc;
}

// ---- sharded tail ---------------------------------------------------------------------------------------------------
extern "C" int vdl_plan_tail_info(vdl_plan *p, int *mergeable, int *fold_ops, int cap) {
  if (!p || !mergeable) return VDL_EINVAL;
  *mergeable = p->tail_ok ? 1 : 0;
  if (p->tail_ok && fold_ops)
    for (int i = 0; i < cap && i < (int)p->outputs.size(); i++) fold_ops[i] = p->nodes[p->outputs[i].node].sub;
  return VDL_OK;
}
extern "C" int vdl_plan_tail_enable(vdl_plan *p, int on) {
  if (!p) return VDL_EINVAL;
  if (on && !p->tail_ok) return vdl_fail(p->ctx, VDL_EUNSUPPORTED, "the plan's outputs are not Folds by runs of one groups vector");
  if (on && (!p->order_key.empty() || p->order_limit >= 0))
    return vdl_fail(p->ctx, VDL_EUNSUPPORTED, "the sharded tail leaves each rank a slice of the result, which an ORDER BY / LIMIT cannot be applied to");
  p->tail_on = on != 0;
  return VDL_OK;
}
extern "C" int vdl_plan_set_order(vdl_plan *p, int nkeys, const int *key_output, const int *descending, int64_t limit) {
  if (!p || nkeys < 0 || (nkeys > 0 && !key_output)) return VDL_EINVAL;
  if (nkeys > VDL_MAX_ORDER_KEYS) return vdl_fail(p->ctx, VDL_EINVAL, "ORDER BY: %d keys (at most %d)", nkeys, VDL_MAX_ORDER_KEYS);
  for (int k = 0; k < nkeys; k++)
    if (key_output[k] < 0 || key_output[k] >= (int)p->outputs.size())
      return vdl_fail(p->ctx, VDL_EINVAL, "ORDER BY key %d: output %d out of range (the plan has %d outputs)", k, key_output[k], (int)p->outputs.size());
  if ((nkeys > 0 || limit >= 0) && p->tail_on)
    return vdl_fail(p->ctx, VDL_EUNSUPPORTED, "the sharded tail leaves each rank a slice of the result, which an ORDER BY / LIMIT cannot be applied to");
  p->order_key.assign(key_output, key_output + nkeys);
  p->order_desc.assign(nkeys, 0);
  for (int k = 0; k < nkeys && descending; k++) p->order_desc[k] = descending[k] ? 1 : 0;
  p->order_limit = limit < 0 ? -1 : limit;
  p->order_heap.assign(nkeys, 0);
  p->order_origin.assign(nkeys, 0);
  return VDL_OK;
}
extern "C" int vdl_plan_set_order_heap(vdl_plan *p, int key, vdl_vec heap, int64_t origin) {
  if (!p) return VDL_EINVAL;
  if (key < 0 || key >= (int)p->order_key.size())
    return vdl_fail(p->ctx, VDL_EINVAL, "ORDER BY key %d out of range (the order has %d keys)", key, (int)p->order_key.size());
  if (heap) {
    Vec *vh = vec_get_any(p->ctx, heap);
    if (!vh) return VDL_EINVAL;
    if (vh->dtype != VDL_U8) return vdl_fail(p->ctx, VDL_EINVAL, "ORDER BY key %d: vector %d is not a string heap (VDL_U8)", key, (int)heap);
  }
  p->order_heap[key] = heap;
  p->order_origin[key] = heap ? origin : 0;
  return VDL_OK;
}
extern "C" int vdl_plan_tail_boundary(vdl_plan *p, int64_t *rec, int cap) {
  if (!p || !rec) return VDL_EINVAL;
  if (!p->tail_on) return vdl_fail(p->ctx, VDL_EINVAL, "vdl_plan_tail_enable first");
  const int k = (int)p->outputs.size();
  if (cap < 4 + 2 * k) return vdl_fail(p->ctx, VDL_EINVAL, "tail record needs %d values", 4 + 2 * k);
  for (int i = 0; i < 4; i++) rec[i] = p->tail_rec[i];
  const i64 runs = p->tail_rec[1];
  for (int i = 0; i < k; i++) {
    const Output &o = p->outputs[i];
    if ((i64)o.len != runs) return vdl_fail(p->ctx, VDL_EINVAL, "sharded tail: output %d has %lld values, the first has %lld", i, (long long)o.len, (long long)runs);
    rec[4 + i] = runs ? out_get(o, 0) : 0;
    rec[4 + k + i] = runs ? out_get(o, runs - 1) : 0;
  }
  return VDL_OK;
}
// The outcome of the boundary merge for this rank: replace the last row of every output (last_row != NULL) and / or give
// up the first row (it continues a group that starts on an earlier rank).  vdl_plan_output then returns the rank's slice.
extern "C" int vdl_plan_tail_apply(vdl_plan *p, int drop_first, const int64_t *last_row) {
  if (!p) return VDL_EINVAL;
  if (!p->tail_on) return vdl_fail(p->ctx, VDL_EINVAL, "vdl_plan_tail_enable first");
  for (size_t i = 0; i < p->outputs.size(); i++) {
    Output &o = p->outputs[i];
    if (o.len == 0 || o.data != o.pinned) continue;
    if (last_row) {
      if (o.dtype == 4) ((int *)o.pinned)[o.len - 1] = (int)last_row[i];      // CHOOSE / MIN / MAX of int32 values stay int32
      else o.pinned[o.len - 1] = last_row[i];
    }
    if (drop_first) { o.data = o.dtype == 4 ? (const i64 *)((const int *)o.pinned + 1) : o.pinned + 1; o.len -= 1; }
  }
  return VDL_OK;
}

extern "C" int vdl_plan_run(vdl_plan *p) {
  VDL_TRY(plan_run_local(p, 1));        // single GPU: every fused scan finalizes itself (one launch per scan)
  return vdl_plan_finish(p, nullptr, 1);
}

extern "C" int vdl_plan_num_outputs(vdl_plan *p) { return p ? (int)p->outputs.size() : 0; }
extern "C" int vdl_plan_output(vdl_plan *p, int i, const char **name, const int64_t **data, int64_t *len) {
  if (!p || i < 0 || i >= (int)p->outputs.size()) return VDL_EINVAL;
  if (data && p->outputs[i].dtype != 8) return vdl_fail(p->ctx, VDL_EINVAL, "output %d was delivered as int32 (typed outputs are on): read it with vdl_plan_output_typed", i);
  if (name) *name = p->outputs[i].name.c_str();
  if (data) *data = p->outputs[i].data;
  if (len) *len = (int64_t)p->outputs[i].len;
  return VDL_OK;
}
extern "C" int vdl_plan_set_typed_outputs(vdl_plan *p, int on) {
  if (!p) return VDL_EINVAL;
  p->typed_outputs = on != 0;
  return VDL_OK;
}
extern "C" int vdl_plan_output_typed(vdl_plan *p, int i, const char **name, const void **data, int64_t *len, int *dtype) {
  if (!p || i < 0 || i >= (int)p->outputs.size()) return VDL_EINVAL;
  if (name) *name = p->outputs[i].name.c_str();
  if (data) *data = p->outputs[i].data;
  if (len) *len = (int64_t)p->outputs[i].len;
  if (dtype) *dtype = p->outputs[i].dtype;
  return VDL_OK;
}

extern "C" int vdl_plan_destroy(vdl_plan *p) {
  if (!p) return VDL_EINVAL;
  free_temps(p);
  for (auto &g : p->groups) if (g.fused) vdl_fused_destroy(g.fused);
  for (auto &o : p->outputs) if (o.pinned) cudaFreeHost(o.pinned);
  for (auto *g : p->pgroups) { if (g->probe) vdl_probe_destroy(g->probe); delete g; }
  for (auto *g : p->egroups) { if (g->probe) vdl_probe_destroy(g->probe); delete g; }
  delete p->join;
  delete p;
  return VDL_OK;
}
