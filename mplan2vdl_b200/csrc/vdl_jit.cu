// Run-time compiled kernels: a generated source is compiled for sm_100a with NVRTC (dlopen'ed: the library has no
// link-time dependency on it) against the headers embedded in the library, loaded through the runtime's library API and
// cached per context.  The fused scan (vdl_fused.cu) and the FK-join probe (vdl_probe.cu) generate theirs; the one of
// vdl_op_map is generated here.
// vdl_op_map: for long vectors the register program is turned into straight-line CUDA C.  The interpreter in vdl_ops.cu
// spends ~15 issue slots per instruction and row on decoding and on its local-memory register file; the specialised kernel
// keeps every value in a register and is bound by the HBM reads of its inputs.  Both take MapArgs, op_ld and binop_apply
// from vdl_device.cuh: the generated source only spells the operands' storage kinds and the ops as literals.
#include <dlfcn.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <map>
#include <string>
#include <vector>

#include "vdl_internal.h"
#include "vdl_embedded.inc"      // the headers a generated source may include, as strings (written by build.py)

namespace {

typedef int (*nvrtcCreateProgram_t)(void **, const char *, const char *, int, const char *const *, const char *const *);
typedef int (*nvrtcCompileProgram_t)(void *, int, const char *const *);
typedef int (*nvrtcGetSize_t)(void *, size_t *);
typedef int (*nvrtcGetData_t)(void *, char *);
typedef int (*nvrtcDestroyProgram_t)(void **);

struct Nvrtc {
  bool tried = false, ok = false;
  nvrtcCreateProgram_t create = nullptr;
  nvrtcCompileProgram_t compile = nullptr;
  nvrtcGetSize_t cubin_size = nullptr, log_size = nullptr;
  nvrtcGetData_t cubin = nullptr, log = nullptr;
  nvrtcDestroyProgram_t destroy = nullptr;
};
Nvrtc g_nvrtc;

bool nvrtc_load() {
  Nvrtc &N = g_nvrtc;
  if (N.tried) return N.ok;
  N.tried = true;
  void *h = nullptr;
  for (const char *name : {"libnvrtc.so.12", "libnvrtc.so", "/usr/local/cuda/lib64/libnvrtc.so.12", "/usr/local/cuda/lib64/libnvrtc.so"})
    if ((h = dlopen(name, RTLD_NOW | RTLD_LOCAL))) break;
  if (!h) return false;
  N.create = (nvrtcCreateProgram_t)dlsym(h, "nvrtcCreateProgram");
  N.compile = (nvrtcCompileProgram_t)dlsym(h, "nvrtcCompileProgram");
  N.cubin_size = (nvrtcGetSize_t)dlsym(h, "nvrtcGetCUBINSize");
  N.cubin = (nvrtcGetData_t)dlsym(h, "nvrtcGetCUBIN");
  N.log_size = (nvrtcGetSize_t)dlsym(h, "nvrtcGetProgramLogSize");
  N.log = (nvrtcGetData_t)dlsym(h, "nvrtcGetProgramLog");
  N.destroy = (nvrtcDestroyProgram_t)dlsym(h, "nvrtcDestroyProgram");
  N.ok = N.create && N.compile && N.cubin_size && N.cubin && N.log_size && N.log && N.destroy;
  return N.ok;
}

struct JitCache {
  std::map<std::string, cudaKernel_t> kernels;   // nullptr: compilation failed before, do not retry
  std::vector<cudaLibrary_t> libs;
};

std::string generate(const MapArgs &m) {
  const vdl_map_desc &d = m.d;
  std::string s = "#include \"vdl_device.cuh\"\n__device__ __forceinline__ i64 row(const MapArgs &m, const i64 i, int *err) {\n";
  char b[512];
  // SSA over the register program: reg -> name of the value it currently holds
  std::vector<std::string> cur(VDL_MAP_MAX_REGS);
  for (int t = 0; t < d.ninstrs; t++) {
    const vdl_map_instr &ins = d.instr[t];
    const std::string v = "v" + std::to_string(t);
    if (ins.op == VDL_MAP_LOAD) {
      snprintf(b, sizeof b, "  const i64 %s = op_ld_k<%d>(m.in[%d], i);\n", v.c_str(), m.in[ins.b].kind, ins.b);
    } else if (ins.op == VDL_MAP_RANGE) {
      snprintf(b, sizeof b, "  const i64 %s = (i64)(%lluull + (u64)i * %lluull);\n", v.c_str(), (unsigned long long)d.imm[ins.a],
               (unsigned long long)d.imm[ins.b]);
    } else if (ins.op == VDL_MAP_GATHER) {
      const char *a = cur[ins.a].c_str();
      snprintf(b, sizeof b, "  i64 %s = 0;\n  if ((u64)%s >= (u64)m.tab_len[%d]) atomicAdd(err, 1); else %s = op_ld_k<%d>(m.tab[%d], %s);\n",
               v.c_str(), a, ins.b, v.c_str(), m.tab[ins.b].kind, ins.b, a);
    } else {
      snprintf(b, sizeof b, "  const i64 %s = binop_apply(%d, %s, %s);\n", v.c_str(), ins.op, cur[ins.a].c_str(), cur[ins.b].c_str());
    }
    s += b;
    cur[ins.dst] = v;
  }
  s += "  return " + cur[d.instr[d.ninstrs - 1].dst] + ";\n}\n";
  s += "extern \"C\" __global__ void __launch_bounds__(256) vdl_map_jit(const __grid_constant__ MapArgs m, i64 *__restrict__ out, const i64 n, int *err) {\n"
       "  const i64 stride = (i64)gridDim.x * 256;\n"
       "  i64 i = (i64)blockIdx.x * 256 + threadIdx.x;\n"
       "  for (; i + stride < n; i += 2 * stride) {\n"
       "    const i64 x = row(m, i, err), y = row(m, i + stride, err);\n"
       "    out[i] = x;\n    out[i + stride] = y;\n  }\n"
       "  if (i < n) out[i] = row(m, i, err);\n}\n";
  return s;
}

// Compile `src` and load its kernel `name`.  nullptr, after a message on stderr, when either fails.
cudaKernel_t compile_and_load(JitCache *jc, const std::string &src, const char *name) {
  std::string log;
  std::vector<char> cubin;
  int status = 0;
  if (vdl_jit_compile(src, &log, &cubin, &status) != VDL_OK) {
    fprintf(stderr, "[vdl jit] NVRTC failed (%d) for %s; the precompiled kernel runs instead.\n%s\n", status, name, log.c_str());
    if (getenv("VDL_DEBUG_JIT")) fprintf(stderr, "%s\n", src.c_str());
    return nullptr;
  }
  cudaLibrary_t lib = nullptr;
  cudaKernel_t k = nullptr;
  if (cudaLibraryLoadData(&lib, cubin.data(), nullptr, nullptr, 0, nullptr, nullptr, 0) != cudaSuccess ||
      cudaLibraryGetKernel(&k, lib, name) != cudaSuccess) {
    fprintf(stderr, "[vdl jit] loading the compiled kernel failed (%s); the interpreter runs instead.\n", cudaGetErrorString(cudaGetLastError()));
    if (lib) cudaLibraryUnload(lib);
    return nullptr;
  }
  jc->libs.push_back(lib);
  return k;
}

}  // namespace

int vdl_jit_compile(const std::string &src, std::string *log, std::vector<char> *cubin, int *status) {
  log->clear();
  if (!nvrtc_load()) return VDL_ENOTFOUND;
  // NVRTC reads only the headers the source includes
  static const char *const headers[] = {EMB_vdl_cuda_h, EMB_vdl_device_cuh, EMB_vdl_fused_kernel_cuh, EMB_vdl_probe_kernel_cuh};
  static const char *const names[] = {"vdl_cuda.h", "vdl_device.cuh", "vdl_fused_kernel.cuh", "vdl_probe_kernel.cuh"};
  Nvrtc &N = g_nvrtc;
  void *prog = nullptr;
  int rc = N.create(&prog, src.c_str(), "vdl_jit.cu", 4, headers, names);
  if (status) *status = rc;
  if (rc != 0) return VDL_ECUDA;
  // -default-device: the public header's (unannotated) function declarations are only declarations here
  const char *opts[] = {"--gpu-architecture=sm_100a", "--std=c++17", "-lineinfo", "-default-device"};
  rc = N.compile(prog, 4, opts);
  if (status) *status = rc;
  size_t ls = 0, cs = 0;
  N.log_size(prog, &ls);
  if (ls > 1) {
    log->resize(ls);
    N.log(prog, &(*log)[0]);
    log->resize(ls - 1);                           // without the terminating NUL
  }
  if (rc == 0) N.cubin_size(prog, &cs);
  if (cubin && cs > 0) {
    cubin->resize(cs);
    N.cubin(prog, cubin->data());
  }
  N.destroy(&prog);
  return rc == 0 && cs > 0 ? VDL_OK : VDL_ECUDA;
}

cudaKernel_t vdl_jit_kernel(vdl_ctx *ctx, const std::string &key, const char *name, size_t smem, const std::function<std::string()> &source) {
  if (!nvrtc_load()) return nullptr;
  if (!ctx->jit) ctx->jit = new JitCache();
  JitCache *jc = (JitCache *)ctx->jit;
  auto it = jc->kernels.find(key);
  if (it == jc->kernels.end()) it = jc->kernels.emplace(key, compile_and_load(jc, source(), name)).first;
  if (it->second && smem > 48 * 1024 &&
      cudaFuncSetAttribute((const void *)it->second, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) {
    cudaGetLastError();
    return nullptr;
  }
  return it->second;
}

// Launches the specialised kernel for `m` on the context's stream.  Returns 1 when it did, 0 when the caller should run
// the interpreter (NVRTC missing, compilation failed, VDL_NO_JIT), negative on a launch error.
int vdl_jit_map_launch(vdl_ctx *ctx, const MapArgs &m, i64 *out, i64 n, int blocks) {
  if (getenv("VDL_NO_JIT")) return 0;
  // key: everything the generated source depends on (the program, its immediates, the operands' storage kinds)
  std::string key = "map|";
  key.append((const char *)&m.d, 4 * sizeof(int32_t));
  key.append((const char *)m.d.instr, (size_t)m.d.ninstrs * sizeof(vdl_map_instr));
  key.append((const char *)m.d.imm, (size_t)m.d.nimms * sizeof(int64_t));
  for (int k = 0; k < m.d.ninputs; k++) key.push_back((char)m.in[k].kind);
  for (int k = 0; k < m.d.ntables; k++) key.push_back((char)m.tab[k].kind);
  cudaKernel_t kh = vdl_jit_kernel(ctx, key, "vdl_map_jit", 0, [&] {
    if (getenv("VDL_DEBUG_JIT")) fprintf(stderr, "[vdl jit] compiling a %d-instruction map program\n", m.d.ninstrs);
    return generate(m);
  });
  if (!kh) return 0;
  int *err = ctx->d_errflag;
  void *args[] = {(void *)&m, (void *)&out, (void *)&n, (void *)&err};
  cudaError_t e = cudaLaunchKernel((const void *)kh, dim3(blocks), dim3(256), args, 0, ctx->stream);
  if (e != cudaSuccess) { vdl_cuda_fail(ctx, e, "launch of a specialised map kernel"); return -1; }
  return 1;
}

// Host-only self-test (no GPU needed): print a program that uses every instruction kind and storage kind as CUDA C and
// compile it with NVRTC for sm_100a.  0 = compiled; VDL_ENOTFOUND = NVRTC not present on this machine; VDL_ECUDA =
// NVRTC rejected the source (the log is copied to `log`).
extern "C" int vdl_jit_selftest(char *log, int log_capacity) {
  if (log && log_capacity > 0) log[0] = 0;
  MapArgs m;
  memset(&m, 0, sizeof m);
  vdl_map_desc &d = m.d;
  d.ninputs = 3; d.ntables = 2; d.nimms = 2;
  d.imm[0] = -5; d.imm[1] = 3;
  m.in[0].kind = 0; m.in[1].kind = 1; m.in[2].kind = 2;
  m.tab[0].kind = 0; m.tab[1].kind = 1;
  int t = 0;
  for (int k = 0; k < 3; k++) d.instr[t++] = vdl_map_instr{VDL_MAP_LOAD, (int16_t)k, 0, (int16_t)k};
  d.instr[t++] = vdl_map_instr{VDL_MAP_RANGE, 3, 0, 1};
  for (int op = VDL_LOGICAL_AND; op <= VDL_MODULO; op++) d.instr[t++] = vdl_map_instr{(int16_t)op, (int16_t)(4 + op % 2), (int16_t)(op % 4), (int16_t)((op + 1) % 4)};
  d.instr[t++] = vdl_map_instr{VDL_MAP_GATHER, 6, 4, 0};
  d.instr[t++] = vdl_map_instr{VDL_MAP_GATHER, 7, 5, 1};
  d.instr[t++] = vdl_map_instr{VDL_ADD, 6, 6, 7};
  d.ninstrs = t;
  std::string l;
  const int rc = vdl_jit_compile(generate(m), &l);
  if (log && log_capacity > 1) snprintf(log, (size_t)log_capacity, "%s", l.c_str());
  return rc;
}

void vdl_jit_destroy(vdl_ctx *ctx) {
  if (!ctx->jit) return;
  JitCache *jc = (JitCache *)ctx->jit;
  for (auto l : jc->libs) cudaLibraryUnload(l);
  delete jc;
  ctx->jit = nullptr;
}
