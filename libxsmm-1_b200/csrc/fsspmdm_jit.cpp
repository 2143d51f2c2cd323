// Create-time kernel baking for FSSPMDM.  Default: the kernel is emitted as PTX text and assembled by the
// driver (cudaLibraryLoadData).  Alternative (LIBXSMM_B200_FSSPMDM_JIT=nvrtc): CUDA C++ compiled by NVRTC, loaded
// lazily with dlopen so that the library itself loads on machines without a CUDA toolkit.  On any failure
// create() falls back to the generic kernel and records the reason.
#include "fsspmdm_jit.h"
#include "common.cuh"
#include <cuda.h>
#include <nvrtc.h>
#include <dlfcn.h>
#include <cstdio>
#include <cstdint>
#include <cstdarg>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>
#include <algorithm>
#include <map>
#include <mutex>

namespace xb {

struct FsJit {
  cudaLibrary_t lib;
  cudaKernel_t kern;
  int cols_per_thread;  // 1, or 2 (float, even pitches: 8-byte accesses)
  int block;
  // strip form (operators whose B rows do not fit the register file): a CTA stages K x 32 columns of B in shared memory by TMA
  int batched;          // 1: (element, column) form with strides (fs_jit_launch_batched)
  int strip;            // 0: register form
  int esz, krows, box_rows, strip_w;
  size_t smem;
};

bool make_tensor_map_2d(CUtensorMap* map, const void* base, int elem_bytes, unsigned long long cols, unsigned long long rows,
                        unsigned long long row_pitch_bytes, unsigned box_cols, unsigned box_rows);

namespace {

struct Nvrtc {
  void* h;
  nvrtcResult (*CreateProgram)(nvrtcProgram*, const char*, const char*, int, const char* const*, const char* const*);
  nvrtcResult (*CompileProgram)(nvrtcProgram, int, const char* const*);
  nvrtcResult (*GetCUBINSize)(nvrtcProgram, size_t*);
  nvrtcResult (*GetCUBIN)(nvrtcProgram, char*);
  nvrtcResult (*GetProgramLogSize)(nvrtcProgram, size_t*);
  nvrtcResult (*GetProgramLog)(nvrtcProgram, char*);
  nvrtcResult (*DestroyProgram)(nvrtcProgram*);
};

Nvrtc* nvrtc()
{
  static Nvrtc api;
  static int state = 0;   // 0 unknown, 1 ok, -1 unavailable
  static std::mutex mtx;
  std::lock_guard<std::mutex> lock(mtx);
  if (0 == state) {
    const char* names[] = { "libnvrtc.so.12", "libnvrtc.so", "/usr/local/cuda/lib64/libnvrtc.so.12", "/usr/local/cuda/lib64/libnvrtc.so" };
    api.h = 0;
    for (size_t i = 0; i < sizeof(names) / sizeof(*names) && 0 == api.h; ++i) api.h = dlopen(names[i], RTLD_NOW | RTLD_LOCAL);
    state = -1;
    if (api.h) {
      *(void**)&api.CreateProgram = dlsym(api.h, "nvrtcCreateProgram");
      *(void**)&api.CompileProgram = dlsym(api.h, "nvrtcCompileProgram");
      *(void**)&api.GetCUBINSize = dlsym(api.h, "nvrtcGetCUBINSize");
      *(void**)&api.GetCUBIN = dlsym(api.h, "nvrtcGetCUBIN");
      *(void**)&api.GetProgramLogSize = dlsym(api.h, "nvrtcGetProgramLogSize");
      *(void**)&api.GetProgramLog = dlsym(api.h, "nvrtcGetProgramLog");
      *(void**)&api.DestroyProgram = dlsym(api.h, "nvrtcDestroyProgram");
      if (api.CreateProgram && api.CompileProgram && api.GetCUBINSize && api.GetCUBIN && api.DestroyProgram) state = 1;
    }
  }
  return 1 == state ? &api : 0;
}

const int kBlock = 128;

void append(std::string& s, const char* fmt, ...)
{
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  s += buf;
}

// The emitted kernel: one thread per CPT consecutive columns of B/C (CPT = 1, or 2 as a vector of two).
// Every B row that the operator touches is loaded once into a named register (coalesced across the warp),
// every output row is then an in-order chain of fused multiply-adds with literal operator values -- the
// rounding sequence of the reference's emitted kernel (generator :227-300) -- and is stored, with a
// streaming store, as soon as it is complete.
void emit_kernel(std::string& s, const char* name, int cpt, int is_double, int M, int K, int beta_one, int skip_empty,
                 const int* rowptr, const int* col, const double* val)
{
  // Only scalar variables are emitted (the two columns of the vector form are split right after the load and
  // joined right before the store): NVRTC's optimiser needs several times longer for thousands of float2 values.
  const char* T = is_double ? "double" : "float";
  char V[16];
  snprintf(V, sizeof(V), "%s%s", T, 2 == cpt ? "2" : "");
  const char* f = is_double ? "fma" : "fmaf";
  std::vector<char> used(K, 0);
  for (int u = 0; u < rowptr[M]; ++u) used[col[u]] = 1;
  append(s, "extern \"C\" __global__ void __launch_bounds__(%d) %s(const %s* __restrict__ B, %s* __restrict__ C, long long ncols, long long ldb, long long ldc)\n{\n", kBlock, name, T, T);
  append(s, "  const long long n = ((long long)blockIdx.x * %d + threadIdx.x) * %d;\n  if (n >= ncols) return;\n", kBlock, cpt);
  append(s, "  const %s* __restrict__ b = B + n;\n  %s* __restrict__ c = C + n;\n  %s ax%s;\n", T, T, T, 2 == cpt ? ", ay" : "");
  for (int k = 0; k < K; ++k) if (used[k]) {
    if (2 == cpt) append(s, "  const %s t%d = __ldcs((const %s*)(b + %dLL * ldb)); const %s b%dx = t%d.x, b%dy = t%d.y;\n", V, k, V, k, T, k, k, k, k);
    else append(s, "  const %s b%dx = __ldcs(b + %dLL * ldb);\n", T, k, k);
  }
  // beta = 1: the C rows of a group are fetched together ahead of the group's chains, so that their latency
  // is paid once per group instead of once per row (loads cannot be hoisted over the stores by the compiler)
  const int group = beta_one ? (is_double ? 8 : 16) : 1;
  for (int m0 = 0; m0 < M; m0 += group) {
    if (beta_one) {
      for (int m = m0; m < M && m < m0 + group; ++m) if (rowptr[m + 1] != rowptr[m]) {
        if (2 == cpt) append(s, "  const %s u%d = __ldcs((const %s*)(c + %dLL * ldc)); const %s c%dx = u%d.x, c%dy = u%d.y;\n", V, m, V, m, T, m, m, m, m);
        else append(s, "  const %s c%dx = __ldcs(c + %dLL * ldc);\n", T, m, m);
      }
    }
    for (int m = m0; m < M && m < m0 + group; ++m) {
      const int lo = rowptr[m], hi = rowptr[m + 1];
      if (hi == lo) {
        if (!skip_empty && !beta_one) {
          if (2 == cpt) append(s, "  __stcs((%s*)(c + %dLL * ldc), make_%s(0, 0));\n", V, m, V);
          else append(s, "  __stcs(c + %dLL * ldc, (%s)0);\n", m, T);
        }
        continue;
      }
      if (beta_one) append(s, 2 == cpt ? "  ax = c%dx; ay = c%dy;\n" : "  ax = c%dx;\n", m, m);
      else append(s, 2 == cpt ? "  ax = 0; ay = 0;\n" : "  ax = 0;\n");
      for (int u = lo; u < hi; ++u) {
        char lit[64];
        if (is_double) {
          long long bits; const double v = val[u];
          memcpy(&bits, &v, 8);
          snprintf(lit, sizeof(lit), "__longlong_as_double(0x%016llxLL)", (unsigned long long)bits);
        }
        else {
          int bits; const float v = (float)val[u];
          memcpy(&bits, &v, 4);
          snprintf(lit, sizeof(lit), "__int_as_float(0x%08x)", (unsigned)bits);
        }
        if (2 == cpt) append(s, "  ax = %s(%s, b%dx, ax); ay = %s(%s, b%dy, ay);\n", f, lit, col[u], f, lit, col[u]);
        else append(s, "  ax = %s(%s, b%dx, ax);\n", f, lit, col[u]);
      }
      if (2 == cpt) append(s, "  __stcs((%s*)(c + %dLL * ldc), make_%s(ax, ay));\n", V, m, V);
      else append(s, "  __stcs(c + %dLL * ldc, ax);\n", m);
    }
  }
  s += "}\n";
}

// vec2: emit the two-columns-per-thread form (8-byte accesses; float only) instead of the one-column form
std::string emit(int is_double, int vec2, int M, int K, int beta_one, int skip_empty,
                 const int* rowptr, const int* col, const double* val)
{
  std::string s;
  s.reserve(160 * (size_t)rowptr[M] + 8192);
  emit_kernel(s, "fs_baked", (vec2 && !is_double) ? 2 : 1, is_double, M, K, beta_one, skip_empty, rowptr, col, val);
  return s;
}

// The same kernel as PTX text.  The driver's JIT (ptxas) assembles thousands of straight-line fused
// multiply-adds in a fraction of the time NVRTC's optimiser needs for the CUDA C++ form (measured: 6.3 s vs
// well under a second for the 150 x 64 / 30 % float operator), which is what keeps create() interactive.
static int fs_prefetch_b()
{
  const char* e = getenv("LIBXSMM_B200_FSSPMDM_PREFETCH_B");   // developer switch: distance of the B prefetch in half waves (default 2 = one wave; 0 = off)
  return (e && *e) ? atoi(e) : 2;
}

static int fs_prefetch_groups()
{
  const char* e = getenv("LIBXSMM_B200_FSSPMDM_PREFETCH");     // developer switch: groups of C rows prefetched ahead (0 = off)
  return (e && *e) ? atoi(e) : 2;
}

// batched: the columns are (element, column-in-element) pairs -- thread n works on element n / J, column n % J, whose B / C
// rows start at slot * stride (the [element][row][column][soa] tensors of the CSR x SoA kernels, SURVEY.md section 8f-1); the
// slot is the element itself, or its entry in a per-element index array (fs_jit_launch_batched)
std::string emit_ptx(int is_double, int vec2, int M, int K, int beta_one, int skip_empty,
                     const int* rowptr, const int* col, const double* val, int batched = 0, int variant = 0)
{
  const int cpt = (vec2 && !is_double && !batched) ? 2 : 1;
  const int esz = is_double ? 8 : 4;
  const char* ty = is_double ? "f64" : "f32";
  std::vector<char> used(K, 0);
  for (int u = 0; u < rowptr[M]; ++u) used[col[u]] = 1;
  std::string s;
  s.reserve(96 * (size_t)rowptr[M] * cpt + 8192);
  // Register-heavy operators (fp64 with ~50 or more used B rows: 100+ registers of B alone): left to itself the assembler interleaves
  // the rows' fma chains until all 255 registers are taken, which leaves two 128-thread CTAs = 8 warps per SM -- too few to keep
  // the FP64 pipe busy (PyFR p4/tet/m6: half its rate).  For those the rows are emitted IL at a time with their chains
  // interleaved explicitly, a bar.warp.sync between the groups keeps the assembler from mixing more, and three CTAs per SM are
  // asked for.  LIBXSMM_B200_FSSPMDM_IL / _MINCTAS (developer switches) override; IL = 0 is the plain row-after-row form.
  int nused = 0;
  for (int k = 0; k < K; ++k) nused += used[k] ? 1 : 0;
  int il = 0, minctas = 0;
  // variant (chosen by the caller, which times the candidates of fs_jit_variants() at create): 0 the plain form, 1 / 2 the explicit
  // form with eight / two rows interleaved.  No variant wins everywhere -- measured on B200, N = 2^20, beta = 0 / 1, plain against
  // eight (beta = 0) or two (beta = 1) rows: p4/tet/m6 362 / 453 -> 300 / 382 us, p5/tet/m460 4674 / 2317 -> 1650 / 2671, p5/tet/m0
  // 522 / 483 -> 714 / 453, p4/tet/m3 226 / 243 -> 239 / 198: what the assembler makes of thousands of straight-line fp64 fmas with
  // hundreds of distinct constants is not predictable from the operator, hence the timing.
  if (is_double && !batched && variant > 0) { il = (1 == variant) ? 8 : 2; minctas = (nused <= 72) ? 3 : 2; }
  { const char* e = getenv("LIBXSMM_B200_FSSPMDM_IL"); if (e && *e) { const int v = atoi(e); if (0 == v || (v >= 2 && v <= 8)) il = v; } }
  { const char* e = getenv("LIBXSMM_B200_FSSPMDM_MINCTAS"); if (e && *e) { const int v = atoi(e); if (0 == v || (v >= 2 && v <= 8)) minctas = v; } }
  s += ".version 8.6\n.target sm_100a\n.address_size 64\n\n";
  // fp64 operators with many distinct values (the reference's dense branch: tet / tri / pri families): a 64-bit literal is not an
  // instruction operand, so the assembler builds each one in (uniform) registers again and again -- a third more instructions, and
  // the values it chooses to keep fill the register file.  Their values go to constant memory instead; the fma takes the
  // constant-bank word as its operand directly.  LIBXSMM_B200_FSSPMDM_CONST=0 (developer switch): literals as before.
  std::vector<unsigned long long> ctab;
  std::map<unsigned long long, int> cidx;
  if (is_double) {
    for (int u = 0; u < rowptr[M]; ++u) {
      unsigned long long bits; const double v = val[u];
      memcpy(&bits, &v, 8);
      if (cidx.find(bits) == cidx.end()) { cidx[bits] = (int)ctab.size(); ctab.push_back(bits); }
    }
  }
  const char* cenv = getenv("LIBXSMM_B200_FSSPMDM_CONST");
  const bool use_const = is_double && ctab.size() > 31 && ctab.size() <= 4096 && ((cenv && *cenv) ? ('1' == *cenv) : (il >= 2));     // by default only with the explicit form (alone it is slower)
  if (use_const) {
    append(s, ".const .align 8 .b64 fsv[%d] = {", (int)ctab.size());
    for (size_t i = 0; i < ctab.size(); ++i) append(s, "%s0x%016llX", i ? ", " : "", ctab[i]);
    s += "};\n\n";
  }
  if (batched) s += ".visible .entry fs_baked(.param .u64 pB, .param .u64 pC, .param .u64 pN, .param .u64 pLDB, .param .u64 pLDC, .param .u64 pJ, .param .u64 pSB, .param .u64 pSC, .param .u64 pIPE, .param .u64 pIB, .param .u64 pIC, .param .u64 pXI, .param .u64 pXS, .param .u64 pCI, .param .u64 pCS)\n";
  else s += ".visible .entry fs_baked(.param .u64 pB, .param .u64 pC, .param .u64 pN, .param .u64 pLDB, .param .u64 pLDC)\n";
  append(s, ".maxntid %d, 1, 1\n", kBlock);
  if (minctas >= 2) append(s, ".minnctapersm %d\n", minctas);
  s += "{\n";
  s += "  .reg .pred %p, %pf;\n  .reg .b32 %r<4>;\n  .reg .b64 %rd<28>;\n";
  if (batched) s += "  .reg .b32 %ri;\n  .reg .b64 %rs<3>;\n";
  append(s, "  .reg .%s %%bx<%d>, %%by<%d>, %%cx<%d>, %%cy<%d>, %%ax, %%ay, %%ai<8>, %%aj<8>, %%kv;\n", ty, K, K, M, M);
  s += "  ld.param.u64 %rd0, [pB];\n  ld.param.u64 %rd1, [pC];\n  ld.param.u64 %rd2, [pN];\n  ld.param.u64 %rd3, [pLDB];\n  ld.param.u64 %rd4, [pLDC];\n";
  s += "  mov.u32 %r0, %ctaid.x;\n  mov.u32 %r1, %tid.x;\n";
  append(s, "  mul.wide.u32 %%rd5, %%r0, %d;\n  cvt.u64.u32 %%rd6, %%r1;\n  add.s64 %%rd5, %%rd5, %%rd6;\n", kBlock);
  if (2 == cpt) s += "  shl.b64 %rd5, %rd5, 1;\n";
  s += "  setp.ge.s64 %p, %rd5, %rd2;\n  @%p bra DONE;\n";
  if (batched) {   // item = n / J, column j = n % J; element e = item / IPE, i = item % IPE: b = B + e * SB + i * IB + j, c likewise
    s += "  ld.param.u64 %rd12, [pJ];\n  ld.param.u64 %rd13, [pSB];\n  ld.param.u64 %rd14, [pSC];\n";
    s += "  ld.param.u64 %rd20, [pIPE];\n  ld.param.u64 %rd21, [pIB];\n  ld.param.u64 %rd22, [pIC];\n";
    s += "  div.u64 %rd15, %rd5, %rd12;\n  mul.lo.s64 %rd16, %rd15, %rd12;\n  sub.s64 %rd16, %rd5, %rd16;\n";      // rd15 = item, rd16 = j
    s += "  div.u64 %rd23, %rd15, %rd20;\n  mul.lo.s64 %rd24, %rd23, %rd20;\n  sub.s64 %rd24, %rd15, %rd24;\n";    // rd23 = e, rd24 = i
    // slots of B and C: e, or idx[e] where the index pointer is not NULL; a slot at or past its count ends the thread
    const char* const pidx[2] = {"pXI", "pCI"};
    const char* const pcnt[2] = {"pXS", "pCS"};
    for (int t = 0; t < 2; ++t) {
      append(s, "  mov.b64 %%rs%d, %%rd23;\n  ld.param.u64 %%rs2, [%s];\n  setp.eq.u64 %%p, %%rs2, 0;\n  @%%p bra SLOT%d;\n", t, pidx[t], t);
      append(s, "  mad.lo.s64 %%rs2, %%rd23, 4, %%rs2;\n  ld.global.u32 %%ri, [%%rs2];\n  cvt.u64.u32 %%rs%d, %%ri;\n", t);
      append(s, "  ld.param.u64 %%rs2, [%s];\n  setp.ge.u64 %%p, %%rs%d, %%rs2;\n  @%%p bra DONE;\nSLOT%d:\n", pcnt[t], t, t);
    }
    s += "  mad.lo.s64 %rd17, %rs0, %rd13, %rd16;\n  mad.lo.s64 %rd17, %rd24, %rd21, %rd17;\n";
    s += "  mad.lo.s64 %rd18, %rs1, %rd14, %rd16;\n  mad.lo.s64 %rd18, %rd24, %rd22, %rd18;\n";
    append(s, "  mad.lo.s64 %%rd0, %%rd17, %d, %%rd0;\n  mad.lo.s64 %%rd1, %%rd18, %d, %%rd1;\n", esz, esz);
  }
  else
  append(s, "  mad.lo.s64 %%rd0, %%rd5, %d, %%rd0;\n  mad.lo.s64 %%rd1, %%rd5, %d, %%rd1;\n", esz, esz);   // b = B + n, c = C + n
  append(s, "  mul.lo.s64 %%rd3, %%rd3, %d;\n  mul.lo.s64 %%rd4, %%rd4, %d;\n", esz, esz);                 // row pitches in bytes
  s += "  and.b32 %r2, %r1, 15;\n  setp.eq.u32 %pf, %r2, 0;\n";                                          // one lane per 128-byte line issues prefetches
  if (il >= 2) s += "  mov.b64 %rd7, %rd0;\n";
  for (int k = 0, kprev = 0; k < K; ++k) if (used[k]) {
    if (il >= 2) {     // explicit form: running pointers everywhere (see the row loop)
      if (k - kprev == 1) s += "  add.s64 %rd7, %rd7, %rd3;\n";
      else if (k != kprev) append(s, "  mad.lo.s64 %%rd7, %%rd3, %d, %%rd7;\n", k - kprev);
      kprev = k;
    }
    else append(s, "  mad.lo.s64 %%rd7, %%rd3, %d, %%rd0;\n", k);
    if (2 == cpt) append(s, "  ld.global.cs.v2.%s {%%bx%d, %%by%d}, [%%rd7];\n", ty, k, k);
    else append(s, "  ld.global.cs.%s %%bx%d, [%%rd7];\n", ty, k);
  }
  // The B rows of the column block one "wave" ahead (number of SMs x this block's columns further on: blocks are
  // scheduled in order) are pulled into L2 now, one lane per 128-byte line: that block's load phase then pays L2
  // latency instead of DRAM latency.  Measured on B200 (fraction of the 6554 GB/s copy peak): 150 x 64 float operator,
  // N = 2^24: 0.854 -> 0.989; double, N = 2^20: 0.960 -> 0.984.  Twice as far ahead is worth nothing (0.88), further
  // is harmful; with beta = 1 the C-row prefetches below already fill the queues and this one costs 1-4 %.
  if (!beta_one && !batched && fs_prefetch_b() > 0) {      // (measured: helps beta = 0, costs 2-4 % with beta = 1, where the C prefetches below already fill the queues)
    s += "  mov.u32 %r3, %nsmid;\n";
    append(s, "  mul.wide.u32 %%rd10, %%r3, %d;\n", fs_prefetch_b() * kBlock * cpt / 2);                                          // columns ahead
    s += "  add.s64 %rd11, %rd5, %rd10;\n  setp.lt.s64 %p, %rd11, %rd2;\n  and.pred %p, %p, %pf;\n";
    append(s, "  mad.lo.s64 %%rd10, %%rd10, %d, %%rd0;\n", esz);
    if (il >= 2) {
      for (int k = 0, kprev = 0; k < K; ++k) if (used[k]) {
        if (k - kprev == 1) s += "  add.s64 %rd10, %rd10, %rd3;\n";
        else if (k != kprev) append(s, "  mad.lo.s64 %%rd10, %%rd3, %d, %%rd10;\n", k - kprev);
        kprev = k;
        s += "  @%p prefetch.global.L2 [%rd10];\n";
      }
    }
    else
    for (int k = 0; k < K; ++k) if (used[k]) append(s, "  mad.lo.s64 %%rd7, %%rd3, %d, %%rd10;\n  @%%p prefetch.global.L2 [%%rd7];\n", k);
  }
  const int group = (il >= 2) ? (beta_one ? ((is_double ? 8 : 16) + il - 1) / il * il : il) : (beta_one ? (is_double ? 8 : 16) : 1);
  // beta = 1: the C rows that will be read are pulled into L2 two groups ahead by prefetch instructions (one lane
  // per 128-byte line, no registers held), so that the group's loads pay the L2 latency instead of the DRAM one
  const int ahead = fs_prefetch_groups();
  auto prefetch_group = [&](int g0) {
    for (int m = g0; m < M && m < g0 + group; ++m) if (rowptr[m + 1] != rowptr[m]) {
      append(s, "  mad.lo.s64 %%rd9, %%rd4, %d, %%rd1;\n  @%%pf prefetch.global.L2 [%%rd9];\n", m);
    }
  };
  if (beta_one && ahead > 0) for (int a = 0; a < ahead; ++a) prefetch_group(a * group);
  int ld_row = 0, st_row = 0;        // explicit form: rows the running load / store pointers (%rd26 / %rd27) stand on
  if (il >= 2) s += "  mov.b64 %rd26, %rd1;\n  mov.b64 %rd27, %rd1;\n";
  for (int m0 = 0; m0 < M; m0 += group) {
    if (beta_one) {
      if (ahead > 0) prefetch_group(m0 + ahead * group);
      for (int m = m0; m < M && m < m0 + group; ++m) if (rowptr[m + 1] != rowptr[m]) {
        if (il >= 2) {       // running pointer (a product per row invites the assembler to compute all row addresses up front and spill them)
          if (m - ld_row == 1) s += "  add.s64 %rd26, %rd26, %rd4;\n";
          else append(s, "  mad.lo.s64 %%rd26, %%rd4, %d, %%rd26;\n", m - ld_row);
          ld_row = m;
          if (2 == cpt) append(s, "  ld.global.cs.v2.%s {%%cx%d, %%cy%d}, [%%rd26];\n", ty, m, m);
          else append(s, "  ld.global.cs.%s %%cx%d, [%%rd26];\n", ty, m);
          continue;
        }
        append(s, "  mad.lo.s64 %%rd8, %%rd4, %d, %%rd1;\n", m);
        if (2 == cpt) append(s, "  ld.global.cs.v2.%s {%%cx%d, %%cy%d}, [%%rd8];\n", ty, m, m);
        else append(s, "  ld.global.cs.%s %%cx%d, [%%rd8];\n", ty, m);
      }
    }
    auto literal = [&](int u, char (&lit)[32]) {      // the operand text of value u (constant-bank form: after loading it)
      if (use_const) {
        unsigned long long bits; const double v = val[u];
        memcpy(&bits, &v, 8);
        append(s, "  ld.const.f64 %%kv, [fsv+%d];\n", 8 * cidx[bits]);
        snprintf(lit, sizeof(lit), "%%kv");
      }
      else if (is_double) {
        unsigned long long bits; const double v = val[u];
        memcpy(&bits, &v, 8);
        snprintf(lit, sizeof(lit), "0d%016llX", bits);
      }
      else {
        unsigned int bits; const float v = (float)val[u];
        memcpy(&bits, &v, 4);
        snprintf(lit, sizeof(lit), "0f%08X", bits);
      }
    };
    if (il >= 2) {
      // explicit form: the non-empty rows of the group il at a time, step j of every chain before step j + 1 of any (each row's
      // own order is unchanged: same bits), stores at the end, then a fence for the assembler's scheduler
      const char* zero = is_double ? "0d0000000000000000" : "0f00000000";
      std::vector<int> rows;
      for (int m = m0; m < M && m < m0 + group; ++m) {
        if (rowptr[m + 1] != rowptr[m]) rows.push_back(m);
        else if (!skip_empty && !beta_one) {
          append(s, "  mad.lo.s64 %%rd8, %%rd4, %d, %%rd1;\n  mov.%s %%ax, %s;\n", m, ty, zero);
          if (2 == cpt) append(s, "  st.global.cs.v2.%s [%%rd8], {%%ax, %%ax};\n", ty);
          else append(s, "  st.global.cs.%s [%%rd8], %%ax;\n", ty);
        }
      }
      for (size_t r0 = 0; r0 < rows.size(); r0 += (size_t)il) {
        const size_t r1 = (r0 + (size_t)il < rows.size()) ? r0 + (size_t)il : rows.size();
        int maxlen = 0;
        for (size_t r = r0; r < r1; ++r) {
          const int m = rows[r], a = (int)(r - r0);
          maxlen = (rowptr[m + 1] - rowptr[m] > maxlen) ? rowptr[m + 1] - rowptr[m] : maxlen;
          if (beta_one) { append(s, "  mov.%s %%ai%d, %%cx%d;\n", ty, a, m); if (2 == cpt) append(s, "  mov.%s %%aj%d, %%cy%d;\n", ty, a, m); }
          else { append(s, "  mov.%s %%ai%d, %s;\n", ty, a, zero); if (2 == cpt) append(s, "  mov.%s %%aj%d, %s;\n", ty, a, zero); }
        }
        for (int j = 0; j < maxlen; ++j) {
          for (size_t r = r0; r < r1; ++r) {
            const int m = rows[r], a = (int)(r - r0), u = rowptr[m] + j;
            if (u >= rowptr[m + 1]) continue;
            char lit[32];
            literal(u, lit);
            append(s, "  fma.rn.%s %%ai%d, %s, %%bx%d, %%ai%d;\n", ty, a, lit, col[u], a);
            if (2 == cpt) append(s, "  fma.rn.%s %%aj%d, %s, %%by%d, %%aj%d;\n", ty, a, lit, col[u], a);
          }
        }
        for (size_t r = r0; r < r1; ++r) {
          const int m = rows[r], a = (int)(r - r0);
          if (m - st_row == 1) s += "  add.s64 %rd27, %rd27, %rd4;\n";
          else if (m != st_row) append(s, "  mad.lo.s64 %%rd27, %%rd4, %d, %%rd27;\n", m - st_row);
          st_row = m;
          if (2 == cpt) append(s, "  st.global.cs.v2.%s [%%rd27], {%%ai%d, %%aj%d};\n", ty, a, a);
          else append(s, "  st.global.cs.%s [%%rd27], %%ai%d;\n", ty, a);
        }
        s += "  bar.warp.sync 0xffffffff;\n";
      }
      continue;
    }
    for (int m = m0; m < M && m < m0 + group; ++m) {
      const int lo = rowptr[m], hi = rowptr[m + 1];
      const char* zero = is_double ? "0d0000000000000000" : "0f00000000";
      if (hi == lo) {
        if (!skip_empty && !beta_one) {
          append(s, "  mad.lo.s64 %%rd8, %%rd4, %d, %%rd1;\n  mov.%s %%ax, %s;\n", m, ty, zero);
          if (2 == cpt) append(s, "  st.global.cs.v2.%s [%%rd8], {%%ax, %%ax};\n", ty);
          else append(s, "  st.global.cs.%s [%%rd8], %%ax;\n", ty);
        }
        continue;
      }
      if (beta_one) {
        append(s, "  mov.%s %%ax, %%cx%d;\n", ty, m);
        if (2 == cpt) append(s, "  mov.%s %%ay, %%cy%d;\n", ty, m);
      }
      else {
        append(s, "  mov.%s %%ax, %s;\n", ty, zero);
        if (2 == cpt) append(s, "  mov.%s %%ay, %s;\n", ty, zero);
      }
      for (int u = lo; u < hi; ++u) {
        char lit[32];
        literal(u, lit);
        append(s, "  fma.rn.%s %%ax, %s, %%bx%d, %%ax;\n", ty, lit, col[u]);
        if (2 == cpt) append(s, "  fma.rn.%s %%ay, %s, %%by%d, %%ay;\n", ty, lit, col[u]);
      }
      append(s, "  mad.lo.s64 %%rd8, %%rd4, %d, %%rd1;\n", m);
      if (2 == cpt) append(s, "  st.global.cs.v2.%s [%%rd8], {%%ax, %%ay};\n", ty);
      else append(s, "  st.global.cs.%s [%%rd8], %%ax;\n", ty);
    }
  }
  s += "DONE:\n  ret;\n}\n";
  return s;
}

// ---- strip form --------------------------------------------------------------------------------------------------------
// For operators with more used B rows than the register file holds (> 100 double / 200 float: every p4..p6 hex / pri PyFR
// operator, e.g. p4/hex/m0 150 x 125, up to p5/hex/m132 216 x 648) the B rows live in SHARED memory instead: a CTA owns 32
// consecutive columns, one thread stages the K x 32 strip with TMA (cp.async.bulk.tensor over the caller's strided panel:
// rows past K and columns past N are zero-filled by the hardware), and every output row is again a straight-line chain of
// fused multiply-adds with literal operator values, its B operand read from shared memory at a literal offset (lane =
// column: conflict-free).  The rows are dealt out to G warps (longest-processing-time first, four rows at a time so that
// four independent chains interleave), each warp running its own section of the emitted code on the same strip; the order
// of the multiply-adds inside a row is the reference's (ascending k).  Per nonzero: one LDS + one FMA.
struct StripPlan { int G, W, box_rows, nboxes, krows; size_t smem; std::vector<std::vector<int> > blocks; };   // blocks[g] = first rows of the 4-row blocks of warp g

const int kStripW = 32;

StripPlan strip_plan(int is_double, int M, int K, const int* rowptr)
{
  StripPlan p;
  const int esz = is_double ? 8 : 4;
  p.nboxes = (K + 255) / 256;                       // a TMA box has at most 256 rows
  p.box_rows = (K + p.nboxes - 1) / p.nboxes;
  p.krows = p.nboxes * p.box_rows;
  p.W = kStripW;                                    // 32 columns per CTA (lane = column); 16 when 32 do not fit shared memory (K > ~900 double)
  p.smem = 128 + (size_t)p.krows * p.W * esz;
  if (p.smem > 227u * 1024u) { p.W = 16; p.smem = 128 + (size_t)p.krows * p.W * esz; }
  const int ctas = (int)((220u * 1024u) / p.smem) < 1 ? 1 : (int)((220u * 1024u) / p.smem);
  int G = (24 + ctas - 1) / ctas;                      // ~24 warps per SM
  const int nblocks = (M + 3) / 4;
  if (G > 8) G = 8;
  if (G > nblocks) G = nblocks;
  if (G < 1) G = 1;
  p.G = G;
  p.blocks.assign((size_t)G, std::vector<int>());
  std::vector<std::pair<int, int> > load;               // (nonzeros, first row) per block, heaviest first
  for (int b = 0; b < nblocks; ++b) {
    const int r0 = 4 * b, r1 = (r0 + 4 < M) ? r0 + 4 : M;
    load.push_back(std::make_pair(rowptr[r1] - rowptr[r0] + 2 * (r1 - r0), r0));
  }
  std::sort(load.begin(), load.end(), [](const std::pair<int, int>& a, const std::pair<int, int>& b) { return a.first != b.first ? a.first > b.first : a.second < b.second; });
  std::vector<long long> tot((size_t)G, 0);
  for (size_t i = 0; i < load.size(); ++i) {
    int best = 0;
    for (int g = 1; g < G; ++g) if (tot[g] < tot[best]) best = g;
    tot[best] += load[i].first;
    p.blocks[best].push_back(load[i].second);
  }
  for (int g = 0; g < G; ++g) std::sort(p.blocks[g].begin(), p.blocks[g].end());
  return p;
}

std::string emit_ptx_strip(int is_double, int M, int K, int beta_one, int skip_empty, const int* rowptr, const int* col, const double* val, const StripPlan& pl)
{
  const int esz = is_double ? 8 : 4;
  const char* ty = is_double ? "f64" : "f32";
  const char* zero = is_double ? "0d0000000000000000" : "0f00000000";
  std::string s;
  s.reserve(80 * (size_t)rowptr[M] + 16384);
  s += ".version 8.6\n.target sm_100a\n.address_size 64\n\n.extern .shared .align 128 .b8 fs_smem[];\n\n";
  s += ".visible .entry fs_baked(.param .align 64 .b8 pMap[128], .param .u64 pC, .param .u64 pN, .param .u64 pLDC)\n";
  append(s, ".maxntid %d, 1, 1\n{\n", pl.G * 32);
  s += "  .reg .pred %p, %pv, %pw;\n  .reg .b32 %r<12>;\n  .reg .b64 %rd<10>;\n";
  append(s, "  .reg .%s %%a<4>, %%b<4>;\n", ty);
  s += "  mov.b64 %rd0, pMap;\n  cvta.param.u64 %rd0, %rd0;\n  ld.param.u64 %rd1, [pC];\n  ld.param.u64 %rd2, [pN];\n  ld.param.u64 %rd3, [pLDC];\n";
  s += "  mov.u32 %r0, %tid.x;\n  mov.u32 %r1, %ctaid.x;\n  mov.u32 %r2, fs_smem;\n";       // %r2: mbarrier, strip at +128
  append(s, "  mul.lo.u32 %%r3, %%r1, %d;\n", pl.W);                                         // first column of the strip
  s += "  setp.ne.u32 %p, %r0, 0;\n  @%p bra INIT_DONE;\n";
  s += "  mbarrier.init.shared::cta.b64 [%r2], 1;\n  fence.mbarrier_init.release.cluster;\n";
  append(s, "  mbarrier.arrive.expect_tx.shared::cta.b64 _, [%%r2], %u;\n", (unsigned)((size_t)pl.krows * pl.W * esz));
  for (int b = 0; b < pl.nboxes; ++b) {
    append(s, "  add.u32 %%r4, %%r2, %u;\n  mov.u32 %%r5, %d;\n", (unsigned)(128 + (size_t)b * pl.box_rows * pl.W * esz), b * pl.box_rows);
    s += "  cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%r4], [%rd0, {%r3, %r5}], [%r2];\n";
  }
  s += "INIT_DONE:\n  bar.sync 0;\n";
  // this lane's column, its validity, its C pointer and its strip address
  append(s, "  and.b32 %%r10, %%r0, 31;\n  and.b32 %%r6, %%r0, %d;\n  shr.u32 %%r7, %%r0, 5;\n  add.u32 %%r8, %%r3, %%r6;\n  cvt.u64.u32 %%rd4, %%r8;\n  setp.lt.s64 %%pv, %%rd4, %%rd2;\n", pl.W - 1);
  if (pl.W < 32) append(s, "  setp.lt.u32 %%p, %%r10, %d;\n  and.pred %%pv, %%pv, %%p;\n", pl.W);      // a 16-column strip: the upper half warp idles
  append(s, "  mad.lo.s64 %%rd1, %%rd4, %d, %%rd1;\n  mul.lo.s64 %%rd3, %%rd3, %d;\n", esz, esz);      // c = C + n; row pitch in bytes
  append(s, "  mad.lo.u32 %%r9, %%r6, %d, %%r2;\n", esz);                                               // strip + lane * esz (the +128 goes into the literal offsets)
  s += "WAIT:\n  mbarrier.try_wait.parity.shared::cta.b64 %pw, [%r2], 0;\n  @%pw bra READY;\n  bra WAIT;\nREADY:\n";
  for (int g = 0; g < pl.G; ++g) {
    if (g + 1 < pl.G) append(s, "  setp.ne.u32 %%p, %%r7, %d;\n  @%%p bra SEC%d;\n", g, g + 1);
    for (size_t bi = 0; bi < pl.blocks[g].size(); ++bi) {
      const int r0 = pl.blocks[g][bi], r1 = (r0 + 4 < M) ? r0 + 4 : M;
      int maxlen = 0;
      for (int m = r0; m < r1; ++m) {
        const int len = rowptr[m + 1] - rowptr[m];
        if (len > maxlen) maxlen = len;
        if (0 == len) continue;
        if (beta_one) {
          append(s, "  mad.lo.s64 %%rd5, %%rd3, %d, %%rd1;\n  mov.%s %%a%d, %s;\n  @%%pv ld.global.cs.%s %%a%d, [%%rd5];\n", m, ty, m - r0, zero, ty, m - r0);
        }
        else append(s, "  mov.%s %%a%d, %s;\n", ty, m - r0, zero);
      }
      for (int j = 0; j < maxlen; ++j) {          // the four chains interleaved: independent accumulators, in-order inside a row
        // a warp-level barrier every 8 steps (32 loads) is a scheduling fence: without it the assembler hoists hundreds of the
        // independent shared-memory loads of a dense row ahead of their multiply-adds and spills them
        if (j > 0 && 0 == (j % 8)) s += "  bar.warp.sync 0xffffffff;\n";
        for (int m = r0; m < r1; ++m) if (rowptr[m] + j < rowptr[m + 1]) {
          const int u = rowptr[m] + j;
          char lit[32];
          if (is_double) { unsigned long long bits; const double v = val[u]; memcpy(&bits, &v, 8); snprintf(lit, sizeof(lit), "0d%016llX", bits); }
          else { unsigned int bits; const float v = (float)val[u]; memcpy(&bits, &v, 4); snprintf(lit, sizeof(lit), "0f%08X", bits); }
          append(s, "  ld.shared.%s %%b%d, [%%r9+%u];\n  fma.rn.%s %%a%d, %s, %%b%d, %%a%d;\n", ty, m - r0, (unsigned)(128 + (size_t)col[u] * pl.W * esz), ty, m - r0, lit, m - r0, m - r0);
        }
      }
      for (int m = r0; m < r1; ++m) {
        const int len = rowptr[m + 1] - rowptr[m];
        if (0 == len) {
          if (!skip_empty && !beta_one) append(s, "  mad.lo.s64 %%rd5, %%rd3, %d, %%rd1;\n  mov.%s %%a0, %s;\n  @%%pv st.global.cs.%s [%%rd5], %%a0;\n", m, ty, zero, ty);
          continue;
        }
        append(s, "  mad.lo.s64 %%rd5, %%rd3, %d, %%rd1;\n  @%%pv st.global.cs.%s [%%rd5], %%a%d;\n", m, ty, m - r0);
      }
    }
    s += "  bra DONE;\n";
    if (g + 1 < pl.G) append(s, "SEC%d:\n", g + 1);
  }
  s += "DONE:\n  ret;\n}\n";
  return s;
}

bool strip_supported(int is_double, int M, int K, const int* rowptr)
{
  (void)is_double;
  return rowptr[M] > 0 && rowptr[M] <= 200000 && strip_plan(is_double, M, K, rowptr).smem <= 227u * 1024u;
}

bool supported(int is_double, int vec2, int M, int K, const int* rowptr, const int* col)
{
  std::vector<char> used(K, 0);
  int nused = 0;
  for (int u = 0; u < rowptr[M]; ++u) if (!used[col[u]]) { used[col[u]] = 1; ++nused; }
  // B rows live in registers: 2 registers per double, 1 per float, out of 255
  // B rows live in registers (2 registers per double, 1 per float, out of 255); the NVRTC form is additionally
  // limited to ~6000 nonzeros in fs_jit_build (compile time grows faster than linearly)
  // (the float kernel that handles two columns per thread holds two registers per row as well)
  return rowptr[M] > 0 && ((is_double || vec2) ? nused <= 100 : nused <= 200) && rowptr[M] <= 40000;
}

std::mutex g_cache_mtx;
std::map<std::string, std::vector<char> > g_cubin_cache;

}  // namespace

// which form fs_jit_build would emit for this operator: 0 none (generic kernel), 1 B rows in registers, 2 B strip in shared memory
int fs_jit_form(int is_double, int vec2, int M, int K, const int* rowptr, const int* col)
{
  if (supported(is_double, vec2, M, K, rowptr, col)) return 1;
  return strip_supported(is_double, M, K, rowptr) ? 2 : 0;
}

char* fs_jit_source(int is_double, int vec2, int M, int K, int beta_one, int skip_empty,
                    const int* rowptr, const int* col, const double* val)
{
  const char* env = getenv("LIBXSMM_B200_FSSPMDM_JIT");
  const bool strip = !supported(is_double, vec2, M, K, rowptr, col) && strip_supported(is_double, M, K, rowptr);
  const std::string s = strip ? emit_ptx_strip(is_double, M, K, beta_one, skip_empty, rowptr, col, val, strip_plan(is_double, M, K, rowptr))
                              : ((env && 'n' == *env) ? emit(is_double, vec2, M, K, beta_one, skip_empty, rowptr, col, val)
                                                      : emit_ptx(is_double, vec2, M, K, beta_one, skip_empty, rowptr, col, val));
  char* out = (char*)malloc(s.size() + 1);
  if (out) memcpy(out, s.c_str(), s.size() + 1);
  return out;
}

// how many emitter variants are worth timing for this operator (1 = only the plain form): fp64 operators in the register form whose
// fma count makes the FP64 pipe, not HBM, the likely bound
int fs_jit_variants(int is_double, int vec2, int M, int K, const int* rowptr, const int* col)
{
  if (!is_double || !supported(is_double, vec2, M, K, rowptr, col)) return 1;
  const char* e = getenv("LIBXSMM_B200_FSSPMDM_TUNE");      // 0: never time, always the plain form
  if (e && '0' == *e) return 1;
  return (rowptr[M] >= 16 * (M + K)) ? 3 : 1;
}

FsJit* fs_jit_build(int is_double, int vec2, int M, int K, int beta_one, int skip_empty,
                    const int* rowptr, const int* col, const double* val, int batched, int variant)
{
  if (batched) vec2 = 0;
  const char* env = getenv("LIBXSMM_B200_FSSPMDM_JIT");
  if (env && '0' == *env) return 0;
  const bool regs_ok = supported(is_double, vec2, M, K, rowptr, col);
  const bool strip = !regs_ok && !batched && strip_supported(is_double, M, K, rowptr);   // B rows in shared memory instead of registers
  if (!regs_ok && !strip) return 0;
  // default: PTX text assembled by the driver (fast); LIBXSMM_B200_FSSPMDM_JIT=nvrtc: CUDA C++ through NVRTC
  const bool use_nvrtc = (env && 'n' == *env) && !strip;
  std::vector<char> cubin;     // cubin (NVRTC) or NUL-terminated PTX text
  StripPlan plan;
  if (strip) {
    plan = strip_plan(is_double, M, K, rowptr);
    const std::string ptx = emit_ptx_strip(is_double, M, K, beta_one, skip_empty, rowptr, col, val, plan);
    cubin.assign(ptx.begin(), ptx.end());
    cubin.push_back(0);
  }
  else if (!use_nvrtc) {
    const std::string ptx = emit_ptx(is_double, vec2, M, K, beta_one, skip_empty, rowptr, col, val, batched, variant);
    cubin.assign(ptx.begin(), ptx.end());
    cubin.push_back(0);
  }
  else {
    if (rowptr[M] > 6000 || batched) return 0;
    Nvrtc* rt = nvrtc();
    if (0 == rt) { set_error(-2, "fsspmdm: NVRTC (libnvrtc.so.12) not found; using the generic kernel"); return 0; }
    const std::string src = emit(is_double, vec2, M, K, beta_one, skip_empty, rowptr, col, val);
    {
      std::lock_guard<std::mutex> lock(g_cache_mtx);
      std::map<std::string, std::vector<char> >::const_iterator it = g_cubin_cache.find(src);
      if (it != g_cubin_cache.end()) cubin = it->second;
    }
    if (cubin.empty()) {
      nvrtcProgram prog = 0;
      if (NVRTC_SUCCESS != rt->CreateProgram(&prog, src.c_str(), "fs_baked.cu", 0, 0, 0)) { set_error(-3, "nvrtcCreateProgram failed"); return 0; }
      const char* opts[] = { "--gpu-architecture=sm_100a", "-lineinfo", "--fmad=false" };
      const nvrtcResult rc = rt->CompileProgram(prog, 3, opts);
      if (NVRTC_SUCCESS != rc) {
        size_t n = 0;
        std::string log;
        if (rt->GetProgramLogSize && NVRTC_SUCCESS == rt->GetProgramLogSize(prog, &n) && n > 1) { log.resize(n); rt->GetProgramLog(prog, &log[0]); }
        set_error(-4, "fsspmdm: NVRTC compile failed (%d): %.300s", (int)rc, log.c_str());
        rt->DestroyProgram(&prog);
        return 0;
      }
      size_t sz = 0;
      if (NVRTC_SUCCESS != rt->GetCUBINSize(prog, &sz) || 0 == sz) { set_error(-5, "nvrtcGetCUBINSize failed"); rt->DestroyProgram(&prog); return 0; }
      cubin.resize(sz);
      rt->GetCUBIN(prog, cubin.data());
      rt->DestroyProgram(&prog);
      std::lock_guard<std::mutex> lock(g_cache_mtx);
      g_cubin_cache[src] = cubin;
    }
  }
  FsJit* j = new FsJit();
  j->block = strip ? plan.G * 32 : kBlock;
  j->cols_per_thread = (vec2 && !is_double && !strip) ? 2 : 1;
  j->batched = batched ? 1 : 0;
  j->strip = strip ? 1 : 0; j->esz = is_double ? 8 : 4; j->krows = K; j->box_rows = strip ? plan.box_rows : 0; j->strip_w = strip ? plan.W : 0; j->smem = strip ? plan.smem : 0;
  cudaError_t e = cudaLibraryLoadData(&j->lib, cubin.data(), 0, 0, 0, 0, 0, 0);
  if (cudaSuccess == e) e = cudaLibraryGetKernel(&j->kern, j->lib, "fs_baked");
  if (cudaSuccess == e && strip && j->smem > 48u * 1024u) e = cudaFuncSetAttribute((const void*)j->kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)j->smem);
  if (cudaSuccess != e) {
    set_error((int)e, "fsspmdm: loading the baked kernel failed: %s", cudaGetErrorString(e));
    (void)cudaGetLastError();
    delete j;
    return 0;
  }
  return j;
}

bool fs_jit_launch(const FsJit* j, const void* dB, void* dC, long long ncols, long long ldb, long long ldc, cudaStream_t stream)
{
  if (j->batched) return false;
  if (j->strip) {
    // the strip form reads B through a TMA tensor map built from the caller's panel: 16-byte aligned base and row pitch
    CUtensorMap map;
    if (!make_tensor_map_2d(&map, dB, j->esz, (unsigned long long)ncols, (unsigned long long)j->krows, (unsigned long long)ldb * j->esz, (unsigned)j->strip_w, (unsigned)j->box_rows)) return false;
    const long long blocks = (ncols + j->strip_w - 1) / j->strip_w;
    void* args[] = { (void*)&map, (void*)&dC, (void*)&ncols, (void*)&ldc };
    const cudaError_t e = cudaLaunchKernel((const void*)j->kern, dim3((unsigned)blocks, 1, 1), dim3((unsigned)j->block, 1, 1), args, j->smem, stream);
    if (cudaSuccess != e) { set_error((int)e, "fsspmdm: baked strip kernel launch failed: %s", cudaGetErrorString(e)); (void)cudaGetLastError(); return false; }
    return true;
  }
  // the 2-column form needs 8-byte aligned rows: even pitches, even column count, aligned bases; a panel that does
  // not qualify goes to the generic kernel (return false)
  if (2 == j->cols_per_thread && !((0 == ((ldb | ldc | ncols) & 1)) && (0 == (((uintptr_t)dB | (uintptr_t)dC) & 7)))) return false;
  const long long per_block = (long long)j->block * j->cols_per_thread;
  const long long blocks = (ncols + per_block - 1) / per_block;
  void* args[] = { (void*)&dB, (void*)&dC, (void*)&ncols, (void*)&ldb, (void*)&ldc };
  const cudaError_t e = cudaLaunchKernel((const void*)j->kern, dim3((unsigned)blocks, 1, 1), dim3((unsigned)j->block, 1, 1), args, 0, stream);
  if (cudaSuccess != e) { set_error((int)e, "fsspmdm: baked kernel launch failed: %s", cudaGetErrorString(e)); return false; }
  return true;
}

bool fs_jit_launch_batched(const FsJit* j, const void* dB, void* dC, long long n_elem, long long items_per_elem, long long cols_per_item, long long ldb, long long ldc,
                           long long stride_b, long long stride_c, long long item_b, long long item_c,
                           const unsigned int* b_index, long long b_slots, const unsigned int* c_index, long long c_slots, cudaStream_t stream)
{
  if (!j->batched) return false;
  long long total = n_elem * items_per_elem * cols_per_item;
  const long long blocks = (total + j->block - 1) / j->block;
  void* args[] = { (void*)&dB, (void*)&dC, (void*)&total, (void*)&ldb, (void*)&ldc, (void*)&cols_per_item, (void*)&stride_b, (void*)&stride_c,
                   (void*)&items_per_elem, (void*)&item_b, (void*)&item_c, (void*)&b_index, (void*)&b_slots, (void*)&c_index, (void*)&c_slots };
  const cudaError_t e = cudaLaunchKernel((const void*)j->kern, dim3((unsigned)blocks, 1, 1), dim3((unsigned)j->block, 1, 1), args, 0, stream);
  if (cudaSuccess != e) { set_error((int)e, "csr_soa: baked kernel launch failed: %s", cudaGetErrorString(e)); (void)cudaGetLastError(); return false; }
  return true;
}

void fs_jit_destroy(FsJit* j)
{
  if (0 == j) return;
  cudaLibraryUnload(j->lib);
  delete j;
}

}  // namespace xb
