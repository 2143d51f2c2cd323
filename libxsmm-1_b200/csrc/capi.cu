// C ABI of libxsmm_b200.so: the 14 reference entry points (include/libxsmm_spmdm.h,
// include/libxsmm_fsspmdm.h) plus the stream-ordered additions (include/libxsmm_b200.h).
// Host logic only; the kernels are in spmdm_kernels.cu / fsspmdm.cu.  No CPU compute path exists:
// every entry point either launches CUDA kernels or records an error.
#include "common.cuh"
#include "../../include/libxsmm_b200.h"
#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <climits>
#include <mutex>
#include <unordered_map>
#include <map>
#include <vector>

namespace xb {

// ---- error state / counters ------------------------------------------------------------------------
static std::mutex g_err_mtx;
static int g_err_code = 0;
static char g_err_msg[1024] = "";
static std::atomic<unsigned long long> g_launches(0);
static std::atomic<unsigned long long> g_err_seq(0);   // bumped by every set_error: lets a call tell its own failures from older, unrelated ones

int verbosity()
{
  static int v = INT_MIN;
  if (INT_MIN == v) {
    const char* e = getenv("LIBXSMM_VERBOSE");   // same switch as the reference (src/libxsmm_main.c:562)
    v = (e && *e) ? atoi(e) : 0;
  }
  return v;
}

void set_error(int code, const char* fmt, ...)
{
  std::lock_guard<std::mutex> lock(g_err_mtx);
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err_msg, sizeof(g_err_msg), fmt, ap);
  va_end(ap);
  g_err_code = (0 != code) ? code : -1;
  g_err_seq.fetch_add(1, std::memory_order_relaxed);
  if (0 != verbosity()) fprintf(stderr, "LIBXSMM_B200 ERROR: %s\n", g_err_msg);
}

void count_launch(int n) { g_launches.fetch_add((unsigned long long)n, std::memory_order_relaxed); }

void ensure_smem_optin(const void* kernel, int bytes)
{
  static std::mutex mtx;
  static std::map<std::pair<const void*, int>, int> done;     // (kernel, device) -> bytes granted
  int dev = 0;
  if (cudaSuccess != cudaGetDevice(&dev)) { (void)cudaGetLastError(); return; }
  std::lock_guard<std::mutex> lock(mtx);
  int& have = done[std::make_pair(kernel, dev)];
  if (have >= bytes) return;
  XB_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
  have = bytes;
}

int device_sm_count()
{
  int dev = 0, sms = 0;
  if (cudaSuccess != cudaGetDevice(&dev) || cudaSuccess != cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev)) { (void)cudaGetLastError(); return 148; }
  return sms > 0 ? sms : 148;
}
static std::atomic<const char*> g_last_compute("");
void note_compute_kernel(const char* name) { g_last_compute.store(name, std::memory_order_relaxed); }

// ---- SPMDM context -----------------------------------------------------------------------------------
constexpr int kExecPanels = 8;   // column panels of the pipelined host path (libxsmm_spmdm_exec_host)
struct SpmdmCtx {
  Geom g;
  int simd_w;
  int max_threads;
  void* arena_base;
  SliceArena arena;
  libxsmm_CSR_sparseslice* table;   // host table of device pointers handed to the caller
  char* staging;                    // device, max_threads slabs
  size_t staging_per_tid;
  std::vector<cudaStream_t> streams;
  std::mutex mtx;
  // whole-problem host path (libxsmm_spmdm_exec_host)
  void* d_a; void* d_b; float* d_c;
  size_t d_a_bytes, d_b_bytes, d_c_bytes;
  cudaStream_t xs[3];
  cudaEvent_t xev[kExecPanels + 1];
  std::vector<cudaEvent_t> xup, xdone;   // per diagonal step of exec_host: uploads landed / tiles computed
  // density feedback: the slicing kernels publish the total nonzero count of the last completed pass into
  // mapped pinned memory; the host uses it (one call late, never for correctness) to avoid enqueueing the
  // kernel twin that will not be selected and the auxiliary arrays only that twin reads
  unsigned long long* h_nnz;      // host view (~0 = unknown)
  unsigned long long* d_nnz;      // device view of the same word
  unsigned long long* d_acc;      // device counters {sum, slices done}
  bool aux_written;               // the auxiliary per-nonzero words of the current slices are valid
  bool dense_written;             // ... and so is their dense tile image
  bool sp_written;                // ... and so are the words of the structured-sparse tensor-core kernel (SliceArena::tcsp)
  float d_seen, d_seen_prev;      // density estimate at the last two multiplies (< 0: unknown): equal-ish = a stable regime
  bool captured;                  // the current slices were (are being) produced under stream capture
  size_t dense_bytes;
};

// 0 unknown (first call), 1 sparse, 2 dense according to the last completed slicing pass and the thresholds of
// launch_compute (common.cuh: tc_density_threshold)
static int density_hint(const SpmdmCtx* c, int is_bf16, bool transb, bool transc)
{
  const unsigned long long n = c->h_nnz ? *(volatile unsigned long long*)c->h_nnz : ~0ull;
  if (~0ull == n) return 0;
  const double thr = xb::tc_density_threshold(0 != is_bf16, transb, transc) * (double)c->g.m * (double)c->g.k;
  return ((double)n < thr) ? 1 : 2;   // either way the result is correct; a wrong guess only costs speed for one call
}

static float density_estimate(const SpmdmCtx* c)
{
  const unsigned long long n = c->h_nnz ? *(volatile unsigned long long*)c->h_nnz : ~0ull;
  return (~0ull == n) ? -1.f : (float)((double)n / ((double)c->g.m * (double)c->g.k));
}

// Called once per multiply: remembers the estimate this multiply sees and tells whether the one before saw about the same.
// When it did not (the matrices going through this handle change density, or this is the first estimate at all), the
// structured-sparse kernel is enqueued together with the dense one and the choice is made on the device (ComputeArgs::sp_guard):
// a dense matrix on the overflow path of K4s would cost milliseconds.
static void density_guard(SpmdmCtx* c, ComputeArgs* a)
{
  const float d = density_estimate(c);
  const float prev = c->d_seen;
  c->d_seen_prev = prev; c->d_seen = d;
  const bool stable = d >= 0.f && prev >= 0.f && prev <= 2.f * d && d <= 2.f * prev;
  a->sp_guard = (stable && !c->captured) ? 0 : 1;      // recorded into a graph: the replay may bring any matrix, the device decides every time
  a->sp_max_nnz = (unsigned long long)(0.03 * (double)c->g.m * (double)c->g.k);
}

static bool stream_is_capturing(cudaStream_t stream)
{
  cudaStreamCaptureStatus st = cudaStreamCaptureStatusNone;
  if (cudaSuccess != cudaStreamIsCapturing(stream, &st)) { (void)cudaGetLastError(); return false; }
  return cudaStreamCaptureStatusNone != st;
}

// dense_image = false: the slicing kernel cannot write the dense tile image (A in CSR or CSC form); an image left by an earlier
// pass is then stale and marked so.
static void slice_policy(SpmdmCtx* c, SliceArgs* a, int is_bf16, bool whole, cudaStream_t stream, bool dense_image = true)
{
  a->acc = c->d_acc; a->host_total = c->d_nnz; a->total_slices = c->g.mb * c->g.kb;
  a->write_dense = 0; a->write_sp = 0;
  if (!whole) {
    // legacy per-block call: the block gets its auxiliary words, its part of a dense image (if any) is now stale.  Whether
    // ALL slices carry auxiliary words is unchanged: they do only if the last whole pass wrote them.
    a->write_aux = 1;
    a->write_sp = 0;
    c->dense_written = false;
    c->sp_written = false;
    return;
  }
  // Under stream capture the decisions must not depend on the handle's history (the graph is replayed on other inputs) and
  // nothing may be allocated: the slices get their auxiliary words, and the dense image too if the handle already owns one;
  // the multiply then enqueues both kernel twins and the choice is made on the device from the slices' own counts.
  const bool capturing = stream_is_capturing(stream);
  c->captured = capturing;
  // the orientation of the multiply that will consume the slices is not known here: the auxiliary words are
  // skipped only when no orientation would take the tensor-core side (bf16: transposed panels always do)
  const bool skip = !capturing && !is_bf16 && 1 == density_hint(c, is_bf16, true, false);
  a->write_aux = skip ? 0 : 1;
  // Dense tile image for the tensor-core kernel (fp32, complete k-blocks; A stored m x k: 16-byte aligned rows): written
  // unless the last pass showed a matrix so sparse (< 1 %) that the CUDA-core kernels will multiply it whatever the
  // orientation of B and C.  Costs ~4 us of extra stores per 2048^2 and takes 50-90 us off the multiply.  Allocated and
  // zeroed on first use (rows and columns of partial tiles are never written and stay zero).
  // (A stored k x m goes through the strip kernel, which writes the image from its shared-memory tile: no alignment rule)
  if (dense_image && !is_bf16 && 0 == (c->g.k % 128) && c->simd_w > 1 && (a->transa || (0 == (a->lda & 3) && 0 == ((uintptr_t)a->a & 15)))) {
    const float d = density_estimate(c);
    if (capturing || d < 0.f || d >= 0.01f) {
      if (0 == c->arena.dense && !capturing) {
        const size_t tiles = (size_t)((c->g.bm + 127) / 128);
        c->dense_bytes = (size_t)c->g.mb * c->g.kb * tiles * 131072;
        if (cudaSuccess == cudaMalloc((void**)&c->arena.dense, c->dense_bytes)) XB_CUDA(cudaMemsetAsync(c->arena.dense, 0, c->dense_bytes, stream));   // once per handle, ordered before the slicing kernel
        else { (void)cudaGetLastError(); c->arena.dense = 0; }
        a->out.dense = c->arena.dense;
      }
      if (c->arena.dense) a->write_dense = 1;
    }
  }
  c->dense_written = (0 != a->write_dense);
  if (a->write_dense && !capturing) a->write_aux = 0;   // the image replaces the per-nonzero words: every tensor-core kernel that could read them reads the image instead
  c->aux_written = (0 != a->write_aux);
  // bf16: the word per nonzero the structured-sparse tensor-core kernel needs (one more array of the arena's capacity,
  // allocated when the first bf16 matrix shows up; never under capture)
  if (is_bf16 && a->write_aux) {
    if (0 == c->arena.tcsp && !capturing) {
      const size_t bytes = (size_t)c->g.mb * c->g.kb * (size_t)c->g.bm * c->g.bk * 4;
      const size_t list_bytes = (size_t)c->g.mb * c->g.kb * xb::kSpOvfCap * sizeof(uint2);
      if (cudaSuccess != cudaMalloc((void**)&c->arena.tcsp, bytes + list_bytes)) { (void)cudaGetLastError(); c->arena.tcsp = 0; }
      else c->arena.ovf_list = (uint2*)((char*)c->arena.tcsp + bytes);
    }
    a->out.tcsp = c->arena.tcsp; a->out.ovf_list = c->arena.ovf_list;
    a->write_sp = c->arena.tcsp ? 1 : 0;
  }
  c->sp_written = dense_image ? slices_get_sp_words(*a) : slices_sparse_get_sp_words(*a);
}

static int compute_policy(const SpmdmCtx* c, int is_bf16, bool transb, bool transc)
{
  if (!c->aux_written && !(c->dense_written && !is_bf16)) return 1;      // the slices carry neither auxiliary words nor the dense image: CUDA cores only
  if (c->captured) return 0;                                             // recorded into a graph: both twins, selected on the device at every replay
  return density_hint(c, is_bf16, transb, transc);
}

static std::mutex g_reg_mtx;
static std::unordered_map<const void*, SpmdmCtx*> g_registry;   // keyed by the slice arena address

static SpmdmCtx* find_ctx(const libxsmm_spmdm_handle* h)
{
  if (0 == h || 0 == h->base_ptr_scratch_A) { set_error(-10, "spmdm: handle not initialised"); return 0; }
  std::lock_guard<std::mutex> lock(g_reg_mtx);
  std::unordered_map<const void*, SpmdmCtx*>::const_iterator it = g_registry.find(h->base_ptr_scratch_A);
  if (it == g_registry.end()) { set_error(-11, "spmdm: unknown handle (not created by libxsmm_spmdm_init or already destroyed)"); return 0; }
  return it->second;
}

static bool is_device_ptr(const void* p)
{
  cudaPointerAttributes at;
  if (cudaSuccess != cudaPointerGetAttributes(&at, p)) { (void)cudaGetLastError(); return false; }
  return cudaMemoryTypeDevice == at.type || cudaMemoryTypeManaged == at.type;
}

static bool is_t(char c) { return 'T' == c || 't' == c; }

// Geometry of the reference (src/libxsmm_spmdm.c:552-608): bm = 512 or 256, bk = 128, bn bound to the
// instantiation (:557-583; here selected by LIBXSMM_B200_SPMDM_BN, default 48 = the AVX2 build every
// GCC build of the reference gets), then bm is lowered one row at a time while the imbalance estimate
// (biggest/mean block work x busiest/mean thread load) exceeds 1.1.
static void spmdm_geometry(int M, int N, int K, int max_threads, int bn, Geom* g)
{
  g->m = M; g->n = N; g->k = K;
  g->bm = (M >= 4096 || M <= 1024) ? 512 : 256;
  g->bn = bn; g->bk = 128;
  g->mb = (M + g->bm - 1) / g->bm;
  g->nb = (N + g->bn - 1) / g->bn;
  g->kb = (K + g->bk - 1) / g->bk;
  const double total = (double)((size_t)M * (size_t)N);
  for (;;) {
    const double per_block = (g->bm * g->bn) / (total / (double)((size_t)g->mb * (size_t)g->nb));
    const int busiest = (g->mb * g->nb + max_threads - 1) / max_threads;
    const double per_thread = busiest / ((double)g->mb * g->nb / max_threads);
    if (!(g->bm > 32 && per_block * per_thread > 1.1)) break;
    --g->bm;
    g->mb = (M + g->bm - 1) / g->bm;
  }
}

static ColModes spmdm_modes(const Geom& g, int simd_w)
{
  ColModes m;
  m.n_full_end = g.n; m.tail_from = g.n;
  if (simd_w > 1 && 0 != (g.n % g.bn)) {   // narrow last block (compute template :72-76)
    m.n_full_end = (g.n / g.bn) * g.bn;
    const int num_n = g.n - m.n_full_end;
    int full_regs = num_n / simd_w;
    if (full_regs > 0 && (full_regs % 2)) --full_regs;
    m.tail_from = m.n_full_end + full_regs * simd_w;
  }
  return m;
}

static cudaStream_t tid_stream(SpmdmCtx* c, int tid)
{
  std::lock_guard<std::mutex> lock(c->mtx);
  if (0 == c->streams[tid]) XB_CUDA(cudaStreamCreateWithFlags(&c->streams[tid], cudaStreamNonBlocking));
  return c->streams[tid];
}

static void slices_whole(const libxsmm_spmdm_handle* handle, char transa, const void* d_a, int is_bf16, cudaStream_t stream)
{
  SpmdmCtx* c = find_ctx(handle);
  if (0 == c) return;
  SliceArgs a;
  a.a = d_a; a.transa = is_t(transa); a.lda = a.transa ? c->g.m : c->g.k; a.is_bf16 = is_bf16;
  a.origin_is_block = 0; a.slice0 = 0; a.slice_step = 1; a.simd_w = c->simd_w; a.g = c->g; a.out = c->arena;
  slice_policy(c, &a, is_bf16, true, stream);
  launch_slices(a, c->g.mb * c->g.kb, stream);
}

// A in CSR or CSC form (device arrays): the argument checks and the slicing policy of both routes.  Returns false, after setting
// the error, when nothing may be launched.
static bool sparse_slices_setup(const libxsmm_spmdm_handle* handle, bool csc, const unsigned int* d_ptr, const unsigned int* d_idx,
                                const void* d_values, long long nnz, int is_bf16, cudaStream_t stream, SliceArgs* a)
{
  SpmdmCtx* c = find_ctx(handle);
  if (0 == c) return false;
  const char* form = csc ? "csc" : "csr";
  if (0 == d_ptr) { set_error(-90, "createSparseSlice_%s: NULL %s", form, csc ? "col_ptr" : "row_ptr"); return false; }
  if (nnz < 0 || nnz > 0xFFFFFFFFll) { set_error(-91, "createSparseSlice_%s: nnz=%lld outside [0, 2^32 - 1]", form, nnz); return false; }
  if (nnz > 0 && (0 == d_idx || 0 == d_values)) {
    set_error(-90, "createSparseSlice_%s: NULL %s or values with nnz=%lld", form, csc ? "row_idx" : "col_idx", nnz);
    return false;
  }
  a->a = 0; a->transa = csc ? 1 : 0; a->lda = csc ? c->g.m : c->g.k; a->is_bf16 = is_bf16;
  a->origin_is_block = 0; a->slice0 = 0; a->slice_step = 1; a->simd_w = c->simd_w; a->g = c->g; a->out = c->arena;
  slice_policy(c, a, is_bf16, true, stream, false);
  return true;
}

// A in CSR form (device arrays): the same slices as slices_whole() for the dense matrix holding these entries, transa = 'N'
static void slices_csr(const libxsmm_spmdm_handle* handle, const unsigned int* d_row_ptr, const unsigned int* d_col_idx,
                       const void* d_values, long long nnz, int is_bf16, cudaStream_t stream)
{
  SliceArgs a;
  if (!sparse_slices_setup(handle, false, d_row_ptr, d_col_idx, d_values, nnz, is_bf16, stream, &a)) return;
  CsrArgs csr;
  csr.row_ptr = d_row_ptr; csr.col_idx = d_col_idx; csr.values = d_values; csr.nnz = (uint32_t)nnz;
  launch_slices_csr(a, csr, stream);
}

// A in CSC form (device arrays; equally the CSR arrays of A stored k x m): the same slices as slices_whole() with transa = 'T' for
// the k x m array holding these entries, and as slices_csr() for A's CSR arrays
static void slices_csc(const libxsmm_spmdm_handle* handle, const unsigned int* d_col_ptr, const unsigned int* d_row_idx,
                       const void* d_values, long long nnz, int is_bf16, cudaStream_t stream)
{
  SliceArgs a;
  if (!sparse_slices_setup(handle, true, d_col_ptr, d_row_idx, d_values, nnz, is_bf16, stream, &a)) return;
  CscArgs csc;
  csc.col_ptr = d_col_ptr; csc.row_idx = d_row_idx; csc.values = d_values; csc.nnz = (uint32_t)nnz;
  launch_slices_csc(a, csc, stream);
}

static void compute_whole(const libxsmm_spmdm_handle* handle, char transb, char transc, float beta,
                          const void* d_b, float* d_c, int is_bf16, cudaStream_t stream)
{
  SpmdmCtx* c = find_ctx(handle);
  if (0 == c) return;
  ComputeArgs a = ComputeArgs();
  a.sl = c->arena; a.b = d_b; a.c = d_c;
  a.transb = is_t(transb); a.transc = is_t(transc); a.is_bf16 = is_bf16;
  a.ldb = a.transb ? c->g.k : c->g.n;
  a.ldc = a.transc ? c->g.m : c->g.n;
  a.beta = beta; a.g = c->g; a.mb_first = 0; a.mb_count = c->g.mb;
  a.row_origin = 0; a.col_origin = 0; a.ncols = c->g.n; a.modes = spmdm_modes(c->g, c->simd_w); a.tc_twin = 0; a.tc_min_nnz = 0; a.tc_hint = compute_policy(c, is_bf16, 0 != a.transb, 0 != a.transc); a.density_hint = density_estimate(c); a.dense_valid = (c->dense_written && !is_bf16) ? 1 : 0; a.aux_valid = c->aux_written ? 1 : 0; a.sp_valid = (c->sp_written && c->aux_written) ? 1 : 0;
  density_guard(c, &a);
  launch_compute(a, stream);
}

// legacy per-block slice creation (reference src/libxsmm_spmdm.c:253-272 / :328-347)
static void slice_block(const libxsmm_spmdm_handle* handle, char transa, const void* a_in, int is_bf16, int block_id, int tid)
{
  SpmdmCtx* c = find_ctx(handle);
  if (0 == c) return;
  const Geom& g = c->g;
  if (block_id < 0 || block_id >= g.mb * g.kb || tid < 0 || tid >= c->max_threads) { set_error(-12, "createSparseSlice: block_id/tid out of range"); return; }
  const cudaStream_t st = tid_stream(c, tid);
  const size_t esz = is_bf16 ? 2 : 4;
  const int kb = block_id / g.mb, mbi = block_id % g.mb;
  const int nrows = (g.bm < g.m - mbi * g.bm) ? g.bm : (g.m - mbi * g.bm);
  const int ncols = (g.bk < g.k - kb * g.bk) ? g.bk : (g.k - kb * g.bk);
  SliceArgs a;
  a.transa = is_t(transa); a.is_bf16 = is_bf16; a.slice0 = block_id; a.slice_step = 1; a.simd_w = c->simd_w; a.g = g; a.out = c->arena;
  if (is_device_ptr(a_in)) {
    a.a = a_in; a.lda = a.transa ? g.m : g.k; a.origin_is_block = 0;
  }
  else {   // host matrix: stage this block in the tid's slab
    char* slab = c->staging + (size_t)tid * c->staging_per_tid;
    if (!a.transa) {
      const char* src = (const char*)a_in + ((size_t)mbi * g.bm * g.k + (size_t)kb * g.bk) * esz;
      XB_CUDA(cudaMemcpy2DAsync(slab, ncols * esz, src, (size_t)g.k * esz, ncols * esz, nrows, cudaMemcpyHostToDevice, st));
      a.lda = ncols;
    }
    else {
      const char* src = (const char*)a_in + ((size_t)kb * g.bk * g.m + (size_t)mbi * g.bm) * esz;
      XB_CUDA(cudaMemcpy2DAsync(slab, nrows * esz, src, (size_t)g.m * esz, nrows * esz, ncols, cudaMemcpyHostToDevice, st));
      a.lda = nrows;
    }
    a.a = slab; a.origin_is_block = 1;
  }
  slice_policy(c, &a, is_bf16, false, (cudaStream_t)0);
  launch_slices(a, 1, st);
  XB_CUDA(cudaStreamSynchronize(st));
}

// legacy per-block compute (reference src/libxsmm_spmdm.c:418-442 / :513-537)
static void compute_block(const libxsmm_spmdm_handle* handle, char transb, char transc, float beta,
                          const void* b_in, float* c_in, int is_bf16, int block_id, int tid)
{
  SpmdmCtx* c = find_ctx(handle);
  if (0 == c) return;
  const Geom& g = c->g;
  if (block_id < 0 || block_id >= g.mb * g.nb || tid < 0 || tid >= c->max_threads) { set_error(-13, "compute: block_id/tid out of range"); return; }
  const cudaStream_t st = tid_stream(c, tid);
  const size_t esz = is_bf16 ? 2 : 4;
  const int mbi = block_id / g.nb, nbi = block_id % g.nb;
  const int m0 = mbi * g.bm, n0 = nbi * g.bn;
  const int num_m = (g.bm < g.m - m0) ? g.bm : (g.m - m0);
  const int num_n = (g.bn < g.n - n0) ? g.bn : (g.n - n0);
  const bool tb = is_t(transb), tc = is_t(transc);
  const bool dev_b = is_device_ptr(b_in), dev_c = is_device_ptr(c_in);
  ComputeArgs a = ComputeArgs();
  a.sl = c->arena; a.transb = tb; a.transc = tc; a.is_bf16 = is_bf16; a.beta = beta; a.g = g;
  a.mb_first = mbi; a.mb_count = 1; a.col_origin = n0; a.ncols = num_n; a.modes = spmdm_modes(g, c->simd_w); a.tc_twin = -1; a.tc_min_nnz = 0; a.tc_hint = 1; a.density_hint = -1.f; a.dense_valid = 0; a.aux_valid = 0; a.sp_valid = 0; a.sp_guard = 0; a.sp_max_nnz = 0;   // legacy block: no tensor-core twin
  char* slab = c->staging + (size_t)tid * c->staging_per_tid;
  const size_t slab_b_bytes = (((size_t)g.k * g.bn * 4) + 255) & ~(size_t)255;
  float* c_stage = (float*)(slab + slab_b_bytes);
  if (dev_b) {
    a.b = (const char*)b_in + (tb ? (size_t)n0 * g.k : (size_t)n0) * esz;
    a.ldb = tb ? g.k : g.n;
  }
  else if (!tb) {
    XB_CUDA(cudaMemcpy2DAsync(slab, num_n * esz, (const char*)b_in + (size_t)n0 * esz, (size_t)g.n * esz, num_n * esz, g.k, cudaMemcpyHostToDevice, st));
    a.b = slab; a.ldb = num_n;
  }
  else {
    XB_CUDA(cudaMemcpyAsync(slab, (const char*)b_in + (size_t)n0 * g.k * esz, (size_t)num_n * g.k * esz, cudaMemcpyHostToDevice, st));
    a.b = slab; a.ldb = g.k;
  }
  if (dev_c) {
    a.c = c_in + (tc ? (size_t)n0 * g.m : (size_t)n0);
    a.ldc = tc ? g.m : g.n; a.row_origin = 0;
  }
  else {
    a.c = c_stage; a.row_origin = m0; a.ldc = tc ? num_m : num_n;
    if (0.f != beta) {
      if (!tc) XB_CUDA(cudaMemcpy2DAsync(c_stage, num_n * 4, c_in + (size_t)m0 * g.n + n0, (size_t)g.n * 4, num_n * 4, num_m, cudaMemcpyHostToDevice, st));
      else XB_CUDA(cudaMemcpy2DAsync(c_stage, num_m * 4, c_in + (size_t)n0 * g.m + m0, (size_t)g.m * 4, num_m * 4, num_n, cudaMemcpyHostToDevice, st));
    }
  }
  launch_compute(a, st);
  if (!dev_c) {
    if (!tc) XB_CUDA(cudaMemcpy2DAsync(c_in + (size_t)m0 * g.n + n0, (size_t)g.n * 4, c_stage, num_n * 4, num_n * 4, num_m, cudaMemcpyDeviceToHost, st));
    else XB_CUDA(cudaMemcpy2DAsync(c_in + (size_t)n0 * g.m + m0, (size_t)g.m * 4, c_stage, num_m * 4, num_m * 4, num_n, cudaMemcpyDeviceToHost, st));
  }
  XB_CUDA(cudaStreamSynchronize(st));
}

}  // namespace xb

using namespace xb;

// =====================================================================================================
// SPMDM
// =====================================================================================================
extern "C" {

void libxsmm_spmdm_init(int M, int N, int K, int max_threads, libxsmm_spmdm_handle* handle,
                        libxsmm_CSR_sparseslice** libxsmm_output_csr)
{
  if (0 == handle) { set_error(-20, "spmdm_init: NULL handle"); return; }
  memset(handle, 0, sizeof(*handle));
  if (libxsmm_output_csr) *libxsmm_output_csr = 0;
  if (M <= 0 || N <= 0 || K <= 0) { set_error(-21, "spmdm_init: empty problem %dx%dx%d", M, N, K); handle->m = M; handle->n = N; handle->k = K; return; }
  if (max_threads < 1) max_threads = 1;
  int bn = 48;
  const char* env = getenv("LIBXSMM_B200_SPMDM_BN");
  if (env && *env) { const int v = atoi(env); if (96 == v || 48 == v || 6 == v) bn = v; }
  SpmdmCtx* c = new SpmdmCtx();
  spmdm_geometry(M, N, K, max_threads, bn, &c->g);
  c->simd_w = (96 == bn) ? 16 : ((48 == bn) ? 8 : 1);
  c->max_threads = max_threads;
  c->streams.assign((size_t)max_threads, (cudaStream_t)0);
  c->d_a = 0; c->d_b = 0; c->d_c = 0; c->d_a_bytes = c->d_b_bytes = c->d_c_bytes = 0;
  c->xs[0] = c->xs[1] = c->xs[2] = 0;
  for (int i = 0; i <= kExecPanels; ++i) c->xev[i] = 0;
  const Geom& g = c->g;
  const size_t ns = (size_t)g.mb * g.kb, cap = (size_t)g.bm * g.bk;
  const size_t row_bytes = ((ns * (g.bm + 1) * 2) + 255) & ~(size_t)255;
  const size_t col_bytes = ns * cap * 2, val_bytes = ns * cap * 4;
  c->arena_base = 0; c->staging = 0; c->table = 0;
  const size_t nnz_bytes = ((ns * 4) + 255) & ~(size_t)255;
  XB_CUDA(cudaMalloc(&c->arena_base, row_bytes + col_bytes + val_bytes + val_bytes + nnz_bytes + nnz_bytes));
  // per-tid staging slab for the legacy per-block entries on HOST matrices: an A block, or a B panel
  // (k x bn) followed by a C tile (bm x bn); the reference's slab holds the latter two (:148-155)
  {
    const size_t a_blk = cap * 4;
    const size_t bc = ((((size_t)g.k * g.bn * 4) + 255) & ~(size_t)255) + (size_t)g.bm * g.bn * 4;
    size_t per = a_blk > bc ? a_blk : bc;
    per = (per + 4095) & ~(size_t)4095;
    c->staging_per_tid = per;
    XB_CUDA(cudaMalloc((void**)&c->staging, per * (size_t)max_threads));
  }
  if (0 == c->arena_base || 0 == c->staging) {   // the reference leaves NULL pointers on failure (:140-144,165-168)
    if (c->arena_base) cudaFree(c->arena_base);
    if (c->staging) cudaFree(c->staging);
    delete c;
    handle->m = M; handle->n = N; handle->k = K;
    return;
  }
  c->arena.rowidx = (uint16_t*)c->arena_base;
  c->arena.colidx = (uint16_t*)((char*)c->arena_base + row_bytes);
  c->arena.values = (float*)((char*)c->arena_base + row_bytes + col_bytes);
  c->arena.tcoff = (uint16_t*)((char*)c->arena_base + row_bytes + col_bytes + val_bytes);
  c->arena.tcpk = (uint32_t*)c->arena.tcoff;     // 4 bytes per entry: bf16 slices keep a 32-bit word per nonzero
  c->arena.slice_nnz = (uint32_t*)((char*)c->arena_base + row_bytes + col_bytes + val_bytes + val_bytes);
  c->arena.slice_ovf = (uint32_t*)((char*)c->arena.slice_nnz + nnz_bytes);
  XB_CUDA(cudaMemset(c->arena.slice_nnz, 0, nnz_bytes + nnz_bytes));
  c->h_nnz = 0; c->d_nnz = 0; c->d_acc = 0; c->aux_written = false; c->dense_written = false; c->sp_written = false; c->d_seen = -1.f; c->d_seen_prev = -1.f; c->captured = false; c->dense_bytes = 0; c->arena.dense = 0; c->arena.tcsp = 0; c->arena.ovf_list = 0;
  if (cudaSuccess == cudaHostAlloc((void**)&c->h_nnz, sizeof(unsigned long long), cudaHostAllocMapped)) {
    *c->h_nnz = ~0ull;
    if (cudaSuccess != cudaHostGetDevicePointer((void**)&c->d_nnz, c->h_nnz, 0)) c->d_nnz = 0;
  }
  else { (void)cudaGetLastError(); c->h_nnz = 0; }
  XB_CUDA(cudaMalloc((void**)&c->d_acc, 2 * sizeof(unsigned long long)));
  if (c->d_acc) XB_CUDA(cudaMemset(c->d_acc, 0, 2 * sizeof(unsigned long long)));
  c->table = (libxsmm_CSR_sparseslice*)malloc(sizeof(libxsmm_CSR_sparseslice) * ns);
  for (size_t s = 0; s < ns; ++s) {
    c->table[s].rowidx = c->arena.rowidx + s * (g.bm + 1);
    c->table[s].colidx = c->arena.colidx + s * cap;
    c->table[s].values = c->arena.values + s * cap;
  }
  handle->m = g.m; handle->n = g.n; handle->k = g.k;
  handle->bm = g.bm; handle->bn = g.bn; handle->bk = g.bk;
  handle->mb = g.mb; handle->nb = g.nb; handle->kb = g.kb;
  handle->datatype = LIBXSMM_SPMDM_DATATYPE_F32;
  handle->base_ptr_scratch_A = (char*)c->arena_base;
  handle->base_ptr_scratch_B_scratch_C = c->staging;
  handle->memory_for_scratch_per_thread = (int)(c->staging_per_tid > (size_t)INT_MAX ? INT_MAX : c->staging_per_tid);
  if (libxsmm_output_csr) *libxsmm_output_csr = c->table;
  {
    std::lock_guard<std::mutex> lock(g_reg_mtx);
    g_registry[c->arena_base] = c;
  }
  if (verbosity() > 0) fprintf(stderr, "LIBXSMM_B200 spmdm_init: %dx%dx%d bm=%d bn=%d bk=%d mb=%d nb=%d kb=%d\n", M, N, K, g.bm, g.bn, g.bk, g.mb, g.nb, g.kb);
}

void libxsmm_spmdm_destroy(libxsmm_spmdm_handle* handle)
{
  if (0 == handle || 0 == handle->base_ptr_scratch_A) return;
  SpmdmCtx* c = 0;
  {
    std::lock_guard<std::mutex> lock(g_reg_mtx);
    std::unordered_map<const void*, SpmdmCtx*>::iterator it = g_registry.find(handle->base_ptr_scratch_A);
    if (it != g_registry.end()) { c = it->second; g_registry.erase(it); }
  }
  if (c) {
    for (size_t i = 0; i < c->streams.size(); ++i) if (c->streams[i]) { cudaStreamSynchronize(c->streams[i]); cudaStreamDestroy(c->streams[i]); }
    for (int i = 0; i < 3; ++i) if (c->xs[i]) { cudaStreamSynchronize(c->xs[i]); cudaStreamDestroy(c->xs[i]); }
    for (int i = 0; i <= kExecPanels; ++i) if (c->xev[i]) cudaEventDestroy(c->xev[i]);
    for (size_t i = 0; i < c->xup.size(); ++i) { if (c->xup[i]) cudaEventDestroy(c->xup[i]); if (c->xdone[i]) cudaEventDestroy(c->xdone[i]); }
    if (c->d_a) cudaFree(c->d_a);
    if (c->d_b) cudaFree(c->d_b);
    if (c->d_c) cudaFree(c->d_c);
    cudaFree(c->arena_base);
    if (c->arena.dense) cudaFree(c->arena.dense);
    if (c->arena.tcsp) cudaFree(c->arena.tcsp);
    cudaFree(c->staging);
    if (c->d_acc) cudaFree(c->d_acc);
    if (c->h_nnz) cudaFreeHost(c->h_nnz);
    free(c->table);
    delete c;
  }
  handle->base_ptr_scratch_A = 0;              // like the reference (:173-179): arenas go, the handle stays
  handle->base_ptr_scratch_B_scratch_C = 0;
}

int libxsmm_spmdm_get_num_createSparseSlice_blocks(const libxsmm_spmdm_handle* handle) { return handle->mb * handle->kb; }
int libxsmm_spmdm_get_num_compute_blocks(const libxsmm_spmdm_handle* handle) { return handle->mb * handle->nb; }

void libxsmm_spmdm_createSparseSlice_fp32_thread(const libxsmm_spmdm_handle* handle, char transa, const float* a,
  libxsmm_CSR_sparseslice* libxsmm_output_csr_a, int block_id, int tid, int nthreads)
{
  (void)libxsmm_output_csr_a; (void)nthreads;
  slice_block(handle, transa, a, 0, block_id, tid);
}

void libxsmm_spmdm_createSparseSlice_bfloat16_thread(const libxsmm_spmdm_handle* handle, char transa, const libxsmm_bfloat16* a,
  libxsmm_CSR_sparseslice* libxsmm_output_csr_a, int block_id, int tid, int nthreads)
{
  (void)libxsmm_output_csr_a; (void)nthreads;
  slice_block(handle, transa, a, 1, block_id, tid);
}

void libxsmm_spmdm_compute_fp32_thread(const libxsmm_spmdm_handle* handle, char transa, char transb, const float* alpha,
  libxsmm_CSR_sparseslice* a_sparse, const float* b, char transc, const float* beta, float* c, int block_id, int tid, int nthreads)
{
  (void)transa; (void)alpha; (void)a_sparse; (void)nthreads;   // transa/alpha unused like the reference (tpl.c:60-61)
  compute_block(handle, transb, transc, *beta, b, c, 0, block_id, tid);
}

void libxsmm_spmdm_compute_bfloat16_thread(const libxsmm_spmdm_handle* handle, char transa, char transb, const libxsmm_bfloat16* alpha,
  libxsmm_CSR_sparseslice* a_sparse, const libxsmm_bfloat16* b, char transc, const libxsmm_bfloat16* beta, float* c,
  int block_id, int tid, int nthreads)
{
  (void)transa; (void)alpha; (void)a_sparse; (void)nthreads;
  // the reference converts the raw 16-bit pattern as an INTEGER (bf16 tpl.c:91,113,164): mirrored
  compute_block(handle, transb, transc, (float)(*beta), b, c, 1, block_id, tid);
}

// ---- stream-ordered whole-problem entries -----------------------------------------------------------
void libxsmm_spmdm_createSparseSlice_fp32_stream(const libxsmm_spmdm_handle* handle, char transa, const float* d_a,
  libxsmm_CSR_sparseslice* libxsmm_output_csr_a, void* stream)
{
  (void)libxsmm_output_csr_a;
  slices_whole(handle, transa, d_a, 0, (cudaStream_t)stream);
}

void libxsmm_spmdm_createSparseSlice_bfloat16_stream(const libxsmm_spmdm_handle* handle, char transa, const libxsmm_bfloat16* d_a,
  libxsmm_CSR_sparseslice* libxsmm_output_csr_a, void* stream)
{
  (void)libxsmm_output_csr_a;
  slices_whole(handle, transa, d_a, 1, (cudaStream_t)stream);
}

void libxsmm_spmdm_createSparseSlice_csr_fp32_stream(const libxsmm_spmdm_handle* handle, const unsigned int* d_row_ptr,
  const unsigned int* d_col_idx, const float* d_values, long long nnz, libxsmm_CSR_sparseslice* libxsmm_output_csr_a, void* stream)
{
  (void)libxsmm_output_csr_a;
  slices_csr(handle, d_row_ptr, d_col_idx, d_values, nnz, 0, (cudaStream_t)stream);
}

void libxsmm_spmdm_createSparseSlice_csr_bfloat16_stream(const libxsmm_spmdm_handle* handle, const unsigned int* d_row_ptr,
  const unsigned int* d_col_idx, const libxsmm_bfloat16* d_values, long long nnz, libxsmm_CSR_sparseslice* libxsmm_output_csr_a,
  void* stream)
{
  (void)libxsmm_output_csr_a;
  slices_csr(handle, d_row_ptr, d_col_idx, d_values, nnz, 1, (cudaStream_t)stream);
}

void libxsmm_spmdm_createSparseSlice_csc_fp32_stream(const libxsmm_spmdm_handle* handle, const unsigned int* d_col_ptr,
  const unsigned int* d_row_idx, const float* d_values, long long nnz, libxsmm_CSR_sparseslice* libxsmm_output_csr_a, void* stream)
{
  (void)libxsmm_output_csr_a;
  slices_csc(handle, d_col_ptr, d_row_idx, d_values, nnz, 0, (cudaStream_t)stream);
}

void libxsmm_spmdm_createSparseSlice_csc_bfloat16_stream(const libxsmm_spmdm_handle* handle, const unsigned int* d_col_ptr,
  const unsigned int* d_row_idx, const libxsmm_bfloat16* d_values, long long nnz, libxsmm_CSR_sparseslice* libxsmm_output_csr_a,
  void* stream)
{
  (void)libxsmm_output_csr_a;
  slices_csc(handle, d_col_ptr, d_row_idx, d_values, nnz, 1, (cudaStream_t)stream);
}

void libxsmm_spmdm_compute_fp32_stream(const libxsmm_spmdm_handle* handle, char transa, char transb, const float* alpha,
  libxsmm_CSR_sparseslice* a_sparse, const float* d_b, char transc, const float* beta, float* d_c, void* stream)
{
  (void)transa; (void)alpha; (void)a_sparse;
  compute_whole(handle, transb, transc, *beta, d_b, d_c, 0, (cudaStream_t)stream);
}

void libxsmm_spmdm_compute_bfloat16_stream(const libxsmm_spmdm_handle* handle, char transa, char transb, const libxsmm_bfloat16* alpha,
  libxsmm_CSR_sparseslice* a_sparse, const libxsmm_bfloat16* d_b, char transc, const libxsmm_bfloat16* beta, float* d_c, void* stream)
{
  (void)transa; (void)alpha; (void)a_sparse;
  compute_whole(handle, transb, transc, (float)(*beta), d_b, d_c, 1, (cudaStream_t)stream);
}

void libxsmm_spmdm_exec_stream(const libxsmm_spmdm_handle* handle, libxsmm_CSR_sparseslice* slices,
  libxsmm_spmdm_datatype datatype, char transa, char transb, char transc, const void* d_a, const void* d_b,
  const void* beta, float* d_c, void* stream)
{
  (void)slices;
  const int is_bf16 = (LIBXSMM_SPMDM_DATATYPE_BFLOAT16 == datatype);
  const float beta_f = is_bf16 ? (float)(*(const libxsmm_bfloat16*)beta) : *(const float*)beta;
  slices_whole(handle, transa, d_a, is_bf16, (cudaStream_t)stream);
  compute_whole(handle, transb, transc, beta_f, d_b, d_c, is_bf16, (cudaStream_t)stream);
}

void libxsmm_spmdm_exec_host(const libxsmm_spmdm_handle* handle, libxsmm_CSR_sparseslice* slices,
  libxsmm_spmdm_datatype datatype, char transa, char transb, char transc, const void* a, const void* b,
  const void* beta, float* c_host)
{
  (void)slices;
  SpmdmCtx* c = find_ctx(handle);
  if (0 == c) return;
  std::lock_guard<std::mutex> lock(c->mtx);
  const Geom& g = c->g;
  const int is_bf16 = (LIBXSMM_SPMDM_DATATYPE_BFLOAT16 == datatype);
  const size_t esz = is_bf16 ? 2 : 4;
  const size_t a_bytes = (size_t)g.m * g.k * esz, b_bytes = (size_t)g.k * g.n * esz, c_bytes = (size_t)g.m * g.n * 4;
  const float beta_f = is_bf16 ? (float)(*(const libxsmm_bfloat16*)beta) : *(const float*)beta;
  const bool tb = is_t(transb), tc = is_t(transc);
  auto grow = [](void** p, size_t* have, size_t need) {       // the recorded size changes only when the allocation succeeded: a later call retries
    if (*have >= need && 0 != *p) return;
    if (*p) cudaFree(*p);
    *p = 0; *have = 0;
    XB_CUDA(cudaMalloc(p, need));
    if (*p) *have = need;
  };
  grow(&c->d_a, &c->d_a_bytes, a_bytes);
  grow(&c->d_b, &c->d_b_bytes, b_bytes);
  grow((void**)&c->d_c, &c->d_c_bytes, c_bytes);
  if (0 == c->xs[0]) {
    for (int i = 0; i < 3; ++i) XB_CUDA(cudaStreamCreateWithFlags(&c->xs[i], cudaStreamNonBlocking));
    for (int i = 0; i < kExecPanels + 1; ++i) XB_CUDA(cudaEventCreateWithFlags(&c->xev[i], cudaEventDisableTiming));
  }
  if (0 == c->d_a || 0 == c->d_b || 0 == c->d_c) return;
  // Three streams: xs[0] uploads, xs[1] kernels, xs[2] downloads (PCIe is full duplex).  The problem is cut
  // into mb row blocks x np column panels.  Diagonal step d uploads A's row block d and B's panel d; that makes
  // the tiles (d, c <= d) and (r < d, d) computable, so the number of finished C tiles grows quadratically
  // while the uploads proceed linearly and the download of C (the largest transfer) starts after 1/mb + 1/np
  // of the inputs instead of after all of A.  Column panels are contiguous row ranges of B / C when those are
  // stored transposed, strided 2-D copies otherwise.
  const ColModes modes = spmdm_modes(g, c->simd_w);
  const bool ta = is_t(transa);
  int np = kExecPanels;
  { const char* e = getenv("LIBXSMM_B200_EXEC_PANELS"); if (e && *e) { const int v = atoi(e); if (v >= 1 && v <= 64) np = v; } }
  // panel boundaries are multiples of 256 columns so that every launch keeps whole CTA tiles and the
  // reference's column modes (defined on global column numbers) are unaffected by the split
  int pw = (((g.n + np - 1) / np) + 255) / 256 * 256;
  if (pw <= 0) pw = 256;
  np = (g.n + pw - 1) / pw;
  const int nd = (g.mb > np) ? g.mb : np;
  if ((int)c->xdone.size() < nd) {
    const size_t old = c->xdone.size();
    c->xdone.resize((size_t)nd, (cudaEvent_t)0); c->xup.resize((size_t)nd, (cudaEvent_t)0);
    for (size_t i = old; i < (size_t)nd; ++i) {
      XB_CUDA(cudaEventCreateWithFlags(&c->xdone[i], cudaEventDisableTiming));
      XB_CUDA(cudaEventCreateWithFlags(&c->xup[i], cudaEventDisableTiming));
    }
  }
  // LIBXSMM_B200_EXEC_TRACE=1: per-step timeline (developer aid; timing events on all three streams)
  static const bool trace = [] { const char* e = getenv("LIBXSMM_B200_EXEC_TRACE"); return e && '1' == *e; }();
  std::vector<cudaEvent_t> tev;
  if (trace) { tev.resize((size_t)(3 * nd + 1)); for (size_t i = 0; i < tev.size(); ++i) XB_CUDA(cudaEventCreate(&tev[i])); XB_CUDA(cudaEventRecord(tev[3 * nd], c->xs[0])); }
  int write_aux = 1, write_dense = 0; bool first_block = true;
  // a rectangle of C: row blocks [r0, r0 + rc) x columns [n0, n0 + w)
  auto rect = [&](int r0, int rc, int n0, int w, int* m0, int* rows) {
    *m0 = r0 * g.bm;
    const int mend = ((r0 + rc) * g.bm < g.m) ? (r0 + rc) * g.bm : g.m;
    *rows = mend - *m0;
    (void)n0; (void)w;
  };
  auto copy_rect = [&](int r0, int rc, int n0, int w, bool up) {
    int m0, rows; rect(r0, rc, n0, w, &m0, &rows);
    if (rows <= 0 || w <= 0) return;
    float* dptr = tc ? (c->d_c + (size_t)n0 * g.m + m0) : (c->d_c + (size_t)m0 * g.n + n0);
    float* hptr = tc ? (c_host + (size_t)n0 * g.m + m0) : (c_host + (size_t)m0 * g.n + n0);
    const size_t pitch = (size_t)(tc ? g.m : g.n) * 4, width = (size_t)(tc ? rows : w) * 4, height = (size_t)(tc ? w : rows);
    if (up) XB_CUDA(cudaMemcpy2DAsync(dptr, pitch, hptr, pitch, width, height, cudaMemcpyHostToDevice, c->xs[0]));
    else XB_CUDA(cudaMemcpy2DAsync(hptr, pitch, dptr, pitch, width, height, cudaMemcpyDeviceToHost, c->xs[2]));
  };
  auto compute_rect = [&](int r0, int rc, int n0, int w) {
    if (rc <= 0 || w <= 0) return;
    ComputeArgs ca = ComputeArgs();
    ca.sl = c->arena; ca.transb = tb; ca.transc = tc; ca.is_bf16 = is_bf16;
    ca.ldb = tb ? g.k : g.n; ca.ldc = tc ? g.m : g.n;
    ca.b = (const char*)c->d_b + (tb ? (size_t)n0 * g.k : (size_t)n0) * esz;
    ca.c = c->d_c + (tc ? (size_t)n0 * g.m : (size_t)n0);
    ca.beta = beta_f; ca.g = g; ca.mb_first = r0; ca.mb_count = rc;
    ca.row_origin = 0; ca.col_origin = n0; ca.ncols = w; ca.modes = modes; ca.tc_twin = 0; ca.tc_min_nnz = 0; ca.tc_hint = compute_policy(c, is_bf16, tb, tc); ca.density_hint = density_estimate(c); ca.dense_valid = (c->dense_written && !is_bf16) ? 1 : 0; ca.aux_valid = c->aux_written ? 1 : 0; ca.sp_valid = (c->sp_written && c->aux_written) ? 1 : 0;
    density_guard(c, &ca);
    launch_compute(ca, c->xs[1]);
  };
  for (int d = 0; d < nd; ++d) {
    // rectangles that become computable in step d: the new row block against all panels uploaded so far
    // (including panel d), and the new panel against all earlier row blocks
    const int row_cols = ((d < np) ? (d + 1) * pw : g.n) < g.n ? ((d < np) ? (d + 1) * pw : g.n) : g.n;   // columns [0, row_cols) of row block d
    const int col_n0 = d * pw, col_w = (d < np) ? ((g.n - col_n0 < pw) ? (g.n - col_n0) : pw) : 0;      // panel d
    const int col_rows = (d < g.mb) ? d : g.mb;                                                          // row blocks [0, col_rows) of panel d
    // ---- uploads of step d ----
    if (d < g.mb) {
      const int m0 = d * g.bm, rows = (g.bm < g.m - m0) ? g.bm : (g.m - m0);
      if (!ta) XB_CUDA(cudaMemcpyAsync((char*)c->d_a + (size_t)m0 * g.k * esz, (const char*)a + (size_t)m0 * g.k * esz, (size_t)rows * g.k * esz, cudaMemcpyHostToDevice, c->xs[0]));
      else XB_CUDA(cudaMemcpy2DAsync((char*)c->d_a + (size_t)m0 * esz, (size_t)g.m * esz, (const char*)a + (size_t)m0 * esz, (size_t)g.m * esz, (size_t)rows * esz, g.k, cudaMemcpyHostToDevice, c->xs[0]));
    }
    if (d < np) {
      char* db = (char*)c->d_b; const char* hb = (const char*)b;
      cudaStream_t sb = c->xs[0];
      if (tb) XB_CUDA(cudaMemcpyAsync(db + (size_t)col_n0 * g.k * esz, hb + (size_t)col_n0 * g.k * esz, (size_t)col_w * g.k * esz, cudaMemcpyHostToDevice, sb));
      else XB_CUDA(cudaMemcpy2DAsync(db + (size_t)col_n0 * esz, (size_t)g.n * esz, hb + (size_t)col_n0 * esz, (size_t)g.n * esz, (size_t)col_w * esz, g.k, cudaMemcpyHostToDevice, sb));
    }
    if (0.f != beta_f) {   // beta != 0: the C rectangles go up before they are needed
      if (d < g.mb) copy_rect(d, 1, 0, row_cols, true);
      if (d < np) copy_rect(0, col_rows, col_n0, col_w, true);
    }
    XB_CUDA(cudaEventRecord(c->xup[d], c->xs[0]));
    if (trace) XB_CUDA(cudaEventRecord(tev[3 * d], c->xs[0]));
    // ---- kernels of step d: at most one slicing launch and two compute launches ----
    XB_CUDA(cudaStreamWaitEvent(c->xs[1], c->xup[d], 0));
    if (d < g.mb) {
      SliceArgs sa;
      sa.a = c->d_a; sa.transa = ta; sa.lda = ta ? g.m : g.k; sa.is_bf16 = is_bf16;
      sa.origin_is_block = 0; sa.slice0 = d; sa.slice_step = g.mb; sa.simd_w = c->simd_w; sa.g = g; sa.out = c->arena;
      slice_policy(c, &sa, is_bf16, true, c->xs[1]);
      if (first_block) { write_aux = sa.write_aux; write_dense = sa.write_dense; first_block = false; }
      sa.write_aux = write_aux;                 // one decision for all row blocks of this multiply
      sa.write_dense = (write_dense && c->arena.dense) ? 1 : 0;
      sa.out = c->arena;
      sa.write_sp = (is_bf16 && write_aux && c->arena.tcsp) ? 1 : 0;
      c->aux_written = (0 != write_aux);
      c->sp_written = slices_get_sp_words(sa);
      c->dense_written = (0 != sa.write_dense);
      c->captured = false;
      launch_slices(sa, g.kb, c->xs[1]);
      compute_rect(d, 1, 0, row_cols);
    }
    if (d < np) compute_rect(0, col_rows, col_n0, col_w);
    XB_CUDA(cudaEventRecord(c->xdone[d], c->xs[1]));
    if (trace) XB_CUDA(cudaEventRecord(tev[3 * d + 1], c->xs[1]));
    // ---- downloads of step d ----
    XB_CUDA(cudaStreamWaitEvent(c->xs[2], c->xdone[d], 0));
    if (d < g.mb) copy_rect(d, 1, 0, row_cols, false);
    if (d < np) copy_rect(0, col_rows, col_n0, col_w, false);
    if (trace) XB_CUDA(cudaEventRecord(tev[3 * d + 2], c->xs[2]));
  }
  XB_CUDA(cudaStreamSynchronize(c->xs[2]));
  XB_CUDA(cudaStreamSynchronize(c->xs[0]));
  if (trace) {
    for (int d = 0; d < nd; ++d) {
      float t[3] = { 0, 0, 0 };
      for (int i = 0; i < 3; ++i) (void)cudaEventElapsedTime(&t[i], tev[3 * nd], tev[3 * d + i]);
      fprintf(stderr, "exec_host step %2d: uploaded %7.3f ms  computed %7.3f ms  downloaded %7.3f ms\n", d, t[0], t[1], t[2]);
    }
    for (size_t i = 0; i < tev.size(); ++i) cudaEventDestroy(tev[i]);
  }
}

// =====================================================================================================
// FSSPMDM
// =====================================================================================================
struct libxsmm_dfsspmdm;
struct libxsmm_sfsspmdm;

// staging contexts of the host-pointer execute path: one per concurrent caller and device, recycled through a free list
struct FsStaging {
  static const int kSlots = 3;
  int device;
  cudaStream_t st[kSlots];
  char* dB[kSlots];
  char* dC[kSlots];
  size_t capB[kSlots], capC[kSlots];
};
static std::mutex g_fs_pool_mtx;
static std::vector<FsStaging*> g_fs_pool;     // idle contexts (all devices)

static FsStaging* fs_staging_acquire()
{
  int dev = 0;
  if (cudaSuccess != cudaGetDevice(&dev)) { (void)cudaGetLastError(); set_error(-32, "fsspmdm_execute: no current device"); return 0; }
  {
    std::lock_guard<std::mutex> lock(g_fs_pool_mtx);
    for (size_t i = 0; i < g_fs_pool.size(); ++i) if (g_fs_pool[i]->device == dev) {
      FsStaging* sg = g_fs_pool[i];
      g_fs_pool.erase(g_fs_pool.begin() + (long)i);
      return sg;
    }
  }
  FsStaging* sg = new FsStaging();
  memset(sg, 0, sizeof(*sg));
  sg->device = dev;
  return sg;
}

static void fs_staging_release(FsStaging* sg)
{
  std::lock_guard<std::mutex> lock(g_fs_pool_mtx);
  g_fs_pool.push_back(sg);
}

static void fs_execute_any(const FsOperator* op, const void* B, void* C)
{
  if (0 == op) { set_error(-30, "fsspmdm_execute: NULL handle"); return; }
  int M, N, K, ldb, ldc, beta_one;
  fs_shape(op, &M, &N, &K, &ldb, &ldc, &beta_one);
  const size_t esz = fs_is_double(op) ? 8 : 4;
  if (is_device_ptr(B) && is_device_ptr(C)) {
    fs_execute(op, B, C, N, ldb, ldc, cudaStreamPerThread);
    XB_CUDA(cudaStreamSynchronize(cudaStreamPerThread));
    return;
  }
  // HOST panels: pipeline column chunks through compact device staging on three streams so that
  // upload, kernel and download of neighbouring chunks overlap.  The staging context (streams + buffers) comes from a
  // pool keyed by device and is held for the duration of the call only: concurrent callers (the reference's driver runs
  // execute from an OpenMP loop over column panels, samples/pyfr/pyfr_driver_asp_reg.c:297-302) each get their own, on
  // the device that is current in THEIR thread, and nothing is serialised behind a global lock.
  FsStaging* sg = fs_staging_acquire();
  if (0 == sg) return;
  long long chunk = 1 << 16;
  if (chunk > N) chunk = N;
  const size_t needB = (size_t)K * chunk * esz, needC = (size_t)M * chunk * esz;
  bool ok = true;
  for (int s = 0; s < FsStaging::kSlots; ++s) {
    if (0 == sg->st[s]) XB_CUDA(cudaStreamCreateWithFlags(&sg->st[s], cudaStreamNonBlocking));
    if (sg->capB[s] < needB) { if (sg->dB[s]) cudaFree(sg->dB[s]); sg->dB[s] = 0; sg->capB[s] = 0; XB_CUDA(cudaMalloc((void**)&sg->dB[s], needB)); if (sg->dB[s]) sg->capB[s] = needB; }
    if (sg->capC[s] < needC) { if (sg->dC[s]) cudaFree(sg->dC[s]); sg->dC[s] = 0; sg->capC[s] = 0; XB_CUDA(cudaMalloc((void**)&sg->dC[s], needC)); if (sg->dC[s]) sg->capC[s] = needC; }
    ok = ok && 0 != sg->st[s] && 0 != sg->dB[s] && 0 != sg->dC[s];
  }
  if (ok) {
    int slot = 0;
    for (long long n0 = 0; n0 < N; n0 += chunk, slot = (slot + 1) % FsStaging::kSlots) {
      const long long w = (N - n0 < chunk) ? (N - n0) : chunk;
      cudaStream_t st = sg->st[slot];
      XB_CUDA(cudaMemcpy2DAsync(sg->dB[slot], w * esz, (const char*)B + n0 * esz, (size_t)ldb * esz, w * esz, K, cudaMemcpyHostToDevice, st));
      if (fs_needs_c_input(op))   // beta == 1, or rows the sparse branch leaves untouched
        XB_CUDA(cudaMemcpy2DAsync(sg->dC[slot], w * esz, (char*)C + n0 * esz, (size_t)ldc * esz, w * esz, M, cudaMemcpyHostToDevice, st));
      fs_execute(op, sg->dB[slot], sg->dC[slot], w, w, w, st);
      XB_CUDA(cudaMemcpy2DAsync((char*)C + n0 * esz, (size_t)ldc * esz, sg->dC[slot], w * esz, w * esz, M, cudaMemcpyDeviceToHost, st));
    }
    for (int s = 0; s < FsStaging::kSlots; ++s) XB_CUDA(cudaStreamSynchronize(sg->st[s]));
  }
  fs_staging_release(sg);
}

libxsmm_dfsspmdm* libxsmm_dfsspmdm_create(libxsmm_blasint M, libxsmm_blasint N, libxsmm_blasint K,
  libxsmm_blasint lda, libxsmm_blasint ldb, libxsmm_blasint ldc, const double alpha, const double beta, const double* a_dense)
{
  if (!(1.0 == alpha)) { set_error(-31, "dfsspmdm_create: alpha must be 1 (reference src/libxsmm_fsspmdm.c:67)"); return 0; }
  return (libxsmm_dfsspmdm*)fs_create(1, M, N, K, lda, ldb, ldc, beta, a_dense);
}

void libxsmm_dfsspmdm_execute(const libxsmm_dfsspmdm* handle, const double* B, double* C) { fs_execute_any((const FsOperator*)handle, B, C); }
void libxsmm_dfsspmdm_destroy(libxsmm_dfsspmdm* handle) { fs_destroy((FsOperator*)handle); }

libxsmm_sfsspmdm* libxsmm_sfsspmdm_create(libxsmm_blasint M, libxsmm_blasint N, libxsmm_blasint K,
  libxsmm_blasint lda, libxsmm_blasint ldb, libxsmm_blasint ldc, const float alpha, const float beta, const float* a_dense)
{
  if (!(1.f == alpha)) { set_error(-31, "sfsspmdm_create: alpha must be 1 (reference src/libxsmm_fsspmdm.c:173)"); return 0; }
  return (libxsmm_sfsspmdm*)fs_create(0, M, N, K, lda, ldb, ldc, (double)beta, a_dense);
}

void libxsmm_sfsspmdm_execute(const libxsmm_sfsspmdm* handle, const float* B, float* C) { fs_execute_any((const FsOperator*)handle, B, C); }
void libxsmm_sfsspmdm_destroy(libxsmm_sfsspmdm* handle) { fs_destroy((FsOperator*)handle); }

void libxsmm_dfsspmdm_execute_stream(const libxsmm_dfsspmdm* handle, const double* d_B, double* d_C, void* stream)
{
  const FsOperator* op = (const FsOperator*)handle;
  if (0 == op) { set_error(-30, "fsspmdm_execute_stream: NULL handle"); return; }
  int M, N, K, ldb, ldc, b1;
  fs_shape(op, &M, &N, &K, &ldb, &ldc, &b1);
  fs_execute(op, d_B, d_C, N, ldb, ldc, (cudaStream_t)stream);
}

void libxsmm_sfsspmdm_execute_stream(const libxsmm_sfsspmdm* handle, const float* d_B, float* d_C, void* stream)
{
  const FsOperator* op = (const FsOperator*)handle;
  if (0 == op) { set_error(-30, "fsspmdm_execute_stream: NULL handle"); return; }
  int M, N, K, ldb, ldc, b1;
  fs_shape(op, &M, &N, &K, &ldb, &ldc, &b1);
  fs_execute(op, d_B, d_C, N, ldb, ldc, (cudaStream_t)stream);
}

int libxsmm_dfsspmdm_is_sparse(const libxsmm_dfsspmdm* handle) { return fs_is_sparse_branch((const FsOperator*)handle); }
int libxsmm_sfsspmdm_is_sparse(const libxsmm_sfsspmdm* handle) { return fs_is_sparse_branch((const FsOperator*)handle); }
int libxsmm_dfsspmdm_is_baked(const libxsmm_dfsspmdm* handle) { return fs_is_baked((const FsOperator*)handle); }
int libxsmm_sfsspmdm_is_baked(const libxsmm_sfsspmdm* handle) { return fs_is_baked((const FsOperator*)handle); }
int libxsmm_sfsspmdm_is_tensor_core(const libxsmm_sfsspmdm* handle) { return fs_is_tensor_core((const FsOperator*)handle); }

// ---- CSR "A sparse" x dense SoA kernels (SURVEY.md section 8f-1) -------------------------------------------------------
// GPU counterpart of libxsmm_create_xcsr_soa + kernel(values, B, C) (reference src/libxsmm_main.c:2423-2447,
// src/generator_spgemm_csr_asparse_soa.c; caller samples/edge/asparse_srsoa.c:148-160), batched over mesh elements because
// one element's [m][n][soa] tensor is far too small for a launch.  Like the reference's descriptor, lda == 0 means A is the
// sparse operand (samples/edge/asparse_srsoa.c) and ldb == 0 means B is (samples/edge/bsparse_srsoa.c); the other operand
// and C are dense SoA tensors.  The operator's values are fixed at create (the reference's kernel re-reads them from its
// argument at every call; its callers pass the same array).
struct libxsmm_b200_csr_soa;
libxsmm_b200_csr_soa* libxsmm_b200_dcsr_soa_create(int M, int N, int K, int lda, int ldb, int ldc, int soa_width, double beta,
  const unsigned int* row_ptr, const unsigned int* column_idx, const double* values)
{ return (libxsmm_b200_csr_soa*)fs_create_csr(1, M, N, K, lda, ldb, ldc, soa_width, beta, row_ptr, column_idx, values); }
libxsmm_b200_csr_soa* libxsmm_b200_scsr_soa_create(int M, int N, int K, int lda, int ldb, int ldc, int soa_width, float beta,
  const unsigned int* row_ptr, const unsigned int* column_idx, const float* values)
{ return (libxsmm_b200_csr_soa*)fs_create_csr(0, M, N, K, lda, ldb, ldc, soa_width, (double)beta, row_ptr, column_idx, values); }
// libxsmm_create_xcsc_soa (reference src/libxsmm_main.c:2450-2474): B sparse in CSC; the handle is executed / destroyed like a CSR one
libxsmm_b200_csr_soa* libxsmm_b200_dcsc_soa_create(int M, int N, int K, int lda, int ldc, int soa_width, double beta,
                                                   const unsigned int* column_ptr, const unsigned int* row_idx, const double* values)
{ return (libxsmm_b200_csr_soa*)fs_create_csc(1, M, N, K, lda, ldc, soa_width, beta, column_ptr, row_idx, values); }
libxsmm_b200_csr_soa* libxsmm_b200_scsc_soa_create(int M, int N, int K, int lda, int ldc, int soa_width, float beta,
                                                   const unsigned int* column_ptr, const unsigned int* row_idx, const float* values)
{ return (libxsmm_b200_csr_soa*)fs_create_csc(0, M, N, K, lda, ldc, soa_width, (double)beta, column_ptr, row_idx, values); }
void libxsmm_b200_csr_soa_execute(const libxsmm_b200_csr_soa* handle, const void* d_B, void* d_C, long long n_elements,
  long long stride_b, long long stride_c, void* stream)
{
  if (0 == handle) { set_error(-63, "csr_soa_execute: NULL handle"); return; }
  const ElemIndex none = {0, 0};
  fs_execute_batched((const FsOperator*)handle, d_B, d_C, n_elements, stride_b, stride_c, none, none, (cudaStream_t)stream);
}
int libxsmm_b200_csr_soa_is_baked(const libxsmm_b200_csr_soa* handle) { return fs_is_baked((const FsOperator*)handle); }
void libxsmm_b200_csr_soa_destroy(libxsmm_b200_csr_soa* handle) { fs_destroy((FsOperator*)handle); }

// ---- dense SoA kernels (rm_soa.cu) ---------------------------------------------------------------------------------------------
// GPU counterparts of libxsmm_create_rm_ac_soa / libxsmm_create_rm_bc_soa (reference src/libxsmm_main.c:2477,2500), batched over
// mesh elements like csr_soa_execute.  Create only checks the descriptor (host only, no CUDA call); execute reads all three
// operands at call time.
struct libxsmm_b200_rm_soa;
static libxsmm_b200_rm_soa* rm_soa_create(int is_double, int form, int M, int N, int K, int lda, int ldb, int ldc, int soa, double beta)
{
  static const char* const nm[2] = {"rm_ac_soa_create", "rm_bc_soa_create"};
  if (M < 1 || N < 1 || K < 1 || soa < 1) { set_error(-80, "%s: empty shape (M=%d N=%d K=%d soa_width=%d)", nm[form], M, N, K, soa); return 0; }
  if (lda < K || ldb < N || ldc < N) { set_error(-81, "%s: pitch smaller than its extent (lda=%d >= K=%d, ldb=%d >= N=%d, ldc=%d >= N)", nm[form], lda, K, ldb, N, ldc); return 0; }
  if (!(0.0 == beta || 1.0 == beta)) { set_error(-82, "%s: beta=%g; it must be 0 or 1 like the reference's JIT", nm[form], beta); return 0; }
  RmSoa* h = new RmSoa();
  h->is_double = is_double; h->form = form; h->M = M; h->N = N; h->K = K; h->lda = lda; h->ldb = ldb; h->ldc = ldc; h->soa = soa;
  h->beta_one = 1.0 == beta;
  return (libxsmm_b200_rm_soa*)h;
}
libxsmm_b200_rm_soa* libxsmm_b200_drm_ac_soa_create(int M, int N, int K, int lda, int ldb, int ldc, int soa_width, double beta)
{ return rm_soa_create(1, 0, M, N, K, lda, ldb, ldc, soa_width, beta); }
libxsmm_b200_rm_soa* libxsmm_b200_srm_ac_soa_create(int M, int N, int K, int lda, int ldb, int ldc, int soa_width, float beta)
{ return rm_soa_create(0, 0, M, N, K, lda, ldb, ldc, soa_width, (double)beta); }
libxsmm_b200_rm_soa* libxsmm_b200_drm_bc_soa_create(int M, int N, int K, int lda, int ldb, int ldc, int soa_width, double beta)
{ return rm_soa_create(1, 1, M, N, K, lda, ldb, ldc, soa_width, beta); }
libxsmm_b200_rm_soa* libxsmm_b200_srm_bc_soa_create(int M, int N, int K, int lda, int ldb, int ldc, int soa_width, float beta)
{ return rm_soa_create(0, 1, M, N, K, lda, ldb, ldc, soa_width, (double)beta); }
void libxsmm_b200_rm_soa_execute(const libxsmm_b200_rm_soa* handle, const void* d_a, const void* d_b, void* d_c, long long n_elements,
  long long stride_a, long long stride_b, long long stride_c, void* stream)
{
  const RmSoa* h = (const RmSoa*)handle;
  if (0 == h) { set_error(-83, "rm_soa_execute: NULL handle"); return; }
  if (n_elements < 0 || stride_a < 0 || stride_b < 0 || stride_c < 0) {
    set_error(-83, "rm_soa_execute: negative count or stride (n_elements=%lld stride_a=%lld stride_b=%lld stride_c=%lld)", n_elements, stride_a, stride_b, stride_c);
    return;
  }
  if (0 == n_elements) return;
  const long long c_extent = ((long long)(h->M - 1) * h->ldc + h->N) * h->soa;
  if (n_elements > 1 && stride_c < c_extent) {
    set_error(-83, "rm_soa_execute: stride_c=%lld is smaller than one element's C (%lld scalars): elements would overlap", stride_c, c_extent);
    return;
  }
  if (0 == d_a || 0 == d_b || 0 == d_c) { set_error(-83, "rm_soa_execute: NULL operand"); return; }
  const ElemIndex none = {0, 0};
  rm_soa_execute(*h, d_a, d_b, d_c, n_elements, stride_a, stride_b, stride_c, none, none, none, (cudaStream_t)stream);
}
void libxsmm_b200_rm_soa_destroy(libxsmm_b200_rm_soa* handle) { delete (RmSoa*)handle; }

// ---- indexed execution of the batched SoA entries ------------------------------------------------------------------------------
// Element e reads operand X at d_X + slot * stride_x with slot = d_x_index[e] (DEVICE array, read at execute time on the stream) or
// e for a NULL index, and writes its C likewise.  An element whose slot in some operand is at or past that operand's slot count is
// skipped on the device.  The host checks below run before any CUDA call; every rejection sets -84 and launches nothing.
static bool soa_index_ok(const char* who, const char* name, const unsigned int* idx, long long slots)
{
  if (0 != idx && (slots < 1 || slots > (1ll << 32))) { set_error(-84, "%s: %s_slots=%lld outside [1, 2^32] for a non-NULL index", who, name, slots); return false; }
  return true;
}
// C slots must not overlap: with a C index whenever more than one slot may be written, without one (slot = element) when more than
// one element runs -- the strided entries' rule
static bool soa_c_disjoint(const char* who, long long n_elements, long long stride_c, long long c_extent, const unsigned int* d_c_index, long long c_slots)
{
  if ((d_c_index ? c_slots > 1 : n_elements > 1) && stride_c < c_extent) {
    set_error(-84, "%s: stride_c=%lld is smaller than one C slot (%lld scalars): slots would overlap", who, stride_c, c_extent);
    return false;
  }
  return true;
}
void libxsmm_b200_csr_soa_execute_indexed(const libxsmm_b200_csr_soa* handle, const void* d_X, void* d_C, long long n_elements,
  long long stride_x, long long stride_c, const unsigned int* d_x_index, long long x_slots, const unsigned int* d_c_index, long long c_slots, void* stream)
{
  static const char* const who = "csr_soa_execute_indexed";
  const FsOperator* o = (const FsOperator*)handle;
  if (0 == o) { set_error(-84, "%s: NULL handle", who); return; }
  if (n_elements < 0 || stride_x < 0 || stride_c < 0) {
    set_error(-84, "%s: negative count or stride (n_elements=%lld stride_x=%lld stride_c=%lld)", who, n_elements, stride_x, stride_c);
    return;
  }
  if (!soa_index_ok(who, "x", d_x_index, x_slots) || !soa_index_ok(who, "c", d_c_index, c_slots)) return;
  if (0 == n_elements) return;
  if (0 == d_X || 0 == d_C) { set_error(-84, "%s: NULL operand", who); return; }
  if (!soa_c_disjoint(who, n_elements, stride_c, fs_soa_c_extent(o), d_c_index, c_slots)) return;
  const ElemIndex ix = {d_x_index, x_slots}, ic = {d_c_index, c_slots};
  fs_execute_batched(o, d_X, d_C, n_elements, stride_x, stride_c, ix, ic, (cudaStream_t)stream);
}
void libxsmm_b200_rm_soa_execute_indexed(const libxsmm_b200_rm_soa* handle, const void* d_a, const void* d_b, void* d_c,
  long long n_elements, long long stride_a, long long stride_b, long long stride_c,
  const unsigned int* d_a_index, long long a_slots, const unsigned int* d_b_index, long long b_slots,
  const unsigned int* d_c_index, long long c_slots, void* stream)
{
  static const char* const who = "rm_soa_execute_indexed";
  const RmSoa* h = (const RmSoa*)handle;
  if (0 == h) { set_error(-84, "%s: NULL handle", who); return; }
  if (n_elements < 0 || stride_a < 0 || stride_b < 0 || stride_c < 0) {
    set_error(-84, "%s: negative count or stride (n_elements=%lld stride_a=%lld stride_b=%lld stride_c=%lld)", who, n_elements, stride_a, stride_b, stride_c);
    return;
  }
  if (!soa_index_ok(who, "a", d_a_index, a_slots) || !soa_index_ok(who, "b", d_b_index, b_slots) || !soa_index_ok(who, "c", d_c_index, c_slots)) return;
  if (0 == n_elements) return;
  if (0 == d_a || 0 == d_b || 0 == d_c) { set_error(-84, "%s: NULL operand", who); return; }
  const long long c_extent = ((long long)(h->M - 1) * h->ldc + h->N) * h->soa;
  if (!soa_c_disjoint(who, n_elements, stride_c, c_extent, d_c_index, c_slots)) return;
  const ElemIndex ia = {d_a_index, a_slots}, ib = {d_b_index, b_slots}, ic = {d_c_index, c_slots};
  rm_soa_execute(*h, d_a, d_b, d_c, n_elements, stride_a, stride_b, stride_c, ia, ib, ic, (cudaStream_t)stream);
}

// ---- fixed 2:4-sparse bf16 and FP8 operators (sp24.cu) --------------------------------------------------------------------
// The shape checks run on the host before any CUDA call (-95); create then compresses A on the device and reports a group
// keeping more than two elements (-96).  Every execute rejection (-97) also comes before anything is enqueued.
struct libxsmm_b200_sp24;
libxsmm_b200_sp24* libxsmm_b200_sp24_create_bfloat16(int M, int K, int lda, const libxsmm_bfloat16* a)
{
  if (M < 1 || K < 1 || lda < K || 0 == a) {
    set_error(-95, "sp24_create_bfloat16: M=%d, K=%d, lda=%d, a=%p: M and K must be at least 1, lda at least K, a not NULL", M, K, lda, (const void*)a);
    return 0;
  }
  return (libxsmm_b200_sp24*)sp24_create(M, K, lda, a, is_device_ptr(a), -1);
}
libxsmm_b200_sp24* libxsmm_b200_sp24_create_fp8(int M, int K, int lda, const unsigned char* a, int format)
{
  if (M < 1 || K < 1 || lda < K || 0 == a || (0 != format && 1 != format)) {
    set_error(-95, "sp24_create_fp8: M=%d, K=%d, lda=%d, a=%p, format=%d: M and K must be at least 1, lda at least K, a not NULL, format 0 (e4m3) or 1 (e5m2)",
              M, K, lda, (const void*)a, format);
    return 0;
  }
  return (libxsmm_b200_sp24*)sp24_create(M, K, lda, a, is_device_ptr(a), format);
}
// the execute checks both kinds share (b_format is checked for FP8 calls only; d_c / d_bias alignment for bf16 C only).
// true: the call has work to enqueue
static bool sp24_execute_ok(const char* who, const Sp24Op* op, bool fp8, char transb, char transc, int N, const void* d_b, int b_format,
                            int ldb, const void* d_c, int ldc, bool bf16_c = false, const void* d_bias = 0)
{
  if (0 == op) { set_error(-97, "%s: NULL handle", who); return false; }
  if (fp8 != (sp24_format(op) >= 0)) {
    set_error(-97, "%s: the handle holds a %s operator (created by sp24_create_%s)", who, fp8 ? "bf16" : "FP8", fp8 ? "bfloat16" : "fp8");
    return false;
  }
  const bool tb = is_t(transb), tc = is_t(transc);
  if (!(tb || 'N' == transb || 'n' == transb) || !(tc || 'N' == transc || 'n' == transc)) {
    set_error(-97, "%s: transb='%c', transc='%c': each must be one of N, n, T, t", who, transb, transc);
    return false;
  }
  if (fp8 && 0 != b_format && 1 != b_format) { set_error(-97, "%s: b_format=%d must be 0 (e4m3) or 1 (e5m2)", who, b_format); return false; }
  if (N < 0) { set_error(-97, "%s: N=%d is negative", who, N); return false; }
  const int M = sp24_rows(op), K = sp24_cols(op);
  if (ldb < (tb ? K : N) || ldc < (tc ? M : N)) {
    set_error(-97, "%s: ldb=%d must be at least %d (%s) and ldc=%d at least %d (%s)", who, ldb, tb ? K : N, tb ? "K" : "N", ldc, tc ? M : N, tc ? "M" : "N");
    return false;
  }
  if (0 == N) return false;
  if (0 == d_b || 0 == d_c) { set_error(-97, "%s: NULL d_b or d_c with N=%d", who, N); return false; }
  const int ldb_unit = fp8 ? 16 : 8;     // elements in 16 bytes
  if (0 != ((uintptr_t)d_b & 15) || 0 != (ldb % ldb_unit)) {
    set_error(-97, "%s: d_b=%p must be 16-byte aligned and ldb=%d a multiple of %d (B is read through TMA)", who, d_b, ldb, ldb_unit);
    return false;
  }
  if (bf16_c && (0 != ((uintptr_t)d_c & 1) || 0 != ((uintptr_t)d_bias & 1))) {
    set_error(-97, "%s: d_c=%p and d_bias=%p must be 2-byte aligned (bf16 elements)", who, d_c, d_bias);
    return false;
  }
  int dev = -1;
  if (cudaSuccess != cudaGetDevice(&dev)) { (void)cudaGetLastError(); dev = -1; }
  if (dev != sp24_device(op)) { set_error(-97, "%s: current device %d, the operator was created on device %d", who, dev, sp24_device(op)); return false; }
  return true;
}
void libxsmm_b200_sp24_execute(const libxsmm_b200_sp24* handle, char transb, char transc, int N,
  const libxsmm_bfloat16* d_b, int ldb, float beta, float* d_c, int ldc, void* stream)
{
  const Sp24Op* op = (const Sp24Op*)handle;
  if (!sp24_execute_ok("sp24_execute", op, false, transb, transc, N, d_b, -2, ldb, d_c, ldc)) return;
  sp24_execute(op, is_t(transb), is_t(transc), N, (const uint16_t*)d_b, ldb, beta, d_c, ldc, (cudaStream_t)stream);
}
void libxsmm_b200_sp24_execute_fp8(const libxsmm_b200_sp24* handle, char transb, char transc, int N,
  const unsigned char* d_b, int b_format, int ldb, float alpha, float beta, float* d_c, int ldc, void* stream)
{
  const Sp24Op* op = (const Sp24Op*)handle;
  if (!sp24_execute_ok("sp24_execute_fp8", op, true, transb, transc, N, d_b, b_format, ldb, d_c, ldc)) return;
  sp24_execute_fp8(op, is_t(transb), is_t(transc), N, d_b, b_format, ldb, alpha, beta, d_c, ldc, (cudaStream_t)stream);
}
void libxsmm_b200_sp24_execute_bf16out(const libxsmm_b200_sp24* handle, char transb, char transc, int N,
  const libxsmm_bfloat16* d_b, int ldb, const libxsmm_bfloat16* d_bias, float beta, libxsmm_bfloat16* d_c, int ldc, void* stream)
{
  const Sp24Op* op = (const Sp24Op*)handle;
  if (!sp24_execute_ok("sp24_execute_bf16out", op, false, transb, transc, N, d_b, -2, ldb, d_c, ldc, true, d_bias)) return;
  sp24_execute_bf16out(op, is_t(transb), is_t(transc), N, (const uint16_t*)d_b, ldb, (const uint16_t*)d_bias, beta, (uint16_t*)d_c, ldc,
                       (cudaStream_t)stream);
}
void libxsmm_b200_sp24_execute_fp8_bf16out(const libxsmm_b200_sp24* handle, char transb, char transc, int N,
  const unsigned char* d_b, int b_format, int ldb, float alpha, const libxsmm_bfloat16* d_bias, float beta,
  libxsmm_bfloat16* d_c, int ldc, void* stream)
{
  const Sp24Op* op = (const Sp24Op*)handle;
  if (!sp24_execute_ok("sp24_execute_fp8_bf16out", op, true, transb, transc, N, d_b, b_format, ldb, d_c, ldc, true, d_bias)) return;
  sp24_execute_fp8_bf16out(op, is_t(transb), is_t(transc), N, d_b, b_format, ldb, alpha, (const uint16_t*)d_bias, beta, (uint16_t*)d_c, ldc,
                           (cudaStream_t)stream);
}
void libxsmm_b200_sp24_destroy(libxsmm_b200_sp24* handle) { sp24_destroy((Sp24Op*)handle); }

// ---- dense SMM dispatch for row-major operators with very many columns (SURVEY.md section 8f-3) ---------------------------
// The reference's callers apply a DENSE fixed operator to a row-major panel with the column-major SMM kernel
//     kernel = libxsmm_dmmdispatch(nblock, M_op, K_op, &ldb_panel, &lda_op, &ldc_panel, alpha, beta, ...)
//     kernel(B_panel + i, A_op, C_panel + i)          for i = 0, nblock, 2 nblock, ...
// (samples/pyfr/pyfr_gemm_rm.c:98-122; libxsmm_[sd]mmdispatch, src/libxsmm_main.c:2166-2195; it is also what
// libxsmm_[sd]fsspmdm_create falls back to, src/libxsmm_fsspmdm.c:134-142).  Column-major C(m x n) = A(m x k) B(k x n) + beta C
// with m = panel columns, n = operator rows, k = operator columns: A[i + l lda] is panel element (row l, column i) and
// B[l + j ldb] is operator element (row j, column l), so the small operand b IS the row-major operator with pitch ldb.
// Here one execute call covers m_total panel columns (all the chunks of the caller's loop).  The small operand is read at
// execute (host or device pointer); the handle keeps the kernel baked for its current CONTENT (fused multiply-add chains
// with literal values, or the tcgen05 kernel for dense float operators) and re-bakes only when the content changes --
// the callers' operators are constant.  Rounding sequence of the reference's SMM kernel: in-order fma over k from C / 0.
struct libxsmm_b200_mm;
struct MmHandle {
  int is_double, m, n, k, lda, ldb, ldc;
  double beta;
  std::mutex mtx;
  unsigned long long hash;
  FsOperator* op;
};

static MmHandle* mm_dispatch(int is_double, int m, int n, int k, const int* lda, const int* ldb, const int* ldc, double alpha, double beta)
{
  const int la = lda ? *lda : m, lb = ldb ? *ldb : k, lc = ldc ? *ldc : m;
  if (m <= 0 || n <= 0 || k <= 0 || la < m || lb < k || lc < m || !(1.0 == alpha) || !(0.0 == beta || 1.0 == beta)) {
    set_error(-70, "mmdispatch: unsupported descriptor (m=%d n=%d k=%d lda=%d ldb=%d ldc=%d alpha=%g beta=%g; alpha must be 1, beta 0 or 1 like the reference's JIT)", m, n, k, la, lb, lc, alpha, beta);
    return 0;
  }
  MmHandle* h = new MmHandle();
  h->is_double = is_double; h->m = m; h->n = n; h->k = k; h->lda = la; h->ldb = lb; h->ldc = lc; h->beta = beta; h->hash = 0; h->op = 0;
  return h;
}

libxsmm_b200_mm* libxsmm_b200_dmmdispatch(int m, int n, int k, const int* lda, const int* ldb, const int* ldc, const double* alpha, const double* beta)
{ return (libxsmm_b200_mm*)mm_dispatch(1, m, n, k, lda, ldb, ldc, alpha ? *alpha : 1.0, beta ? *beta : 1.0); }   // LIBXSMM_ALPHA = LIBXSMM_BETA = 1
libxsmm_b200_mm* libxsmm_b200_smmdispatch(int m, int n, int k, const int* lda, const int* ldb, const int* ldc, const float* alpha, const float* beta)
{ return (libxsmm_b200_mm*)mm_dispatch(0, m, n, k, lda, ldb, ldc, alpha ? (double)*alpha : 1.0, beta ? (double)*beta : 1.0); }

void libxsmm_b200_mm_execute(libxsmm_b200_mm* handle, const void* d_a, const void* b, void* d_c, long long m_total, void* stream)
{
  MmHandle* h = (MmHandle*)handle;
  if (0 == h || 0 == d_a || 0 == b || 0 == d_c) { set_error(-71, "mm_execute: NULL argument"); return; }
  if (m_total <= 0) return;
  const size_t esz = h->is_double ? 8 : 4;
  const size_t nb = ((size_t)(h->n - 1) * h->ldb + h->k) * esz;      // the operator as it lies in memory: n rows of pitch ldb
  std::vector<unsigned char> host(nb);
  if (is_device_ptr(b)) {
    XB_CUDA(cudaMemcpyAsync(host.data(), b, nb, cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    XB_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
  }
  else memcpy(host.data(), b, nb);
  unsigned long long hash = 1469598103934665603ull;                      // FNV-1a over the operator's elements (not the pitch padding)
  for (int j = 0; j < h->n; ++j) {
    const unsigned char* row = host.data() + (size_t)j * h->ldb * esz;
    for (size_t z = 0; z < (size_t)h->k * esz; ++z) { hash ^= row[z]; hash *= 1099511628211ull; }
  }
  std::lock_guard<std::mutex> lock(h->mtx);
  if (0 == h->op || hash != h->hash) {
    if (h->op) { XB_CUDA(cudaStreamSynchronize((cudaStream_t)stream)); fs_destroy(h->op); h->op = 0; }
    h->op = fs_create(h->is_double, h->n, -1 /* any column count */, h->k, h->ldb, h->lda, h->ldc, h->beta, host.data());
    h->hash = hash;
    if (0 == h->op) return;
  }
  fs_execute(h->op, d_a, d_c, m_total, h->lda, h->ldc, (cudaStream_t)stream);
}

const char* libxsmm_b200_mm_kernel(const libxsmm_b200_mm* handle)
{
  const MmHandle* h = (const MmHandle*)handle;
  if (0 == h || 0 == h->op) return "none";
  return fs_is_tensor_core(h->op) ? "fs_tc_kernel" : (fs_is_baked(h->op) ? "fs_baked" : "fs_generic_kernel");
}

void libxsmm_b200_mm_release(libxsmm_b200_mm* handle)
{
  MmHandle* h = (MmHandle*)handle;
  if (0 == h) return;
  if (h->op) fs_destroy(h->op);
  delete h;
}

// =====================================================================================================
// service
// =====================================================================================================
int libxsmm_b200_last_error(void) { std::lock_guard<std::mutex> lock(g_err_mtx); return g_err_code; }
const char* libxsmm_b200_last_error_string(void) { return g_err_msg; }
void libxsmm_b200_clear_error(void) { std::lock_guard<std::mutex> lock(g_err_mtx); g_err_code = 0; g_err_msg[0] = 0; }
unsigned long long libxsmm_b200_launch_count(void) { return g_launches.load(); }
const char* libxsmm_b200_last_compute_kernel(void) { return g_last_compute.load(); }

void* libxsmm_b200_host_alloc(size_t bytes)
{
  void* p = 0;
  if (cudaSuccess != cudaMallocHost(&p, bytes)) { (void)cudaGetLastError(); set_error(-40, "host_alloc(%zu) failed", bytes); return 0; }
  return p;
}
void libxsmm_b200_host_free(void* p) { if (p) cudaFreeHost(p); }

void* libxsmm_b200_device_alloc(size_t bytes)
{
  void* p = 0;
  if (cudaSuccess != cudaMalloc(&p, bytes ? bytes : 1)) { (void)cudaGetLastError(); set_error(-41, "device_alloc(%zu) failed", bytes); return 0; }
  return p;
}
void libxsmm_b200_device_free(void* p) { if (p) cudaFree(p); }
int libxsmm_b200_memcpy_h2d(void* d, const void* s, size_t n) { const cudaError_t e = cudaMemcpy(d, s, n, cudaMemcpyHostToDevice); if (e) set_error((int)e, "memcpy_h2d: %s", cudaGetErrorString(e)); return (int)e; }
int libxsmm_b200_memcpy_d2h(void* d, const void* s, size_t n) { const cudaError_t e = cudaMemcpy(d, s, n, cudaMemcpyDeviceToHost); if (e) set_error((int)e, "memcpy_d2h: %s", cudaGetErrorString(e)); return (int)e; }
int libxsmm_b200_memset(void* d, int v, size_t n) { const cudaError_t e = cudaMemset(d, v, n); if (e) set_error((int)e, "memset: %s", cudaGetErrorString(e)); return (int)e; }
int libxsmm_b200_synchronize(void) { const cudaError_t e = cudaDeviceSynchronize(); if (e) set_error((int)e, "synchronize: %s", cudaGetErrorString(e)); return (int)e; }
int libxsmm_b200_device_count(void) { int n = 0; if (cudaSuccess != cudaGetDeviceCount(&n)) { (void)cudaGetLastError(); return 0; } return n; }
int libxsmm_b200_set_device(int device) { const cudaError_t e = cudaSetDevice(device); if (e) set_error((int)e, "set_device: %s", cudaGetErrorString(e)); return (int)e; }

void* libxsmm_b200_stream_create(void) { cudaStream_t s = 0; XB_CUDA(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking)); return (void*)s; }
void libxsmm_b200_stream_destroy(void* s) { if (s) cudaStreamDestroy((cudaStream_t)s); }
int libxsmm_b200_stream_synchronize(void* s) { const cudaError_t e = cudaStreamSynchronize((cudaStream_t)s); if (e) set_error((int)e, "stream_synchronize: %s", cudaGetErrorString(e)); return (int)e; }
void* libxsmm_b200_event_create(void) { cudaEvent_t ev = 0; XB_CUDA(cudaEventCreate(&ev)); return (void*)ev; }
void libxsmm_b200_event_destroy(void* ev) { if (ev) cudaEventDestroy((cudaEvent_t)ev); }
int libxsmm_b200_event_record(void* ev, void* s) { const cudaError_t e = cudaEventRecord((cudaEvent_t)ev, (cudaStream_t)s); if (e) set_error((int)e, "event_record: %s", cudaGetErrorString(e)); return (int)e; }
int libxsmm_b200_event_synchronize(void* ev) { const cudaError_t e = cudaEventSynchronize((cudaEvent_t)ev); if (e) set_error((int)e, "event_synchronize: %s", cudaGetErrorString(e)); return (int)e; }
float libxsmm_b200_event_elapsed_ms(void* a, void* b) { float ms = -1.f; const cudaError_t e = cudaEventElapsedTime(&ms, (cudaEvent_t)a, (cudaEvent_t)b); if (e) { set_error((int)e, "event_elapsed: %s", cudaGetErrorString(e)); return -1.f; } return ms; }
int libxsmm_b200_memcpy_h2d_async(void* d, const void* s, size_t n, void* st) { const cudaError_t e = cudaMemcpyAsync(d, s, n, cudaMemcpyHostToDevice, (cudaStream_t)st); if (e) set_error((int)e, "memcpy_h2d_async: %s", cudaGetErrorString(e)); return (int)e; }
int libxsmm_b200_memcpy_d2h_async(void* d, const void* s, size_t n, void* st) { const cudaError_t e = cudaMemcpyAsync(d, s, n, cudaMemcpyDeviceToHost, (cudaStream_t)st); if (e) set_error((int)e, "memcpy_d2h_async: %s", cudaGetErrorString(e)); return (int)e; }
int libxsmm_b200_memset_async(void* d, int v, size_t n, void* st) { const cudaError_t e = cudaMemsetAsync(d, v, n, (cudaStream_t)st); if (e) set_error((int)e, "memset_async: %s", cudaGetErrorString(e)); return (int)e; }
int libxsmm_b200_graph_begin(void* st) { const cudaError_t e = cudaStreamBeginCapture((cudaStream_t)st, cudaStreamCaptureModeThreadLocal); if (e) set_error((int)e, "graph_begin: %s", cudaGetErrorString(e)); return (int)e; }
void* libxsmm_b200_graph_end(void* st)
{
  cudaGraph_t g = 0; cudaGraphExec_t x = 0;
  cudaError_t e = cudaStreamEndCapture((cudaStream_t)st, &g);
  if (cudaSuccess == e) e = cudaGraphInstantiate(&x, g, 0);
  if (g) cudaGraphDestroy(g);
  if (e) { set_error((int)e, "graph_end: %s", cudaGetErrorString(e)); return 0; }
  return (void*)x;
}
int libxsmm_b200_graph_launch(void* x, void* st) { const cudaError_t e = cudaGraphLaunch((cudaGraphExec_t)x, (cudaStream_t)st); if (e) set_error((int)e, "graph_launch: %s", cudaGetErrorString(e)); return (int)e; }
void libxsmm_b200_graph_destroy(void* x) { if (x) cudaGraphExecDestroy((cudaGraphExec_t)x); }

// ---- host-only planning entries (no CUDA calls; usable without a GPU) --------------------------------
int libxsmm_b200_spmdm_geometry(int M, int N, int K, int max_threads, int bn, int* geom)
{
  if (M <= 0 || N <= 0 || K <= 0 || 0 == geom) return -1;
  if (max_threads < 1) max_threads = 1;
  Geom g;
  spmdm_geometry(M, N, K, max_threads, bn, &g);
  geom[0] = g.m; geom[1] = g.n; geom[2] = g.k; geom[3] = g.bm; geom[4] = g.bn; geom[5] = g.bk;
  geom[6] = g.mb; geom[7] = g.nb; geom[8] = g.kb;
  return 0;
}

int libxsmm_b200_fsspmdm_plan(int is_double, int M, int N, int K, int lda, int ldb, int ldc, double beta,
                              const void* a_dense, long long* info)
{
  FsOperator* o = fs_plan(is_double, M, N, K, lda, ldb, ldc, beta, a_dense);
  if (0 == o) return -1;
  if (info) fs_plan_info(o, info);
  fs_destroy(o);
  return 0;
}

char* libxsmm_b200_fsspmdm_kernel_source(int is_double, int M, int N, int K, int lda, int ldb, int ldc, double beta,
                                         const void* a_dense)
{
  FsOperator* o = fs_plan(is_double, M, N, K, lda, ldb, ldc, beta, a_dense);
  if (0 == o) return 0;
  char* src = fs_kernel_source(o);
  fs_destroy(o);
  return src;
}

void libxsmm_b200_free_string(char* s) { free(s); }

// ---- MatrixMarket operators (SURVEY.md section 8f-2) ----------------------------------------------------
// Same file convention as the reference's reader (src/generator_spgemm_csr_reader.c:46-169 and the PyFR driver's
// copy, samples/pyfr/pyfr_driver_asp_reg.c:47-158): '%' comment lines, one "rows cols nnz" line, then nnz lines
// "row col value" with 1-based indices; rows without entries are allowed.  The reference assumes the entries
// are sorted by row; here they are bucketed by row (stable), which is the identity on sorted files.
int libxsmm_b200_csr_read_mtx(const char* path, unsigned int** row_ptr, unsigned int** col_idx, double** values,
                              unsigned int* rows, unsigned int* cols, unsigned int* nnz)
{
  if (0 == path || 0 == row_ptr || 0 == col_idx || 0 == values || 0 == rows || 0 == cols || 0 == nnz) return -1;
  *row_ptr = 0; *col_idx = 0; *values = 0; *rows = *cols = *nnz = 0;
  FILE* f = fopen(path, "r");
  if (0 == f) { set_error(-40, "csr_read_mtx: cannot open %s", path); return -40; }
  char line[1024];
  unsigned int nr = 0, nc = 0, ne = 0;
  bool header = false;
  std::vector<unsigned int> er, ec;
  std::vector<double> ev;
  int rc = 0;
  while (0 == rc && 0 != fgets(line, (int)sizeof(line), f)) {
    if (strlen(line) + 1 >= sizeof(line)) { rc = -41; break; }                  // over-long line (reference: CSR_READ_LEN)
    const char* q = line;
    while (' ' == *q || '\t' == *q) ++q;
    if ('%' == *q || '\n' == *q || '\r' == *q || 0 == *q) continue;
    if (!header) {
      if (3 != sscanf(q, "%u %u %u", &nr, &nc, &ne) || 0 == nr || 0 == nc || 0 == ne) { rc = -42; break; }   // reference: CSR_READ_DESC
      header = true;
      er.reserve(ne); ec.reserve(ne); ev.reserve(ne);
    }
    else {
      unsigned int r = 0, cidx = 0; double v = 0;
      if (3 != sscanf(q, "%u %u %lf", &r, &cidx, &v)) { rc = -43; break; }                                      // reference: CSR_READ_ELEMS
      if (0 == r || 0 == cidx || r > nr || cidx > nc) { rc = -44; break; }
      er.push_back(r - 1); ec.push_back(cidx - 1); ev.push_back(v);
    }
  }
  fclose(f);
  if (0 == rc && (!header || er.size() != (size_t)ne)) rc = -45;                                                 // reference: CSR_LEN
  if (0 != rc) { set_error(rc, "csr_read_mtx: %s is not a valid MatrixMarket coordinate file (code %d)", path, rc); return rc; }
  unsigned int* rp = (unsigned int*)malloc(sizeof(unsigned int) * ((size_t)nr + 1));
  unsigned int* ci = (unsigned int*)malloc(sizeof(unsigned int) * ne);
  double* va = (double*)malloc(sizeof(double) * ne);
  if (0 == rp || 0 == ci || 0 == va) { free(rp); free(ci); free(va); set_error(-46, "csr_read_mtx: out of memory"); return -46; }
  memset(rp, 0, sizeof(unsigned int) * ((size_t)nr + 1));
  for (unsigned int i = 0; i < ne; ++i) ++rp[er[i] + 1];
  for (unsigned int i = 0; i < nr; ++i) rp[i + 1] += rp[i];
  std::vector<unsigned int> fill(rp, rp + nr);
  for (unsigned int i = 0; i < ne; ++i) { const unsigned int d = fill[er[i]]++; ci[d] = ec[i]; va[d] = ev[i]; }
  *row_ptr = rp; *col_idx = ci; *values = va; *rows = nr; *cols = nc; *nnz = ne;
  return 0;
}

void libxsmm_b200_csr_free(unsigned int* row_ptr, unsigned int* col_idx, double* values) { free(row_ptr); free(col_idx); free(values); }

// operator file -> dense row-major A (lda = cols) -> the ordinary create(); duplicates in the file overwrite like
// the drivers' own densification (samples/pyfr/pyfr_driver_asp_reg.c:226-238)
static void* fsspmdm_create_mtx(int is_double, const char* path, int N, int ldb, int ldc, double beta, int* M_out, int* K_out)
{
  unsigned int *rp = 0, *ci = 0, nr = 0, nc = 0, ne = 0; double* va = 0;
  if (0 != libxsmm_b200_csr_read_mtx(path, &rp, &ci, &va, &nr, &nc, &ne)) return 0;
  void* h = 0;
  if (is_double) {
    std::vector<double> a((size_t)nr * nc, 0.0);
    for (unsigned int r = 0; r < nr; ++r) for (unsigned int j = rp[r]; j < rp[r + 1]; ++j) a[(size_t)r * nc + ci[j]] = va[j];
    h = libxsmm_dfsspmdm_create((int)nr, N, (int)nc, (int)nc, ldb, ldc, 1.0, beta, a.data());
  }
  else {
    std::vector<float> a((size_t)nr * nc, 0.f);
    for (unsigned int r = 0; r < nr; ++r) for (unsigned int j = rp[r]; j < rp[r + 1]; ++j) a[(size_t)r * nc + ci[j]] = (float)va[j];
    h = libxsmm_sfsspmdm_create((int)nr, N, (int)nc, (int)nc, ldb, ldc, 1.f, (float)beta, a.data());
  }
  if (M_out) *M_out = (int)nr;
  if (K_out) *K_out = (int)nc;
  libxsmm_b200_csr_free(rp, ci, va);
  return h;
}
libxsmm_dfsspmdm* libxsmm_b200_dfsspmdm_create_mtx(const char* path, int N, int ldb, int ldc, double beta, int* M, int* K)
{ return (libxsmm_dfsspmdm*)fsspmdm_create_mtx(1, path, N, ldb, ldc, beta, M, K); }
libxsmm_sfsspmdm* libxsmm_b200_sfsspmdm_create_mtx(const char* path, int N, int ldb, int ldc, float beta, int* M, int* K)
{ return (libxsmm_sfsspmdm*)fsspmdm_create_mtx(0, path, N, ldb, ldc, (double)beta, M, K); }

// ---- fused caller step (SURVEY.md section 8f-4) ----------------------------------------------------------
// What TensorFlow's sparse_matmul_op builds around the reference (documentation/tensorflow.md:241-250): a cache of
// handles keyed by the problem shape, and slice creation + compute as one call.  Here the key also holds the stream,
// because a handle's slice arena must not be shared by multiplies that may run concurrently.
struct MatmulKey {
  int m, n, k, threads; void* stream;
  bool operator<(const MatmulKey& o) const {
    if (m != o.m) return m < o.m; if (n != o.n) return n < o.n; if (k != o.k) return k < o.k;
    if (threads != o.threads) return threads < o.threads; return stream < o.stream;
  }
};
struct MatmulEntry { libxsmm_spmdm_handle handle; libxsmm_CSR_sparseslice* slices; unsigned long long last_use; };
static std::mutex g_mm_mtx;
static std::map<MatmulKey, MatmulEntry*> g_mm_cache;
static unsigned long long g_mm_clock = 0;
static const size_t kMatmulCacheMax = 16;

int libxsmm_b200_sparse_matmul(libxsmm_spmdm_datatype datatype, char transa, char transb, char transc, int M, int N, int K,
  int max_threads, const void* d_a, const void* d_b, const void* beta, float* d_c, void* stream)
{
  if (M <= 0 || N <= 0 || K <= 0 || 0 == d_a || 0 == d_b || 0 == d_c || 0 == beta) { set_error(-50, "sparse_matmul: bad argument"); return -50; }
  if (max_threads < 1) max_threads = 1;
  MatmulEntry* e = 0;
  {
    std::lock_guard<std::mutex> lock(g_mm_mtx);
    const MatmulKey key = { M, N, K, max_threads, stream };
    std::map<MatmulKey, MatmulEntry*>::iterator it = g_mm_cache.find(key);
    if (it == g_mm_cache.end()) {
      if (g_mm_cache.size() >= kMatmulCacheMax) {      // evict the least recently used handle (its stream is drained first)
        std::map<MatmulKey, MatmulEntry*>::iterator old = g_mm_cache.begin();
        for (std::map<MatmulKey, MatmulEntry*>::iterator j = g_mm_cache.begin(); j != g_mm_cache.end(); ++j) if (j->second->last_use < old->second->last_use) old = j;
        XB_CUDA(cudaStreamSynchronize((cudaStream_t)old->first.stream));
        libxsmm_spmdm_destroy(&old->second->handle);
        delete old->second;
        g_mm_cache.erase(old);
      }
      e = new MatmulEntry();
      memset(&e->handle, 0, sizeof(e->handle)); e->slices = 0;
      libxsmm_spmdm_init(M, N, K, max_threads, &e->handle, &e->slices);
      if (0 == e->handle.base_ptr_scratch_A) { delete e; return -51; }
      g_mm_cache[key] = e;
    }
    else e = it->second;
    e->last_use = ++g_mm_clock;
  }
  const unsigned long long seq = g_err_seq.load(std::memory_order_relaxed);
  libxsmm_spmdm_exec_stream(&e->handle, e->slices, datatype, transa, transb, transc, d_a, d_b, beta, d_c, stream);
  return (seq == g_err_seq.load(std::memory_order_relaxed)) ? 0 : libxsmm_b200_last_error();   // an older, unrelated sticky error is not this call's failure
}

int libxsmm_b200_sparse_matmul_cache_entries(void)
{
  std::lock_guard<std::mutex> lock(g_mm_mtx);
  return (int)g_mm_cache.size();
}

void libxsmm_b200_sparse_matmul_cache_clear(void)
{
  std::lock_guard<std::mutex> lock(g_mm_mtx);
  for (std::map<MatmulKey, MatmulEntry*>::iterator j = g_mm_cache.begin(); j != g_mm_cache.end(); ++j) {
    (void)cudaStreamSynchronize((cudaStream_t)j->first.stream);
    libxsmm_spmdm_destroy(&j->second->handle);
    delete j->second;
  }
  g_mm_cache.clear();
}

}  // extern "C"
