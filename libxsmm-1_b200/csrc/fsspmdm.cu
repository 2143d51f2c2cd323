// FSSPMDM: a fixed sparse operator A (M x K) baked at create time, applied to a dense B with
// very many columns:  C[:, 0:N] = A * B[:, 0:N] + beta * C   (beta in {0,1}).
// Replaces reference src/libxsmm_fsspmdm.c (create :48-257, execute :260-291, destroy :294-329)
// and the kernel emitted by src/generator_spgemm_csr_asparse_reg.c:196-300.
#include "common.cuh"
#include <algorithm>
#include "fsspmdm_jit.h"
#include <vector>
#include <cstring>
#include <cstdlib>
#include <cmath>
#include <cstdio>

namespace xb {

struct FsTc;
bool fs_tc_supported(int is_double, int M, int K);
FsTc* fs_tc_build(int M, int K, int lda, int beta_one, const float* a_dense);
bool fs_tc_launch(const FsTc* t, const void* dB, void* dC, long long ncols, long long ldb, long long ldc, cudaStream_t stream);
void fs_tc_destroy(FsTc* t);

struct FsOperator {
  // leading fields mirror the reference's private handle (src/libxsmm_main.h:695-715) so that code
  // peeking at M/N/K/ldb/ldc/N_chunksize/a_dense keeps working; a_dense == NULL <=> sparse branch.
  int M, N, K, ldb, ldc, N_chunksize;
  void* a_dense;      // DEVICE copy of the packed M x K operator (dense branch only)
  void* kernel;       // opaque: the baked kernel (FsJit*) or NULL
  // ---- private ----
  int is_double;
  int beta_one;
  int sparse_branch;  // the branch the reference would take (decides empty-row behaviour)
  int nnz, n_unique;
  long long x86_code_size;   // bytes the reference's generator would emit (0 if not evaluated)
  int* d_rowptr;      // M+1
  int* d_col;         // per nonzero: column index
  void* d_val;        // per nonzero: value as executed (double or float)
  std::vector<int> rowptr, col;
  std::vector<double> val;
  FsJit* jit;
  FsTc* tc;            // tensor-core kernel for dense float operators (fsspmdm_tc.cu), or NULL
  // CSR x SoA (fs_create_csr): the batched apply sees every element as `items` items of `item_cols` columns
  long long items, item_cols, item_b, item_c;
};

// ---- branch rule of the reference ------------------------------------------------------------------
// x86 bytes the reference's sparse_reg generator would emit; the sparse branch exists only while this
// fits its 128 KiB JIT buffer (src/libxsmm_main.c:66-67).  Displacement sizes follow the encoder
// (src/generator_x86_instructions.c:52-77): none if 0, one byte if a multiple of the operand size
// within +-127 units, else four.  Byte-exact against the reference (tests pin the threshold).
static int fs_disp(long long off, int unit)
{
  if (0 == off) return 0;
  if (0 == (off % unit) && off / unit <= 127 && off / unit >= -128) return 1;
  return 4;
}
static long long fs_x86_code_size(const FsOperator& o)
{
  long long sz = 40 + (long long)o.n_unique * 76;
  for (int m = 0; m < o.M; ++m) {
    const int lo = o.rowptr[m], hi = o.rowptr[m + 1];
    const long long coff = (long long)m * o.ldc * 8;
    if (hi == lo) continue;
    sz += o.beta_one ? (6 + fs_disp(coff, 64)) : 6;
    sz += 3 + fs_disp(coff + 64, 1);
    for (int u = lo; u < hi; ++u) {
      const long long boff = (long long)o.col[u] * o.ldb * 8;
      sz += 6 + fs_disp(boff, 64) + 3 + fs_disp(boff + 64, 1);
    }
    sz += 6 + fs_disp(coff, 64);
  }
  return sz;
}

// ---- generic kernel: operator streamed from global memory (warp-uniform addresses), B through L1 ----
struct FsDev {
  int M, beta_one, skip_empty;
  long long ldb, ldc;
  long long J, sb, sc;   // batched form (CSR x SoA): columns per item and element strides; J = 0: plain column panel
  long long ipe, ib, ic; // items per element and item strides
  ElemIndex xb, xc;      // batched form: slots of B and C per element (fs_execute_batched)
  const int* rowptr;
  const int* col;
  const void* val;
};

template <typename T, int VEC>
__global__ void __launch_bounds__(256) fs_generic_kernel(const FsDev p, const T* __restrict__ B, T* __restrict__ C, long long ncols)
{
  const long long n = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * VEC;
  if (n >= ncols) return;
  const T* __restrict__ val = (const T*)p.val;
  long long nb = n, nc = n;
  if (p.J > 0) {   // (element, item, column) form: VEC == 1
    const long long item = n / p.J, j = n - item * p.J, e = item / p.ipe, i = item - e * p.ipe;
    const long long sb = p.xb.idx ? (long long)p.xb.idx[e] : e, sc = p.xc.idx ? (long long)p.xc.idx[e] : e;
    if (sb >= p.xb.slots || sc >= p.xc.slots) return;
    nb = sb * p.sb + i * p.ib + j; nc = sc * p.sc + i * p.ic + j;
  }
  const T* Bn = B + nb;
  for (int m = 0; m < p.M; ++m) {
    const int lo = __ldg(p.rowptr + m), hi = __ldg(p.rowptr + m + 1);
    if (hi == lo && p.skip_empty) continue;
    T* crow = C + (long long)m * p.ldc + nc;
    T acc[VEC];
    if (p.beta_one) {
#pragma unroll
      for (int e = 0; e < VEC; ++e) acc[e] = (n + e < ncols) ? crow[e] : (T)0;
    }
    else {
#pragma unroll
      for (int e = 0; e < VEC; ++e) acc[e] = (T)0;
    }
    for (int j = lo; j < hi; ++j) {
      const T v = __ldg(val + j);
      const T* brow = Bn + (long long)__ldg(p.col + j) * p.ldb;
#pragma unroll
      for (int e = 0; e < VEC; ++e) {
        const T b = (n + e < ncols) ? __ldg(brow + e) : (T)0;
        acc[e] = fma(v, b, acc[e]);
      }
    }
#pragma unroll
    for (int e = 0; e < VEC; ++e) if (n + e < ncols) crow[e] = acc[e];
  }
}

// ---- create -------------------------------------------------------------------------------------------
template <typename T>
static void fs_build_csr(FsOperator& o, const T* a, int lda)
{
  o.rowptr.assign(o.M + 1, 0);
  for (int i = 0; i < o.M; ++i) {
    o.rowptr[i] = (int)o.col.size();
    for (int j = 0; j < o.K; ++j) {
      const T v = a[(size_t)i * lda + j];
      if (v != (T)0) { o.col.push_back(j); o.val.push_back((double)v); }   // NaN kept, -0 dropped (:88-116)
    }
  }
  o.rowptr[o.M] = (int)o.col.size();
  o.nnz = (int)o.col.size();
}

// Host-only part of create(): contract check, CSR, unique-value table, branch rule.  No CUDA calls,
// so that it can be exercised (and is, tests/test_host_logic.py) on a machine without a GPU.
FsOperator* fs_plan(int is_double, int M, int N, int K, int lda, int ldb, int ldc, double beta, const void* a_dense)
{
  // the reference asserts this contract (src/libxsmm_fsspmdm.c:65-71) and calls a NULL kernel when it
  // is violated in a release build; here a violation is an error and create returns NULL.
  // N < 0: no contract on the column count (the dense dispatch entry, capi.cu: the caller's panels may have any width)
  const bool free_n = (N < 0);
  if (M <= 0 || K <= 0 || (!free_n && (N < 16 || 0 != (N % 16) || N > ldb || N > ldc)) || K > lda || 0 == a_dense
      || !(beta == 0.0 || beta == 1.0)) {
    set_error(-1, "fsspmdm_create: contract violated (M=%d N=%d K=%d lda=%d ldb=%d ldc=%d beta=%g)", M, N, K, lda, ldb, ldc, beta);
    return 0;
  }
  FsOperator* o = new FsOperator();
  o->M = M; o->N = N; o->K = K; o->ldb = ldb; o->ldc = ldc;
  o->a_dense = 0; o->kernel = 0; o->jit = 0; o->tc = 0;
  o->is_double = is_double; o->beta_one = (1.0 == beta);
  o->d_rowptr = 0; o->d_col = 0; o->d_val = 0;
  if (is_double) fs_build_csr(*o, (const double*)a_dense, lda); else fs_build_csr(*o, (const float*)a_dense, lda);

  // unique-value table of the sparse_reg generator (:125-150); for a NaN value the search "hits"
  // every entry and the LAST one wins, i.e. the emitted kernel multiplies with that entry instead.
  o->n_unique = 0;
  o->sparse_branch = 0;
  o->x86_code_size = 0;
  if (is_double && o->nnz > 0 && !free_n) {   // (the dense dispatch entry is the dense SMM kernel by definition: no sparse_reg branch)
    std::vector<double> table;
    std::vector<double> exec_val(o->val);
    table.push_back(o->val[0]);
    for (int u = 1; u < o->nnz && (int)table.size() <= 32; ++u) {
      int hit = -1;
      for (int z = 0; z < (int)table.size(); ++z) if (!(table[z] < o->val[u]) && !(table[z] > o->val[u])) hit = z;
      if (hit < 0) table.push_back(o->val[u]); else exec_val[u] = table[hit];
    }
    o->n_unique = (int)table.size();
    if (o->n_unique <= 31) {
      o->x86_code_size = fs_x86_code_size(*o);
      if (o->x86_code_size <= 131072) {
        o->sparse_branch = 1;
        o->val.swap(exec_val);
      }
    }
  }
  o->N_chunksize = o->sparse_branch ? 8 : 16;   // what the reference reports (:119,133,225,239)
  return o;
}

FsOperator* fs_create(int is_double, int M, int N, int K, int lda, int ldb, int ldc, double beta, const void* a_dense)
{
  FsOperator* o = fs_plan(is_double, M, N, K, lda, ldb, ldc, beta, a_dense);
  if (0 == o) return 0;

  // device side of the operator
  const size_t nalloc = (size_t)(o->nnz > 0 ? o->nnz : 1);
  XB_CUDA(cudaMalloc(&o->d_rowptr, sizeof(int) * (M + 1)));
  XB_CUDA(cudaMalloc(&o->d_col, sizeof(int) * nalloc));
  XB_CUDA(cudaMalloc(&o->d_val, 8 * nalloc));
  if (0 == o->d_rowptr || 0 == o->d_col || 0 == o->d_val) { fs_destroy(o); return 0; }
  XB_CUDA(cudaMemcpy(o->d_rowptr, o->rowptr.data(), sizeof(int) * (M + 1), cudaMemcpyHostToDevice));
  if (o->nnz > 0) XB_CUDA(cudaMemcpy(o->d_col, o->col.data(), sizeof(int) * (size_t)o->nnz, cudaMemcpyHostToDevice));
  if (o->nnz > 0) {
    if (is_double) XB_CUDA(cudaMemcpy(o->d_val, o->val.data(), 8 * (size_t)o->nnz, cudaMemcpyHostToDevice));
    else {
      std::vector<float> vf(o->val.begin(), o->val.end());
      XB_CUDA(cudaMemcpy(o->d_val, vf.data(), 4 * (size_t)o->nnz, cudaMemcpyHostToDevice));
    }
  }
  if (!o->sparse_branch) {   // dense branch keeps a packed copy of A like the reference (:136-142)
    const size_t esz = is_double ? 8 : 4;
    std::vector<char> packed((size_t)M * K * esz);
    for (int i = 0; i < M; ++i) memcpy(&packed[(size_t)i * K * esz], (const char*)a_dense + (size_t)i * lda * esz, (size_t)K * esz);
    XB_CUDA(cudaMalloc(&o->a_dense, packed.size()));
    if (o->a_dense) XB_CUDA(cudaMemcpy(o->a_dense, packed.data(), packed.size(), cudaMemcpyHostToDevice));
  }
  // Dense float operators: once the FMA pipe, not HBM, bounds the baked kernel (more than ~4 nonzeros per byte
  // moved per column), the apply is a dense contraction and goes to the tensor cores (3xTF32, fsspmdm_tc.cu).
  // Measured on B200, 150 x 64, N = 2^22: tensor cores 625 us at any density (round 1: 819; beta = 1: 1067 us, was 6388);
  // baked 652 / 716 / 996 / 1367 / 1767 us at 30 / 35 / 40 / 45-50 / 60 % -> break-even ~30 % (beta = 0; the rule below keeps its margin).
  // LIBXSMM_B200_FSSPMDM_TC=1 forces that kernel for every eligible operator, =0 disables it.
  if (fs_tc_supported(is_double, M, K)) {
    const char* e = getenv("LIBXSMM_B200_FSSPMDM_TC");
    const double bytes_per_col = 4.0 * (K + M * (o->beta_one ? 2.0 : 1.0));
    const bool want = (e && *e) ? ('1' == *e) : ((double)o->nnz > 4.0 * bytes_per_col);
    if (want) o->tc = fs_tc_build(M, K, lda, o->beta_one, (const float*)a_dense);
  }
  // bake the operator into a specialised kernel (the GPU counterpart of the reference's JIT)
  // (not when the tensor-core kernel took the operator: panels it cannot take fall back to the generic kernel)
  if (0 == o->tc) {
    const int vec2 = (0 == ((ldb | ldc) & 1)) ? 1 : 0;
    o->jit = fs_jit_build(is_double, vec2, M, K, o->beta_one, o->sparse_branch /*skip empty rows*/, o->rowptr.data(), o->col.data(), o->val.data());
    // fma-heavy fp64 operators (the dense tet / tri families): the emitter has three forms and none wins everywhere, so the
    // candidates are timed here, once, on a scratch panel, and the fastest is kept (the reference spends its create on a JIT too)
    const int nvar = o->jit ? fs_jit_variants(is_double, vec2, M, K, o->rowptr.data(), o->col.data()) : 1;
    if (nvar > 1) {
      const long long nt = (N > 0 && N < (1 << 17)) ? ((N + 15) / 16 * 16) : (1 << 17);
      void* sb = 0; void* sc = 0;
      cudaEvent_t e0 = 0, e1 = 0;
      if (cudaSuccess == cudaMalloc(&sb, (size_t)K * nt * 8) && cudaSuccess == cudaMalloc(&sc, (size_t)M * nt * 8) &&
          cudaSuccess == cudaEventCreate(&e0) && cudaSuccess == cudaEventCreate(&e1)) {
        cudaMemset(sb, 0, (size_t)K * nt * 8); cudaMemset(sc, 0, (size_t)M * nt * 8);
        auto time_of = [&](FsJit* j) -> float {
          float best = 1e30f;
          if (!fs_jit_launch(j, sb, sc, nt, nt, nt, 0)) return best;
          for (int rep = 0; rep < 3; ++rep) {
            cudaEventRecord(e0, 0);
            fs_jit_launch(j, sb, sc, nt, nt, nt, 0);
            cudaEventRecord(e1, 0);
            float ms = 1e30f;
            if (cudaSuccess == cudaEventSynchronize(e1) && cudaSuccess == cudaEventElapsedTime(&ms, e0, e1) && ms < best) best = ms;
          }
          return best;
        };
        float tbest = time_of(o->jit);
        int vbest = 0;
        for (int v = 1; v < nvar; ++v) {
          FsJit* cand = fs_jit_build(is_double, vec2, M, K, o->beta_one, o->sparse_branch, o->rowptr.data(), o->col.data(), o->val.data(), 0, v);
          if (0 == cand) continue;
          const float t = time_of(cand);
          if (t < 0.97f * tbest) { fs_jit_destroy(o->jit); o->jit = cand; tbest = t; vbest = v; }
          else fs_jit_destroy(cand);
        }
        if (verbosity() > 0) fprintf(stderr, "LIBXSMM_B200 fsspmdm: %dx%d nnz=%d: emitter variant %d of %d (%.1f us for %lld columns)\n", M, K, o->nnz, vbest, nvar, tbest * 1e3f, nt);
      }
      (void)cudaGetLastError();
      if (e0) cudaEventDestroy(e0);
      if (e1) cudaEventDestroy(e1);
      if (sb) cudaFree(sb);
      if (sc) cudaFree(sc);
    }
  }
  o->kernel = o->jit;
  if (verbosity() > 0) {
    fprintf(stderr, "LIBXSMM_B200 fsspmdm: %dx%d nnz=%d unique=%d branch=%s kernel=%s\n", M, K, o->nnz, o->n_unique,
            o->sparse_branch ? "sparse" : "dense", o->jit ? "baked" : "generic");
  }
  return o;
}

void fs_execute(const FsOperator* o, const void* dB, void* dC, long long ncols, long long ldb, long long ldc, cudaStream_t stream)
{
  if (0 == o || ncols <= 0) return;
  count_launch(1);
  if (o->tc && fs_tc_launch(o->tc, dB, dC, ncols, ldb, ldc, stream)) { note_compute_kernel("fs_tc_kernel"); return; }
  if (o->jit && fs_jit_launch(o->jit, dB, dC, ncols, ldb, ldc, stream)) { note_compute_kernel("fs_baked"); return; }
  note_compute_kernel("fs_generic_kernel");
  FsDev d;
  d.M = o->M; d.beta_one = o->beta_one; d.skip_empty = o->sparse_branch;
  d.ldb = ldb; d.ldc = ldc; d.rowptr = o->d_rowptr; d.col = o->d_col; d.val = o->d_val;
  d.J = 0; d.sb = 0; d.sc = 0; d.ipe = 1; d.ib = 0; d.ic = 0;
  d.xb.idx = 0; d.xb.slots = 0; d.xc.idx = 0; d.xc.slots = 0;
  const int threads = 256;
  if (o->is_double) {
    const bool v2 = (0 == (ldb & 1)) && (0 == (ldc & 1)) && (0 == (((uintptr_t)dB | (uintptr_t)dC) & 15));
    if (v2) {
      const long long blocks = (ncols + 2 * threads - 1) / (2 * threads);
      fs_generic_kernel<double, 2><<<(unsigned)blocks, threads, 0, stream>>>(d, (const double*)dB, (double*)dC, ncols);
    }
    else {
      const long long blocks = (ncols + threads - 1) / threads;
      fs_generic_kernel<double, 1><<<(unsigned)blocks, threads, 0, stream>>>(d, (const double*)dB, (double*)dC, ncols);
    }
  }
  else {
    const bool v4 = (0 == (ldb & 3)) && (0 == (ldc & 3)) && (0 == (((uintptr_t)dB | (uintptr_t)dC) & 15));
    if (v4) {
      const long long blocks = (ncols + 4 * threads - 1) / (4 * threads);
      fs_generic_kernel<float, 4><<<(unsigned)blocks, threads, 0, stream>>>(d, (const float*)dB, (float*)dC, ncols);
    }
    else {
      const long long blocks = (ncols + threads - 1) / threads;
      fs_generic_kernel<float, 1><<<(unsigned)blocks, threads, 0, stream>>>(d, (const float*)dB, (float*)dC, ncols);
    }
  }
  XB_CUDA(cudaGetLastError());
}

// device copy of the operator rows (for the generic kernel) + the baked, batched kernel: common tail of the SoA creators
static FsOperator* fs_finish_soa(FsOperator* o)
{
  const size_t nalloc = (size_t)(o->nnz > 0 ? o->nnz : 1);
  XB_CUDA(cudaMalloc(&o->d_rowptr, sizeof(int) * (o->M + 1)));
  XB_CUDA(cudaMalloc(&o->d_col, sizeof(int) * nalloc));
  XB_CUDA(cudaMalloc(&o->d_val, 8 * nalloc));
  if (0 == o->d_rowptr || 0 == o->d_col || 0 == o->d_val) { fs_destroy(o); return 0; }
  XB_CUDA(cudaMemcpy(o->d_rowptr, o->rowptr.data(), sizeof(int) * (o->M + 1), cudaMemcpyHostToDevice));
  if (o->nnz > 0) {
    XB_CUDA(cudaMemcpy(o->d_col, o->col.data(), sizeof(int) * (size_t)o->nnz, cudaMemcpyHostToDevice));
    if (o->is_double) XB_CUDA(cudaMemcpy(o->d_val, o->val.data(), 8 * (size_t)o->nnz, cudaMemcpyHostToDevice));
    else { std::vector<float> vf(o->val.begin(), o->val.end()); XB_CUDA(cudaMemcpy(o->d_val, vf.data(), 4 * (size_t)o->nnz, cudaMemcpyHostToDevice)); }
  }
  if (o->M > 0) o->jit = fs_jit_build(o->is_double, 0, o->M, o->K, o->beta_one, o->sparse_branch, o->rowptr.data(), o->col.data(), o->val.data(), 1 /*batched*/);
  o->kernel = o->jit;
  return o;
}


// ---- CSR x dense SoA (SURVEY.md section 8f-1) ----------------------------------------------------------------------------
// The operator arrives as CSR (reference libxsmm_create_xcsr_soa, src/libxsmm_main.c:2423-2447) and is applied to
// [row][column][soa] tensors.  Arithmetic of the reference's emitted kernel (src/generator_spgemm_csr_asparse_soa.c:
// 213-420): per row with nonzeros an in-order chain of fused multiply-adds from C (beta != 0) or from zero; rows without
// nonzeros are skipped.  With the SoA lanes as innermost columns this IS the fixed-operator apply over N * soa columns
// with row pitches ldb * soa / ldc * soa, so it reuses the baked kernel (batched over mesh elements).
FsOperator* fs_create_csr(int is_double, int M, int N, int K, int lda, int ldb, int ldc, int soa, double beta,
                          const unsigned int* rowptr, const unsigned int* colidx, const void* values)
{
  // like the reference's descriptor: lda == 0 <=> A is the sparse operand (CSR over its M rows), ldb == 0 <=> B is (CSR over its K rows)
  const bool a_sparse = (0 == lda && ldb > 0), b_sparse = (lda > 0 && 0 == ldb);
  if (M <= 0 || N <= 0 || K <= 0 || soa <= 0 || !(a_sparse || b_sparse) || ldc < N || (a_sparse && ldb < N) || (b_sparse && lda < K)
      || 0 == rowptr || 0 == colidx || 0 == values
      || !(0.0 == beta || 1.0 == beta)) {   // the reference's descriptor (libxsmm_gemm_descriptor_dinit) exists for beta 0 and 1 only
    set_error(-60, "csr_soa_create: bad argument (M=%d N=%d K=%d lda=%d ldb=%d ldc=%d soa=%d beta=%g; exactly one of lda / ldb is 0)", M, N, K, lda, ldb, ldc, soa, beta);
    return 0;
  }
  const int srows = a_sparse ? M : K, scols = a_sparse ? K : N;       // shape of the sparse operand
  for (int r = 0; r < srows; ++r) if (rowptr[r + 1] < rowptr[r]) { set_error(-61, "csr_soa_create: row pointers not monotone"); return 0; }
  for (unsigned int z = rowptr[0]; z < rowptr[srows]; ++z) if (a_sparse && colidx[z] >= (unsigned int)scols) { set_error(-62, "csr_soa_create: column index out of range"); return 0; }
  FsOperator* o = new FsOperator();
  o->a_dense = 0; o->kernel = 0; o->jit = 0; o->tc = 0;
  o->is_double = is_double; o->beta_one = (0.0 != beta);
  o->d_rowptr = 0; o->d_col = 0; o->d_val = 0;
  o->n_unique = 0; o->x86_code_size = 0; o->N_chunksize = soa;
  auto value_at = [&](unsigned int z) -> double { return is_double ? ((const double*)values)[z] : (double)((const float*)values)[z]; };
  if (a_sparse) {
    // C[m][(n, s)] = sum_z a[z] B[col z][(n, s)]: the operator is A itself, an item is a whole element with N * soa columns
    o->M = M; o->K = K; o->N = N * soa; o->ldb = ldb * soa; o->ldc = ldc * soa;
    o->items = 1; o->item_cols = (long long)N * soa; o->item_b = 0; o->item_c = 0;
    o->sparse_branch = 1;                                          // rows without nonzeros are skipped (generator_spgemm_csr_asparse_soa.c:249)
    o->rowptr.assign(M + 1, 0);
    for (int m = 0; m <= M; ++m) o->rowptr[m] = (int)(rowptr[m] - rowptr[0]);
    o->nnz = o->rowptr[M];
    o->col.resize((size_t)o->nnz); o->val.resize((size_t)o->nnz);
    for (int z = 0; z < o->nnz; ++z) { o->col[z] = (int)colidx[rowptr[0] + z]; o->val[z] = value_at(rowptr[0] + z); }
  }
  else {
    // C[m][n][s] = sum_k A[m][k][s] b[k][n]: for one m this is the operator B^T applied to the item A[m] = [k][soa]; an
    // element has M items of soa columns, lda * soa / ldc * soa apart.  Row n of B^T holds column n of B in ascending k, the
    // order of the reference's k loop (generator_spgemm_csr_bsparse_soa.c:208-292).  The reference works on columns
    // 0 .. ncols-1 only, ncols = 1 + the largest column index of any nonzero (:161-167): empty columns below ncols are
    // written, columns from ncols on are never touched -- so B^T gets ncols rows, not N.  Nonzeros with column >= N count
    // towards ncols but are not multiplied (:213,233).
    int ncols = 0;
    for (unsigned int z = rowptr[0]; z < rowptr[K]; ++z) if (colidx[z] >= (unsigned int)ncols) ncols = (int)colidx[z] + 1;
    if (ncols > ldc) { set_error(-62, "csr_soa_create: column index %d of B reaches past ldc=%d", ncols - 1, ldc); fs_destroy(o); return 0; }
    o->M = ncols; o->K = K; o->N = soa; o->ldb = soa; o->ldc = soa;
    o->items = M; o->item_cols = soa; o->item_b = (long long)lda * soa; o->item_c = (long long)ldc * soa;
    o->sparse_branch = 0;
    std::vector<int> cnt((size_t)ncols + 1, 0);
    for (unsigned int z = rowptr[0]; z < rowptr[K]; ++z) if (colidx[z] < (unsigned int)N) ++cnt[colidx[z] + 1];
    o->rowptr.assign((size_t)ncols + 1, 0);
    for (int n = 0; n < ncols; ++n) o->rowptr[n + 1] = o->rowptr[n] + cnt[n + 1];
    o->nnz = o->rowptr[ncols];
    o->col.resize((size_t)o->nnz); o->val.resize((size_t)o->nnz);
    std::vector<int> fill(o->rowptr.begin(), o->rowptr.end() - 1);
    for (int k = 0; k < K; ++k) for (unsigned int z = rowptr[k]; z < rowptr[k + 1]; ++z) if (colidx[z] < (unsigned int)N) {
      const int d = fill[colidx[z]]++;
      o->col[d] = k; o->val[d] = value_at(z);
    }
  }
  return fs_finish_soa(o);
}

// libxsmm_create_xcsc_soa (reference src/libxsmm_main.c:2450-2474, src/generator_spgemm_csc_bsparse_soa.c:143-435; caller
// samples/edge/bsparse_scsoa.c:327-354): B sparse in CSC (column pointers over its N columns, row indices = k), A dense
// [m][lda][soa], C [m][ldc][soa].  The generator walks k = 0 .. K-1 and, per column of the chunk, takes the FIRST entry of the column
// whose row index equals k (:270-279): one fused multiply-add per (k, n) in ascending k whatever the order inside the column, later
// duplicates and rows >= K never used.  Its trailing-empty-column rule (:185-190) cannot fire -- the loop does not stop at the first
// match, so the last assignment is always n -- hence all N columns are written (unlike the CSR form above).
FsOperator* fs_create_csc(int is_double, int M, int N, int K, int lda, int ldc, int soa, double beta,
                          const unsigned int* colptr, const unsigned int* rowidx, const void* values)
{
  if (M <= 0 || N <= 0 || K <= 0 || soa <= 0 || lda < K || ldc < N || 0 == colptr || 0 == rowidx || 0 == values || !(0.0 == beta || 1.0 == beta)) {
    set_error(-60, "csc_soa_create: bad argument (M=%d N=%d K=%d lda=%d ldc=%d soa=%d beta=%g)", M, N, K, lda, ldc, soa, beta);
    return 0;
  }
  for (int n = 0; n < N; ++n) if (colptr[n + 1] < colptr[n]) { set_error(-61, "csc_soa_create: column pointers not monotone"); return 0; }
  FsOperator* o = new FsOperator();
  o->a_dense = 0; o->kernel = 0; o->jit = 0; o->tc = 0;
  o->is_double = is_double; o->beta_one = (0.0 != beta);
  o->d_rowptr = 0; o->d_col = 0; o->d_val = 0;
  o->n_unique = 0; o->x86_code_size = 0; o->N_chunksize = soa;
  o->M = N; o->K = K; o->N = soa; o->ldb = soa; o->ldc = soa;
  o->items = M; o->item_cols = soa; o->item_b = (long long)lda * soa; o->item_c = (long long)ldc * soa;
  o->sparse_branch = 0;
  o->rowptr.assign((size_t)N + 1, 0);
  std::vector<std::pair<unsigned int, unsigned int> > ent;     // (k, position) of one column
  for (int n = 0; n < N; ++n) {
    ent.clear();
    for (unsigned int z = colptr[n]; z < colptr[n + 1]; ++z) if (rowidx[z] < (unsigned int)K) ent.push_back(std::make_pair(rowidx[z], z));
    std::stable_sort(ent.begin(), ent.end(), [](const std::pair<unsigned int, unsigned int>& x, const std::pair<unsigned int, unsigned int>& y) { return x.first < y.first; });
    for (size_t i = 0; i < ent.size(); ++i) {
      if (i > 0 && ent[i].first == ent[i - 1].first) continue;          // the first entry with this k wins
      o->col.push_back((int)ent[i].first);
      o->val.push_back(is_double ? ((const double*)values)[ent[i].second] : (double)((const float*)values)[ent[i].second]);
    }
    o->rowptr[n + 1] = (int)o->col.size();
  }
  o->nnz = o->rowptr[N];
  return fs_finish_soa(o);
}

// ib / ic: the slot of every element's B and C (no index: the element itself, never skipped)
void fs_execute_batched(const FsOperator* o, const void* dB, void* dC, long long n_elem, long long stride_b, long long stride_c,
                        ElemIndex ib, ElemIndex ic, cudaStream_t stream)
{
  if (0 == o || n_elem <= 0 || o->M <= 0) return;   // B sparse without a single nonzero: the reference's kernel touches nothing
  if (0 == ib.idx) ib.slots = n_elem;
  if (0 == ic.idx) ic.slots = n_elem;
  count_launch(1);
  if (o->jit && fs_jit_launch_batched(o->jit, dB, dC, n_elem, o->items, o->item_cols, o->ldb, o->ldc, stride_b, stride_c, o->item_b, o->item_c,
                                      ib.idx, ib.slots, ic.idx, ic.slots, stream)) { note_compute_kernel("fs_baked (batched)"); return; }
  note_compute_kernel("fs_generic_kernel (batched)");
  FsDev d;
  d.M = o->M; d.beta_one = o->beta_one; d.skip_empty = o->sparse_branch;
  d.ldb = o->ldb; d.ldc = o->ldc; d.rowptr = o->d_rowptr; d.col = o->d_col; d.val = o->d_val;
  d.J = o->item_cols; d.sb = stride_b; d.sc = stride_c; d.ipe = o->items; d.ib = o->item_b; d.ic = o->item_c;
  d.xb = ib; d.xc = ic;
  const int threads = 256;
  const long long total = n_elem * o->items * o->item_cols, blocks = (total + threads - 1) / threads;
  if (o->is_double) fs_generic_kernel<double, 1><<<(unsigned)blocks, threads, 0, stream>>>(d, (const double*)dB, (double*)dC, total);
  else fs_generic_kernel<float, 1><<<(unsigned)blocks, threads, 0, stream>>>(d, (const float*)dB, (float*)dC, total);
  XB_CUDA(cudaGetLastError());
}

void fs_destroy(FsOperator* o)
{
  if (0 == o) return;
  if (o->tc) fs_tc_destroy(o->tc);
  if (o->jit) fs_jit_destroy(o->jit);
  if (o->d_rowptr) cudaFree(o->d_rowptr);
  if (o->d_col) cudaFree(o->d_col);
  if (o->d_val) cudaFree(o->d_val);
  if (o->a_dense) cudaFree(o->a_dense);
  delete o;
}

int fs_is_sparse_branch(const FsOperator* o) { return o ? o->sparse_branch : 0; }
int fs_is_baked(const FsOperator* o) { return (o && o->jit) ? 1 : 0; }
int fs_is_tensor_core(const FsOperator* o) { return (o && o->tc) ? 1 : 0; }
int fs_needs_c_input(const FsOperator* o)
{
  if (0 == o) return 0;
  if (o->beta_one) return 1;
  if (o->sparse_branch) for (int m = 0; m < o->M; ++m) if (o->rowptr[m] == o->rowptr[m + 1]) return 1;   // untouched rows
  return 0;
}
int fs_is_double(const FsOperator* o) { return o ? o->is_double : 0; }
long long fs_soa_c_extent(const FsOperator* o)
{
  if (o->M <= 0) return 0;     // B sparse without a nonzero: nothing is written
  return (o->items - 1) * o->item_c + (long long)(o->M - 1) * o->ldc + o->item_cols;
}
void fs_plan_info(const FsOperator* o, long long* info)
{
  info[0] = o->nnz; info[1] = o->n_unique; info[2] = o->sparse_branch; info[3] = o->x86_code_size; info[4] = o->N_chunksize;
  info[5] = fs_jit_form(o->is_double, (0 == ((o->ldb | o->ldc) & 1)) ? 1 : 0, o->M, o->K, o->rowptr.data(), o->col.data());
}
char* fs_kernel_source(const FsOperator* o)
{
  return fs_jit_source(o->is_double, (0 == ((o->ldb | o->ldc) & 1)) ? 1 : 0, o->M, o->K, o->beta_one, o->sparse_branch, o->rowptr.data(), o->col.data(), o->val.data());
}
void fs_shape(const FsOperator* o, int* M, int* N, int* K, int* ldb, int* ldc, int* beta_one)
{
  *M = o->M; *N = o->N; *K = o->K; *ldb = o->ldb; *ldc = o->ldc; *beta_one = o->beta_one;
}

}  // namespace xb
