// Dense SoA kernels (DESIGN.md section 8): the GPU counterparts of libxsmm_create_rm_ac_soa / libxsmm_create_rm_bc_soa, batched
// over mesh elements.  One operand of every element is an SoA tensor [R][ld][soa] (A in the ac form, B in the bc form), the
// other a plain row-major matrix (b, a), C is [M][ldc][soa].  Every output is one chain of fused multiply-adds over k
// ascending, from C (beta = 1) or +0 (beta = 0), zeros included: the arithmetic of the reference's generated code.
//
// Both forms are one kernel.  A thread owns a lane (r, s) of the SoA operand -- r = m (ac) or n (bc) -- and a register block of
// kRB entries j of the other output dimension (n for ac, m for bc); at each k it reads X[r][k][s] (ac) or X[k][r][s] (bc) once
// and the kRB plain-operand values it meets as broadcasts.  A persistent grid walks the elements.
//   staged: the element's SoA operand arrives in shared memory by one 1-D bulk copy (cp.async.bulk, mbarrier completion),
//           double-buffered so that the next element's copy overlaps this element's multiply-adds; the plain operand is
//           copied once per CTA (stride 0) or per element with cp.async into a second double buffer.
//   direct: the same inner loop on global memory, for operands the bulk copy cannot address (16-byte alignment of the base,
//           the element stride and the size) and for shapes whose double buffer does not fit in shared memory.
// Indexed execute (kIx = true): element e takes its operands from slot index[e] of each (slot e where an index is NULL); an element
// with a slot at or past that operand's slot count is skipped, nothing of it read or written.  The strided entry instantiates
// the kernels with kIx = false, which compiles to the plain element loop.
#include "common.cuh"
#include "ptx.cuh"
#include <algorithm>

namespace xb {
namespace {

constexpr int kRB = 8;              // register block: outputs per thread along j
constexpr int kMaxThreads = 512;

struct RmArgs {
  const void* x; const void* p; void* c;      // SoA operand, plain operand, C (element 0)
  long long sx, sp, sc, n_elem;               // element strides in scalars
  int L, soa, J, K;                           // lanes (rows of the SoA operand's lane dimension x soa), register dimension, depth
  long long xs_l, xs_k;                       // X[lane row][k]: lr * xs_l + k * xs_k + s
  long long ps_k, ps_j;                       // P[k][j]:        k * ps_k + j * ps_j
  long long cs_l, cs_j;                       // C[lane row][j]: lr * cs_l + j * cs_j + s
  int nblk;                                   // register blocks per lane
  long long x_elems, p_elems;                 // extents of one element's X and P (scalars)
  int x_buf, p_buf;                           // staged: shared-memory scalars per X / P buffer (X rounded up to 16 bytes)
  int beta_one;
  const unsigned int *xi, *pi, *ci;           // per-element slots of X, P, C, or NULL (slot = element)
  long long x_slots, p_slots, c_slots;        // slots at or past these skip the element
};

// the slot of element e in an operand with index idx (NULL: e); whether every slot of e is in range
template <bool kIx>
__device__ __forceinline__ long long rm_slot(const unsigned int* idx, long long e) { return (kIx && idx) ? (long long)idx[e] : e; }
template <bool kIx>
__device__ __forceinline__ bool rm_runs(const RmArgs& a, long long e)
{
  return !kIx || (rm_slot<kIx>(a.xi, e) < a.x_slots && rm_slot<kIx>(a.pi, e) < a.p_slots && rm_slot<kIx>(a.ci, e) < a.c_slots);
}

__device__ __forceinline__ void cp_async_elem(void* dst, const double* src)
{ asm volatile("cp.async.ca.shared.global [%0], [%1], 8;\n" ::"r"(smem_u32(dst)), "l"(src) : "memory"); }
__device__ __forceinline__ void cp_async_elem(void* dst, const float* src)
{ asm volatile("cp.async.ca.shared.global [%0], [%1], 4;\n" ::"r"(smem_u32(dst)), "l"(src) : "memory"); }
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_prev() { asm volatile("cp.async.wait_group 1;\n" ::: "memory"); }

__device__ __forceinline__ double xfma(double x, double y, double acc) { return __fma_rn(x, y, acc); }
__device__ __forceinline__ float xfma(float x, float y, float acc) { return __fmaf_rn(x, y, acc); }

// One work item of one element: lane (lr, s), outputs j0 .. j0 + kRB - 1.  X and P are the element's operands in shared memory
// (offsets I = int) or in global memory (I = long long); the chain of multiply-adds is the same either way.  Entries j >= J are
// computed on a clamped column and never stored.
template <typename T, typename I>
__device__ __forceinline__ void rm_item(const RmArgs& a, const T* __restrict__ X, const T* __restrict__ P, T* __restrict__ C, int item)
{
  const int blk = item / a.L, lane = item - blk * a.L;
  const int lr = lane / a.soa, s = lane - lr * a.soa;
  const int j0 = blk * kRB;
  const I xs_k = (I)a.xs_k, ps_k = (I)a.ps_k;
  const T* xp = X + (I)lr * (I)a.xs_l + s;
  I po[kRB];
  T acc[kRB];
  T* cp = C + lr * a.cs_l + s;
#pragma unroll
  for (int r = 0; r < kRB; ++r) {
    const int j = min(j0 + r, a.J - 1);
    po[r] = (I)j * (I)a.ps_j;
    acc[r] = (T)0;
    if (a.beta_one && j0 + r < a.J) acc[r] = cp[(long long)(j0 + r) * a.cs_j];
  }
#pragma unroll 1
  for (int k = 0; k < a.K; ++k) {
    const T x = xp[(I)k * xs_k];
    const T* pk = P + (I)k * ps_k;
#pragma unroll
    for (int r = 0; r < kRB; ++r) acc[r] = xfma(x, pk[po[r]], acc[r]);
  }
#pragma unroll
  for (int r = 0; r < kRB; ++r)
    if (j0 + r < a.J) cp[(long long)(j0 + r) * a.cs_j] = acc[r];
}

template <typename T, bool kIx>
__global__ void __launch_bounds__(kMaxThreads) rm_soa_direct_kernel(RmArgs a)
{
  const int items = a.L * a.nblk;
  for (long long e = blockIdx.x; e < a.n_elem; e += gridDim.x) {
    if (!rm_runs<kIx>(a, e)) continue;
    const T* X = (const T*)a.x + rm_slot<kIx>(a.xi, e) * a.sx;
    const T* P = (const T*)a.p + rm_slot<kIx>(a.pi, e) * a.sp;
    T* C = (T*)a.c + rm_slot<kIx>(a.ci, e) * a.sc;
    for (int i = threadIdx.x; i < items; i += blockDim.x) rm_item<T, long long>(a, X, P, C, i);
  }
}

template <typename T, bool kIx>
__global__ void __launch_bounds__(kMaxThreads, 2) rm_soa_staged_kernel(RmArgs a)
{
  extern __shared__ __align__(16) unsigned char smem[];
  T* xbuf = (T*)smem;                                   // [2][x_buf]
  T* pbuf = xbuf + 2 * a.x_buf;                         // [1 or 2][p_buf]
  __shared__ uint64_t bar[2];
  const int tid = threadIdx.x, items = a.L * a.nblk;
  const bool p_shared = 0 == a.sp;
  const uint32_t xbytes = (uint32_t)a.x_elems * sizeof(T);
  const T* gx = (const T*)a.x;
  const T* gp = (const T*)a.p;
  long long e = blockIdx.x;
  if (e >= a.n_elem) return;
  if (0 == tid) { mbar_init(&bar[0], 1); mbar_init(&bar[1], 1); mbar_fence_init(); }
  // Whether an element is computed is decided by a barrier reduction over the whole CTA, so that the thread issuing its bulk
  // copy and every thread waiting for it agree.  The decision for the element of iteration it + 1 is taken at the end of
  // iteration it - 1 (the prologue for it = 0), before issue() starts its copies.
  const long long g = gridDim.x;
  auto decide = [&](long long el) {
    if (kIx) return 0 != __syncthreads_and(el < a.n_elem && rm_runs<kIx>(a, el));
    __syncthreads();
    return true;                                        // (unused: issue() tests el < n_elem itself)
  };
  bool run = kIx ? decide(e) : true;
  bool run_next = decide(e + g);
  // element el lands in buffer b: X by the bulk copy, a per-element P by cp.async (one group per thread and iteration, empty for
  // a skipped element and past the last one, so that wait_group 1 always means "everything but the newest")
  auto issue = [&](long long el, int b, bool go) {
    if (kIx ? go : el < a.n_elem) {
      if (0 == tid) {
        mbar_arrive_expect_tx(&bar[b], xbytes);
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n"
                     ::"r"(smem_u32(xbuf + b * a.x_buf)), "l"(gx + rm_slot<kIx>(a.xi, el) * a.sx), "r"(xbytes), "r"(smem_u32(&bar[b])) : "memory");
      }
      if (!p_shared) {
        const T* src = gp + rm_slot<kIx>(a.pi, el) * a.sp;
        for (int i = tid; i < a.p_elems; i += blockDim.x) cp_async_elem(pbuf + b * a.p_buf + i, src + i);
      }
    }
    if (!p_shared) cp_async_commit();
  };
  if (p_shared)
    for (int i = tid; i < a.p_elems; i += blockDim.x) pbuf[i] = gp[i];
  issue(e, 0, run);
  // bit b of parity: phase of the next completion of bar[b], flipped for every copy issued into (and waited on in) buffer b (without
  // skipped elements every iteration fills its buffer, and the phase follows from the iteration number)
  uint32_t parity = 0;
  for (int it = 0; e < a.n_elem; e += g, ++it) {
    const int b = it & 1;
    issue(e + g, b ^ 1, run_next);
    if (!p_shared) cp_async_wait_prev();
    if (!kIx || run) {
      mbar_wait(&bar[b], kIx ? (parity >> b) & 1u : (uint32_t)(it >> 1) & 1u);
      parity ^= 1u << b;
      __syncthreads();                                  // cp.async data of the other threads (and the shared P) visible
      const T* X = xbuf + b * a.x_buf;
      const T* P = p_shared ? pbuf : pbuf + b * a.p_buf;
      T* C = (T*)a.c + rm_slot<kIx>(a.ci, e) * a.sc;
      for (int i = tid; i < items; i += blockDim.x) rm_item<T, int>(a, X, P, C, i);
    }
    run = run_next;
    run_next = decide(e + 2 * g);                       // (its barrier: buffer b is read out before iteration it + 1 refills it)
    if (0 == tid) fence_proxy_async();
  }
}

template <typename T, bool kIx>
void launch(const RmArgs& a0, bool staged, cudaStream_t stream)
{
  RmArgs a = a0;
  const int items = a.L * a.nblk;
  const int rounds = (items + kMaxThreads - 1) / kMaxThreads;
  const int threads = ((items + rounds - 1) / rounds + 31) / 32 * 32;
  int per_sm = 1;
  size_t smem = 0;
  if (staged) {
    a.x_buf = (int)((a.x_elems * (long long)sizeof(T) + 15) / 16 * 16 / (long long)sizeof(T));
    a.p_buf = (int)a.p_elems;
    smem = ((size_t)2 * a.x_buf + (size_t)(0 == a.sp ? 1 : 2) * a.p_buf) * sizeof(T);
    ensure_smem_optin((const void*)rm_soa_staged_kernel<T, kIx>, (int)smem);
    XB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, rm_soa_staged_kernel<T, kIx>, threads, smem));
  }
  else XB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, rm_soa_direct_kernel<T, kIx>, threads, 0));
  const long long grid = std::min<long long>(a.n_elem, (long long)std::max(per_sm, 1) * device_sm_count());
  if (staged) rm_soa_staged_kernel<T, kIx><<<(unsigned)grid, threads, smem, stream>>>(a);
  else rm_soa_direct_kernel<T, kIx><<<(unsigned)grid, threads, 0, stream>>>(a);
  XB_CUDA(cudaGetLastError());
}

}  // namespace

// bytes of shared memory one CTA of the staged kernel may use (the opt-in maximum of the device)
static int smem_limit()
{
  int dev = 0, v = 0;
  if (cudaSuccess != cudaGetDevice(&dev) || cudaSuccess != cudaDeviceGetAttribute(&v, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev)) {
    (void)cudaGetLastError();
    return 0;
  }
  return v - 1024;        // the kernel's static barriers and the runtime's reserve
}

void rm_soa_execute(const RmSoa& h, const void* d_a, const void* d_b, void* d_c, long long n_elem, long long stride_a,
                    long long stride_b, long long stride_c, ElemIndex ia, ElemIndex ib, ElemIndex ic, cudaStream_t stream)
{
  const bool ac = 0 == h.form;
  const size_t esz = h.is_double ? 8 : 4;
  RmArgs a = {};
  a.c = d_c; a.sc = stride_c; a.n_elem = n_elem; a.soa = h.soa; a.K = h.K; a.beta_one = h.beta_one;
  if (ac) {         // X = A [M][lda][soa], P = b [K][ldb], j = n
    a.x = d_a; a.sx = stride_a; a.p = d_b; a.sp = stride_b;
    a.L = h.M * h.soa; a.J = h.N;
    a.xs_l = (long long)h.lda * h.soa; a.xs_k = h.soa; a.ps_k = h.ldb; a.ps_j = 1;
    a.cs_l = (long long)h.ldc * h.soa; a.cs_j = h.soa;
    a.x_elems = ((long long)(h.M - 1) * h.lda + h.K) * h.soa; a.p_elems = (long long)(h.K - 1) * h.ldb + h.N;
    a.xi = ia.idx; a.x_slots = ia.slots; a.pi = ib.idx; a.p_slots = ib.slots;
  }
  else {            // X = B [K][ldb][soa], P = a [M][lda], j = m
    a.x = d_b; a.sx = stride_b; a.p = d_a; a.sp = stride_a;
    a.L = h.N * h.soa; a.J = h.M;
    a.xs_l = h.soa; a.xs_k = (long long)h.ldb * h.soa; a.ps_k = 1; a.ps_j = h.lda;
    a.cs_l = h.soa; a.cs_j = (long long)h.ldc * h.soa;
    a.x_elems = ((long long)(h.K - 1) * h.ldb + h.N) * h.soa; a.p_elems = (long long)(h.M - 1) * h.lda + h.K;
    a.xi = ib.idx; a.x_slots = ib.slots; a.pi = ia.idx; a.p_slots = ia.slots;
  }
  a.ci = ic.idx; a.c_slots = ic.slots;
  if (0 == a.xi) a.x_slots = n_elem;                    // no index: slot e < n_elem, never skipped
  if (0 == a.pi) a.p_slots = n_elem;
  if (0 == a.ci) a.c_slots = n_elem;
  a.nblk = (a.J + kRB - 1) / kRB;
  const size_t xbytes = (size_t)a.x_elems * esz;
  const size_t smem = 2 * ((xbytes + 15) / 16 * 16) + (size_t)(0 == a.sp ? 1 : 2) * (size_t)a.p_elems * esz;
  const bool staged = 0 == ((uintptr_t)a.x & 15) && 0 == ((size_t)a.sx * esz) % 16 && 0 == xbytes % 16 && smem <= (size_t)smem_limit();
  static const char* const names[2][2] = {{"rm_soa_ac (direct)", "rm_soa_ac (staged)"}, {"rm_soa_bc (direct)", "rm_soa_bc (staged)"}};
  note_compute_kernel(names[ac ? 0 : 1][staged ? 1 : 0]);
  count_launch(1);
  const bool ix = a.xi || a.pi || a.ci;
  if (h.is_double) (ix ? launch<double, true> : launch<double, false>)(a, staged, stream);
  else (ix ? launch<float, true> : launch<float, false>)(a, staged, stream);
}

}  // namespace xb
