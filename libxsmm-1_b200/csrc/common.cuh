// Shared declarations of the B200-native SPMDM / FSSPMDM implementation (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stddef.h>
#include <stdlib.h>

namespace xb {

// ---- sticky error state (reference entry points return void: src/libxsmm_spmdm.c:140-142) ----
void set_error(int code, const char* fmt, ...);
int verbosity();
void count_launch(int n);
// Opt-in to more than 48 KiB of dynamic shared memory, once per (kernel, device); callers may race (the legacy
// *_thread entries are called from OpenMP regions) and a process may drive several devices.
void ensure_smem_optin(const void* kernel, int bytes);
int device_sm_count();
void note_compute_kernel(const char* name);   // which spmdm compute / fsspmdm kernel the last call enqueued (reported by bench.py)

#define XB_CUDA(call)                                                                      \
  do {                                                                                     \
    cudaError_t xb_e_ = (call);                                                            \
    if (cudaSuccess != xb_e_) {                                                            \
      xb::set_error((int)xb_e_, "%s:%d: %s -> %s", __FILE__, __LINE__, #call,              \
                    cudaGetErrorString(xb_e_));                                            \
    }                                                                                      \
  } while (0)

// ---- SPMDM ----------------------------------------------------------------------------------
// Block geometry, same meaning as the fields of libxsmm_spmdm_handle
// (reference include/libxsmm_spmdm.h:42-60).
struct Geom { int m, n, k, bm, bn, bk, mb, nb, kb; };

// Flat device layout of the CSR slice arena.  Slice s = kb*mb + mb owns
//   rowidx[s*(bm+1) ..], colidx[s*bm*bk ..], values[s*bm*bk ..]
// (same logical arrays as reference src/libxsmm_spmdm.c:126-136; the byte packing differs
// because the reference leaves `values` only 2-byte aligned).
struct SliceArena {
  uint16_t* rowidx;
  uint16_t* colidx;
  float* values;
  uint32_t* slice_nnz;   // auxiliary: true nonzero count of every slice (the u16 row pointers wrap at 65536)
  uint16_t* tcoff;   // auxiliary (not part of the reference's slice), same indexing as colidx: where the nonzero
                     // goes in the tensor-core branch's shared-memory A tile (fp32 slices: xb_tc_pack)
  uint32_t* tcpk;    // the same memory seen as 32-bit words (bf16 slices: xb_tc16_pack, value and position in one word)
  uint32_t* slice_ovf;   // auxiliary: overflow entries (see tcsp) of every slice, written by the slicing kernel that writes tcsp
  uint2* ovf_list;       // auxiliary: the first kSpOvfCap overflow entries of every slice, in no particular order: {row in the slice | k in the slice << 16, value bits}
  uint32_t* tcsp;    // auxiliary, bf16 slices sliced by the wide kernel: one more word per nonzero for the 2:4 structured-sparse
                     // tensor-core kernel (spmdm_compute_tc16s.cu): metadata of the row's 16-k span << 16 | overflow << 15 |
                     // position of the kept element in the compressed A tile (xb_sp_pos)
  float* dense;      // auxiliary, optional (fp32 slices of dense matrices): the slice once more as the tensor-core kernel's
                     // shared-memory image -- per (slice, 128-row tile, 64-k half) 64 KiB: a_hi chunk 0, 1, a_lo chunk 0, 1,
                     // each [128 rows x 32 k] fp32, K-major, SWIZZLE_128B -- so that K4 fetches a half with one bulk copy
                     // instead of rebuilding it from (column, value) pairs.  0 until a dense matrix shows up.
};

// Tensor-core branch (spmdm_compute_tc.cu): A is rebuilt per k-block as two K-halves (k < 64, k >= 64), each
// two K-major SWIZZLE_128B chunks of [128 rows x 32 k] fp32 (16 KiB).  For a nonzero at block-local row r
// and column k: bit 15 = half, bits 0..14 = word offset inside the half (chunk, 8-row group, row, 16-byte
// unit XOR row, word).  Rows are taken modulo the 128-row tile.
#if defined(__CUDACC__)
__host__ __device__ __forceinline__ uint16_t xb_tc_pack(int r, int k)
{
  const int row = r & 127, kk = k & 31;
  const uint32_t off = (uint32_t)(((k >> 5) & 1) * 16384 + (row >> 3) * 1024 + (row & 7) * 128 + ((((kk >> 2) ^ (row & 7)) & 7) << 4) + ((kk & 3) << 2));
  return (uint16_t)((off >> 2) | ((uint32_t)(k >> 6) << 15));
}
#endif

// bf16 slices (spmdm_compute_tc16*.cu): the A tile is [128 rows x 64 k] bf16 per K-half, K-major SWIZZLE_128B
// (16 KiB).  One word per nonzero: bf16 value << 16 | half << 15 | (byte offset inside the half) >> 1.
#if defined(__CUDACC__)
__host__ __device__ __forceinline__ uint32_t xb_tc16_pack(int r, int k, uint32_t f32_bits)
{
  const uint32_t row = (uint32_t)r & 127u, kk = (uint32_t)k & 63u;
  const uint32_t off = (row >> 3) * 1024u + (row & 7u) * 128u + ((((kk >> 3) ^ row) & 7u) << 4) + ((kk & 7u) << 1);
  return (f32_bits & 0xFFFF0000u) | ((((uint32_t)k >> 6) & 1u) << 15) | (off >> 1);
}
#endif

// 2:4 structured-sparse tensor-core kernel (spmdm_compute_tc16s.cu, tcgen05.mma.sp kind::f16): of every four consecutive k
// of a row the tensor core takes two KEPT elements plus a 4-bit nibble (position of the first | position of the second << 2,
// first < second).  A group of four with one nonzero at p keeps it in slot p & 1 under the nibble (0,1) or (2,3); with two or
// more nonzeros the first two are kept and the others are OVERFLOW entries, which a CUDA-core pass adds afterwards.
// Compressed A tile per (128 rows, 128 k): [128 rows x 64 kept bf16], K-major SWIZZLE_128B (16 KiB).
#if defined(__CUDACC__)
__host__ __device__ __forceinline__ uint32_t xb_sp_pos(uint32_t row, uint32_t slot)   // (byte offset in the compressed tile) >> 1
{
  return (((row >> 3) & 15u) * 1024u + (row & 7u) * 128u + ((((slot >> 3) ^ row) & 7u) << 4) + ((slot & 7u) << 1)) >> 1;
}
// nibble of a group from its 4-bit nonzero mask (table of 16 nibbles in two words)
__host__ __device__ __forceinline__ uint32_t xb_sp_nibble(uint32_t gm)
{
  return (((gm & 8u) ? 0x498E4DCEu : 0x498E4444u) >> ((gm & 7u) * 4u)) & 15u;
}
// slot (0 / 1) of the nonzero at position p of a group with mask gm; bit 1 set: overflow (third or fourth nonzero)
__host__ __device__ __forceinline__ uint32_t xb_sp_slot(uint32_t gm, uint32_t p)
{
#if defined(__CUDA_ARCH__)
  const uint32_t rank = (uint32_t)__popc(gm & ((1u << p) - 1u));
#else
  const uint32_t rank = (uint32_t)__builtin_popcount(gm & ((1u << p) - 1u));
#endif
  if (0 == (gm & (gm - 1u))) return p & 1u;
  return rank >= 2u ? 3u : rank;
}
// Metadata image of a compressed tile (2 KiB, the operand of tcgen05.cp.128x128b: tensor-memory lane L at byte 16 L): byte
// offset of the 16-bit metadata word of (row, 16-k span), from the position xb_sp_pos of any kept element of that span.
// Lane = row % 8 + 8 * (span % 2) + 16 * (row / 16), column = span / 2, upper half word for rows 8..15 of 16.
__host__ __device__ __forceinline__ uint32_t xb_sp_meta_off(uint32_t pos)
{
  const uint32_t r7 = (pos >> 6) & 7u, span = ((pos >> 3) & 7u) ^ r7;
  const uint32_t tl = r7 + ((span & 1u) << 3) + ((pos >> 10) << 4);
  return tl * 16u + (span >> 1) * 4u + ((pos >> 8) & 2u);
}
#endif

constexpr int kSpOvfCap = 256;        // overflow entries listed per slice (SliceArena::ovf_list); a slice with more is walked by its row pointers instead

constexpr int kSliceStripRows = 64;   // rows of one slice handled by one CTA of the slicing kernel

struct SliceArgs {
  const void* a;        // dense A (float or bf16 bits)
  long long lda;        // elements between consecutive rows ('N') or consecutive k ('T')
  int transa;           // 0: A is m x k row-major, 1: A is stored k x m
  int is_bf16;
  int origin_is_block;  // 1: `a` already points at the block's first element (legacy staged block)
  int slice0;           // slice handled by the first CTA (cluster) of the launch
  int slice_step;       // slice of CTA i = slice0 + i*slice_step (1: consecutive slices; mb: all k-blocks of one row block)
  int simd_w;           // vector width of the reference instantiation mirrored (NaN rule)
  Geom g;
  SliceArena out;
  // density feedback for the host (see capi.cu: a lagging hint that only steers which kernels are enqueued):
  // every slice adds its count to acc[0] and bumps acc[1]; the CTA that completes the set publishes the total
  // to *host_total (mapped pinned memory) and resets the counters
  unsigned long long* acc;
  unsigned long long* host_total;
  int total_slices;
  int write_aux;        // 0: skip the auxiliary per-nonzero words (tensor-core kernels will not be enqueued)
  int write_dense;      // 1: also write the dense tile image (SliceArena::dense; fp32, transa = 'N', complete k-blocks)
  int write_sp;         // 1: also write the per-nonzero word of the structured-sparse tensor-core kernel (SliceArena::tcsp; wide bf16 kernel only)
};

#if defined(__CUDACC__)
__device__ __forceinline__ void xb_publish_nnz(const SliceArgs& p, unsigned long long slice_total)
{
  if (0 == p.acc) return;
  atomicAdd(p.acc, slice_total);
  __threadfence();
  const unsigned long long done = atomicAdd(p.acc + 1, 1ull);
  if (done + 1 == (unsigned long long)p.total_slices) {
    const unsigned long long total = atomicExch(p.acc, 0ull);
    p.acc[1] = 0ull;
    if (p.host_total) { *(volatile unsigned long long*)p.host_total = total; __threadfence_system(); }
  }
}
#endif

// mode boundaries of the reference's narrow last block (compute template :72-76,372-434)
struct ColModes { int n_full_end; int tail_from; };

// Density (nnz / (M*K)) from which the tensor-core twin takes over, measured on B200 (2048^3 and 4096^3):
//   bf16: the CTA-pair kernel costs the same at any density and orientation (93 us for 4096^3, 28 us for 2048^3); the
//         TMA CUDA-core kernel (N/N/N) is ahead of it below ~0.5 %, the generic one (transb / transc) never is.
//   fp32: 3xTF32 costs 70-78 us for 2048^3 when the slices carry their dense image (the CTA-pair kernel; matrices the
//         last slicing pass found below 1 % dense are sliced without it)
//         and ~104 us / ~180 us without it (single-CTA kernel, patching / wiping variant); the TMA kernel (N/N/N) is
//         ahead below ~2.8 %, the generic one below ~1 % (transc) and never (transb).
inline double tc_density_threshold(bool is_bf16, bool transb, bool transc)
{
  if (is_bf16) return (transb || transc) ? 0.0 : 0.005;
  return transb ? 0.0 : (transc ? 0.01 : 0.028);
}

struct ComputeArgs {
  SliceArena sl;
  const void* b;      // local column 0 / k 0
  long long ldb;      // 'N': elements between k rows; 'T': elements between n rows
  float* c;           // local row 0 / local column 0
  long long ldc;      // 'N': elements between m rows; 'T': elements between n rows
  int transb, transc, is_bf16;
  float beta;
  Geom g;
  int mb_first, mb_count;   // row blocks computed
  int row_origin;           // global row that local C row 0 corresponds to
  int col_origin;           // global column that local column 0 corresponds to
  int ncols;                // local columns computed
  ColModes modes;           // in GLOBAL column numbering
  // sparse / tensor-core twin launches: both kernels are enqueued, each CTA sums slice_nnz and only the
  // selected kernel does the work (dense <=> total nnz >= tc_min_nnz).  tc_twin = 0: no twin, always run.
  int tc_twin;
  unsigned long long tc_min_nnz;
  int aux_valid;        // the slices' per-nonzero auxiliary words (tcoff / tcpk) were written for ALL slices by the pass these slices come from
  int sp_valid;         // ... and so were the words of the structured-sparse kernel (tcsp)
  // Guarded pair K4s | K4p: the host's density estimate has just changed (or is one observation old), so it may be a dense matrix
  // that arrives: both kernels are enqueued, each sums the slices' counts, K4s (sp_guard = 1) works iff nnz <= sp_max_nnz,
  // K4p (sp_guard = 2) iff nnz > sp_max_nnz.  0: no guard (stable estimate: K4s alone).
  int sp_guard;
  unsigned long long sp_max_nnz;
  int dense_valid;      // the slices' dense tile image (SliceArena::dense) was written by the slicing pass these slices come from
  float density_hint;   // host's lagging estimate of nnz / (M*K) from the last completed slicing pass, < 0: unknown (performance only)
  int debug_flags;  // developer timing aid (LIBXSMM_B200_K2S_DEBUG; results are wrong when set): 1 = skip the multiply-adds, 2 = skip the B tile loads
  int tc_hint;      // host's lagging density hint: 0 unknown / borderline (enqueue both twins), 1 clearly sparse (CUDA cores only), 2 clearly dense (tensor cores only)
};

#if defined(__CUDACC__)
// total nonzero count over all slices, evaluated redundantly by every CTA (ns is a few hundred at most)
__device__ __forceinline__ unsigned long long xb_total_nnz(const uint32_t* slice_nnz, int ns)
{
  __shared__ unsigned long long xb_nnz_s;
  if (threadIdx.x < 32) {
    unsigned long long t = 0;
    for (int i = (int)threadIdx.x; i < ns; i += 32) t += slice_nnz[i];
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) t += __shfl_xor_sync(0xffffffffu, t, d);
    if (0 == threadIdx.x) xb_nnz_s = t;
  }
  __syncthreads();
  return xb_nnz_s;
}
#endif

#if defined(__CUDACC__)
// Launch with programmatic stream serialization: the grid may be scheduled while the kernel in front of it in the stream is
// still draining; the kernel itself waits (ptx.cuh: pdl_wait) before it touches anything that kernel wrote or still reads.
// LIBXSMM_B200_PDL=0: plain stream order.
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, Args&&... args)
{
  static const bool pdl = [] { const char* e = getenv("LIBXSMM_B200_PDL"); return !(e && '0' == *e); }();
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = stream;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization; at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at; cfg.numAttrs = pdl ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}
#endif

void launch_slices(const SliceArgs& args, int nslices, cudaStream_t stream);
// A in CSR form (device arrays, 0-based, columns ascending within a row): row_ptr[m + 1], col_idx[nnz], values[nnz] (float or
// bf16 bits).  launch_slices_csr writes every slice of args.g exactly as launch_slices would for the dense matrix holding these
// entries (transa = 'N'), except the dense tile image; args.write_sp is honoured only for bf16 with k % 128 == 0 and simd_w > 1.
struct CsrArgs { const unsigned int* row_ptr; const unsigned int* col_idx; const void* values; uint32_t nnz; };
void launch_slices_csr(const SliceArgs& args, const CsrArgs& csr, cudaStream_t stream);
// A in CSC form (device arrays, 0-based, rows ascending within a column): col_ptr[k + 1], row_idx[nnz], values[nnz].
// launch_slices_csc writes what launch_slices_csr writes for the same A, and launch_slices for the k x m array holding these
// entries with transa = 'T', except the dense tile image.
struct CscArgs { const unsigned int* col_ptr; const unsigned int* row_idx; const void* values; uint32_t nnz; };
void launch_slices_csc(const SliceArgs& args, const CscArgs& csc, cudaStream_t stream);
bool slices_sparse_get_sp_words(const SliceArgs& args);                  // would launch_slices_csr() / _csc() write tcsp for these arguments?
void launch_compute(const ComputeArgs& args, cudaStream_t stream);
bool launch_compute_tma(const ComputeArgs& args, bool partial, cudaStream_t stream);
bool launch_compute_sp(const ComputeArgs& args, cudaStream_t stream);    // K2s: order-preserving TMA-ring kernel (spmdm_compute_sp.cu)
bool launch_compute_tc(const ComputeArgs& args, cudaStream_t stream);
bool launch_compute_tc16p(const ComputeArgs& args, cudaStream_t stream);  // tcgen05 branch for bf16 inputs: CTA-pair kernel
bool launch_compute_tc16s(const ComputeArgs& args, cudaStream_t stream);  // 2:4 structured-sparse CTA-pair kernel (needs SliceArena::tcsp)
bool slices_get_sp_words(const SliceArgs& args);                          // would launch_slices() write tcsp for these arguments?
bool launch_compute_tcq(const ComputeArgs& args, cudaStream_t stream);    // fp32 CTA-pair kernel (needs the slices' dense image)  // CTA-pair (cta_group::2) persistent form of it

// ---- FSSPMDM --------------------------------------------------------------------------------
struct FsOperator;   // fsspmdm.cu
FsOperator* fs_plan(int is_double, int M, int N, int K, int lda, int ldb, int ldc, double beta, const void* a_dense);   // host only
void fs_plan_info(const FsOperator* o, long long* info);
char* fs_kernel_source(const FsOperator* o);
FsOperator* fs_create(int is_double, int M, int N, int K, int lda, int ldb, int ldc, double beta, const void* a_dense);
FsOperator* fs_create_csr(int is_double, int M, int N, int K, int lda, int ldb, int ldc, int soa, double beta,
                          const unsigned int* rowptr, const unsigned int* colidx, const void* values);
FsOperator* fs_create_csc(int is_double, int M, int N, int K, int lda, int ldc, int soa, double beta,
                          const unsigned int* colptr, const unsigned int* rowidx, const void* values);
// the slot of every element in one operand of the batched SoA entries: idx[e] (a DEVICE array) or, for idx = NULL, e itself;
// an element with a slot at or past `slots` is skipped
struct ElemIndex { const unsigned int* idx; long long slots; };
void fs_execute_batched(const FsOperator* o, const void* dB, void* dC, long long n_elem, long long stride_b, long long stride_c,
                        ElemIndex ib, ElemIndex ic, cudaStream_t stream);
void fs_execute(const FsOperator* op, const void* dB, void* dC, long long ncols, long long ldb, long long ldc, cudaStream_t stream);
int fs_is_sparse_branch(const FsOperator* o);
int fs_is_baked(const FsOperator* o);
int fs_is_tensor_core(const FsOperator* o);
int fs_needs_c_input(const FsOperator* o);
int fs_is_double(const FsOperator* o);
long long fs_soa_c_extent(const FsOperator* o);   // scalars from the first to past the last C entry one element of a csr_soa handle writes
void fs_shape(const FsOperator* o, int* M, int* N, int* K, int* ldb, int* ldc, int* beta_one);
void fs_destroy(FsOperator* op);

// ---- fixed 2:4-sparse bf16 and FP8 operators (sp24.cu); arguments checked by capi.cu ---------------------------------------------
struct Sp24Op;
Sp24Op* sp24_create(int M, int K, int lda, const void* a, bool a_on_device, int format);     // format: -1 bf16, 0 e4m3, 1 e5m2
void sp24_execute(const Sp24Op* op, bool transb, bool transc, int N, const uint16_t* d_b, int ldb, float beta, float* d_c, int ldc, cudaStream_t stream);
void sp24_execute_fp8(const Sp24Op* op, bool transb, bool transc, int N, const unsigned char* d_b, int b_format, int ldb, float alpha, float beta,
                      float* d_c, int ldc, cudaStream_t stream);
void sp24_execute_bf16out(const Sp24Op* op, bool transb, bool transc, int N, const uint16_t* d_b, int ldb, const uint16_t* d_bias, float beta,
                          uint16_t* d_c, int ldc, cudaStream_t stream);
void sp24_execute_fp8_bf16out(const Sp24Op* op, bool transb, bool transc, int N, const unsigned char* d_b, int b_format, int ldb, float alpha,
                              const uint16_t* d_bias, float beta, uint16_t* d_c, int ldc, cudaStream_t stream);
int sp24_format(const Sp24Op* op);
int sp24_device(const Sp24Op* op);
int sp24_rows(const Sp24Op* op);
int sp24_cols(const Sp24Op* op);
void sp24_destroy(Sp24Op* op);

// ---- dense SoA kernels (rm_soa.cu) ----------------------------------------------------------
// form 0: ac (A and C are [row][ld][soa], b is plain row-major), 1: bc (B and C are SoA, a is plain)
struct RmSoa { int is_double, form, M, N, K, lda, ldb, ldc, soa, beta_one; };
void rm_soa_execute(const RmSoa& h, const void* d_a, const void* d_b, void* d_c, long long n_elem, long long stride_a,
                    long long stride_b, long long stride_c, ElemIndex ia, ElemIndex ib, ElemIndex ic, cudaStream_t stream);

}  // namespace xb
