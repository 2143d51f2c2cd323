// SPMDM kernels for sm_100a:
//   K1  spmdm_slice_kernel    dense A -> CSR slices   (reference createSparseSlice templates)
//   K2  spmdm_compute_kernel  C = beta*C + slices * B (reference compute templates)
// Hand-written CUDA; no library calls on the data path.
#include "common.cuh"
#include "ptx.cuh"
#include <map>
#include <cooperative_groups.h>
#include <mutex>
#include <cstdlib>

namespace cg = cooperative_groups;

namespace xb {

// =================================================================================================
// K1: slice compaction.
// One cluster of CTAs per slice (bm x 128 block of A), one CTA per strip of 64 rows.  The strip
// is staged once in shared memory (coalesced 16-byte loads; transposed on the fly for transa='T'),
// every warp then owns rows: 4 ballots per row give the per-lane exclusive prefix in ascending
// column order, a warp scan gives row offsets inside the strip, and strip totals are exchanged
// between the CTAs of the cluster through distributed shared memory so that every CTA knows its
// base offset inside the slice without a second kernel.
// Bit-exact with reference src/template/libxsmm_spmdm_createSparseSlice_{fp32,bfloat16}_thread.tpl.c:
// row pointers, column indices and values in [0, nnz) of every slice.
// =================================================================================================
constexpr int K1_THREADS = 256;
constexpr int K1_WARPS = K1_THREADS / 32;
constexpr int K1_R = kSliceStripRows;
constexpr int K1_TPITCH = K1_R + 1;   // pitch of the transposed tile (conflict-free column reads)

// Non-zero test of the reference: vector loops use an ordered compare (NaN dropped,
// src/libxsmm_spmdm_begin_avx2.h:54), the scalar remainder keeps NaN (fp32 tpl.c:129-133).
__device__ __forceinline__ bool k1_keep(float v, int k, int vec_end)
{
  return (v < 0.f || v > 0.f) || (k >= vec_end && v != v);
}

__global__ void __launch_bounds__(K1_THREADS) spmdm_slice_kernel(const SliceArgs p)
{
  cg::cluster_group cluster = cg::this_cluster();
  __shared__ __align__(16) uint32_t tile[128 * K1_TPITCH];
  __shared__ uint32_t row_cnt[K1_R];
  __shared__ uint32_t row_off[K1_R];
  __shared__ uint32_t strip_tot[8];

  const Geom& g = p.g;
  const int s = p.slice0 + (int)blockIdx.y * p.slice_step;
  const int kb = s / g.mb, mbi = s - kb * g.mb;
  const int nrows = min(g.bm, g.m - mbi * g.bm);
  const int ncols = min(g.bk, g.k - kb * g.bk);
  int vec_end = p.is_bf16 ? (ncols / (4 * p.simd_w)) * (4 * p.simd_w) : (ncols / p.simd_w) * p.simd_w;
  if (p.simd_w <= 1) vec_end = 0;
  const int strip = (int)blockIdx.x, nstrips = (int)gridDim.x;
  const int r0 = strip * K1_R;
  const int rcount = max(0, min(K1_R, nrows - r0));
  const int tid = (int)threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const long long origin = p.origin_is_block ? 0ll
    : (p.transa ? ((long long)kb * g.bk * p.lda + (long long)mbi * g.bm)
                : ((long long)mbi * g.bm * p.lda + (long long)kb * g.bk));

  // ---- stage the strip: tile holds fp32 bit patterns (bf16 widened by <<16) --------------------
  if (!p.transa) {
    if (!p.is_bf16) {
      const float* A = (const float*)p.a + origin + (long long)r0 * p.lda;
      const bool vec = (0 == (p.lda & 3)) && (0 == ((uintptr_t)A & 15));
      for (int idx = tid; idx < rcount * 32; idx += K1_THREADS) {
        const int r = idx >> 5, k = (idx & 31) * 4;
        const float* src = A + (long long)r * p.lda + k;
        uint4 w = make_uint4(0, 0, 0, 0);
        if (vec && k + 3 < ncols) w = __ldg((const uint4*)src);
        else {
          if (k < ncols) w.x = __float_as_uint(__ldg(src));
          if (k + 1 < ncols) w.y = __float_as_uint(__ldg(src + 1));
          if (k + 2 < ncols) w.z = __float_as_uint(__ldg(src + 2));
          if (k + 3 < ncols) w.w = __float_as_uint(__ldg(src + 3));
        }
        *(uint4*)&tile[r * 128 + k] = w;
      }
    }
    else {
      const uint16_t* A = (const uint16_t*)p.a + origin + (long long)r0 * p.lda;
      const bool vec = (0 == (p.lda & 3)) && (0 == ((uintptr_t)A & 7));
      for (int idx = tid; idx < rcount * 32; idx += K1_THREADS) {
        const int r = idx >> 5, k = (idx & 31) * 4;
        const uint16_t* src = A + (long long)r * p.lda + k;
        uint4 w = make_uint4(0, 0, 0, 0);
        if (vec && k + 3 < ncols) {
          const uint2 raw = __ldg((const uint2*)src);
          w.x = raw.x << 16; w.y = raw.x & 0xFFFF0000u; w.z = raw.y << 16; w.w = raw.y & 0xFFFF0000u;
        }
        else {
          if (k < ncols) w.x = (uint32_t)__ldg(src) << 16;
          if (k + 1 < ncols) w.y = (uint32_t)__ldg(src + 1) << 16;
          if (k + 2 < ncols) w.z = (uint32_t)__ldg(src + 2) << 16;
          if (k + 3 < ncols) w.w = (uint32_t)__ldg(src + 3) << 16;
        }
        *(uint4*)&tile[r * 128 + k] = w;
      }
    }
  }
  else {  // A stored k x m: consecutive rows of the slice are contiguous in memory: four of them per load
    const size_t esz = p.is_bf16 ? 2 : 4;
    const bool vec = (0 == (p.lda & 3)) && (0 == (((uintptr_t)p.a + (size_t)(origin + r0) * esz) & (p.is_bf16 ? 7 : 15)));
    for (int idx = tid; idx < ncols * (K1_R / 4); idx += K1_THREADS) {
      const int k = idx / (K1_R / 4), r = (idx - k * (K1_R / 4)) * 4;
      const long long at = origin + (long long)k * p.lda + r0 + r;
      uint32_t* dst = &tile[k * K1_TPITCH + r];
      if (vec && r + 3 < rcount) {
        if (p.is_bf16) {
          const uint2 raw = __ldg((const uint2*)((const uint16_t*)p.a + at));
          dst[0] = raw.x << 16; dst[1] = raw.x & 0xFFFF0000u; dst[2] = raw.y << 16; dst[3] = raw.y & 0xFFFF0000u;
        }
        else {
          const uint4 raw = __ldg((const uint4*)((const float*)p.a + at));
          dst[0] = raw.x; dst[1] = raw.y; dst[2] = raw.z; dst[3] = raw.w;
        }
      }
      else {
        for (int e = 0; e < 4; ++e) {
          if (r + e < rcount) dst[e] = p.is_bf16 ? ((uint32_t)__ldg((const uint16_t*)p.a + at + e) << 16) : __float_as_uint(__ldg((const float*)p.a + at + e));
        }
      }
    }
  }
  __syncthreads();

  // ---- pass 1: per-row counts -------------------------------------------------------------------
  for (int r = warp; r < rcount; r += K1_WARPS) {
    uint32_t c = 0;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int k = 32 * j + lane;
      const float v = __uint_as_float(p.transa ? tile[k * K1_TPITCH + r] : tile[r * 128 + k]);
      const bool keep = (k < ncols) && k1_keep(v, k, vec_end);
      c += __popc(__ballot_sync(0xffffffffu, keep));
    }
    if (0 == lane) row_cnt[r] = c;
  }
  __syncthreads();

  // ---- strip-local exclusive scan of the 64 row counts (warp 0, two rows per lane) ---------------
  uint32_t total = 0;
  if (0 == warp) {
    const uint32_t a0 = (2 * lane < rcount) ? row_cnt[2 * lane] : 0u;
    const uint32_t a1 = (2 * lane + 1 < rcount) ? row_cnt[2 * lane + 1] : 0u;
    uint32_t inc = a0 + a1;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const uint32_t t = __shfl_up_sync(0xffffffffu, inc, d);
      if (lane >= d) inc += t;
    }
    row_off[2 * lane] = inc - (a0 + a1);
    row_off[2 * lane + 1] = inc - a1;
    total = inc;   // valid in lane 31
  }

  // ---- exchange strip totals across the cluster (distributed shared memory) ----------------------
  cluster.sync();   // every CTA of the cluster is resident before remote shared memory is touched
  if (31 == tid) {
    for (int q = 0; q < nstrips; ++q) *cluster.map_shared_rank(&strip_tot[strip], q) = total;
  }
  cluster.sync();
  uint32_t base = 0, slice_total = 0;
  for (int q = 0; q < strip; ++q) base += strip_tot[q];
  for (int q = 0; q < nstrips; ++q) slice_total += strip_tot[q];
  // a completely full 512 x 128 slice wraps the reference's u16 counter (template :72): its last row pointer reads 0 and
  // the reference's multiply sees row 511 as EMPTY.  The dense image mirrors that (the CSR arrays do by construction).
  const bool wrapped = slice_total >= 65536u;

  // ---- pass 2: write row pointers, column indices, values ---------------------------------------
  uint16_t* ro = p.out.rowidx + (size_t)s * (g.bm + 1);
  uint16_t* co = p.out.colidx + (size_t)s * g.bm * g.bk;
  float* va = p.out.values + (size_t)s * g.bm * g.bk;
  uint16_t* ri = p.out.tcoff + (size_t)s * g.bm * g.bk;
  uint32_t* rk = p.out.tcpk + (size_t)s * g.bm * g.bk;
  const uint32_t lt = (1u << lane) - 1u;
  for (int r = warp; r < rcount; r += K1_WARPS) {
    uint32_t pos = base + row_off[r];
    if (0 == lane) ro[r0 + r] = (uint16_t)pos;   // u16 like the reference's counter (tpl.c:72,78)
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int k = 32 * j + lane;
      const float v = __uint_as_float(p.transa ? tile[k * K1_TPITCH + r] : tile[r * 128 + k]);
      const bool keep = (k < ncols) && k1_keep(v, k, vec_end);
      const uint32_t bal = __ballot_sync(0xffffffffu, keep);
      if (keep) {
        const uint32_t q = pos + __popc(bal & lt);
        co[q] = (uint16_t)k;
        va[q] = v;
        if (p.write_aux) {
          if (p.is_bf16) rk[q] = xb_tc16_pack(r0 + r, k, __float_as_uint(v));
          else ri[q] = xb_tc_pack(r0 + r, k);
        }
      }
      if (p.write_dense && !p.is_bf16) {
        // dense tile image (see SliceArena::dense): the 32 lanes cover one 128-byte image row of chunk j & 1 of half
        // j >> 1 (16-byte units permuted by the swizzle, same line): a_hi, and a_lo 32 KiB further on
        const int rr = r0 + r, trow = rr & 127;
        float* img = p.out.dense + ((size_t)s * ((g.bm + 127) / 128) + (size_t)(rr >> 7)) * 32768
                   + (size_t)(j >> 1) * 16384 + (size_t)(j & 1) * 4096
                   + (size_t)(trow >> 3) * 256 + (size_t)(trow & 7) * 32 + (size_t)((((lane >> 2) ^ trow) & 7) * 4 + (lane & 3));
        const bool in_image = keep && !(wrapped && rr == g.bm - 1);
        const float vh = in_image ? __uint_as_float(__float_as_uint(v) & 0xFFFFE000u) : 0.f;
        img[0] = vh;
        img[8192] = in_image ? (v - vh) : 0.f;
      }
      pos += __popc(bal);
    }
  }
  if (strip == nstrips - 1 && 0 == tid) {
    ro[nrows] = (uint16_t)(base + strip_tot[strip]);
    p.out.slice_nnz[s] = base + strip_tot[strip];
    xb_publish_nnz(p, base + strip_tot[strip]);
  }
}

// -------------------------------------------------------------------------------------------------
// K1 for transa = 'N' (A stored m x k): one CTA per slice, a warp owns a contiguous range of rows.
// Pass 1 streams the rows (one 16-byte / 8-byte load per lane per row, four rows in flight per warp) and
// only counts; the per-warp totals are scanned once per CTA; pass 2 re-reads the rows (now L1/L2
// resident), rebuilds the ballots and writes row pointers, column indices and values.  A is read from
// HBM exactly once; no cluster, one __syncthreads.
// -------------------------------------------------------------------------------------------------
constexpr int K1N_THREADS = 1024;
constexpr int K1N_WARPS = K1N_THREADS / 32;

// A lane holds four consecutive elements (columns lane*4 .. lane*4+3) of a row "as loaded": four fp32
// words, or two words of packed bf16 pairs; widen() gives the fp32 bit patterns (bf16 << 16).
template <bool BF16> struct K1Raw;
template <> struct K1Raw<false> {
  typedef uint4 raw_t;
  static __device__ __forceinline__ raw_t zero() { return make_uint4(0, 0, 0, 0); }
  static __device__ __forceinline__ raw_t load(const void* a, long long lda, int row, int lane, int ncols, bool vec)
  {
    const int k = lane * 4;
    const float* src = (const float*)a + (long long)row * lda + k;
    uint4 w = make_uint4(0, 0, 0, 0);
    if (vec && k + 3 < ncols) w = __ldg((const uint4*)src);
    else {
      if (k < ncols) w.x = __float_as_uint(__ldg(src));
      if (k + 1 < ncols) w.y = __float_as_uint(__ldg(src + 1));
      if (k + 2 < ncols) w.z = __float_as_uint(__ldg(src + 2));
      if (k + 3 < ncols) w.w = __float_as_uint(__ldg(src + 3));
    }
    return w;
  }
  static __device__ __forceinline__ uint4 widen(raw_t r) { return r; }
};
template <> struct K1Raw<true> {
  typedef uint2 raw_t;
  static __device__ __forceinline__ raw_t zero() { return make_uint2(0, 0); }
  static __device__ __forceinline__ raw_t load(const void* a, long long lda, int row, int lane, int ncols, bool vec)
  {
    const int k = lane * 4;
    const uint16_t* src = (const uint16_t*)a + (long long)row * lda + k;
    uint2 r = make_uint2(0, 0);
    if (vec && k + 3 < ncols) r = __ldg((const uint2*)src);
    else {
      if (k < ncols) r.x = (uint32_t)__ldg(src);
      if (k + 1 < ncols) r.x |= (uint32_t)__ldg(src + 1) << 16;
      if (k + 2 < ncols) r.y = (uint32_t)__ldg(src + 2);
      if (k + 3 < ncols) r.y |= (uint32_t)__ldg(src + 3) << 16;
    }
    return r;
  }
  static __device__ __forceinline__ uint4 widen(raw_t r) { return make_uint4(r.x << 16, r.x & 0xFFFF0000u, r.y << 16, r.y & 0xFFFF0000u); }
};

// Exclusive scan of the CW warp totals of a CTA on top of `base` (the kept elements of the rows before the CTA's): the first
// output position of this warp's rows, and the running total after the CTA's rows.  wtot: CW words of shared memory.
struct K1Scan { uint32_t pos; uint32_t slice_total; };

template <int CW>
__device__ __forceinline__ K1Scan k1_scan(uint32_t warp_total, uint32_t* wtot, uint32_t base)
{
  const int tid = (int)threadIdx.x, warp = tid >> 5, lane = tid & 31;
  if (0 == lane) wtot[warp] = warp_total;
  __syncthreads();
  const uint32_t t = (lane < CW) ? wtot[lane] : 0u;
  uint32_t inc = t;
#pragma unroll
  for (int d = 1; d < CW; d <<= 1) {
    const uint32_t u = __shfl_up_sync(0xffffffffu, inc, d);
    if (lane >= d) inc += u;
  }
  const uint32_t cta_total = __shfl_sync(0xffffffffu, inc, CW - 1);
  K1Scan r;
  r.pos = base + __shfl_sync(0xffffffffu, inc - t, warp);
  r.slice_total = base + cta_total;
  return r;
}

// keep-mask of the lane's four elements.  FULL = complete 128-column block whose columns are all inside the
// reference's vector loops: kept iff ordered-nonzero, i.e. |v| > 0 (NaN and -0.0 dropped, denormals kept).
template <bool FULL>
__device__ __forceinline__ uint32_t k1n_mask(uint4 w, int lane, int ncols, int vec_end)
{
  if (FULL) {
    return (fabsf(__uint_as_float(w.x)) > 0.f ? 1u : 0u) | (fabsf(__uint_as_float(w.y)) > 0.f ? 2u : 0u)
         | (fabsf(__uint_as_float(w.z)) > 0.f ? 4u : 0u) | (fabsf(__uint_as_float(w.w)) > 0.f ? 8u : 0u);
  }
  const int k = lane * 4;
  uint32_t m = 0;
  if (k < ncols && k1_keep(__uint_as_float(w.x), k, vec_end)) m |= 1u;
  if (k + 1 < ncols && k1_keep(__uint_as_float(w.y), k + 1, vec_end)) m |= 2u;
  if (k + 2 < ncols && k1_keep(__uint_as_float(w.z), k + 2, vec_end)) m |= 4u;
  if (k + 3 < ncols && k1_keep(__uint_as_float(w.w), k + 3, vec_end)) m |= 8u;
  return m;
}

// ROWS = rows a warp handles (>= rows per warp).  KEEP: the rows stay in registers between the two phases; at 16 rows
// phase 2 re-reads them (fp32 slices of 512 rows do not fit the register file).
template <bool BF16, bool FULL, int ROWS>
__global__ void __launch_bounds__(K1N_THREADS, 1) spmdm_slice_n_kernel(const SliceArgs p)
{
  typedef K1Raw<BF16> Raw;
  typedef typename Raw::raw_t raw_t;
  constexpr bool KEEP = ROWS <= 8;
  __shared__ uint32_t wtot[K1N_WARPS];
  pdl_wait();          // launch_pdl: the slices may still be read by the multiply in front of this kernel in the stream
  pdl_trigger();       // ... and the multiply behind it may be scheduled (it waits in turn)
  const Geom& g = p.g;
  const int s = p.slice0 + (int)blockIdx.x * p.slice_step;
  const int kb = s / g.mb, mbi = s - kb * g.mb;
  const int nrows = min(g.bm, g.m - mbi * g.bm);
  const int ncols = min(g.bk, g.k - kb * g.bk);
  int vec_end = BF16 ? (ncols / (4 * p.simd_w)) * (4 * p.simd_w) : (ncols / p.simd_w) * p.simd_w;
  if (p.simd_w <= 1) vec_end = 0;
  const int tid = (int)threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int rpw = (g.bm + K1N_WARPS - 1) / K1N_WARPS;      // rows per warp (<= 16 because bm <= 512)
  const int row_lo = warp * rpw, row_hi = min(nrows, row_lo + rpw);
  const size_t esz = BF16 ? 2 : 4;
  const long long origin = p.origin_is_block ? 0ll : ((long long)mbi * g.bm * p.lda + (long long)kb * g.bk);
  const char* A = (const char*)p.a + origin * (long long)esz;
  const bool vec = (0 == (p.lda & 3)) && (0 == ((uintptr_t)A & (BF16 ? 7 : 15)));

  // ---- phase 1: load, test, count ---------------------------------------------------------------------
  raw_t w[KEEP ? ROWS : 8];
  uint32_t masks[(ROWS + 7) / 8];        // 4 bits per row
#pragma unroll
  for (int j = 0; j < (ROWS + 7) / 8; ++j) masks[j] = 0;
#pragma unroll
  for (int j0 = 0; j0 < ROWS; j0 += 8) {
#pragma unroll
    for (int j = 0; j < 8; ++j)
      w[KEEP ? j0 + j : j] = (row_lo + j0 + j < row_hi) ? Raw::load(A, p.lda, row_lo + j0 + j, lane, ncols, vec) : Raw::zero();
#pragma unroll
    for (int j = 0; j < 8; ++j)
      masks[(j0 + j) / 8] |= k1n_mask<FULL>(Raw::widen(w[KEEP ? j0 + j : j]), lane, ncols, vec_end) << (4 * ((j0 + j) % 8));
  }
  uint32_t mine = 0;
#pragma unroll
  for (int j = 0; j < (ROWS + 7) / 8; ++j) mine += __popc(masks[j]);
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) mine += __shfl_xor_sync(0xffffffffu, mine, d);
  const K1Scan sc = k1_scan<K1N_WARPS>(mine, wtot, 0u);
  uint32_t pos = sc.pos;   // first output position of this warp's rows
  // completely full 512 x 128 slice: the reference's u16 counter wraps and its multiply sees the last row as empty
  const bool wrapped = sc.slice_total >= 65536u;
  if (0 == tid) {
    p.out.rowidx[(size_t)s * (g.bm + 1) + nrows] = (uint16_t)sc.slice_total;   // u16 like the reference's counter
    p.out.slice_nnz[s] = sc.slice_total;
    xb_publish_nnz(p, sc.slice_total);
  }

  // ---- phase 2: positions and stores -----------------------------------------------------------------------
  uint16_t* ro = p.out.rowidx + (size_t)s * (g.bm + 1);
  uint16_t* co = p.out.colidx + (size_t)s * g.bm * g.bk;
  float* va = p.out.values + (size_t)s * g.bm * g.bk;
  uint16_t* ri = p.out.tcoff + (size_t)s * g.bm * g.bk;
  uint32_t* rk = p.out.tcpk + (size_t)s * g.bm * g.bk;
  const uint32_t lt = (1u << lane) - 1u;
  const int k = lane * 4;
  const bool aux = (0 != p.write_aux);
#pragma unroll
  for (int j = 0; j < ROWS; ++j) {
    if (row_lo + j < row_hi) {     // warp-uniform
      const uint32_t m = (masks[j / 8] >> (4 * (j % 8))) & 15u;
      const uint4 v = Raw::widen(KEEP ? w[KEEP ? j : 0] : Raw::load(A, p.lda, row_lo + j, lane, ncols, vec));
      // lane order = column order: count the kept elements of lower lanes with one ballot per bit of the
      // per-lane count (0..4)
      const uint32_t nm = __popc(m);
      const uint32_t b0 = __ballot_sync(0xffffffffu, nm & 1u), b1 = __ballot_sync(0xffffffffu, nm & 2u), b2 = __ballot_sync(0xffffffffu, nm & 4u);
      uint32_t q = pos + __popc(b0 & lt) + 2 * __popc(b1 & lt) + 4 * __popc(b2 & lt);
      if (0 == lane) ro[row_lo + j] = (uint16_t)pos;
      if (!BF16 && FULL && p.write_dense) {
        // the row's piece of the tensor-core kernel's A image: this lane's four columns are one 16-byte swizzle
        // unit of the [128 rows x 32 k] chunk (lane >> 3) & 1 of the 64-k half lane >> 4; a_hi, then a_lo 32 KiB on
        const int rr = row_lo + j, trow = rr & 127;
        float* img = p.out.dense + ((size_t)s * ((g.bm + 127) / 128) + (size_t)(rr >> 7)) * 32768
                   + (size_t)(lane >> 4) * 16384 + (size_t)((lane >> 3) & 1) * 4096
                   + (size_t)(trow >> 3) * 256 + (size_t)(trow & 7) * 32 + (size_t)(((lane & 7) ^ (trow & 7)) * 4);
        uint4 hi, lo;
        const uint32_t mraw = (masks[j / 8] >> (4 * (j % 8))) & 15u;
        const uint32_t m = (wrapped && rr == g.bm - 1) ? 0u : mraw;   // the image mirrors the wrapped row pointer: row 511 of a full slice is empty
        hi.x = (m & 1u) ? (v.x & 0xFFFFE000u) : 0u; lo.x = (m & 1u) ? __float_as_uint(__uint_as_float(v.x) - __uint_as_float(hi.x)) : 0u;
        hi.y = (m & 2u) ? (v.y & 0xFFFFE000u) : 0u; lo.y = (m & 2u) ? __float_as_uint(__uint_as_float(v.y) - __uint_as_float(hi.y)) : 0u;
        hi.z = (m & 4u) ? (v.z & 0xFFFFE000u) : 0u; lo.z = (m & 4u) ? __float_as_uint(__uint_as_float(v.z) - __uint_as_float(hi.z)) : 0u;
        hi.w = (m & 8u) ? (v.w & 0xFFFFE000u) : 0u; lo.w = (m & 8u) ? __float_as_uint(__uint_as_float(v.w) - __uint_as_float(hi.w)) : 0u;
        *(uint4*)img = hi;
        *(uint4*)(img + 8192) = lo;
      }
      if (m) {   // few lanes hold nonzeros in the sparse regime: one divergent region per row
        const int rr = row_lo + j;
        // auxiliary per-nonzero word: position in the tcgen05 branch's A tile (bf16 slices: value and position)
        if (m & 1u) { co[q] = (uint16_t)k; va[q] = __uint_as_float(v.x); if (aux) { if (BF16) rk[q] = xb_tc16_pack(rr, k, v.x); else ri[q] = xb_tc_pack(rr, k); } ++q; }
        if (m & 2u) { co[q] = (uint16_t)(k + 1); va[q] = __uint_as_float(v.y); if (aux) { if (BF16) rk[q] = xb_tc16_pack(rr, k + 1, v.y); else ri[q] = xb_tc_pack(rr, k + 1); } ++q; }
        if (m & 4u) { co[q] = (uint16_t)(k + 2); va[q] = __uint_as_float(v.z); if (aux) { if (BF16) rk[q] = xb_tc16_pack(rr, k + 2, v.z); else ri[q] = xb_tc_pack(rr, k + 2); } ++q; }
        if (m & 8u) { co[q] = (uint16_t)(k + 3); va[q] = __uint_as_float(v.w); if (aux) { if (BF16) rk[q] = xb_tc16_pack(rr, k + 3, v.w); else ri[q] = xb_tc_pack(rr, k + 3); } }
      }
      pos += __popc(b0) + 2 * __popc(b1) + 4 * __popc(b2);
    }
  }
}

// -------------------------------------------------------------------------------------------------
// K1x: bf16, transa = 'N', complete 128-column blocks with 16-byte aligned rows.  A lane holds SIXTEEN consecutive elements
// (two 16-byte loads), so a row is a quarter of a warp and one iteration of the positioning phase covers four rows; the keep
// test runs on the packed bf16 pairs with carry arithmetic (no widening, no per-element compare).  Same two phases and the same
// outputs as the generic kernel, bit for bit, at about a third of its instructions (it is instruction-issue bound).  Measured on
// C2: one 16-byte word per lane 25.1 us, two 23.2 us, four 23.1 us.
// -------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t k1w_mask8(uint4 w)
{
  // per 16-bit half h (sign dropped): kept iff 1 <= h <= 0x7F80, i.e. nonzero and not NaN (ordered compare of the
  // reference's vector loops: src/libxsmm_spmdm_begin_avx2.h:54); denormals and Inf kept, -0.0 dropped.
  // Carry arithmetic leaves the verdict of the low / high half in bit 15 / 31 of k; the eight verdict bits are then
  // collected in column order with two byte permutes and a multiply (bit 7 of four bytes -> one nibble).
  const uint32_t v[4] = { w.x, w.y, w.z, w.w };
  uint32_t k[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const uint32_t t = v[i] & 0x7FFF7FFFu;
    const uint32_t nz = t + 0x7FFF7FFFu;          // bit 15 / 31 set iff the half is nonzero
    const uint32_t nan = t + 0x007F007Fu;         // bit 15 / 31 set iff the half is > 0x7F80
    k[i] = nz & ~nan;
  }
  const uint32_t r01 = __byte_perm(k[0], k[1], 0x7531);   // bytes holding bit 15 and 31 of k0, k1: elements 0..3
  const uint32_t r23 = __byte_perm(k[2], k[3], 0x7531);   // elements 4..7
  const uint32_t lo = (((r01 >> 7) & 0x01010101u) * 0x01020408u) >> 24;
  const uint32_t hi = (((r23 >> 7) & 0x01010101u) * 0x01020408u) >> 24;
  return lo | (hi << 4);
}

// CW < 32: one CTA of CW warps walks the 32 / CW parts of its slice one after the other (the running total is the next part's
// base), so that two 16-warp CTAs fit an SM and one's loads overlap the other's arithmetic.
//
// Sparse regime (at most 32 candidate lanes in a warp's rows, i.e. up to about 2 % density): a lane whose 16 elements are all
// +-0 keeps nothing, and at 1 % density that is 85 % of the lanes.  One cheap test per lane (any half with a magnitude bit set)
// and one ballot per iteration list the candidate lanes; in (iteration, lane) order they are exactly the output order.  The
// candidates' 32 bytes are compacted through the warp's stage, lane t runs the exact keep test on candidate t, and a warp scan of
// the counts gives every output index and every row pointer.  Denser warps take the per-lane path (warp-uniform branch).
template <int ROWS, int CW>
__global__ void __launch_bounds__(CW * 32, (32 == CW) ? 1 : 2) spmdm_slice_bf16x_kernel(const SliceArgs p)
{
  constexpr int NW = 2;                      // 16-byte words per lane
  constexpr int SEQ = 32 / CW;               // parts of the slice walked by the CTA in turn
  constexpr int LPR = 16 / NW;               // lanes per row
  constexpr int RPI = 32 / LPR;              // rows per iteration
  constexpr int ITS = (ROWS + RPI - 1) / RPI;
  __shared__ uint32_t wtot[CW];
  constexpr int SCAP = 64;                   // records per warp of the per-lane path: all 16 rows of a warp at once up to 3 % density
  constexpr int CCAP = 128;                  // records per warp of the compacted path (the candidates' words take the same 1 KiB first)
  __shared__ uint4 stage_mem[CW][2 * 32];    // per warp: 32 candidates x 32 bytes, then the records of its outputs (stage and spread)
  __shared__ uint32_t csrc_mem[CW][32];      // per warp: where candidate t came from, as record bits: lane << 4 | iteration << 9
  // programmatic dependent launch (launch_slices): the slices this kernel overwrites may still be read by the multiply in front of
  // it in the stream -- wait for it before anything else; the multiply behind it may be scheduled from now on (it waits in turn)
  pdl_wait();
  pdl_trigger();
  const Geom& g = p.g;
  const int s = p.slice0 + (int)blockIdx.x * p.slice_step;
  const int kb = s / g.mb, mbi = s - kb * g.mb;
  const int nrows = min(g.bm, g.m - mbi * g.bm);
  const int tid = (int)threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int qr = lane / LPR, hl = lane % LPR;       // row inside the group, segment of the row
  const int rpw = (g.bm + K1N_WARPS - 1) / K1N_WARPS;
  const uint32_t lt = (1u << lane) - 1u;
  uint2* stg = (uint2*)stage_mem[warp];
  uint32_t seq_base = 0;                     // kept elements of the parts already done
#pragma unroll 1
  for (int pass = 0; pass < SEQ; ++pass) {
  const int row_lo = (pass * CW + warp) * rpw, row_hi = min(nrows, row_lo + rpw);
  const long long origin = p.origin_is_block ? 0ll : ((long long)mbi * g.bm * p.lda + (long long)kb * g.bk);
  const uint16_t* A = (const uint16_t*)p.a + origin + hl * (8 * NW);

  // ---- phase 1: load, test, count ---------------------------------------------------------------------
  uint4 w[ITS][NW];
#pragma unroll
  for (int it = 0; it < ITS; ++it) {
    const int r = row_lo + RPI * it + qr;
    const uint4* src = (const uint4*)(A + (long long)r * p.lda);
#pragma unroll
    for (int j = 0; j < NW; ++j) w[it][j] = (r < row_hi) ? __ldg(src + j) : make_uint4(0, 0, 0, 0);
  }
  // candidate lanes: some half has a magnitude bit set.  The others hold only +-0, which the keep rule drops.
  uint32_t cb[ITS], cb0[ITS], ncand = 0;
#pragma unroll
  for (int it = 0; it < ITS; ++it) {
    uint32_t o = 0;
#pragma unroll
    for (int j = 0; j < NW; ++j) o |= w[it][j].x | w[it][j].y | w[it][j].z | w[it][j].w;
    cb[it] = __ballot_sync(0xffffffffu, 0 != (o & 0x7FFF7FFFu));
    cb0[it] = ncand;
    ncand += __popc(cb[it]);
  }
  const bool compact = ncand <= 32u;         // warp-uniform
  uint32_t masks[ITS];
  // compacted: lane t's candidate: its keep mask, origin, first output in the warp, and its words in w[0] (the two paths share
  // the registers that stay live across the scan)
  uint32_t cm = 0, csrc = 0, cex = 0;
  uint4 (&cw)[NW] = w[0];
  // ... and for the warp's row i = RPI * it + qr held by lane i: the index of its first candidate, or ncand when none follows
  uint32_t rci = 0;
  uint32_t mine = 0;
  if (compact) {
    const int itr = lane / RPI;
    const uint32_t above = (1u << (LPR * (lane % RPI))) - 1u;      // the lanes of the rows above it in its group
#pragma unroll
    for (int it = 0; it < ITS; ++it) rci += __popc(cb[it] & ((it < itr) ? 0xFFFFFFFFu : ((it == itr) ? above : 0u)));
#pragma unroll
    for (int it = 0; it < ITS; ++it) {
      if ((cb[it] >> lane) & 1u) {
        const uint32_t t = cb0[it] + __popc(cb[it] & lt);
#pragma unroll
        for (int j = 0; j < NW; ++j) stage_mem[warp][NW * t + j] = w[it][j];
        csrc_mem[warp][t] = ((uint32_t)lane << 4) | ((uint32_t)it << 9);
      }
    }
    __syncwarp();
#pragma unroll
    for (int j = 0; j < NW; ++j) cw[j] = make_uint4(0, 0, 0, 0);
    if ((uint32_t)lane < ncand) {
#pragma unroll
      for (int j = 0; j < NW; ++j) { cw[j] = stage_mem[warp][NW * lane + j]; cm |= k1w_mask8(cw[j]) << (8 * j); }
      csrc = csrc_mem[warp][lane];
    }
    const uint32_t cnt = __popc(cm);
    uint32_t inc = cnt;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const uint32_t u = __shfl_up_sync(0xffffffffu, inc, d);
      if (lane >= d) inc += u;
    }
    cex = inc - cnt;                         // lanes past the candidates: the warp's total
    mine = __shfl_sync(0xffffffffu, inc, 31);
  }
  else {
#pragma unroll
    for (int it = 0; it < ITS; ++it) {
      uint32_t m = 0;
#pragma unroll
      for (int j = 0; j < NW; ++j) m |= k1w_mask8(w[it][j]) << (8 * j);
      masks[it] = m;
      mine += __popc(m);
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) mine += __shfl_xor_sync(0xffffffffu, mine, d);
  }
  const uint32_t warp_total = mine;
  if (0 == pass && 0 == tid && p.write_sp && p.out.tcsp) p.out.slice_ovf[s] = 0;   // counted below, after the scan's barrier
  const K1Scan sc = k1_scan<CW>(mine, wtot, seq_base);
  seq_base = sc.slice_total;
  uint32_t pos = sc.pos;
  if (SEQ - 1 == pass && 0 == tid) {
    p.out.rowidx[(size_t)s * (g.bm + 1) + nrows] = (uint16_t)sc.slice_total;   // u16 like the reference's counter
    p.out.slice_nnz[s] = sc.slice_total;
    xb_publish_nnz(p, sc.slice_total);
  }

  // ---- phase 2: positions and stores -----------------------------------------------------------------------
  uint16_t* ro = p.out.rowidx + (size_t)s * (g.bm + 1);
  uint16_t* co = p.out.colidx + (size_t)s * g.bm * g.bk;
  float* va = p.out.values + (size_t)s * g.bm * g.bk;
  uint32_t* rk = p.out.tcpk + (size_t)s * g.bm * g.bk;
  const bool aux = (0 != p.write_aux);
  // word per nonzero for the structured-sparse tensor-core kernel: a lane's 16 elements are exactly the four groups of four
  // whose nibbles make one 16-bit metadata word of the row, so everything is known to the lane (common.cuh: xb_sp_*)
  const bool spw = (0 != p.write_sp) && (0 != p.out.tcsp);
  uint32_t* sp = p.out.tcsp + (size_t)s * g.bm * g.bk;
  auto spread = [&](const uint2 rec, const uint32_t q) {      // everything one output costs, by whichever lane gets it
    const uint32_t vb = rec.x & 0xFFFF0000u, ms = rec.x & 0xFFFFu, e16 = rec.y & 15u, sl = (rec.y >> 4) & 31u, its = rec.y >> 9;
    const uint32_t rs = (uint32_t)row_lo + (uint32_t)RPI * its + sl / LPR, hs = sl % LPR, rowm = rs & 127u, k = hs * 16u + e16;
    co[q] = (uint16_t)k;
    va[q] = __uint_as_float(vb);
    if (aux) rk[q] = xb_tc16_pack((int)rs, (int)k, vb);
    if (spw) {
      uint32_t meta16 = 0;
#pragma unroll
      for (int gi = 0; gi < 4; ++gi) meta16 |= xb_sp_nibble((ms >> (4 * gi)) & 15u) << (16 + 4 * gi);
      const uint32_t gi = e16 >> 2, slot = xb_sp_slot((ms >> (4u * gi)) & 15u, e16 & 3u);
      sp[q] = meta16 | ((slot & 2u) << 14) | xb_sp_pos(rowm, hs * 8u + 2u * gi + (slot & 1u));
      if (slot & 2u) {     // rare: third / fourth nonzero of its group of four.  Counted per slice; the first kSpOvfCap are listed
        const uint32_t idx = atomicAdd(p.out.slice_ovf + s, 1u);
        if (idx < (uint32_t)kSpOvfCap) p.out.ovf_list[(size_t)s * kSpOvfCap + idx] = make_uint2(rs | (k << 16), vb);
      }
    }
  };
  if (compact) {
    // row pointers: lane i takes the warp's row i, whose first output is that of its first candidate (or the warp's total when
    // no candidate follows it)
    const uint32_t off = __shfl_sync(0xffffffffu, cex, rci & 31u);
    if (lane < ROWS && row_lo + lane < row_hi) ro[row_lo + lane] = (uint16_t)(pos + (rci < 32u ? off : warp_total));
    // stage and spread: lane t drops its candidate's kept elements as 8-byte records {value | the lane's 16-bit mask,
    // element | lane << 4 | iteration << 9} at their output index, then lane t does all the work for output t
    for (uint32_t c0 = 0; c0 < warp_total; c0 += (uint32_t)CCAP) {      // one round below ~6 % density
      if (cm) {
        uint32_t i = cex - c0;                  // unsigned: outputs before this round wrap around
        for (uint32_t mm = cm; mm; mm &= mm - 1u, ++i) {
          if (i < (uint32_t)CCAP) {
            const int e = __ffs((int)mm) - 1;
            const uint4 v = (e & 8) ? cw[NW - 1] : cw[0];
            const uint32_t pr = (e & 4) ? ((e & 2) ? v.w : v.z) : ((e & 2) ? v.y : v.x);
            const uint32_t vb = (e & 1) ? (pr & 0xFFFF0000u) : (pr << 16);
            stg[i] = make_uint2(vb | cm, (uint32_t)e | csrc);
          }
        }
      }
      __syncwarp();
      const uint32_t nc = min((uint32_t)CCAP, warp_total - c0);
      for (uint32_t t = (uint32_t)lane; t < nc; t += 32u) spread(stg[t], pos + c0 + t);
      __syncwarp();                             // the stage is rewritten by the next round
    }
  }
  else {
  const uint32_t before = (1u << (LPR * qr)) - 1u;             // the lanes of the rows above it in the group
  uint32_t wdone = 0;                      // outputs of this warp's earlier iterations
  const uint32_t pos0 = pos;               // first output of this warp
#pragma unroll
  for (int it = 0; it < ITS; ++it) {
    if (row_lo + RPI * it < row_hi) {      // warp-uniform
      const uint32_t m = masks[it];
      const uint32_t nm = __popc(m);       // 0 .. 8 * NW
      const uint32_t b0 = __ballot_sync(0xffffffffu, nm & 1u), b1 = __ballot_sync(0xffffffffu, nm & 2u);
      // a lane keeping four or more of its elements is rare in the sparse regime: the upper count bits are voted on
      // only then (warp-uniform branch)
      const bool big = 0 != __any_sync(0xffffffffu, nm >= 4u);
      uint32_t b2 = 0, b3 = 0, b4 = 0, b5 = 0;
      if (big) {
        b2 = __ballot_sync(0xffffffffu, nm & 4u); b3 = __ballot_sync(0xffffffffu, nm & 8u);
        b4 = __ballot_sync(0xffffffffu, nm & 16u); b5 = __ballot_sync(0xffffffffu, nm & 32u);
      }
      auto kept = [&](uint32_t lanes) -> uint32_t {     // kept elements held by the given lanes
        uint32_t c = __popc(b0 & lanes) + 2 * __popc(b1 & lanes);
        if (big) c += 4 * __popc(b2 & lanes) + 8 * __popc(b3 & lanes) + 16 * __popc(b4 & lanes) + 32 * __popc(b5 & lanes);
        return c;
      };
      const uint32_t rowpos = pos + kept(before);
      const int r = row_lo + RPI * it + qr;
      if (0 == hl && r < row_hi) ro[r] = (uint16_t)rowpos;
      // Stage and spread as in the compacted path, one iteration at a time, without the compaction.  When the warp's 16 rows
      // hold at most SCAP nonzeros (always below 3 % density) all four iterations are staged first and spread in one pass after
      // the loop.
      const uint32_t tot = kept(0xFFFFFFFFu);
      if (tot) {                                        // warp-uniform
        const uint32_t ex = kept(lt);                   // this lane's first output of the iteration (lane order = (row, column) order)
        const bool all_at_once = warp_total <= (uint32_t)SCAP;
        for (uint32_t c0 = 0; c0 < tot; c0 += 32u) {    // one chunk below ~6 % density
          if (m) {
            uint32_t i = all_at_once ? (wdone + ex) : (ex - c0);
#pragma unroll
            for (int j = 0; j < NW; ++j) {
              const uint32_t v[4] = { w[it][j].x, w[it][j].y, w[it][j].z, w[it][j].w };
              for (uint32_t mm = (m >> (8 * j)) & 0xFFu; mm; mm &= mm - 1u, ++i) {
                if (all_at_once || i < 32u) {           // unsigned: outputs before this chunk wrap around
                  const int e = __ffs((int)mm) - 1;
                  const uint32_t pr = (e & 4) ? ((e & 2) ? v[3] : v[2]) : ((e & 2) ? v[1] : v[0]);
                  const uint32_t vb = (e & 1) ? (pr & 0xFFFF0000u) : (pr << 16);
                  stg[i] = make_uint2(vb | m, (uint32_t)(8 * j + e) | ((uint32_t)lane << 4) | ((uint32_t)it << 9));
                }
              }
            }
          }
          if (all_at_once) break;
          __syncwarp();
          if (c0 + (uint32_t)lane < tot) spread(stg[lane], pos + c0 + (uint32_t)lane);
          __syncwarp();                                 // the stage is rewritten by the next chunk / iteration
        }
      }
      pos += tot; wdone += tot;
    }
  }
  if (warp_total <= (uint32_t)SCAP && warp_total > 0) {     // all iterations staged: one spread pass
    __syncwarp();
    for (uint32_t c0 = 0; c0 < warp_total; c0 += 32u)
      if (c0 + (uint32_t)lane < warp_total) spread(stg[c0 + lane], pos0 + c0 + (uint32_t)lane);
  }
  }
  if (SEQ > 1) __syncthreads();             // wtot and the stages are reused by the next part
  }
}

// K1x takes a slicing pass over bf16 A (transa = 'N') whose blocks are all complete 128-column blocks inside the reference's
// vector loops and whose rows are 16-byte aligned.  It is the only slicing kernel that writes SliceArena::tcsp.
static bool k1x_takes(const SliceArgs& a)
{
  return !a.transa && a.is_bf16 && !a.origin_is_block && 0 == (a.g.k % 128) && a.simd_w > 1 && 0 == (a.lda & 7) && 0 == ((uintptr_t)a.a & 15);
}

bool slices_get_sp_words(const SliceArgs& args)
{
  return k1x_takes(args) && 0 != args.write_sp && 0 != args.out.tcsp;
}

template <bool BF16, int ROWS>
static void launch_slice_n(const SliceArgs& args, int nslices, bool full, cudaStream_t stream)
{
  if (full) XB_CUDA(launch_pdl(spmdm_slice_n_kernel<BF16, true, ROWS>, dim3((unsigned)nslices), dim3(K1N_THREADS), 0, stream, args));
  else XB_CUDA(launch_pdl(spmdm_slice_n_kernel<BF16, false, ROWS>, dim3((unsigned)nslices), dim3(K1N_THREADS), 0, stream, args));
}

void launch_slices(const SliceArgs& args, int nslices, cudaStream_t stream)
{
  if (nslices <= 0) return;
  if (!args.transa) {
    count_launch(1);
    const int rpw = (args.g.bm + K1N_WARPS - 1) / K1N_WARPS;
    if (k1x_takes(args)) {
      // 512-row slices: one 16-warp CTA that does the two halves of its slice one after the other, two such CTAs per SM (all
      // 256 slices of a 4096^2 matrix resident at once instead of 1.73 waves of 32-warp CTAs): 1.1 us less per C2 step
      if (rpw <= 8) XB_CUDA(launch_pdl(spmdm_slice_bf16x_kernel<8, 32>, dim3((unsigned)nslices), dim3(K1N_THREADS), 0, stream, args));
      else XB_CUDA(launch_pdl(spmdm_slice_bf16x_kernel<16, 16>, dim3((unsigned)nslices), dim3(512), 0, stream, args));
    }
    else {
      // FULL: every slice is a complete 128-column block inside the reference's vector loops (k % 128 == 0
      // makes the NaN rule of the scalar remainder unreachable)
      const bool full = (0 == (args.g.k % 128)) && (args.simd_w > 1);
      if (args.is_bf16) {
        if (rpw <= 8) launch_slice_n<true, 8>(args, nslices, full, stream);
        else launch_slice_n<true, 16>(args, nslices, full, stream);
      }
      else {
        if (rpw <= 8) launch_slice_n<false, 8>(args, nslices, full, stream);
        else launch_slice_n<false, 16>(args, nslices, full, stream);
      }
    }
    XB_CUDA(cudaGetLastError());
    return;
  }
  const int nstrips = (args.g.bm + K1_R - 1) / K1_R;   // <= 8 because bm <= 512
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)nstrips, (unsigned)nslices, 1);
  cfg.blockDim = dim3(K1_THREADS, 1, 1);
  cfg.dynamicSmemBytes = 0;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = (unsigned)nstrips;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  count_launch(1);
  XB_CUDA(cudaLaunchKernelEx(&cfg, spmdm_slice_kernel, args));
}

// -------------------------------------------------------------------------------------------------
// K1c: A given in CSR form (transa = 'N') -> the same slices as K1n / K1x write for the dense matrix holding these entries.
// One CTA per slice, one thread per row of it.  With sorted columns the slice's entries of a row are one contiguous range of
// col_idx, found by two binary searches; the CTA then walks the concatenation of its rows' ranges ("candidates", already in
// output order) 512 at a time, one candidate per thread, and a block scan of the keep verdicts gives each kept entry its
// output index.  Row pointers come from per-row kept counts.  Malformed input (row_ptr not monotone or past nnz, columns
// unsorted, duplicated or >= K) gives unspecified slices but stays inside the arrays: every row range is clamped to
// [0, nnz] and to at most ncols candidates, and a candidate is kept only if its column lies in the slice.
// -------------------------------------------------------------------------------------------------
constexpr int K1C_THREADS = 512;      // >= bm: one row per thread
constexpr int K1C_WARPS = K1C_THREADS / 32;

// first index in [lo, hi) whose column is >= c (hi if none); on unsorted columns some index in [lo, hi]
__device__ __forceinline__ uint32_t k1c_lower_bound(const unsigned int* col, uint32_t lo, uint32_t hi, uint32_t c)
{
  while (lo < hi) {
    const uint32_t mid = lo + ((hi - lo) >> 1);
    if (__ldg(col + mid) < c) lo = mid + 1; else hi = mid;
  }
  return lo;
}

// block-wide exclusive scan of one value per thread; returns the thread's prefix, *total the sum.  wtot: K1C_WARPS words.
__device__ __forceinline__ uint32_t k1c_scan(uint32_t v, uint32_t* wtot, uint32_t* total)
{
  const int tid = (int)threadIdx.x, warp = tid >> 5, lane = tid & 31;
  uint32_t inc = v;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const uint32_t u = __shfl_up_sync(0xffffffffu, inc, d);
    if (lane >= d) inc += u;
  }
  __syncthreads();                       // wtot may still be read by the previous scan
  if (31 == lane) wtot[warp] = inc;
  __syncthreads();
  uint32_t base = 0, sum = 0;
#pragma unroll
  for (int w = 0; w < K1C_WARPS; ++w) { const uint32_t t = wtot[w]; base += (w < warp) ? t : 0u; sum += t; }
  *total = sum;
  return base + inc - v;
}

template <bool BF16>
__device__ __forceinline__ uint32_t k1c_bits(const void* values, uint32_t j)
{
  if (BF16) return (uint32_t)__ldg((const uint16_t*)values + j) << 16;
  return __float_as_uint(__ldg((const float*)values + j));
}

template <bool BF16>
__global__ void __launch_bounds__(K1C_THREADS, 2) spmdm_slice_csr_kernel(const SliceArgs p, const CsrArgs a)
{
  __shared__ uint32_t cbeg[K1C_THREADS];       // first candidate of the row in col_idx
  __shared__ uint32_t coff[K1C_THREADS + 1];   // exclusive scan of the rows' candidate counts
  __shared__ uint32_t kcnt[K1C_THREADS];       // kept entries of the row
  __shared__ uint32_t wtot[K1C_WARPS];
  pdl_wait();          // launch_pdl: the slices may still be read by the multiply in front of this kernel in the stream
  pdl_trigger();       // ... and the multiply behind it may be scheduled (it waits in turn)
  const Geom& g = p.g;
  const int s = (int)blockIdx.x;
  const int kb = s / g.mb, mbi = s - kb * g.mb;
  const int nrows = min(g.bm, g.m - mbi * g.bm);
  const int ncols = min(g.bk, g.k - kb * g.bk);
  int vec_end = BF16 ? (ncols / (4 * p.simd_w)) * (4 * p.simd_w) : (ncols / p.simd_w) * p.simd_w;
  if (p.simd_w <= 1) vec_end = 0;
  const uint32_t c0 = (uint32_t)kb * (uint32_t)g.bk, c1 = c0 + (uint32_t)ncols;
  const int tid = (int)threadIdx.x, lane = tid & 31;
  const bool spw = BF16 && (0 != p.write_sp) && (0 != p.out.tcsp) && 0 == (g.k % 128) && p.simd_w > 1;
  if (spw && 0 == tid) p.out.slice_ovf[s] = 0;     // counted below, after the first barrier

  // ---- the row's candidate range --------------------------------------------------------------------------
  uint32_t n = 0;
  if (tid < nrows) {
    const int gr = mbi * g.bm + tid;
    const uint32_t lo = min(__ldg(a.row_ptr + gr), a.nnz);
    const uint32_t hi = max(lo, min(__ldg(a.row_ptr + gr + 1), a.nnz));
    const uint32_t b = k1c_lower_bound(a.col_idx, lo, hi, c0);
    const uint32_t e = k1c_lower_bound(a.col_idx, b, (hi - b > (uint32_t)ncols) ? b + (uint32_t)ncols : hi, c1);
    cbeg[tid] = b;
    n = e - b;
  }
  kcnt[tid] = 0;
  uint32_t ncand;
  coff[tid] = k1c_scan(n, wtot, &ncand);
  if (0 == tid) coff[K1C_THREADS] = ncand;
  __syncthreads();

  // ---- walk the candidates in output order ------------------------------------------------------------------
  uint16_t* co = p.out.colidx + (size_t)s * g.bm * g.bk;
  float* va = p.out.values + (size_t)s * g.bm * g.bk;
  uint16_t* ri = p.out.tcoff + (size_t)s * g.bm * g.bk;
  uint32_t* rk = p.out.tcpk + (size_t)s * g.bm * g.bk;
  uint32_t* sp = p.out.tcsp + (size_t)s * g.bm * g.bk;
  const bool aux = (0 != p.write_aux);
  uint32_t base = 0;
  for (uint32_t i0 = 0; i0 < ncand; i0 += K1C_THREADS) {      // block-uniform
    const uint32_t i = i0 + (uint32_t)tid;
    bool keep = false;
    int r = 0;
    uint32_t j = 0, k = 0, vb = 0;
    if (i < ncand) {
      int lo = 0, hi = nrows - 1;                  // last row whose first candidate is <= i (it owns i: empty rows are skipped)
      while (lo < hi) { const int mid = (lo + hi + 1) >> 1; if (coff[mid] <= i) lo = mid; else hi = mid - 1; }
      r = lo;
      j = cbeg[r] + (i - coff[r]);
      const uint32_t col = __ldg(a.col_idx + j);
      vb = k1c_bits<BF16>(a.values, j);
      k = col - c0;
      keep = (col >= c0) && (col < c1) && k1_keep(__uint_as_float(vb), (int)k, vec_end);
    }
    uint32_t nkept;
    const uint32_t q = base + k1c_scan(keep ? 1u : 0u, wtot, &nkept);
    base += nkept;
    // per-row kept counts: one shared-memory add per row and warp
    const unsigned same = __match_any_sync(0xffffffffu, keep ? r : -1);
    const unsigned kept_lanes = __ballot_sync(0xffffffffu, keep) & same;
    if (keep && lane == __ffs((int)kept_lanes) - 1) atomicAdd(&kcnt[r], (uint32_t)__popc(kept_lanes));
    if (keep) {
      co[q] = (uint16_t)k;
      va[q] = __uint_as_float(vb);
      if (aux) { if (BF16) rk[q] = xb_tc16_pack(r, (int)k, vb); else ri[q] = xb_tc_pack(r, (int)k); }
      if (BF16 && spw) {
        // the kept-mask of the row's 16-k span holding k (K1x: one lane's 16 elements), from the entry's neighbours in the row
        const uint32_t span = k & ~15u, rb = cbeg[r], re = cbeg[r] + (coff[r + 1] - coff[r]);
        uint32_t ms = 1u << (k & 15u);
        for (uint32_t t = j; t > rb; --t) {
          const uint32_t cn = __ldg(a.col_idx + t - 1);
          if (cn < c0 + span || cn >= c0 + span + 16u) break;
          if (k1_keep(__uint_as_float(k1c_bits<BF16>(a.values, t - 1)), 0, vec_end)) ms |= 1u << ((cn - c0) & 15u);
        }
        for (uint32_t t = j + 1; t < re; ++t) {
          const uint32_t cn = __ldg(a.col_idx + t);
          if (cn < c0 + span || cn >= c0 + span + 16u) break;
          if (k1_keep(__uint_as_float(k1c_bits<BF16>(a.values, t)), 0, vec_end)) ms |= 1u << ((cn - c0) & 15u);
        }
        const uint32_t e16 = k & 15u, hs = k >> 4, rowm = (uint32_t)r & 127u;
        uint32_t meta16 = 0;
#pragma unroll
        for (int gi = 0; gi < 4; ++gi) meta16 |= xb_sp_nibble((ms >> (4 * gi)) & 15u) << (16 + 4 * gi);
        const uint32_t gi = e16 >> 2, slot = xb_sp_slot((ms >> (4u * gi)) & 15u, e16 & 3u);
        sp[q] = meta16 | ((slot & 2u) << 14) | xb_sp_pos(rowm, hs * 8u + 2u * gi + (slot & 1u));
        if (slot & 2u) {     // third / fourth nonzero of its group of four: counted per slice, the first kSpOvfCap listed
          const uint32_t idx = atomicAdd(p.out.slice_ovf + s, 1u);
          if (idx < (uint32_t)kSpOvfCap) p.out.ovf_list[(size_t)s * kSpOvfCap + idx] = make_uint2((uint32_t)r | (k << 16), vb);
        }
      }
    }
  }

  // ---- row pointers (u16 like the reference's counter), the slice's count, density feedback -------------------------
  __syncthreads();
  uint32_t total;
  const uint32_t rp = k1c_scan(tid < nrows ? kcnt[tid] : 0u, wtot, &total);
  uint16_t* ro = p.out.rowidx + (size_t)s * (g.bm + 1);
  if (tid < nrows) ro[tid] = (uint16_t)rp;
  if (0 == tid) {
    ro[nrows] = (uint16_t)total;
    p.out.slice_nnz[s] = total;
    xb_publish_nnz(p, total);
  }
}

// -------------------------------------------------------------------------------------------------
// K1t: A given in CSC form (col_ptr[k + 1], row_idx[nnz]; also the CSR arrays of A stored k x m) -> the same slices as the dense
// slicer writes for transa = 'T' on the k x m array holding these entries, and as K1c writes for the CSR arrays of A.  One CTA
// of K1c's shape per slice.  A column lists its rows in ascending order, a slice lists each row's columns in ascending order; the
// transpose goes through a shared bitmask of the slice's kept entries (bm x 128 bits) instead of a sort or scratch memory:
//   1. thread t < ncols finds column c0 + t's entries in the slice's rows (two binary searches, at most nrows candidates); a
//      block scan lays the columns' ranges end to end;
//   2. the CTA walks the candidates 512 at a time, tests each and sets its bit in its row's mask (shared atomicOr);
//   3. thread r scans the popcount of row r's mask into the row pointers;
//   4. a second walk writes every kept entry (r, k) at rowstart[r] + the kept bits of row r below k.
// Placement depends only on the mask: the output is deterministic, and for any input an entry's index is below its row's end,
// at most bm * bk.  Malformed input (col_ptr not monotone or past nnz, rows unsorted, duplicated or >= M) gives unspecified
// slices but stays inside the arrays: column ranges are clamped to [0, nnz] and to nrows candidates, a candidate is kept only if
// its row lies in the slice, and the duplicates of an entry set one bit and write one slot.
// -------------------------------------------------------------------------------------------------
template <bool BF16>
__global__ void __launch_bounds__(K1C_THREADS, 2) spmdm_slice_csc_kernel(const SliceArgs p, const CscArgs a)
{
  __shared__ __align__(16) uint32_t kmask[K1C_THREADS][4];   // kept columns of each row of the slice
  __shared__ uint32_t rstart[K1C_THREADS];                   // first output of each row
  __shared__ uint32_t cbeg[128];                             // first candidate of the column in row_idx
  __shared__ uint32_t coff[128];                             // exclusive scan of the columns' candidate counts
  __shared__ uint32_t wtot[K1C_WARPS];
  pdl_wait();          // launch_pdl: the slices may still be read by the multiply in front of this kernel in the stream
  pdl_trigger();       // ... and the multiply behind it may be scheduled (it waits in turn)
  const Geom& g = p.g;
  const int s = (int)blockIdx.x;
  const int kb = s / g.mb, mbi = s - kb * g.mb;
  const int nrows = min(g.bm, g.m - mbi * g.bm);
  const int ncols = min(g.bk, g.k - kb * g.bk);
  int vec_end = BF16 ? (ncols / (4 * p.simd_w)) * (4 * p.simd_w) : (ncols / p.simd_w) * p.simd_w;
  if (p.simd_w <= 1) vec_end = 0;
  const uint32_t c0 = (uint32_t)kb * (uint32_t)g.bk;
  const uint32_t r0 = (uint32_t)mbi * (uint32_t)g.bm, r1 = r0 + (uint32_t)nrows;
  const int tid = (int)threadIdx.x;
  const bool spw = BF16 && (0 != p.write_sp) && (0 != p.out.tcsp) && 0 == (g.k % 128) && p.simd_w > 1;
  if (spw && 0 == tid) p.out.slice_ovf[s] = 0;     // counted in step 4, after the first barrier

  // ---- 1. the column's candidate range ------------------------------------------------------------------------
  uint32_t n = 0;
  if (tid < ncols) {
    const uint32_t gc = c0 + (uint32_t)tid;
    const uint32_t lo = min(__ldg(a.col_ptr + gc), a.nnz);
    const uint32_t hi = max(lo, min(__ldg(a.col_ptr + gc + 1), a.nnz));
    const uint32_t b = k1c_lower_bound(a.row_idx, lo, hi, r0);
    const uint32_t e = k1c_lower_bound(a.row_idx, b, (hi - b > (uint32_t)nrows) ? b + (uint32_t)nrows : hi, r1);
    cbeg[tid] = b;
    n = e - b;
  }
  *(uint4*)kmask[tid] = make_uint4(0, 0, 0, 0);
  uint32_t ncand;
  const uint32_t off = k1c_scan(n, wtot, &ncand);
  if (tid < ncols) coff[tid] = off;
  __syncthreads();

  // the candidate i < ncand: its column (the last one whose first candidate is <= i: empty columns are skipped), row and value
  auto candidate = [&](uint32_t i, int* c, uint32_t* r, uint32_t* vb) {
    int lo = 0, hi = ncols - 1;
    while (lo < hi) { const int mid = (lo + hi + 1) >> 1; if (coff[mid] <= i) lo = mid; else hi = mid - 1; }
    const uint32_t j = cbeg[lo] + (i - coff[lo]);
    *c = lo;
    *r = __ldg(a.row_idx + j) - r0;              // rows outside the slice wrap to >= nrows
    *vb = k1c_bits<BF16>(a.values, j);
    return *r < (uint32_t)nrows && k1_keep(__uint_as_float(*vb), lo, vec_end);
  };

  // ---- 2. the kept-mask of every row -----------------------------------------------------------------------------
  for (uint32_t i = (uint32_t)tid; i < ncand; i += K1C_THREADS) {
    int c;
    uint32_t r, vb;
    if (candidate(i, &c, &r, &vb)) atomicOr(&kmask[r][c >> 5], 1u << (c & 31));
  }
  __syncthreads();

  // ---- 3. row pointers (u16 like the reference's counter), the slice's count, density feedback -------------------------
  uint32_t cnt = 0;
  if (tid < nrows) { const uint4 m = *(const uint4*)kmask[tid]; cnt = __popc(m.x) + __popc(m.y) + __popc(m.z) + __popc(m.w); }
  uint32_t total;
  const uint32_t rp = k1c_scan(cnt, wtot, &total);
  rstart[tid] = rp;
  uint16_t* ro = p.out.rowidx + (size_t)s * (g.bm + 1);
  if (tid < nrows) ro[tid] = (uint16_t)rp;
  if (0 == tid) {
    ro[nrows] = (uint16_t)total;
    p.out.slice_nnz[s] = total;
    xb_publish_nnz(p, total);
  }
  __syncthreads();

  // ---- 4. place the kept entries -----------------------------------------------------------------------------------
  uint16_t* co = p.out.colidx + (size_t)s * g.bm * g.bk;
  float* va = p.out.values + (size_t)s * g.bm * g.bk;
  uint16_t* ri = p.out.tcoff + (size_t)s * g.bm * g.bk;
  uint32_t* rk = p.out.tcpk + (size_t)s * g.bm * g.bk;
  uint32_t* sp = p.out.tcsp + (size_t)s * g.bm * g.bk;
  const bool aux = (0 != p.write_aux);
  for (uint32_t i = (uint32_t)tid; i < ncand; i += K1C_THREADS) {
    int c;
    uint32_t r, vb;
    if (!candidate(i, &c, &r, &vb)) continue;
    const uint4 m = *(const uint4*)kmask[r];
    const uint32_t k = (uint32_t)c, w = k >> 5, mw = (w & 2) ? ((w & 1) ? m.w : m.z) : ((w & 1) ? m.y : m.x);
    const uint32_t q = rstart[r] + __popc(mw & ((1u << (k & 31u)) - 1u))
                     + (w > 0 ? __popc(m.x) : 0u) + (w > 1 ? __popc(m.y) : 0u) + (w > 2 ? __popc(m.z) : 0u);
    co[q] = (uint16_t)k;
    va[q] = __uint_as_float(vb);
    if (aux) { if (BF16) rk[q] = xb_tc16_pack((int)r, (int)k, vb); else ri[q] = xb_tc_pack((int)r, (int)k); }
    if (BF16 && spw) {
      const uint32_t ms = (mw >> (k & 16u)) & 0xFFFFu;      // the kept-mask of the row's 16-k span holding k (K1x: one lane's 16 elements)
      const uint32_t e16 = k & 15u, hs = k >> 4, rowm = r & 127u;
      uint32_t meta16 = 0;
#pragma unroll
      for (int gi = 0; gi < 4; ++gi) meta16 |= xb_sp_nibble((ms >> (4 * gi)) & 15u) << (16 + 4 * gi);
      const uint32_t gi = e16 >> 2, slot = xb_sp_slot((ms >> (4u * gi)) & 15u, e16 & 3u);
      sp[q] = meta16 | ((slot & 2u) << 14) | xb_sp_pos(rowm, hs * 8u + 2u * gi + (slot & 1u));
      if (slot & 2u) {     // third / fourth nonzero of its group of four: counted per slice, the first kSpOvfCap listed
        const uint32_t idx = atomicAdd(p.out.slice_ovf + s, 1u);
        if (idx < (uint32_t)kSpOvfCap) p.out.ovf_list[(size_t)s * kSpOvfCap + idx] = make_uint2(r | (k << 16), vb);
      }
    }
  }
}

// K1c and K1t write tcsp under K1x's geometric condition: complete 128-column blocks inside the reference's vector loops
bool slices_sparse_get_sp_words(const SliceArgs& args)
{
  return args.is_bf16 && 0 == (args.g.k % 128) && args.simd_w > 1 && 0 != args.write_sp && 0 != args.out.tcsp;
}

void launch_slices_csr(const SliceArgs& args, const CsrArgs& csr, cudaStream_t stream)
{
  const int nslices = args.g.mb * args.g.kb;
  if (nslices <= 0) return;
  count_launch(1);
  if (args.is_bf16) XB_CUDA(launch_pdl(spmdm_slice_csr_kernel<true>, dim3((unsigned)nslices), dim3(K1C_THREADS), 0, stream, args, csr));
  else XB_CUDA(launch_pdl(spmdm_slice_csr_kernel<false>, dim3((unsigned)nslices), dim3(K1C_THREADS), 0, stream, args, csr));
}

void launch_slices_csc(const SliceArgs& args, const CscArgs& csc, cudaStream_t stream)
{
  const int nslices = args.g.mb * args.g.kb;
  if (nslices <= 0) return;
  count_launch(1);
  if (args.is_bf16) XB_CUDA(launch_pdl(spmdm_slice_csc_kernel<true>, dim3((unsigned)nslices), dim3(K1C_THREADS), 0, stream, args, csc));
  else XB_CUDA(launch_pdl(spmdm_slice_csc_kernel<false>, dim3((unsigned)nslices), dim3(K1C_THREADS), 0, stream, args, csc));
}

// =================================================================================================
// K2: sliced SpMM.
// CTA = 16 warps x RPW rows of one row block (mb) x BN = 32*VEC columns.  Per k-block the
// 128 x BN panel of B is staged in shared memory (double buffered, cp.async 16-byte copies;
// transposed on the fly for transb='T'; bf16 kept as bf16 and widened in registers).  A warp
// owns RPW consecutive rows -- their nonzeros are contiguous in the slice, so the warp fetches
// them with coalesced 32-wide loads and broadcasts (column, value) by shuffle -- and a lane owns
// VEC consecutive columns: one 16-byte shared-memory read and VEC fused multiply-adds per nonzero.
// Per output element this is the reference's rounding sequence: start from beta*C, one fma per
// nonzero in ascending (kb, column) order (compute template :309-370).  PARTIAL = true is the
// variant for the columns of the narrow last block that the reference accumulates per k-block
// from zero and then adds (:372-434).
// =================================================================================================
constexpr int K2_THREADS = 512;
constexpr int K2_WARPS = K2_THREADS / 32;

template <bool BF16> struct K2Elem { typedef float type; };
template <> struct K2Elem<true> { typedef uint16_t type; };

__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gsrc)
{
  const uint32_t d = (uint32_t)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(d), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::: "memory"); }
template <int N> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N) : "memory"); }

template <bool BF16, int VEC>
__device__ __forceinline__ void k2_fma_row(float (&acc)[VEC], const unsigned char* brow, float val)
{
  if (!BF16) {
    const float4 b = *(const float4*)brow;
    acc[0] = fmaf(val, b.x, acc[0]); acc[1] = fmaf(val, b.y, acc[1]);
    acc[2] = fmaf(val, b.z, acc[2]); acc[3] = fmaf(val, b.w, acc[3]);
  }
  else {
    const uint4 b = *(const uint4*)brow;
    const uint32_t w[4] = { b.x, b.y, b.z, b.w };
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      acc[2 * e] = fmaf(val, __uint_as_float(w[e] << 16), acc[2 * e]);
      acc[2 * e + 1] = fmaf(val, __uint_as_float(w[e] & 0xFFFF0000u), acc[2 * e + 1]);
    }
  }
}

template <bool BF16, bool PARTIAL, int RPW>
__global__ void __launch_bounds__(K2_THREADS, 1) spmdm_compute_kernel(const ComputeArgs p)
{
  typedef typename K2Elem<BF16>::type elem_t;
  constexpr int VEC = BF16 ? 8 : 4;
  constexpr int BN = 32 * VEC;
  constexpr int TM = K2_WARPS * RPW;
  constexpr int ROWB = BN * (int)sizeof(elem_t);   // 512 bytes per tile row
  constexpr int TILEB = 128 * ROWB;                // 64 KiB per stage
  constexpr int CPITCH = BN + 1;
  extern __shared__ __align__(128) unsigned char smem[];

  const Geom& g = p.g;
  if (p.tc_twin > 0 && xb_total_nnz(p.sl.slice_nnz, g.mb * g.kb) >= p.tc_min_nnz) return;   // the tensor-core twin does this multiply
  const int tid = (int)threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int tiles_per_mb = (g.bm + TM - 1) / TM;
  const int mbi = p.mb_first + (int)blockIdx.y / tiles_per_mb;
  const int ml0 = ((int)blockIdx.y % tiles_per_mb) * TM;       // first block-local row of the CTA
  const int rows_in_block = min(g.bm, g.m - mbi * g.bm);
  if (ml0 >= rows_in_block) return;
  const int tile_rows = min(TM, rows_in_block - ml0);
  const int n0 = (int)blockIdx.x * BN;                        // local column of the CTA
  const int mycol = n0 + lane * VEC;
  const int wrow0 = ml0 + warp * RPW;                         // block-local first row of the warp
  const int nvalid = max(0, min(RPW, rows_in_block - wrow0));
  const int crow0 = mbi * g.bm + ml0 - p.row_origin;          // local C row of the CTA's first row
  const size_t cap = (size_t)g.bm * g.bk;

  float acc[RPW][VEC];
  float run[PARTIAL ? RPW : 1][PARTIAL ? VEC : 1];
  (void)run;

  // ---- start value: 0, C or beta*C (reference compute template :81-212) --------------------------
  const bool cvec = (0 == (p.ldc & 3)) && (0 == ((uintptr_t)p.c & 15));
  if (0.f == p.beta) {
#pragma unroll
    for (int i = 0; i < RPW; ++i)
#pragma unroll
      for (int e = 0; e < VEC; ++e) acc[i][e] = 0.f;
  }
  else {
    if (p.transc) {  // C stored n x m: stage the tile through shared memory for coalesced reads
      float* Cs = (float*)smem;
      for (int idx = tid; idx < BN * TM; idx += K2_THREADS) {
        const int n = idx / TM, r = idx - n * TM;
        float v = 0.f;
        if (r < tile_rows && n0 + n < p.ncols) v = p.c[(size_t)(n0 + n) * p.ldc + crow0 + r];
        Cs[r * CPITCH + n] = v;
      }
      __syncthreads();
#pragma unroll
      for (int i = 0; i < RPW; ++i)
#pragma unroll
        for (int e = 0; e < VEC; ++e) acc[i][e] = Cs[(warp * RPW + i) * CPITCH + lane * VEC + e];
      __syncthreads();
    }
    else {
#pragma unroll
      for (int i = 0; i < RPW; ++i) {
        const float* src = p.c + (size_t)(crow0 + warp * RPW + i) * p.ldc + mycol;
        if (i < nvalid && cvec && mycol + VEC <= p.ncols) {
#pragma unroll
          for (int q = 0; q < VEC / 4; ++q) {
            const float4 v = *(const float4*)(src + 4 * q);
            acc[i][4 * q] = v.x; acc[i][4 * q + 1] = v.y; acc[i][4 * q + 2] = v.z; acc[i][4 * q + 3] = v.w;
          }
        }
        else {
#pragma unroll
          for (int e = 0; e < VEC; ++e) acc[i][e] = (i < nvalid && mycol + e < p.ncols) ? src[e] : 0.f;
        }
      }
    }
    if (1.f != p.beta) {
#pragma unroll
      for (int i = 0; i < RPW; ++i)
#pragma unroll
        for (int e = 0; e < VEC; ++e) acc[i][e] = p.beta * acc[i][e];
    }
  }
  if (PARTIAL) {
#pragma unroll
    for (int i = 0; i < RPW; ++i)
#pragma unroll
      for (int e = 0; e < VEC; ++e) { run[i][e] = acc[i][e]; acc[i][e] = 0.f; }
  }

  // ---- B panel loader -----------------------------------------------------------------------------
  const elem_t* Bg = (const elem_t*)p.b;
  constexpr int EPC = 16 / (int)sizeof(elem_t);   // elements per 16-byte chunk
  const bool bvec = (0 == (p.ldb % EPC)) && (0 == ((uintptr_t)p.b & 15));
  auto fill = [&](int kb, unsigned char* dst) {
    const int k0 = kb * g.bk;
    const int numk = min(g.bk, g.k - k0);
    if (!p.transb) {   // B stored k x n: a tile row is 32 chunks of 16 bytes
      for (int idx = tid; idx < numk * 32; idx += K2_THREADS) {
        const int kk = idx >> 5, ch = idx & 31;
        const int nl = n0 + ch * EPC;
        const elem_t* src = Bg + (size_t)(k0 + kk) * p.ldb + nl;
        elem_t* d = (elem_t*)(dst + kk * ROWB) + ch * EPC;
        if (bvec && nl + EPC <= p.ncols) cp_async16(d, src);
        else {
#pragma unroll
          for (int e = 0; e < EPC; ++e) d[e] = (nl + e < p.ncols) ? src[e] : (elem_t)0;
        }
      }
    }
    else {             // B stored n x k: a thread walks k for one column, 16 bytes at a time
      constexpr int CPT = K2_THREADS / BN;         // k-chunks in flight per pass
      const int n = tid % BN, c0 = tid / BN;
      const bool in = (n0 + n < p.ncols);
      const elem_t* srow = Bg + (size_t)(n0 + n) * p.ldb + k0;
      for (int ch = c0; ch * EPC < numk; ch += CPT) {
        const int kk = ch * EPC;
        __align__(16) elem_t v[EPC];
        if (in && bvec && kk + EPC <= numk && 0 == (k0 % EPC)) {
          const uint4 raw = *(const uint4*)(srow + kk);
          *(uint4*)v = raw;
        }
        else {
#pragma unroll
          for (int e = 0; e < EPC; ++e) v[e] = (in && kk + e < numk) ? srow[kk + e] : (elem_t)0;
        }
#pragma unroll
        for (int e = 0; e < EPC; ++e) if (kk + e < numk) ((elem_t*)(dst + (kk + e) * ROWB))[n] = v[e];
      }
    }
  };

  // ---- main loop over k blocks ----------------------------------------------------------------------
  fill(0, smem);
  cp_async_commit();
  for (int kb = 0; kb < g.kb; ++kb) {
    unsigned char* cur = smem + (kb & 1) * TILEB;
    if (kb + 1 < g.kb) fill(kb + 1, smem + ((kb + 1) & 1) * TILEB);
    cp_async_commit();
    cp_async_wait<1>();
    __syncthreads();

    if (nvalid > 0) {
      const int s = kb * g.mb + mbi;
      const uint16_t* ro = p.sl.rowidx + (size_t)s * (g.bm + 1) + wrow0;
      const uint16_t* cp = p.sl.colidx + s * cap;
      const float* vp = p.sl.values + s * cap;
      int myrp = 0;
      if (lane <= RPW) myrp = (int)ro[min(lane, nvalid)];
      int rs[RPW + 1];
#pragma unroll
      for (int i = 0; i <= RPW; ++i) rs[i] = __shfl_sync(0xffffffffu, myrp, i);
#pragma unroll
      for (int i = 1; i <= RPW; ++i) rs[i] = max(rs[i], rs[i - 1]);   // wrapped u16 pointer: empty row (tpl.c:292-297)
      const int pend = rs[RPW];
      const unsigned char* bbase = cur + lane * 16;
      for (int p0 = rs[0]; p0 < pend; p0 += 32) {
        const int q = p0 + lane;
        uint32_t off_l = 0; float val_l = 0.f;
        if (q < pend) { off_l = (uint32_t)cp[q] * ROWB; val_l = vp[q]; }
#pragma unroll
        for (int i = 0; i < RPW; ++i) {
          const int lo = max(rs[i], p0) - p0, hi = min(rs[i + 1], p0 + 32) - p0;
          for (int t = lo; t < hi; ++t) {
            const uint32_t off = __shfl_sync(0xffffffffu, off_l, t);
            const float val = __shfl_sync(0xffffffffu, val_l, t);
            k2_fma_row<BF16, VEC>(acc[i], bbase + off, val);
          }
        }
      }
      if (PARTIAL) {
#pragma unroll
        for (int i = 0; i < RPW; ++i)
#pragma unroll
          for (int e = 0; e < VEC; ++e) { run[i][e] = acc[i][e] + run[i][e]; acc[i][e] = 0.f; }
      }
    }
    __syncthreads();
  }
  cp_async_wait<0>();
  if (PARTIAL) {
#pragma unroll
    for (int i = 0; i < RPW; ++i)
#pragma unroll
      for (int e = 0; e < VEC; ++e) acc[i][e] = run[i][e];
  }

  // ---- write C --------------------------------------------------------------------------------------
  if (p.transc) {
    float* Cs = (float*)smem;
#pragma unroll
    for (int i = 0; i < RPW; ++i)
#pragma unroll
      for (int e = 0; e < VEC; ++e) Cs[(warp * RPW + i) * CPITCH + lane * VEC + e] = acc[i][e];
    __syncthreads();
    for (int idx = tid; idx < BN * TM; idx += K2_THREADS) {
      const int n = idx / TM, r = idx - n * TM;
      if (r < tile_rows && n0 + n < p.ncols) p.c[(size_t)(n0 + n) * p.ldc + crow0 + r] = Cs[r * CPITCH + n];
    }
  }
  else {
#pragma unroll
    for (int i = 0; i < RPW; ++i) {
      if (i < nvalid) {
        float* dst = p.c + (size_t)(crow0 + warp * RPW + i) * p.ldc + mycol;
        if (cvec && mycol + VEC <= p.ncols) {
#pragma unroll
          for (int q = 0; q < VEC / 4; ++q)
            *(float4*)(dst + 4 * q) = make_float4(acc[i][4 * q], acc[i][4 * q + 1], acc[i][4 * q + 2], acc[i][4 * q + 3]);
        }
        else {
#pragma unroll
          for (int e = 0; e < VEC; ++e) if (mycol + e < p.ncols) dst[e] = acc[i][e];
        }
      }
    }
  }
}

template <bool BF16, bool PARTIAL, int RPW>
static void launch_compute_variant(const ComputeArgs& a, cudaStream_t stream)
{
  constexpr int VEC = BF16 ? 8 : 4;
  constexpr int BN = 32 * VEC;
  constexpr int TM = K2_WARPS * RPW;
  const size_t tiles = 2 * 128 * (size_t)BN * (BF16 ? 2 : 4);
  const size_t cstage = (size_t)TM * (BN + 1) * 4;
  const size_t smem = tiles > cstage ? tiles : cstage;
  auto kern = spmdm_compute_kernel<BF16, PARTIAL, RPW>;
  ensure_smem_optin((const void*)kern, (int)smem);
  const int tiles_per_mb = (a.g.bm + TM - 1) / TM;
  const dim3 grid((unsigned)((a.ncols + BN - 1) / BN), (unsigned)(a.mb_count * tiles_per_mb), 1);
  count_launch(1);
  if (!PARTIAL) note_compute_kernel("spmdm_compute_kernel");
  kern<<<grid, K2_THREADS, smem, stream>>>(a);
  XB_CUDA(cudaGetLastError());
}

// Splits the column range into the reference's accumulation modes and launches each part:
//   [0, n_full_end)          full-width blocks: in-order fma chain
//   [n_full_end, tail_from)  narrow block, vector part: per-kb partial sums
//   [tail_from, N)           narrow block, scalar part: in-order fma chain (GCC contracts += b*v)
// The narrow last block forks onto a side stream.  The stream and the two events of the fork / join are created once per
// (host thread, device): a process may drive several devices, callers may run concurrently, and nothing is created or
// destroyed on the hot path (which also keeps the pattern legal under stream capture).
struct SideCtx { cudaStream_t stream; cudaEvent_t fork, join; };
static SideCtx* side_ctx()
{
  static thread_local std::map<int, SideCtx*> per_device;
  int dev = 0;
  if (cudaSuccess != cudaGetDevice(&dev)) { (void)cudaGetLastError(); return 0; }
  SideCtx*& c = per_device[dev];
  if (0 == c) {
    c = new SideCtx();
    c->stream = 0; c->fork = 0; c->join = 0;
    XB_CUDA(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
    XB_CUDA(cudaEventCreateWithFlags(&c->fork, cudaEventDisableTiming));
    XB_CUDA(cudaEventCreateWithFlags(&c->join, cudaEventDisableTiming));
  }
  return (c->stream && c->fork && c->join) ? c : 0;
}

// LIBXSMM_B200_SPMDM_TC: "0" never use the tensor-core branch, "1" always (when the panel qualifies),
// unset / anything else: by density -- total nnz >= tc_density_threshold() of M*K (common.cuh), decided on the device.
static int tc_mode()
{
  const char* e = getenv("LIBXSMM_B200_SPMDM_TC");
  if (0 == e || 0 == *e) return 2;
  return ('0' == *e) ? 0 : (('1' == *e) ? 1 : 2);
}

// bf16 tensor-core branch: the 2:4 structured-sparse kernel (K4s) when it qualifies, else the CTA-pair kernel (K4p)
static bool launch_tc_bf16(const ComputeArgs& a, cudaStream_t stream)
{
  if (launch_compute_tc16s(a, stream)) {                 // 2:4 structured-sparse form (low density, slices from the wide kernel)
    const char* fe = getenv("LIBXSMM_B200_TC16_SPARSE");
    if (a.sp_guard && !(fe && '1' == *fe)) {             // the estimate is fresh or has just moved: the dense kernel stands by (ComputeArgs::sp_guard)
      ComputeArgs g2 = a;
      g2.sp_guard = 2;
      if (launch_compute_tc16p(g2, stream)) note_compute_kernel("guarded: spmdm_compute_tc16s_kernel | spmdm_compute_tc16p_kernel (selected on the device by nnz)");
    }
    return true;
  }
  return launch_compute_tc16p(a, stream);
}

// fp32 tensor-core branch: the CTA-pair kernel (K4q) when the slices carry their dense image, else the single-CTA kernel (K4)
static bool launch_tc_f32(const ComputeArgs& a, cudaStream_t stream)
{
  return launch_compute_tcq(a, stream) || launch_compute_tc(a, stream);
}

static void launch_part(const ComputeArgs& a, bool partial, cudaStream_t stream)
{
  if (!partial && launch_compute_sp(a, stream)) return;  // K2s: TMA ring, list-driven row walk (spmdm_compute_sp.cu)
  if (launch_compute_tma(a, partial, stream)) return;   // K2: the narrow-block parts and what K2s refuses (spmdm_compute_tma.cu)
  if (a.is_bf16) {
    if (partial) launch_compute_variant<true, true, 4>(a, stream);
    else launch_compute_variant<true, false, 8>(a, stream);
  }
  else {
    if (partial) launch_compute_variant<false, true, 4>(a, stream);
    else launch_compute_variant<false, false, 8>(a, stream);
  }
}

void launch_compute(const ComputeArgs& args, cudaStream_t stream)
{
  if (args.ncols <= 0 || args.mb_count <= 0) return;
  // Tensor-core twin (fp32, N/N/N, aligned panels): the dense kernel is enqueued next to the sparse ones and
  // every CTA of both reads the slices' nonzero counts; only the selected side does the work.
  ComputeArgs targs = args;
  int mode = (0 == args.tc_twin) ? tc_mode() : 0;
  if (2 == mode && 1 == args.tc_hint) mode = 0;      // clearly sparse last time: do not even enqueue the dense twin
  targs.tc_twin = 0;
  if (2 == mode && 2 == args.tc_hint) {              // clearly dense last time: the tensor-core kernel alone (correct for any density)
    if (args.is_bf16 ? launch_tc_bf16(targs, stream) : launch_tc_f32(targs, stream)) return;
  }
  if (mode > 0) {
    targs.tc_twin = 1;
    targs.tc_min_nnz = (1 == mode) ? 0ull : (unsigned long long)(tc_density_threshold(0 != args.is_bf16, 0 != args.transb, 0 != args.transc) * (double)args.g.m * (double)args.g.k);
    if (!(args.is_bf16 ? launch_tc_bf16(targs, stream) : launch_tc_f32(targs, stream))) targs.tc_twin = 0;
    else if (1 == mode) return;   // forced: nothing for the sparse kernels to do
  }
  const ComputeArgs& args2 = targs;
  const int c_lo = args.col_origin, c_hi = args.col_origin + args.ncols;
  const int cut[4] = { c_lo, min(max(args.modes.n_full_end, c_lo), c_hi), min(max(args.modes.tail_from, c_lo), c_hi), c_hi };
  // the narrow last block (at most bn - 1 columns, two small launches) runs on a side stream, forked from
  // and joined back into `stream`, so that it overlaps the main launch instead of serialising behind it
  SideCtx* sc = ((cut[3] > cut[1]) && (cut[1] > cut[0])) ? side_ctx() : 0;
  const bool narrow = 0 != sc;
  cudaStream_t side = stream;
  if (narrow) {
    side = sc->stream;
    XB_CUDA(cudaEventRecord(sc->fork, stream));
    XB_CUDA(cudaStreamWaitEvent(side, sc->fork, 0));
  }
  for (int part = 2; part >= 0; --part) {
    const int lo = cut[part], hi = cut[part + 1];
    if (hi <= lo) continue;
    ComputeArgs a = args2;
    const size_t esz = args.is_bf16 ? 2 : 4;
    const long long shift = lo - c_lo;
    a.b = (const char*)args.b + (args.transb ? (size_t)shift * args.ldb * esz : (size_t)shift * esz);
    a.c = args.c + (args.transc ? (size_t)shift * args.ldc : (size_t)shift);
    a.col_origin = lo;
    a.ncols = hi - lo;
    launch_part(a, 1 == part, (0 == part) ? stream : side);
  }
  if (args2.tc_twin > 0) note_compute_kernel(args.is_bf16 ? "twin: spmdm_compute_tc16p_kernel | spmdm_compute_tma_kernel (selected on the device by nnz)"
                                                          : "twin: spmdm_compute_tc_kernel | spmdm_compute_tma_kernel (selected on the device by nnz)");
  if (narrow) {
    XB_CUDA(cudaEventRecord(sc->join, side));
    XB_CUDA(cudaStreamWaitEvent(stream, sc->join, 0));
  }
}

}  // namespace xb
