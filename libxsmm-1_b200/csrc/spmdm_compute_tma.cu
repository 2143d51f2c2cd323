// K2 fast path: sliced SpMM with the B panel staged by TMA (sm_100a).
//
//   C[tile rows, tile cols] = beta*C + sum_kb slice(kb, mb)[tile rows, :] * B[kb*128 .. +128, tile cols]
//
// CTA = CW warps.  One elected lane (warp 0) also acts as producer: it streams the 128 x BN tiles of B
// (k-block after k-block) into a STAGES-deep shared-memory ring with cp.async.bulk.tensor (TMA; rows past K
// and columns past N are zero-filled by the hardware, so there is no bounds code on the load path) and
// signals each stage through an mbarrier; consumer warps release a stage through a second mbarrier, so
// the warps of a CTA are never synchronised as a block and drift freely over the ring.
// A consumer warp owns R consecutive rows of the row block and 32*VEC columns (a lane owns VEC consecutive
// columns: one 16-byte -- or 8-byte -- shared-memory read and VEC fused multiply-adds per nonzero).  The
// rows' nonzeros are contiguous in the slice; row pointers are fetched two k-blocks ahead and the first 32
// nonzeros one k-block ahead, so that global-memory latency is off the critical path in the sparse regime.
// Per output element the rounding sequence is the reference's: start from beta*C, one fma per nonzero in
// ascending (kb, column) order (reference src/template/libxsmm_spmdm_compute_fp32_thread.tpl.c:309-370).
// Only full-width reference blocks, transb = transc = 'N' and 16-byte aligned panels come here; everything
// else stays on the generic kernel in spmdm_kernels.cu.
#include "common.cuh"
#include "ptx.cuh"
#include <mutex>

namespace xb {

template <bool BF16, int VEC> struct BVec;
template <> struct BVec<false, 4> {
  static __device__ __forceinline__ void fma(float (&acc)[4], const unsigned char* brow, float val)
  {
    const float4 b = *(const float4*)brow;
    acc[0] = fmaf(val, b.x, acc[0]); acc[1] = fmaf(val, b.y, acc[1]);
    acc[2] = fmaf(val, b.z, acc[2]); acc[3] = fmaf(val, b.w, acc[3]);
  }
};
template <> struct BVec<false, 2> {
  static __device__ __forceinline__ void fma(float (&acc)[2], const unsigned char* brow, float val)
  {
    const float2 b = *(const float2*)brow;
    acc[0] = fmaf(val, b.x, acc[0]); acc[1] = fmaf(val, b.y, acc[1]);
  }
};
template <> struct BVec<true, 8> {
  static __device__ __forceinline__ void fma(float (&acc)[8], const unsigned char* brow, float val)
  {
    const uint4 b = *(const uint4*)brow;
    const uint32_t w[4] = { b.x, b.y, b.z, b.w };
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      acc[2 * e] = fmaf(val, __uint_as_float(w[e] << 16), acc[2 * e]);
      acc[2 * e + 1] = fmaf(val, __uint_as_float(w[e] & 0xFFFF0000u), acc[2 * e + 1]);
    }
  }
};
template <> struct BVec<true, 4> {
  static __device__ __forceinline__ void fma(float (&acc)[4], const unsigned char* brow, float val)
  {
    const uint2 b = *(const uint2*)brow;
    acc[0] = fmaf(val, __uint_as_float(b.x << 16), acc[0]);
    acc[1] = fmaf(val, __uint_as_float(b.x & 0xFFFF0000u), acc[1]);
    acc[2] = fmaf(val, __uint_as_float(b.y << 16), acc[2]);
    acc[3] = fmaf(val, __uint_as_float(b.y & 0xFFFF0000u), acc[3]);
  }
};

// row pointers of R+1 consecutive rows live in lanes 0..R; a wrapped u16 pointer (reference quirk: the
// counter of a completely full slice wraps, template :72) must read as "empty row": running maximum.
template <int R>
__device__ __forceinline__ int rp_monotone(int rp, int lane)
{
  const int nxt = __shfl_down_sync(0xffffffffu, rp, 1);
  if (__any_sync(0xffffffffu, lane < R && nxt < rp)) {
#pragma unroll
    for (int d = 1; d <= R; d <<= 1) {
      const int t = __shfl_up_sync(0xffffffffu, rp, d);
      if (lane >= d) rp = max(rp, t);
    }
  }
  return rp;
}

template <bool BF16, int VEC, int R, int CW, int STAGES, bool PARTIAL>
__global__ void __launch_bounds__(CW * 32, 1)
spmdm_compute_tma_kernel(const __grid_constant__ CUtensorMap tmB, const ComputeArgs p)
{
  constexpr int ESZ = BF16 ? 2 : 4;
  constexpr int BN = 32 * VEC;
  constexpr int TM = CW * R;
  constexpr int ROWB = BN * ESZ;
  constexpr int STAGEB = 128 * ROWB;
  constexpr int LANEB = VEC * ESZ;
  extern __shared__ __align__(128) unsigned char smem[];
  uint64_t* full = (uint64_t*)(smem + (size_t)STAGES * STAGEB);
  uint64_t* empty = full + STAGES;

  const Geom& g = p.g;
  if (p.tc_twin > 0 && xb_total_nnz(p.sl.slice_nnz, g.mb * g.kb) >= p.tc_min_nnz) return;   // the tensor-core twin does this multiply
  const int tid = (int)threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int tiles_per_mb = (g.bm + TM - 1) / TM;
  const int mbi = p.mb_first + (int)blockIdx.y / tiles_per_mb;
  const int ml0 = ((int)blockIdx.y % tiles_per_mb) * TM;
  const int rows_in_block = min(g.bm, g.m - mbi * g.bm);
  if (ml0 >= rows_in_block) return;
  const int n0 = (int)blockIdx.x * BN;

  if (0 == tid) {
#pragma unroll
    for (int s = 0; s < STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], CW); }
    mbar_fence_init();
  }
  __syncthreads();

  // ---------------- producer role: lane 0 of warp 0, interleaved with its consumer work ----------------
  // tile t goes to stage t % STAGES; refilling a stage waits until every warp has released its previous
  // contents (empty barrier, one arrival per warp)
  const bool is_producer = (0 == tid);
  auto produce = [&](int t) {
    if (t < g.kb) {
      const int s = t % STAGES, f = t / STAGES;
      if (f > 0) mbar_wait(&empty[s], (f - 1) & 1);
      mbar_arrive_expect_tx(&full[s], STAGEB);
      tma_load_2d(smem + (size_t)s * STAGEB, &tmB, n0, t * g.bk, &full[s]);
    }
  };
  if (is_producer) {
    tma_prefetch_desc(&tmB);
    for (int t = 0; t < STAGES - 1; ++t) produce(t);
  }

  // ---------------- consumers ----------------
  const int mycol = n0 + lane * VEC;
  const int wrow0 = ml0 + warp * R;
  const int nvalid = max(0, min(R, rows_in_block - wrow0));
  const size_t crow0 = (size_t)(mbi * g.bm + wrow0 - p.row_origin);
  const size_t cap = (size_t)g.bm * g.bk;
  const bool colfull = (VEC >= 4) && (mycol + VEC <= p.ncols);   // 16-byte vector path

  float acc[R][VEC];
  if (0.f == p.beta) {
#pragma unroll
    for (int i = 0; i < R; ++i)
#pragma unroll
      for (int e = 0; e < VEC; ++e) acc[i][e] = 0.f;
  }
  else {
#pragma unroll
    for (int i = 0; i < R; ++i) {
      const float* src = p.c + (crow0 + i) * p.ldc + mycol;
      if (i < nvalid && colfull) {
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
    if (1.f != p.beta) {
#pragma unroll
      for (int i = 0; i < R; ++i)
#pragma unroll
        for (int e = 0; e < VEC; ++e) acc[i][e] = p.beta * acc[i][e];
    }
  }

  // PARTIAL (narrow last block of the reference, vector part): per k-block a fresh sum, then one add
  // into the running value (compute template :372-434)
  float run[PARTIAL ? R : 1][PARTIAL ? VEC : 1];
  (void)run;
  if (PARTIAL) {
#pragma unroll
    for (int i = 0; i < R; ++i)
#pragma unroll
      for (int e = 0; e < VEC; ++e) { run[PARTIAL ? i : 0][PARTIAL ? e : 0] = acc[i][e]; acc[i][e] = 0.f; }
  }

  // slice s = kb*mb + mbi: the three pointers advance by one "kb" stride per iteration
  const size_t rp_stride = (size_t)g.mb * (g.bm + 1);
  const size_t nz_stride = (size_t)g.mb * cap;
  const bool rp_lane = (lane <= R) && (nvalid > 0);
  const uint16_t* rpp = p.sl.rowidx + (size_t)mbi * (g.bm + 1) + wrow0 + min(lane, nvalid);   // row pointers, k-block kb+2
  const uint16_t* cpn = p.sl.colidx + (size_t)mbi * cap + lane;                                // nonzeros, k-block kb+1
  const float* vpn = p.sl.values + (size_t)mbi * cap + lane;

  int rp_cur = rp_lane ? (int)__ldg(rpp) : 0;
  rpp += rp_stride;
  int rp_nxt = (rp_lane && 1 < g.kb) ? (int)__ldg(rpp) : 0;
  rpp += rp_stride;
  rp_cur = rp_monotone<R>(rp_cur, lane);
  uint32_t col_c = 0; float val_c = 0.f;     // lane q holds nonzero (first + q) of the warp's rows, current k-block
  {
    const int s0 = __shfl_sync(0xffffffffu, rp_cur, 0), e0 = __shfl_sync(0xffffffffu, rp_cur, R);
    if (s0 + lane < e0) { col_c = __ldg(cpn + s0); val_c = __ldg(vpn + s0); }
  }
  cpn += nz_stride; vpn += nz_stride;

  for (int kb = 0; kb < g.kb; ++kb) {
    if (is_producer) produce(kb + STAGES - 1);
    // ---- prefetch: row pointers of kb+2, first 32 nonzeros of kb+1 (consumed one iteration later) --------
    const int rp_nn = (rp_lane && kb + 2 < g.kb) ? (int)__ldg(rpp) : 0;
    rpp += rp_stride;
    rp_nxt = rp_monotone<R>(rp_nxt, lane);
    uint32_t col_n = 0; float val_n = 0.f;
    {
      const int s1 = __shfl_sync(0xffffffffu, rp_nxt, 0), e1 = __shfl_sync(0xffffffffu, rp_nxt, R);
      if (s1 + lane < e1) { col_n = __ldg(cpn + s1); val_n = __ldg(vpn + s1); }   // e1 == s1 == 0 past the last k-block
    }
    const int first = __shfl_sync(0xffffffffu, rp_cur, 0);
    const int total = __shfl_sync(0xffffffffu, rp_cur, R) - first;
    const int rel = rp_cur - first;            // lane i: offset of row i's first nonzero inside the warp's range
    // ---- wait for the B tile of this k-block ---------------------------------------------------------------
    const int s = kb % STAGES;
    mbar_wait(&full[s], (kb / STAGES) & 1);
    const unsigned char* bbase = smem + (size_t)s * STAGEB + lane * LANEB;
    uint32_t off_c = col_c * ROWB;

    if (total <= 32) {   // sparse regime: everything the warp needs is already in registers
      int lo = 0;
#pragma unroll
      for (int i = 0; i < R; ++i) {
        const int hi = __shfl_sync(0xffffffffu, rel, i + 1);
#pragma unroll 1
        for (int t = lo; t < hi; ++t) {
          const uint32_t off = __shfl_sync(0xffffffffu, off_c, t);
          const float val = __shfl_sync(0xffffffffu, val_c, t);
          BVec<BF16, VEC>::fma(acc[i], bbase + off, val);
        }
        lo = hi;
      }
    }
    else {               // denser rows: walk the range in chunks of 32 nonzeros, later chunks fetched in line
      const uint16_t* cpk = cpn - nz_stride + first;   // this k-block (cpn points at kb+1, lane included)
      const float* vpk = vpn - nz_stride + first;
      for (int p0 = 0; p0 < total; p0 += 32) {
        if (0 != p0) {
          off_c = 0; val_c = 0.f;
          if (p0 + lane < total) { off_c = (uint32_t)__ldg(cpk + p0) * ROWB; val_c = __ldg(vpk + p0); }
        }
#pragma unroll
        for (int i = 0; i < R; ++i) {
          const int lo = max(__shfl_sync(0xffffffffu, rel, i), p0) - p0;
          const int hi = min(__shfl_sync(0xffffffffu, rel, i + 1), p0 + 32) - p0;
          for (int t = lo; t < hi; ++t) {
            const uint32_t off = __shfl_sync(0xffffffffu, off_c, t);
            const float val = __shfl_sync(0xffffffffu, val_c, t);
            BVec<BF16, VEC>::fma(acc[i], bbase + off, val);
          }
        }
      }
    }
    __syncwarp();
    if (0 == lane) mbar_arrive(&empty[s]);
    if (PARTIAL) {
#pragma unroll
      for (int i = 0; i < R; ++i)
#pragma unroll
        for (int e = 0; e < VEC; ++e) { run[PARTIAL ? i : 0][PARTIAL ? e : 0] = acc[i][e] + run[PARTIAL ? i : 0][PARTIAL ? e : 0]; acc[i][e] = 0.f; }
    }
    cpn += nz_stride; vpn += nz_stride;
    rp_cur = rp_nxt; rp_nxt = rp_nn; col_c = col_n; val_c = val_n;
  }
  if (PARTIAL) {
#pragma unroll
    for (int i = 0; i < R; ++i)
#pragma unroll
      for (int e = 0; e < VEC; ++e) acc[i][e] = run[PARTIAL ? i : 0][PARTIAL ? e : 0];
  }

  // ---- write C (each element exactly once: streaming stores) ---------------------------------------------
#pragma unroll
  for (int i = 0; i < R; ++i) {
    if (i < nvalid) {
      float* dst = p.c + (crow0 + i) * p.ldc + mycol;
      if (colfull) {
#pragma unroll
        for (int q = 0; q < VEC / 4; ++q)
          st_global_cs_f4(dst + 4 * q, make_float4(acc[i][4 * q], acc[i][4 * q + 1], acc[i][4 * q + 2], acc[i][4 * q + 3]));
      }
      else {
#pragma unroll
        for (int e = 0; e < VEC; ++e) if (mycol + e < p.ncols) dst[e] = acc[i][e];
      }
    }
  }
}

// ---- host side ---------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_tiled()
{
  static EncodeTiledFn fn = 0;
  static std::once_flag once;
  std::call_once(once, [] {
    void* f = 0;
    cudaDriverEntryPointQueryResult q;
    if (cudaSuccess == cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &q) && cudaDriverEntryPointSuccess == q) fn = (EncodeTiledFn)f;
    else (void)cudaGetLastError();
  });
  return fn;
}

bool make_tensor_map_2d(CUtensorMap* map, const void* base, int elem_bytes, unsigned long long cols, unsigned long long rows,
                        unsigned long long row_pitch_bytes, unsigned box_cols, unsigned box_rows)
{
  EncodeTiledFn fn = encode_tiled();
  if (0 == fn) return false;
  if (0 != ((uintptr_t)base & 15) || 0 != (row_pitch_bytes & 15) || box_cols > 256 || box_rows > 256) return false;
  const CUtensorMapDataType dt = (2 == elem_bytes) ? CU_TENSOR_MAP_DATA_TYPE_UINT16
                               : ((4 == elem_bytes) ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_FLOAT64);
  const cuuint64_t gdim[2] = { cols, rows };
  const cuuint64_t gstr[1] = { row_pitch_bytes };
  const cuuint32_t box[2] = { box_cols, box_rows };
  const cuuint32_t estr[2] = { 1, 1 };
  const CUresult r = fn(map, dt, 2, const_cast<void*>(base), gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                        CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return CUDA_SUCCESS == r;
}

bool make_tensor_map_2d_sw128(CUtensorMap* map, const void* base, int elem_bytes, unsigned long long cols, unsigned long long rows,
                              unsigned long long row_pitch_bytes, unsigned box_cols, unsigned box_rows, bool atom32)
{
  // atom32: 128-byte swizzle with 32-byte atoms (the only layout tcgen05 accepts for MN-major TF32 operands)
  EncodeTiledFn fn = encode_tiled();
  if (0 == fn) return false;
  if (0 != ((uintptr_t)base & 15) || 0 != (row_pitch_bytes & 15) || box_cols * elem_bytes != 128 || box_rows > 256) return false;
  const CUtensorMapDataType dt = (2 == elem_bytes) ? CU_TENSOR_MAP_DATA_TYPE_UINT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32;
  const cuuint64_t gdim[2] = { cols, rows };
  const cuuint64_t gstr[1] = { row_pitch_bytes };
  const cuuint32_t box[2] = { box_cols, box_rows };
  const cuuint32_t estr[2] = { 1, 1 };
  const CUresult r = fn(map, dt, 2, const_cast<void*>(base), gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                        atom32 ? CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B : CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return CUDA_SUCCESS == r;
}

// one-byte elements (FP8 operands), boxes of box_cols = swizzle_bytes (64 or 128) columns
bool make_tensor_map_2d_u8(CUtensorMap* map, const void* base, unsigned long long cols, unsigned long long rows,
                           unsigned long long row_pitch_bytes, unsigned box_cols, unsigned box_rows, int swizzle_bytes)
{
  EncodeTiledFn fn = encode_tiled();
  if (0 == fn) return false;
  if (0 != ((uintptr_t)base & 15) || 0 != (row_pitch_bytes & 15) || (int)box_cols != swizzle_bytes || box_rows > 256 ||
      (64 != swizzle_bytes && 128 != swizzle_bytes)) return false;
  const cuuint64_t gdim[2] = { cols, rows };
  const cuuint64_t gstr[1] = { row_pitch_bytes };
  const cuuint32_t box[2] = { box_cols, box_rows };
  const cuuint32_t estr[2] = { 1, 1 };
  const CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, const_cast<void*>(base), gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                        128 == swizzle_bytes ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return CUDA_SUCCESS == r;
}

template <bool BF16, int VEC, int R, int CW, int STAGES, bool PARTIAL>
static bool launch_tma_variant(const ComputeArgs& a, cudaStream_t stream)
{
  constexpr int ESZ = BF16 ? 2 : 4;
  constexpr int BN = 32 * VEC;
  constexpr int TM = CW * R;
  constexpr size_t smem = (size_t)STAGES * 128 * BN * ESZ + 2 * STAGES * sizeof(uint64_t);
  CUtensorMap map;
  if (!make_tensor_map_2d(&map, a.b, ESZ, (unsigned long long)a.ncols, (unsigned long long)a.g.k,
                          (unsigned long long)a.ldb * ESZ, BN, 128)) return false;
  auto kern = spmdm_compute_tma_kernel<BF16, VEC, R, CW, STAGES, PARTIAL>;
  ensure_smem_optin((const void*)kern, (int)smem);
  const int tiles_per_mb = (a.g.bm + TM - 1) / TM;
  const dim3 grid((unsigned)((a.ncols + BN - 1) / BN), (unsigned)(a.mb_count * tiles_per_mb), 1);
  count_launch(1);
  if (!PARTIAL) note_compute_kernel("spmdm_compute_tma_kernel");
  kern<<<grid, CW * 32, smem, stream>>>(map, a);
  XB_CUDA(cudaGetLastError());
  return true;
}

// returns false when the panel does not qualify (caller then uses the generic kernel).
// partial = the reference's narrow-block vector columns (per-k-block partial sums).
bool launch_compute_tma(const ComputeArgs& a, bool partial, cudaStream_t stream)
{
  if (a.transb || a.transc) return false;
  if (0 != ((uintptr_t)a.c & 15) || 0 != (a.ldc & 3)) return false;
  if (partial) {   // at most bn - 1 columns: one narrow column tile, many short row tiles
    return a.is_bf16 ? launch_tma_variant<true, 4, 4, 8, 4, true>(a, stream) : launch_tma_variant<false, 2, 4, 8, 4, true>(a, stream);
  }
  if (a.ncols <= 32) {   // scalar tail of the narrow block: in-order chain, few columns
    return a.is_bf16 ? launch_tma_variant<true, 4, 4, 8, 4, false>(a, stream) : launch_tma_variant<false, 2, 4, 8, 4, false>(a, stream);
  }
  return a.is_bf16 ? launch_tma_variant<true, 8, 8, 16, 3, false>(a, stream) : launch_tma_variant<false, 4, 8, 16, 3, false>(a, stream);
}

}  // namespace xb
