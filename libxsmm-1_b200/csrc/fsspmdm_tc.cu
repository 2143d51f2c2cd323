// K4f: tensor-core branch of sfsspmdm for DENSE fixed operators (fp32, K <= 64, M <= 192), sm_100a.
//
// The reference always applies a float operator through its dense SMM kernel (src/libxsmm_fsspmdm.c:240-248,
// SREG is F64-only: src/libxsmm_main.c:1418).  For sparse operators the create-time baked FMA kernel is already
// bound by HBM; once the operator is dense enough that the FMA pipe becomes the bound (about half full for
// 150 x 64), the apply really is a dense contraction and goes to tcgen05:
//
//     D[n, m] = sum_k  B[k, n0 + n] * A[m, k]          (128 columns of the panel x M operator rows per tile)
//
//   * "A" operand = the B tile as it lies in memory ([k][n], n contiguous -> MN-major TF32 operand, TMA boxes of
//     32 columns with the 128B/32B-atom swizzle), "B" operand = the operator (K-major, SWIZZLE_128B), resident in
//     shared memory for the whole persistent CTA.
//   * 3xTF32: operator hi/lo split once at create time; b_lo = b - trunc(b) by four worker warps per tile, into ONE
//     buffer that serves both raw B stages (written once the MMAs of the tile before have completed).
//   * accumulator [128 lanes = columns][M_pad TMEM columns], double buffered: the epilogue of tile t overlaps the MMAs
//     of tile t+1.  Epilogue (EPI = 2, default): tcgen05.ld (thread = panel column, registers = operator rows) ->
//     shared-memory staging box of 32 rows x 128 columns -> TMA store (beta = 1: TMA reduce-add; C is never read by
//     the SM).  Per-thread stores (EPI = 1, also what an unaligned C gets; EPI = 0: the round-1 loop) left 600 line
//     stores per tile waiting in the load / store unit for DRAM, in front of the b_lo warps' shared-memory
//     instructions, so that stores and loads + MMAs ran one after the other (0.67-0.72 of HBM; now 0.88).
//   * 22 warps: TMA (+ L2 prefetch instructions two tiles ahead), MMA, four for b_lo, sixteen for the epilogue.
// Not the reference's rounding sequence; contract 1e-5 relative (observed ~2e-6; at most 24 accumulations).
#include "common.cuh"
#include "tc_common.cuh"
#include <vector>
#include <cstring>
#include <cstdlib>

namespace xb {

constexpr int FT_BN = 128;                  // panel columns per tile (UMMA M)
constexpr int FT_STAGES = 2;                // raw B tiles in flight; ONE b_lo buffer serves them in turn
constexpr int FT_WORKERS = 4;               // warps that write b_lo for the next tile
constexpr int FT_EPI = 16;                  // epilogue warps: four per TMEM lane quarter, taking the 32-row chunks of the operator in turn
constexpr int FT_THREADS = (2 + FT_WORKERS + FT_EPI) * 32;
constexpr int FT_STAGE_HALF = 64 * FT_BN * 4;          // 32 KiB: 64 k x 128 columns fp32
constexpr int FT_SMEM_B = 0;                           // FT_STAGES raw tiles
constexpr int FT_SMEM_LO = FT_STAGES * FT_STAGE_HALF;  // b_lo of the tile the tensor core works on (next)
constexpr int FT_CBOX_ROWS = 32;                       // rows of C per TMA store box
constexpr int FT_CBOX = FT_CBOX_ROWS * FT_BN * 4;      // 16 KiB: [32 rows][128 columns] fp32, plain row-major
constexpr int FT_SMEM_CBOX = FT_SMEM_LO + FT_STAGE_HALF;        // two staging boxes for C (EPI = 2)
constexpr int FT_SMEM_OP = FT_SMEM_CBOX + 2 * FT_CBOX; // operator: chunk 0 hi, chunk 1 hi, chunk 0 lo, chunk 1 lo (M_pad x 128 B each)

struct FsTcArgs {
  const float* B; float* C;
  const unsigned char* op_packed;   // 4 planes of M_pad x 128 B, already swizzled
  long long ncols, ldb, ldc;
  int M, M_pad, K, beta_one;
  int pf_mode;                      // 0: L2 prefetch through the TMA unit, 1: prefetch instructions of the producer warp
  int pf_dist;                      // the tile this many of the CTA's steps ahead is pulled into L2
  int debug;                        // developer timing aid (LIBXSMM_B200_K4F_DEBUG; results are wrong when set): 1 no b_lo, 2 no C stores, 4 no MMAs, 8 no B loads
};

template <int EPI>
__global__ void __launch_bounds__(FT_THREADS, 1)
fsspmdm_tc_kernel(const __grid_constant__ CUtensorMap tmB, const __grid_constant__ CUtensorMap tmC, const FsTcArgs p)
{
  extern __shared__ __align__(1024) unsigned char smem[];
  const int plane = p.M_pad * 128;
  unsigned char* sop = smem + FT_SMEM_OP;
  uint64_t* bar = (uint64_t*)(sop + 4 * plane);
  // Shared memory holds the operator (80 KiB for 150 rows) and 128 KiB of B.  Two stages of {raw, lo} left 64 KiB of loads in
  // flight per SM and no room for anything else.  Two raw stages and ONE b_lo buffer instead (b_lo of tile t + 1 is written once the
  // MMAs of tile t have completed: the tensor core idles for that half microsecond of the 2.5 us a tile may take), which frees 32 KiB
  // for two staging boxes of C (EPI = 2): the epilogue's 600 line stores per tile, waiting in the load / store unit for DRAM, held up
  // the shared-memory instructions of the b_lo warps behind them, so that stores and loads + MMAs ran one after the other.
  uint64_t* b_full = bar;            // [<= 3] TMA landed
  uint64_t* b_free = bar + 3;        // [<= 3] MMAs that read the stage have completed
  uint64_t* b_split = bar + 6;       // [1] workers wrote b_lo of the next tile
  uint64_t* lo_free = bar + 7;       // [1] MMAs that read b_lo have completed
  uint64_t* acc_full = bar + 8;      // [2] tile's MMAs completed
  uint64_t* acc_free = bar + 10;     // [2] epilogue drained the accumulator
  uint32_t* tmem_slot = (uint32_t*)(bar + 12);

  const int tid = (int)threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const long long ntiles = (p.ncols + FT_BN - 1) / FT_BN;
  const uint32_t sbase = smem_u32(smem);
  const int nks = (p.K + 7) / 8;     // k-steps of 8
  auto tile_of = [&](long long i) -> long long { return (long long)blockIdx.x + i * (long long)gridDim.x; };      // the i-th tile of this CTA

  if (0 == tid) {
#pragma unroll
    for (int i = 0; i < FT_STAGES; ++i) { mbar_init(&b_full[i], 1); mbar_init(&b_free[i], 1); }
    mbar_init(b_split, FT_WORKERS); mbar_init(lo_free, 1);
#pragma unroll
    for (int i = 0; i < 2; ++i) { mbar_init(&acc_full[i], 1); mbar_init(&acc_free[i], FT_EPI); }
    mbar_fence_init();
  }
  if (1 == warp) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;\n" ::"r"(smem_u32(tmem_slot)), "r"(512) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n" ::: "memory");
  }
  // the operator (already in UMMA layout) becomes resident
  for (int i = tid; i < 4 * plane / 16; i += FT_THREADS) ((uint4*)sop)[i] = __ldg((const uint4*)p.op_packed + i);
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_d = *tmem_slot;

  if (0 == warp) {
    if (0 == lane) tma_prefetch_desc(&tmB);
    long long it = 0;
    for (long long t = tile_of(0); t < ntiles; t = tile_of(++it)) {
      const int s = (int)(it % FT_STAGES);
      if (0 == lane) {
        if (it >= FT_STAGES) mbar_wait(&b_free[s], (uint32_t)(((it / FT_STAGES) - 1) & 1));
        if (p.debug & 8) mbar_arrive(&b_full[s]);
        else {
          mbar_arrive_expect_tx(&b_full[s], FT_STAGE_HALF);
          unsigned char* dst = smem + FT_SMEM_B + s * FT_STAGE_HALF;
#pragma unroll
          for (int j = 0; j < 4; ++j) tma_load_2d(dst + j * (64 * 128), &tmB, (int)(t * FT_BN) + 32 * j, 0, &b_full[s]);
        }
      }
      if (p.debug & 8) continue;
      // A tile this CTA will need after the ones in flight: into L2 now (with C's stores filling the DRAM queues a tile fetched
      // from DRAM takes several microseconds to arrive).
      const long long tn = tile_of(it + p.pf_dist);
      if (tn < ntiles) {
        if (0 == p.pf_mode) {          // through the TMA unit (measured: these requests queue in front of the next tile's loads)
          if (0 == lane) {
#pragma unroll
            for (int j = 0; j < 4; ++j) tma_prefetch_l2_2d(&tmB, (int)(tn * FT_BN) + 32 * j, 0);
          }
        }
        else {                         // prefetch instructions of the whole warp: one per 128-byte line, four lines per row of B
          __syncwarp();
          const long long c0 = tn * FT_BN + 32 * (lane & 3);
          if (c0 < p.ncols) {
            for (int k = lane >> 2; k < p.K; k += 8) asm volatile("prefetch.global.L2 [%0];\n" ::"l"(p.B + (long long)k * p.ldb + c0) : "memory");
          }
        }
      }
    }
  }
  else if (1 == warp) {
    if (0 == lane) {
      // D = F32, A = B = TF32, A MN-major (the B tile), B K-major (the operator), M = 128, N = M_pad
      const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | (1u << 15) | (0u << 16) | ((uint32_t)(p.M_pad >> 3) << 17) | ((uint32_t)(FT_BN >> 4) << 24);
      long long it = 0;
      for (long long t = tile_of(0); t < ntiles; t = tile_of(++it)) {
        const int s = (int)(it % FT_STAGES), ab = (int)(it & 1);
        if (it >= 2) mbar_wait(&acc_free[ab], (uint32_t)(((it >> 1) - 1) & 1));
        mbar_wait(b_split, (uint32_t)(it & 1));
        tc_fence_after();
        const uint32_t x_hi = sbase + FT_SMEM_B + s * FT_STAGE_HALF, x_lo = sbase + FT_SMEM_LO;
        const uint32_t tacc = tmem_d + (uint32_t)(ab * 256);
        for (int ks = 0; ks < nks; ++ks) {
          // tile operand (MN-major, 128B/32B-atom swizzle): 8 k = 1024 B; 32-column blocks 64*128 B apart, 4-k groups 512 B
          const uint64_t dxh = tc_smem_desc(x_hi + ks * 1024, 64 * 128, 512, 1);
          const uint64_t dxl = tc_smem_desc(x_lo + ks * 1024, 64 * 128, 512, 1);
          // operator (K-major, SWIZZLE_128B): chunk = ks / 4 (32 k each), 8 k = 32 B inside the 128-byte rows
          const uint32_t o = sbase + FT_SMEM_OP + (uint32_t)((ks >> 2) * plane + (ks & 3) * 32);
          const uint64_t doh = tc_smem_desc(o, 16, 1024, 2);
          const uint64_t dol = tc_smem_desc(o + 2 * plane, 16, 1024, 2);
          if (p.debug & 4) continue;
          tc_mma_tf32(tacc, dxh, doh, idesc, ks > 0 ? 1u : 0u);
          tc_mma_tf32(tacc, dxl, doh, idesc, 1u);
          tc_mma_tf32(tacc, dxh, dol, idesc, 1u);
        }
        tc_commit(&b_free[s]);
        tc_commit(lo_free);
        tc_commit(&acc_full[ab]);
      }
    }
  }
  else if (warp < 2 + FT_WORKERS) {
    // ---------------- b_lo = b - trunc_tf32(b) for every tile (same swizzled addresses) ----------------
    const int wt = tid - 64;                      // 0..127
    long long it = 0;
    for (long long t = tile_of(0); t < ntiles; t = tile_of(++it)) {
      const int s = (int)(it % FT_STAGES);
      mbar_wait(&b_full[s], (uint32_t)((it / FT_STAGES) & 1));
      if (it >= 1) mbar_wait(lo_free, (uint32_t)((it - 1) & 1));       // the MMAs of the tile before have read b_lo
      const uint4* src = (const uint4*)(smem + FT_SMEM_B + s * FT_STAGE_HALF);
      uint4* dst = (uint4*)(smem + FT_SMEM_LO);
#pragma unroll 4
      for (int i = wt; i < FT_STAGE_HALF / 16; i += FT_WORKERS * 32) {
        if (p.debug & 1) break;
        const uint4 b = src[i];
        uint4 l;
        l.x = __float_as_uint(__uint_as_float(b.x) - __uint_as_float(b.x & 0xFFFFE000u));
        l.y = __float_as_uint(__uint_as_float(b.y) - __uint_as_float(b.y & 0xFFFFE000u));
        l.z = __float_as_uint(__uint_as_float(b.z) - __uint_as_float(b.z & 0xFFFFE000u));
        l.w = __float_as_uint(__uint_as_float(b.w) - __uint_as_float(b.w & 0xFFFFE000u));
        dst[i] = l;
      }
      fence_proxy_async();
      __syncwarp();
      if (0 == lane) mbar_arrive(b_split);
    }
  }
  else {
    // ---------------- epilogue: thread = panel column, registers = operator rows ----------------
    // A worker's instruction stream is one dependent chain of memory instructions (each tens of cycles next to the
    // UMMA operand traffic), so the 150 row stores of a tile are spread over sixteen warps: four per TMEM
    // lane quarter, taking the 32-row chunks in turn.
    const int quarter = warp & 3, part = (warp - 2 - FT_WORKERS) >> 2;
    long long it = 0;
    if (2 == EPI) {
      // C through the store engine: the sixteen warps put 32 rows x 128 columns of the tile into a staging box (thread = column,
      // eight rows per warp: conflict-free 4-byte stores), one thread hands the box to TMA (beta = 1: as a reduction, C is never
      // read by the SM) and the next 32 rows go to the other box.  Nothing of the epilogue waits in the load / store unit for DRAM.
      const int ew = warp - 2 - FT_WORKERS;                 // 0..15
      const bool issuer = (0 == ew) && (0 == lane);
      const int nbox = (p.M + FT_CBOX_ROWS - 1) / FT_CBOX_ROWS;
      const uint32_t tq = tmem_d + ((uint32_t)(quarter * 32) << 16);
      uint32_t nb = 0;                                      // boxes issued so far (parity picks the staging box)
      for (long long t = tile_of(0); t < ntiles; t = tile_of(++it)) {
        const int ab = (int)(it & 1);
        mbar_wait(&acc_full[ab], (uint32_t)((it >> 1) & 1));
        tc_fence_after();
        for (int b = 0; b < nbox; ++b, ++nb) {
          unsigned char* box = smem + FT_SMEM_CBOX + (nb & 1u) * FT_CBOX;
          uint32_t v[8];
          tc_ld8_nowait(tq + (uint32_t)(ab * 256 + FT_CBOX_ROWS * b + 8 * part), v);
          tc_wait_ld();
          tc_pin8(v);
          if (b == nbox - 1) {                              // the accumulator is in registers: hand it back
            tc_fence_before();
            __syncwarp();
            if (0 == lane) mbar_arrive(&acc_free[ab]);
          }
          // the box is free once the store engine has read its previous content out (the issuing thread waited for that after
          // handing over the box before this one)
          asm volatile("bar.sync 1, %0;\n" ::"n"(FT_EPI * 32) : "memory");
#pragma unroll
          for (int j = 0; j < 8; ++j) *(uint32_t*)(box + ((8 * part + j) * FT_BN + quarter * 32 + lane) * 4) = v[j];
          fence_proxy_async();
          asm volatile("bar.sync 2, %0;\n" ::"n"(FT_EPI * 32) : "memory");
          if (issuer && !(p.debug & 2)) {
            if (p.beta_one)
              asm volatile("cp.reduce.async.bulk.tensor.2d.global.shared::cta.add.tile.bulk_group [%0, {%1, %2}], [%3];\n"
                           ::"l"(&tmC), "r"((int)(t * FT_BN)), "r"(FT_CBOX_ROWS * b), "r"(smem_u32(box)) : "memory");
            else
              asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%1, %2}], [%3];\n"
                           ::"l"(&tmC), "r"((int)(t * FT_BN)), "r"(FT_CBOX_ROWS * b), "r"(smem_u32(box)) : "memory");
            asm volatile("cp.async.bulk.commit_group;\n" ::: "memory");
            asm volatile("cp.async.bulk.wait_group.read 1;\n" ::: "memory");      // the OTHER box (the next one to be filled) has been read out
          }
        }
      }
      if (issuer) asm volatile("cp.async.bulk.wait_group.read 0;\n" ::: "memory");
    }
    else if (0 == EPI) {
      for (long long t = tile_of(0); t < ntiles; t = tile_of(++it)) {
        const int ab = (int)(it & 1);
        mbar_wait(&acc_full[ab], (uint32_t)((it >> 1) & 1));
        tc_fence_after();
        const long long col = t * FT_BN + quarter * 32 + lane;
        for (int m0 = 32 * part; m0 < p.M; m0 += 32 * (FT_EPI / 4)) {
          uint32_t v[32];
          tc_ld32(tmem_d + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(ab * 256 + m0), v);
          if (col < p.ncols && !(p.debug & 2)) {
#pragma unroll
            for (int j = 0; j < 32; ++j) {
              if (m0 + j < p.M) {
                float* dst = p.C + (long long)(m0 + j) * p.ldc + col;
                const float r = __uint_as_float(v[j]);
                __stcs(dst, p.beta_one ? (r + __ldcs(dst)) : r);
              }
            }
          }
        }
        tc_fence_before();
        __syncwarp();
        if (0 == lane) mbar_arrive(&acc_free[ab]);
      }
    }
    else {
      // The operator's rows in chunks of eight, dealt round-robin to the four warps of a lane quarter (150 rows: 40 / 40 / 40 / 30).
      // All of a warp's chunks are fetched from tensor memory first, the accumulator is handed back to the tensor core, and only
      // then the rows are stored: one pointer stepping by ldc, no per-row branch in full chunks; for beta = 1 the eight C
      // values of a chunk are all requested before the first is used.
      const int nchunk = (p.M + 7) >> 3;
      const uint32_t tq = tmem_d + ((uint32_t)(quarter * 32) << 16);
      const long long ldc = p.ldc;
      for (long long t = tile_of(0); t < ntiles; t = tile_of(++it)) {
        const int ab = (int)(it & 1);
        if (p.beta_one && tile_of(it + 1) < ntiles) {
          // beta = 1: the lines of C this warp will read for the CTA's NEXT tile go into L2 now (lane = row of a chunk)
          const long long cn = tile_of(it + 1) * FT_BN + quarter * 32;
          if (cn < p.ncols) {
#pragma unroll
            for (int r = 0; r < 2; ++r) {
              const int i = 4 * r + (lane >> 3), m = 8 * (part + 4 * i) + (lane & 7);
              if (i < 6 && m < p.M) asm volatile("prefetch.global.L2 [%0];\n" ::"l"(p.C + (long long)m * ldc + cn) : "memory");
            }
          }
        }
        mbar_wait(&acc_full[ab], (uint32_t)((it >> 1) & 1));
        tc_fence_after();
        const long long col = t * FT_BN + quarter * 32 + lane;
        float* dst = p.C + (long long)(8 * part) * ldc + col;
        const bool live = col < p.ncols && !(p.debug & 2);
#pragma unroll
        for (int h = 0; h < 2; ++h) {          // M_pad <= 192: at most 24 chunks, six per warp, fetched three at a time
          uint32_t v[3][8];
#pragma unroll
          for (int i = 0; i < 3; ++i) if (part + 4 * (3 * h + i) < nchunk) tc_ld8_nowait(tq + (uint32_t)(ab * 256 + 8 * (part + 4 * (3 * h + i))), v[i]);
          tc_wait_ld();
#pragma unroll
          for (int i = 0; i < 3; ++i) tc_pin8(v[i]);
          if (1 == h) {                        // the accumulator is in registers: hand it back before the stores
            tc_fence_before();
            __syncwarp();
            if (0 == lane) mbar_arrive(&acc_free[ab]);
          }
          if (live) {
#pragma unroll
            for (int i = 0; i < 3; ++i) {
              const int m0 = 8 * (part + 4 * (3 * h + i));
              if (m0 + 8 <= p.M) {
                if (p.beta_one) {      // the eight C values of the chunk are all requested before the first is used
                  float o[8];
#pragma unroll
                  for (int j = 0; j < 8; ++j) o[j] = __ldcs(dst + j * ldc);
#pragma unroll
                  for (int j = 0; j < 8; ++j) __stcs(dst + j * ldc, __uint_as_float(v[i][j]) + o[j]);
                }
                else {
#pragma unroll
                  for (int j = 0; j < 8; ++j) __stcs(dst + j * ldc, __uint_as_float(v[i][j]));
                }
              }
              else {
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                  if (m0 + j < p.M) {
                    const float r = __uint_as_float(v[i][j]);
                    __stcs(dst + j * ldc, p.beta_one ? (r + __ldcs(dst + j * ldc)) : r);
                  }
                }
              }
              dst += 32 * ldc;
            }
          }
        }
      }
    }
  }
  __syncthreads();
  if (1 == warp) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;\n" ::"r"(tmem_d), "r"(512) : "memory");
  }
}

bool make_tensor_map_2d_sw128(CUtensorMap* map, const void* base, int elem_bytes, unsigned long long cols, unsigned long long rows,
                              unsigned long long row_pitch_bytes, unsigned box_cols, unsigned box_rows, bool atom32);

// ---- host side ---------------------------------------------------------------------------------------------
struct FsTc { unsigned char* d_op; int M, M_pad, K, beta_one; size_t smem; int sms; int epi, pf_mode, pf_dist, debug; };

bool make_tensor_map_2d(CUtensorMap* map, const void* base, int elem_bytes, unsigned long long cols, unsigned long long rows,
                        unsigned long long row_pitch_bytes, unsigned box_cols, unsigned box_rows);

static int fs_tc_mpad(int M) { return (M + 15) / 16 * 16; }

// can this operator use the tensor-core kernel at all?
bool fs_tc_supported(int is_double, int M, int K) { return !is_double && K >= 1 && K <= 64 && M >= 1 && fs_tc_mpad(M) <= 192; }

FsTc* fs_tc_build(int M, int K, int lda, int beta_one, const float* a_dense)
{
  FsTc* t = new FsTc();
  t->M = M; t->K = K; t->M_pad = fs_tc_mpad(M); t->beta_one = beta_one; t->d_op = 0;
  const int plane = t->M_pad * 128;
  std::vector<unsigned char> packed((size_t)4 * plane, 0);
  for (int m = 0; m < M; ++m) for (int k = 0; k < K; ++k) {
    const float v = a_dense[(size_t)m * lda + k];
    unsigned int bits; memcpy(&bits, &v, 4);
    bits &= 0xFFFFE000u;
    float hi; memcpy(&hi, &bits, 4);
    const float lo = v - hi;
    const int chunk = k >> 5, kk = k & 31;
    const size_t off = (size_t)chunk * plane + (size_t)(m >> 3) * 1024 + (size_t)(m & 7) * 128 + (size_t)((((kk >> 2) ^ (m & 7)) & 7) << 4) + (size_t)((kk & 3) << 2);
    memcpy(&packed[off], &hi, 4);
    memcpy(&packed[(size_t)2 * plane + off], &lo, 4);
  }
  XB_CUDA(cudaMalloc((void**)&t->d_op, packed.size()));
  if (0 == t->d_op) { delete t; return 0; }
  XB_CUDA(cudaMemcpy(t->d_op, packed.data(), packed.size(), cudaMemcpyHostToDevice));
  t->smem = (size_t)FT_SMEM_OP + (size_t)4 * plane + 256;
  int dev = 0; cudaDeviceProp prop;
  t->sms = 148;
  if (cudaSuccess == cudaGetDevice(&dev) && cudaSuccess == cudaGetDeviceProperties(&prop, dev)) t->sms = prop.multiProcessorCount;
  ensure_smem_optin((const void*)fsspmdm_tc_kernel<0>, (int)((size_t)FT_SMEM_OP + (size_t)4 * 192 * 128 + 256));
  ensure_smem_optin((const void*)fsspmdm_tc_kernel<1>, (int)((size_t)FT_SMEM_OP + (size_t)4 * 192 * 128 + 256));
  ensure_smem_optin((const void*)fsspmdm_tc_kernel<2>, (int)((size_t)FT_SMEM_OP + (size_t)4 * 192 * 128 + 256));
  const char* e = getenv("LIBXSMM_B200_K4F_EPI");        // 0: the round-1 epilogue (32-row chunks, per-row address arithmetic)
  t->epi = (e && *e >= '0' && *e <= '2') ? (*e - '0') : 2;       // 2: C through TMA store boxes; 1: per-thread stores, 8-row chunks; 0: the round-1 epilogue
  e = getenv("LIBXSMM_B200_K4F_PF");
  t->pf_dist = (e && atoi(e) >= 2) ? atoi(e) : 2;       // measured with the TMA-store epilogue: 2 / 3 / 4 / 6 tiles ahead 624 / 624 / 698 / 784 us (further ahead the lines are evicted by C's stream before they are used)
  e = getenv("LIBXSMM_B200_K4F_PFMODE");
  t->pf_mode = (e && '0' == *e) ? 0 : 1;
  e = getenv("LIBXSMM_B200_K4F_DEBUG");
  t->debug = e ? atoi(e) : 0;
  return t;
}

bool fs_tc_launch(const FsTc* t, const void* dB, void* dC, long long ncols, long long ldb, long long ldc, cudaStream_t stream)
{
  if (0 == t || ncols <= 0) return false;
  if (0 != ((uintptr_t)dB & 15) || 0 != ((ldb * 4) & 15)) return false;
  CUtensorMap map;
  if (!make_tensor_map_2d_sw128(&map, dB, 4, (unsigned long long)ncols, (unsigned long long)t->K, (unsigned long long)ldb * 4, 32, 64, true)) return false;
  FsTcArgs a;
  a.B = (const float*)dB; a.C = (float*)dC; a.op_packed = t->d_op; a.ncols = ncols; a.ldb = ldb; a.ldc = ldc;
  a.M = t->M; a.M_pad = t->M_pad; a.K = t->K; a.beta_one = t->beta_one; a.pf_dist = t->pf_dist; a.pf_mode = t->pf_mode; a.debug = t->debug;
  const long long ntiles = (ncols + FT_BN - 1) / FT_BN;
  const unsigned grid = (unsigned)(ntiles < t->sms ? ntiles : t->sms);
  // C as a tensor of (ncols, M) for the store engine: rows past M and columns past ncols of a box are clipped by the hardware
  CUtensorMap cmap = map;
  int epi = t->epi;
  // The store engine clips a box at the tensor's last column only to a 16-byte boundary: with ncols not a multiple of four
  // it would write (beta = 0: zeros) or read-modify-write (beta = 1) up to three columns past the panel, which belong to the
  // caller (the dense dispatch entry takes any column count).  Per-thread stores write exactly [0, ncols).
  if (0 != (ncols & 3)) epi = (0 == epi) ? 0 : 1;
  if (2 == epi &&!make_tensor_map_2d(&cmap, dC, 4, (unsigned long long)ncols, (unsigned long long)t->M, (unsigned long long)ldc * 4, FT_BN, FT_CBOX_ROWS)) { cmap = map; epi = 1; }   // unaligned C
  if (2 == epi) fsspmdm_tc_kernel<2><<<grid, FT_THREADS, t->smem, stream>>>(map, cmap, a);
  else if (1 == epi) fsspmdm_tc_kernel<1><<<grid, FT_THREADS, t->smem, stream>>>(map, cmap, a);
  else fsspmdm_tc_kernel<0><<<grid, FT_THREADS, t->smem, stream>>>(map, cmap, a);
  XB_CUDA(cudaGetLastError());
  return true;
}

void fs_tc_destroy(FsTc* t)
{
  if (0 == t) return;
  if (t->d_op) cudaFree(t->d_op);
  delete t;
}

}  // namespace xb
