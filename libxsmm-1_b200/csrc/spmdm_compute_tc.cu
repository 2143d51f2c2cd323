// K4: tensor-core branch of the spmdm compute step for the DENSE regime (fp32 inputs), sm_100a.
//
//   C[128 rows, 128 cols] = beta*C + sum_kb densify(slice(kb, mb))[128 x 128] * B[kb*128 .. +128, 128 cols]
//
// The CSR slice block is scattered back into a dense, 128B-swizzled K-major shared-memory tile and fed to
// tcgen05.mma (kind::tf32, M = 128, N = 128, K = 8) with the accumulator in TMEM.  fp32 accuracy comes from
// the error-compensated 3xTF32 split: a = a_hi + a_lo, b = b_hi + b_lo with the *_hi parts representable in
// TF32, and D += a_hi*b_hi + a_hi*b_lo + a_lo*b_hi (the dropped a_lo*b_lo term is 2^-22 relative).
//   * A_hi / A_lo: built by the worker warps from (colidx, values) of the slice, once per k-block.
//   * B: 32 x 128 chunks by TMA (SWIZZLE_128B_ATOM_32B, MN-major operand: four boxes of 32 columns), two stages;
//     the raw chunk serves as b_hi (the tensor core ignores the low 13 mantissa bits), the workers write
//     b_lo = b - trunc(b) into a second buffer with the same swizzled addressing.
//   * one thread issues the MMAs; tcgen05.commit releases B stages / the A tile / signals the epilogue.
//   * every k-block's accumulator is drained into registers by tcgen05.ld (thread = row, 32 columns per
//     instruction) while the next k-block's MMAs run into the other TMEM buffer; epilogue: + beta*C, 16-byte stores.
// This branch does NOT keep the reference's rounding sequence (tensor-core accumulation order); it is used
// where the relative-error contract (1e-5) is the bar.  It never touches operands the reference would skip
// in a way that changes finite results: dropped (zero) entries of A are exact zeros in the dense tile.
#include "common.cuh"
#include "tc_common.cuh"

namespace xb {

constexpr int TC_BM = 128;          // rows per CTA (UMMA M)
constexpr int TC_BN = 128;          // columns per CTA (UMMA N)
constexpr int TC_KC = 32;           // k per B chunk = one 128-byte swizzle row of fp32
constexpr int TC_NB = 3;            // B stages
constexpr int TC_WORKERS = 16;      // worker warps (densify, split, drain, epilogue)
constexpr int TC_WT = TC_WORKERS * 32;
constexpr int TC_THREADS = (2 + TC_WORKERS) * 32;
constexpr int TC_A_CHUNK = TC_BM * 128;             // bytes of one 128 x 32 fp32 K-major tile (16 KiB)
constexpr int TC_A_HALF = 4 * TC_A_CHUNK;           // one half of a k-block (64 k): hi chunks 0,1 then lo chunks 0,1 (64 KiB)
constexpr int TC_B_CHUNK = TC_KC * TC_BN * 4;       // bytes of one 32 x 128 fp32 chunk (16 KiB)
constexpr int TC_SMEM_A = 0;                                        // two halves, double buffered: 128 KiB
constexpr int TC_SMEM_B = 2 * TC_A_HALF;                            // stage s: raw at +s*32K, lo at +s*32K+16K
constexpr int TC_SMEM_BAR = TC_SMEM_B + TC_NB * 2 * TC_B_CHUNK;     // 224 KiB
constexpr int TC_SMEM_BYTES = TC_SMEM_BAR + 256;

// TC_NQ = nonzeros a worker thread keeps in registers per k-block; HIST = it also remembers where it put the previous
// k-block's and clears those instead of wiping the half.  <8, true> for slices up to ~25 % dense (measured on 2048^3 at
// 10 %: 174 -> 139 us), <16, false> for denser ones (at 50 % the short register list sends half the nonzeros through
// the memory loop: 183 -> 211 us); the register file (576 threads) does not hold 16 + 16 + 16.
// DENSEA = the slicing kernel also left the dense tile image of the slices (SliceArena::dense): a half of A is then
// one 64 KiB bulk copy issued by the producer thread and nobody rebuilds anything.
template <int TC_NQ, bool HIST, bool DENSEA>
__global__ void __launch_bounds__(TC_THREADS, 1)
spmdm_compute_tc_kernel(const __grid_constant__ CUtensorMap tmB, const ComputeArgs p)
{
  extern __shared__ __align__(1024) unsigned char smem[];
  uint64_t* bar = (uint64_t*)(smem + TC_SMEM_BAR);
  uint64_t* b_full = bar;            // [3] TMA landed (tx bytes)
  uint64_t* b_split = bar + 3;       // [3] workers wrote b_lo
  uint64_t* b_free = bar + 6;        // [3] MMAs that read the stage have completed
  uint64_t* a_ready = bar + 9;       // [2] workers built the A half (k 0..63 / 64..127 of the k-block)
  uint64_t* a_free = bar + 11;       // [2] MMAs that read the A half have completed
  uint64_t* acc_full = bar + 13;     // [2] the k-block's MMAs into accumulator buffer (kb & 1) have completed
  uint64_t* acc_free = bar + 15;     // [2] the workers have drained that buffer
  uint32_t* tmem_slot = (uint32_t*)(bar + 17);

  const Geom& g = p.g;
  if (p.tc_twin > 0 && xb_total_nnz(p.sl.slice_nnz, g.mb * g.kb) < p.tc_min_nnz) return;   // sparse regime: the CUDA-core twin does this multiply
  const int tid = (int)threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int tiles_per_mb = (g.bm + TC_BM - 1) / TC_BM;
  const int mbi = p.mb_first + (int)blockIdx.y / tiles_per_mb;
  const int ml0 = ((int)blockIdx.y % tiles_per_mb) * TC_BM;
  const int rows_in_block = min(g.bm, g.m - mbi * g.bm);
  if (ml0 >= rows_in_block) return;
  const int tile_rows = min(TC_BM, rows_in_block - ml0);
  const int n0 = (int)blockIdx.x * TC_BN;
  const int nsteps = g.kb * 2;       // one step = one half k-block = two B chunks
  const uint32_t sbase = smem_u32(smem);

  if (0 == tid) {
#pragma unroll
    for (int i = 0; i < TC_NB; ++i) { mbar_init(&b_full[i], 1); mbar_init(&b_split[i], HIST ? TC_WORKERS / 2 : TC_WORKERS); mbar_init(&b_free[i], 1); }
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      mbar_init(&a_ready[i], DENSEA ? 1 : (HIST ? TC_WORKERS / 2 : TC_WORKERS)); mbar_init(&a_free[i], 1);
      mbar_init(&acc_full[i], 1); mbar_init(&acc_free[i], TC_WORKERS);
    }
    mbar_fence_init();
  }
  if (1 == warp) {   // TMEM: 2 x 128 columns of fp32 accumulators (one warp allocates and later frees)
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;\n" ::"r"(smem_u32(tmem_slot)), "r"(256) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_d = *tmem_slot;

  if (0 == warp) {
    // ---------------- TMA producer: B chunks through a 3-stage ring ----------------
    if (0 == lane) {
      tma_prefetch_desc(&tmB);
      const int tiles_per_mb_img = (g.bm + 127) / 128;
      for (int c = 0; c < nsteps * 2; ++c) {
        if (DENSEA && 0 == (c & 1)) {      // first chunk of a step: the step's A half straight from the dense image
          const int t = c >> 1, kb = t >> 1, h = t & 1;
          if (kb > 0) mbar_wait(&a_free[h], (kb - 1) & 1);
          const float* src = p.sl.dense + ((size_t)(kb * g.mb + mbi) * tiles_per_mb_img + (size_t)(ml0 >> 7)) * 32768 + (size_t)h * 16384;
          mbar_arrive_expect_tx(&a_ready[h], TC_A_HALF);
          asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n"
                       ::"r"(smem_u32(smem + TC_SMEM_A + h * TC_A_HALF)), "l"(src), "r"((uint32_t)TC_A_HALF), "r"(smem_u32(&a_ready[h])) : "memory");
        }
        const int s = c % TC_NB, f = c / TC_NB;
        if (f > 0) mbar_wait(&b_free[s], (f - 1) & 1);
        mbar_arrive_expect_tx(&b_full[s], TC_B_CHUNK);
        unsigned char* dst = smem + TC_SMEM_B + s * 2 * TC_B_CHUNK;
        if (p.transb) tma_load_2d(dst, &tmB, c * TC_KC, n0, &b_full[s]);   // B stored n x k: one box of 128 n-rows x 32 k (K-major operand)
        else {
#pragma unroll
          for (int j = 0; j < 4; ++j) tma_load_2d(dst + j * (TC_KC * 128), &tmB, n0 + 32 * j, c * TC_KC, &b_full[s]);
        }
      }
    }
  }
  else if (1 == warp) {
    // ---------------- MMA issuer ----------------
    if (0 == lane) {
      // instruction descriptor (cute/arch/mma_sm100_desc.hpp InstrDescriptor): D = F32, A = B = TF32,
      // A K-major, B MN-major, N = 128, M = 128
      // (B stored n x k, transb = 'T', is a K-major operand: plain SWIZZLE_128B rows of 32 k)
      const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | (0u << 15) | ((p.transb ? 0u : 1u) << 16) | ((uint32_t)(TC_BN >> 3) << 17) | ((uint32_t)(TC_BM >> 4) << 24);
      const uint32_t b_kstep = p.transb ? 32u : 1024u, b_lbo = p.transb ? 16u : (uint32_t)(TC_KC * 128), b_sbo = p.transb ? 1024u : 512u, b_lay = p.transb ? 2u : 1u;
      for (int t = 0; t < nsteps; ++t) {
        const int kb = t >> 1, h = t & 1;
        // The accumulator of a k-block is drained into registers by the workers (IEEE adds) instead of being
        // carried in TMEM over the whole K loop: the tensor core truncates on every accumulation, and over
        // K/8*3 accumulations that bias would exceed the 1e-5 contract.  Two TMEM buffers alternate.
        const uint32_t tmem_acc = tmem_d + (uint32_t)((kb & 1) * TC_BN);
        if (0 == h && kb >= 2) mbar_wait(&acc_free[kb & 1], ((kb >> 1) - 1) & 1);
        mbar_wait(&a_ready[h], kb & 1);
#pragma unroll
        for (int j = 0; j < 2; ++j) {
          const int c = 2 * t + j, s = c % TC_NB;
          mbar_wait(&b_split[s], (c / TC_NB) & 1);
          tc_fence_after();
          const uint32_t a_hi = sbase + TC_SMEM_A + h * TC_A_HALF + j * TC_A_CHUNK;
          const uint32_t a_lo = a_hi + 2 * TC_A_CHUNK;
          const uint32_t b_hi = sbase + TC_SMEM_B + s * 2 * TC_B_CHUNK;
          const uint32_t b_lo = b_hi + TC_B_CHUNK;
#pragma unroll
          for (int ks = 0; ks < 4; ++ks) {
            // A (K-major, SWIZZLE_128B): 8 k = 32 bytes further inside the 128-byte rows; 8-row groups 1024 B apart
            const uint64_t dah = tc_smem_desc(a_hi + ks * 32, 16, 1024, 2);
            const uint64_t dal = tc_smem_desc(a_lo + ks * 32, 16, 1024, 2);
            // B (MN-major TF32: only the 128-byte swizzle with 32-byte atoms exists; pinned with tools/umma_probe):
            // atoms of 4 k x 128 B, k groups 512 B apart (SBO), 32-column blocks 4096 B apart (LBO); 8 k = 1024 B
            const uint64_t dbh = tc_smem_desc(b_hi + ks * b_kstep, b_lbo, b_sbo, b_lay);
            const uint64_t dbl = tc_smem_desc(b_lo + ks * b_kstep, b_lbo, b_sbo, b_lay);
            tc_mma_tf32(tmem_acc, dah, dbh, idesc, (h > 0 || j > 0 || ks > 0) ? 1u : 0u);
            tc_mma_tf32(tmem_acc, dah, dbl, idesc, 1u);
            tc_mma_tf32(tmem_acc, dal, dbh, idesc, 1u);
          }
          tc_commit(&b_free[s]);
        }
        tc_commit(&a_free[h]);
        if (1 == h) tc_commit(&acc_full[kb & 1]);
      }
    }
  }
  else {
    // ---------------- workers: densify A, split B, drain accumulators, epilogue ----------------
    const int w = warp - 2;                       // 0..15
    // HIST (sparse) variant: the sixteen worker warps split the per-step jobs -- warps 0-7 rebuild the A half, warps
    // 8-15 write b_lo -- and all of them drain; a worker's instruction stream is one dependent chain of memory
    // instructions, so two shorter chains side by side beat one long one.  The dense variant keeps all sixteen on
    // every job (the rebuild of a dense half needs all the threads it can get).
    constexpr int DW = HIST ? TC_WT / 2 : TC_WT;  // threads on the densify job / on the split job
    const bool do_dens = !DENSEA && (!HIST || w < TC_WORKERS / 2), do_split = !HIST || w >= TC_WORKERS / 2;
    const int wt = HIST ? ((tid - 64) & (DW - 1)) : (tid - 64);   // index within the job's threads
    const size_t cap = (size_t)g.bm * g.bk;
    // this thread's part of the output: row (quarter*32 + lane), 32 columns; warp w may touch TMEM lanes
    // 32*(w%4) .. +31, and the four warps that share a lane quarter take 32 columns each
    const int quarter = warp & 3;
    const int row = quarter * 32 + lane;
    const int cgrp = (w >> 2) * 32;
    float run[32];
#pragma unroll
    for (int j = 0; j < 32; ++j) run[j] = 0.f;
    auto drain = [&](int kbd) {                   // run += accumulator of k-block kbd
      mbar_wait(&acc_full[kbd & 1], (kbd >> 1) & 1);
      tc_fence_after();
      uint32_t v[32];
      tc_ld32(tmem_d + ((uint32_t)(quarter * 32) << 16) + (uint32_t)((kbd & 1) * TC_BN + cgrp), v);
#pragma unroll
      for (int j = 0; j < 32; ++j) run[j] += __uint_as_float(v[j]);
      tc_fence_before();
      __syncwarp();
      if (0 == lane) mbar_arrive(&acc_free[kbd & 1]);
    };
    // The tile's nonzeros of one k-block are one contiguous range of the slice.  Thread wt owns nonzeros
    // first + wt + i*TC_WT; the first TC_NQ of them are fetched ONCE per k-block into registers (packed
    // row|column and value), well before they are needed, and scattered twice (k < 64, k >= 64).
    uint32_t pk[TC_NQ]; float vv[TC_NQ];       // raw loads only: nothing here may consume them (no stall on the fetch)
    uint32_t hk[HIST ? TC_NQ : 1];             // positions of the previous k-block's nonzeros (this thread's share)
    int first = 0, last = 0, n_prev = 0;
    auto fetch = [&](int kbf) {
      const int sidx = kbf * g.mb + mbi;
      const uint16_t* ro = p.sl.rowidx + (size_t)sidx * (g.bm + 1) + ml0;
      const uint16_t* ri = p.sl.tcoff + sidx * cap;
      const float* va = p.sl.values + sidx * cap;
      first = (int)__ldg(ro);
      last = (int)__ldg(ro + tile_rows);
      if (last < first) last = (int)__ldg(ro + tile_rows - 1);   // wrapped u16 counter of a full slice: last row reads as empty
#pragma unroll
      for (int i = 0; i < TC_NQ; ++i) {
        const int q = first + wt + i * DW;
        pk[i] = 0; vv[i] = 0.f;
        if (q < last) { pk[i] = (uint32_t)__ldg(ri + q); vv[i] = __ldg(va + q); }
      }
    };
    if (do_dens) fetch(0);
    for (int t = 0; t < nsteps; ++t) {
      const int kb = t >> 1, h = t & 1;
      // (1) A half: wait until the MMAs that read this buffer (previous k-block) are done, zero, scatter.
      //     The other half is being multiplied meanwhile.
      if (do_dens) {
      if (kb > 0) mbar_wait(&a_free[h], (kb - 1) & 1);
      unsigned char* abuf = smem + TC_SMEM_A + h * TC_A_HALF;
      // The half still holds the same half of the previous k-block.  If all of that k-block's nonzeros were in
      // registers (hk), the thread clears exactly what it wrote (at 10 % density 1.6 stores per thread instead of a
      // 64 KiB wipe that competes with the operand reads for shared memory); otherwise the half is wiped.
      bool wipe = true;
      if constexpr (HIST) {
        if (kb > 0 && n_prev <= TC_NQ * DW) {
          wipe = false;
#pragma unroll
          for (int i = 0; i < TC_NQ; ++i) {
            if (i * DW >= n_prev) break;                     // uniform
            if (wt + i * DW < n_prev && (int)((hk[i] >> 15) & 1u) == h) {
              const uint32_t off = (hk[i] & 0x7FFFu) << 2;
              *(float*)(abuf + off) = 0.f;
              *(float*)(abuf + 2 * TC_A_CHUNK + off) = 0.f;
            }
          }
        }
      }
      if (wipe) {
        uint4* z = (uint4*)abuf;
#pragma unroll
        for (int i = 0; i < TC_A_HALF / 16 / DW; ++i) z[wt + i * DW] = make_uint4(0, 0, 0, 0);
      }
      asm volatile("bar.sync 1, %0;\n" ::"n"(DW) : "memory");   // clearing complete before the scatter (another thread may write there)
      auto put = [&](uint32_t t, float v) {   // t = xb_tc_pack(row, k): half in bit 15, word offset below
        if ((int)((t >> 15) & 1u) == h) {
          const uint32_t off = (t & 0x7FFFu) << 2;
          const float vh = __uint_as_float(__float_as_uint(v) & 0xFFFFE000u);
          *(float*)(abuf + off) = vh;
          *(float*)(abuf + 2 * TC_A_CHUNK + off) = v - vh;
        }
      };
#pragma unroll
      for (int i = 0; i < TC_NQ; ++i) {
        const int q = first + wt + i * DW;
        if (q < last) put(pk[i], vv[i]);
      }
      if (first + TC_NQ * DW < last) {   // denser than TC_NQ*DW nonzeros per tile: the rest straight from memory
        const int sidx = kb * g.mb + mbi;
        const uint16_t* ri = p.sl.tcoff + sidx * cap;
        const float* va = p.sl.values + sidx * cap;
#pragma unroll 2
        for (int q = first + wt + TC_NQ * DW; q < last; q += DW) put((uint32_t)__ldg(ri + q), __ldg(va + q));
      }
      fence_proxy_async();       // generic-proxy writes -> visible to the tensor core's async-proxy reads
      __syncwarp();
      if (0 == lane) mbar_arrive(&a_ready[h]);
      if constexpr (HIST) {
        if (1 == h) {            // this k-block's positions become the history its successor clears
          n_prev = last - first;
#pragma unroll
          for (int i = 0; i < TC_NQ; ++i) hk[i] = pk[i];
        }
      }
      if (1 == h && kb + 1 < g.kb) fetch(kb + 1);   // registers are free again: next k-block's nonzeros, consumed a step later
      }
      // (2) the two B chunks of this step: b_lo = b - trunc_tf32(b), same (swizzled) addresses
      if (do_split) {
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        const int c = 2 * t + j, s = c % TC_NB;
        mbar_wait(&b_full[s], (c / TC_NB) & 1);
        const uint4* src = (const uint4*)(smem + TC_SMEM_B + s * 2 * TC_B_CHUNK);
        uint4* dst = (uint4*)(smem + TC_SMEM_B + s * 2 * TC_B_CHUNK + TC_B_CHUNK);
#pragma unroll
        for (int i = 0; i < TC_B_CHUNK / 16 / DW; ++i) {
          const uint4 b = src[wt + i * DW];
          uint4 l;
          l.x = __float_as_uint(__uint_as_float(b.x) - __uint_as_float(b.x & 0xFFFFE000u));
          l.y = __float_as_uint(__uint_as_float(b.y) - __uint_as_float(b.y & 0xFFFFE000u));
          l.z = __float_as_uint(__uint_as_float(b.z) - __uint_as_float(b.z & 0xFFFFE000u));
          l.w = __float_as_uint(__uint_as_float(b.w) - __uint_as_float(b.w & 0xFFFFE000u));
          dst[wt + i * DW] = l;
        }
        fence_proxy_async();
        __syncwarp();
        if (0 == lane) mbar_arrive(&b_split[s]);
      }
      }
      // (3) drain the previous k-block's accumulator while this k-block's MMAs run
      if (0 == h && kb > 0) drain(kb - 1);
    }
    drain(g.kb - 1);
    // (4) epilogue: + beta*C.  C stored m x n: 16-byte streaming stores along the thread's row; C stored n x m
    // (transc = 'T'): the 32 lanes of a warp hold 32 consecutive m, so every store instruction is one full line
    const size_t crow = (size_t)(mbi * g.bm + ml0 + row - p.row_origin);
    if (row < tile_rows) {
      if (p.transc) {
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          const int col = n0 + cgrp + j;
          if (col < p.ncols) {
            float* dst = p.c + (size_t)col * p.ldc + crow;
            *dst = (0.f != p.beta) ? fmaf(p.beta, *dst, run[j]) : run[j];
          }
        }
      }
      else {
        float* dst = p.c + crow * p.ldc + n0 + cgrp;
#pragma unroll
        for (int j = 0; j < 32; j += 4) {
          const int col = n0 + cgrp + j;
          float4 o = make_float4(run[j], run[j + 1], run[j + 2], run[j + 3]);
          if (col + 3 < p.ncols) {
            if (0.f != p.beta) {
              const float4 cin = *(const float4*)(dst + j);
              o.x = fmaf(p.beta, cin.x, o.x); o.y = fmaf(p.beta, cin.y, o.y); o.z = fmaf(p.beta, cin.z, o.z); o.w = fmaf(p.beta, cin.w, o.w);
            }
            st_global_cs_f4(dst + j, o);
          }
          else {
            const float e[4] = { o.x, o.y, o.z, o.w };
#pragma unroll
            for (int t2 = 0; t2 < 4; ++t2) if (col + t2 < p.ncols) dst[j + t2] = (0.f != p.beta) ? fmaf(p.beta, dst[j + t2], e[t2]) : e[t2];
          }
        }
      }
    }
    tc_fence_before();
  }
  __syncthreads();
  if (1 == warp) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;\n" ::"r"(tmem_d), "r"(256) : "memory");
  }
}

bool make_tensor_map_2d_sw128(CUtensorMap* map, const void* base, int elem_bytes, unsigned long long cols, unsigned long long rows,
                              unsigned long long row_pitch_bytes, unsigned box_cols, unsigned box_rows, bool atom32);

// returns false when the panel does not qualify (caller falls back to the CUDA-core kernels)
bool launch_compute_tc(const ComputeArgs& a, cudaStream_t stream)
{
  if (a.is_bf16) return false;
  if (!a.transc && (0 != ((uintptr_t)a.c & 15) || 0 != (a.ldc & 3))) return false;
  CUtensorMap map;
  if (a.transb) {   // B stored n x k: inner dimension k, box 32 k x 128 n, plain 128-byte swizzle
    if (!make_tensor_map_2d_sw128(&map, a.b, 4, (unsigned long long)a.g.k, (unsigned long long)a.ncols, (unsigned long long)a.ldb * 4, 32, TC_BN, false)) return false;
  }
  else if (!make_tensor_map_2d_sw128(&map, a.b, 4, (unsigned long long)a.ncols, (unsigned long long)a.g.k, (unsigned long long)a.ldb * 4, 32, TC_KC, true)) return false;
  // performance-only choice (every instantiation is complete): the host's estimate is one call old at most
  const bool sparse_variant = a.density_hint >= 0.f && a.density_hint < 0.25f;
  const bool image = 0 != a.dense_valid && 0 != a.sl.dense;   // the slicing pass left the A image: nothing to rebuild
  if (!image && 0 == a.aux_valid) return false;   // neither the image nor the per-nonzero words: the CUDA-core kernels multiply these slices
  const void* kern = image ? (const void*)spmdm_compute_tc_kernel<16, false, true>
                   : (sparse_variant ? (const void*)spmdm_compute_tc_kernel<8, true, false> : (const void*)spmdm_compute_tc_kernel<16, false, false>);
  ensure_smem_optin(kern, TC_SMEM_BYTES);
  const int tiles_per_mb = (a.g.bm + TC_BM - 1) / TC_BM;
  const dim3 grid((unsigned)((a.ncols + TC_BN - 1) / TC_BN), (unsigned)(a.mb_count * tiles_per_mb), 1);
  count_launch(1);
  note_compute_kernel(image ? "spmdm_compute_tc_kernel (dense image)" : "spmdm_compute_tc_kernel");
  if (image) spmdm_compute_tc_kernel<16, false, true><<<grid, TC_THREADS, TC_SMEM_BYTES, stream>>>(map, a);
  else if (sparse_variant) spmdm_compute_tc_kernel<8, true, false><<<grid, TC_THREADS, TC_SMEM_BYTES, stream>>>(map, a);
  else spmdm_compute_tc_kernel<16, false, false><<<grid, TC_THREADS, TC_SMEM_BYTES, stream>>>(map, a);
  XB_CUDA(cudaGetLastError());
  return true;
}

}  // namespace xb
