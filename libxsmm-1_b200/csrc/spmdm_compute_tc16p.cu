// K4p: CTA-pair (tcgen05 cta_group::2), persistent tensor-core kernel of the spmdm compute step for bf16 inputs.
//
//   C[256 rows, 256 cols] = beta*C + sum_kb densify(slices(kb, rows))[256 x 128] * B[kb*128 .. +128, 256 cols]
//
// What bounded the single-CTA kernel this one replaced (K4h, 164 us for 4096^3 against 93 us here; measured with its
// stages switched off one at a time): B travels L2 -> SM once per 128 output rows (1.07 GB for 4096^3, 8.4 TB/s at the 128 us the bare
// MMA + TMA pipeline needs), the zero-fill of the A tile competes with the operand reads for shared memory, and
// the epilogue of a tile is not overlapped with anything.  This kernel changes all three:
//   * two CTAs of one TPC share every MMA (M = 256: 128 rows each, N = 256: each CTA stages 128 columns of B).
//     B crosses L2 -> SM once per 256 rows and each SM writes / reads half the B bytes.
//   * persistent: one CTA pair per TPC walks over its tiles; the accumulator is double buffered in TMEM
//     (2 x 256 columns), so the epilogue warps drain tile i while the tensor core works on tile i + 1.
//   * the A tile is never zero-filled: a worker thread owns one row, remembers (in shared memory) where it put
//     the nonzeros of the k-block that used the buffer before and clears exactly those before it writes the new
//     ones.  No synchronisation among the workers; at 1 % density that is ~1.3 stores per row and k-block
//     instead of 32 KiB of zero-fill.
// Roles per CTA (14 warps): warp 0 TMA producer, warp 1 MMA issuer (leader CTA only) and TMEM owner, warps 2-9
// densify (two groups taking k-blocks in turn, thread = row), warps 10-13 epilogue (warp % 4 = TMEM lane quarter).
// Like the fp32 branch this kernel keeps the 1e-2 contract of the bf16 path, not the reference's rounding sequence;
// LIBXSMM_B200_SPMDM_TC=0 selects the order-preserving CUDA-core kernels.
#include "common.cuh"
#include "tc_common.cuh"
#include <cstdlib>

namespace xb {

constexpr int P_BM = 128;                       // rows per CTA
constexpr int P_BN = 256;                       // columns per pair tile
constexpr int P_BNH = 128;                      // columns of B staged per CTA
constexpr int P_KH = 64;                        // k per stage = one 128-byte swizzle row of bf16
constexpr int P_NG = 2;                         // worker groups (four warps each) taking k-blocks in turn
constexpr int P_NB = 6;                         // B stages
constexpr int P_NA = 4;                         // A k-block buffers (two 64-k halves each); = 2 * P_NG: a worker's register set always meets the same buffer
constexpr int P_NQ = 4;                         // nonzeros per thread and k-block kept in registers (4 x 128 per tile: 3 % density)
constexpr int P_A_HALF = P_BM * 128;            // 16 KiB
constexpr int P_A_BUF = 2 * P_A_HALF;           // 32 KiB
constexpr int P_B_STAGE = P_KH * P_BNH * 2;     // 16 KiB
constexpr int P_THREADS = (2 + 4 * P_NG + 4) * 32;
constexpr int P_SMEM_A = 0;
constexpr int P_SMEM_B = P_SMEM_A + P_NA * P_A_BUF;
constexpr int P_SMEM_BAR = P_SMEM_B + P_NB * P_B_STAGE;
static_assert(P_NA == 2 * P_NG, "register set <-> A buffer pairing");
constexpr int P_SMEM_BYTES = P_SMEM_BAR + 256;

struct PairTile { int mbi, ml0, rows, n0; };

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(P_THREADS, 1)
spmdm_compute_tc16p_kernel(const __grid_constant__ CUtensorMap tmB, const ComputeArgs p)
{
  extern __shared__ __align__(1024) unsigned char smem[];
  uint64_t* bar = (uint64_t*)(smem + P_SMEM_BAR);
  uint64_t* b_full = bar;                   // [NB] leader: both halves of the B stage landed
  uint64_t* b_free = b_full + P_NB;         // [NB] both: MMAs that read the stage have completed
  uint64_t* a_ready = b_free + P_NB;        // [NA] leader: the workers of both CTAs built the k-block
  uint64_t* a_free = a_ready + P_NA;        // [NA] both: MMAs that read the k-block have completed
  uint64_t* acc_full = a_free + P_NA;       // [2]  both: all MMAs of the tile have completed
  uint64_t* acc_empty = acc_full + 2;       // [2]  leader: the epilogue warps of both CTAs drained the accumulator
  uint32_t* tmem_slot = (uint32_t*)(acc_empty + 2);

  const Geom& g = p.g;
  if (p.tc_twin > 0 || 2 == p.sp_guard) {    // the twin / guard decision reads the slices' counts
    pdl_wait();
    const unsigned long long total = xb_total_nnz(p.sl.slice_nnz, g.mb * g.kb);
    if (p.tc_twin > 0 && total < p.tc_min_nnz) return;      // uniform over the grid
    if (2 == p.sp_guard && total <= p.sp_max_nnz) return;   // the structured-sparse kernel enqueued in front of this one has multiplied
  }
  const int tid = (int)threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t rank = cluster_rank();
  const int pair = (int)blockIdx.x >> 1, npairs = (int)gridDim.x >> 1;
  const int tiles_per_mb = (g.bm + P_BM - 1) / P_BM;
  const int ctiles_m = p.mb_count * tiles_per_mb;
  const int pair_m = (ctiles_m + 1) >> 1;
  const int n_tiles = (p.ncols + P_BN - 1) / P_BN;
  const int total = pair_m * n_tiles;
  const int nkb = g.kb;
  const uint32_t sbase = smem_u32(smem);

  auto tile_of = [&](int idx) -> PairTile {
    PairTile t;
    const int ct = 2 * (idx % pair_m) + (int)rank;
    t.n0 = (idx / pair_m) * P_BN;
    t.mbi = p.mb_first + ct / tiles_per_mb;
    t.ml0 = (ct % tiles_per_mb) * P_BM;
    t.rows = 0;
    if (ct < ctiles_m) t.rows = max(0, min(P_BM, min(g.bm, g.m - t.mbi * g.bm) - t.ml0));
    return t;
  };

  // Work list of this pair: q full tiles, then -- when the remaining tiles are at most half as many as the pairs --
  // one HALF tile (128 of the 256 columns), so that no pair idles through the last round (4096^3 on 74 pairs:
  // 256 tiles = 3 rounds + 34 tiles -> 68 half tiles).  Measured gain 4 us of 108, not the 12 a half-cost round would
  // give: a half tile needs its k-blocks at twice the rate and is bound by the densifying warps, not the tensor core.
  const int wq = total / npairs, wrem = total - wq * npairs;
  const bool wsplit = !p.transb && wrem > 0 && 2 * wrem <= npairs;
  const int nwork = wq + ((wsplit ? (pair < 2 * wrem) : (pair < wrem)) ? 1 : 0);
  auto work_idx = [&](int i) -> int { return i < wq ? pair + i * npairs : wq * npairs + (wsplit ? (pair >> 1) : pair); };
  auto work_half = [&](int i) -> int { return (i < wq || !wsplit) ? -1 : (pair & 1); };

  if (0 == tid) {
#pragma unroll
    for (int i = 0; i < P_NB; ++i) { mbar_init(&b_full[i], 1); mbar_init(&b_free[i], 1); }
#pragma unroll
    for (int i = 0; i < P_NA; ++i) { mbar_init(&a_ready[i], 8); mbar_init(&a_free[i], 1); }
#pragma unroll
    for (int i = 0; i < 2; ++i) { mbar_init(&acc_full[i], 1); mbar_init(&acc_empty[i], 8); }
    mbar_fence_init();
  }
  if (1 == warp) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;\n" ::"r"(smem_u32(tmem_slot)), "r"(512) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;\n" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_d = *tmem_slot;
  if (p.tc_twin <= 0 && 2 != p.sp_guard) pdl_wait();       // barriers, tensor memory and the cluster hand-shake were set up while the kernel in front was still finishing

  if (0 == warp) {
    // ---------------- TMA producer: this CTA's 128 columns of every B stage ----------------
    if (0 == lane) {
      tma_prefetch_desc(&tmB);
      uint32_t gs = 0;
      for (int wi = 0; wi < nwork; ++wi) {
        const int idx = work_idx(wi), half = work_half(wi);
        const int n0 = (idx / pair_m) * P_BN + (half < 0 ? (int)rank * P_BNH : half * P_BNH + (int)rank * (P_BNH / 2));
        for (int t = 0; t < 2 * nkb; ++t, ++gs) {
          const uint32_t s = gs % P_NB, f = gs / P_NB;
          if (f > 0) mbar_wait(&b_free[s], (f - 1) & 1);
          if (0 == rank) mbar_arrive_expect_tx(&b_full[s], half < 0 ? 2 * P_B_STAGE : P_B_STAGE);
          const uint32_t lbar = map_to_cta(&b_full[s], 0);
          unsigned char* dst = smem + P_SMEM_B + s * P_B_STAGE;
          if (p.transb) tma_load_2d_pair(dst, &tmB, t * P_KH, n0, lbar);             // B stored n x k: 128 n-rows x 64 k
          else {
            tma_load_2d_pair(dst, &tmB, n0, t * P_KH, lbar);                         // 64 k-rows x 64 columns
            if (half < 0) tma_load_2d_pair(dst + P_KH * 128, &tmB, n0 + 64, t * P_KH, lbar);
          }
        }
      }
    }
  }
  else if (1 == warp) {
    // ---------------- MMA issuer (leader CTA) ----------------
    if (0 == rank && 0 == lane) {
      // D = F32, A = B = BF16, A K-major, B MN-major ('N') or K-major ('T'), N = 256, M = 256 (pair)
      const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((p.transb ? 0u : 1u) << 16) | ((uint32_t)(P_BN >> 3) << 17) | ((uint32_t)((2 * P_BM) >> 4) << 24);
      const uint32_t b_kstep = p.transb ? 32u : 2048u, b_lbo = p.transb ? 16u : (uint32_t)(P_KH * 128), b_sbo = 1024u;
      uint32_t gs = 0, gk = 0, it = 0;
      for (int wi = 0; wi < nwork; ++wi, ++it) {
        const uint32_t acc = it & 1;
        // a half tile is the same instruction with N = 128: each CTA stages one 64-column block
        const uint32_t idesc_w = (work_half(wi) < 0) ? idesc : ((idesc & ~(0x3Fu << 17)) | ((uint32_t)(P_BNH >> 3) << 17));
        if (it >= 2) mbar_wait(&acc_empty[acc], ((it >> 1) - 1) & 1);
        tc_fence_after();
        const uint32_t tacc = tmem_d + acc * P_BN;
        for (int kbi = 0; kbi < nkb; ++kbi, ++gk) {
          const uint32_t j = gk % P_NA;
          mbar_wait(&a_ready[j], (gk / P_NA) & 1);
#pragma unroll
          for (int h = 0; h < 2; ++h, ++gs) {
            const uint32_t s = gs % P_NB;
            mbar_wait(&b_full[s], (gs / P_NB) & 1);
            tc_fence_after();
            const uint32_t a_base = sbase + P_SMEM_A + j * P_A_BUF + h * P_A_HALF;
            const uint32_t b_base = sbase + P_SMEM_B + s * P_B_STAGE;
#pragma unroll
            for (int ks = 0; ks < 4; ++ks) {
              const uint64_t da = tc_smem_desc(a_base + ks * 32, 16, 1024, 2);
              const uint64_t db = tc_smem_desc(b_base + ks * b_kstep, b_lbo, b_sbo, 2);
              tc_mma_bf16_pair(tacc, da, db, idesc_w, (kbi > 0 || h > 0 || ks > 0) ? 1u : 0u);
            }
            tc_commit_pair(&b_free[s]);
          }
          tc_commit_pair(&a_free[j]);
        }
        tc_commit_pair(&acc_full[acc]);
      }
    }
  }
  else if (warp < 2 + 4 * P_NG) {
    // ---------------- workers: group grp (128 threads) builds k-blocks grp, grp + NG, ... ----------------
    // The nonzeros of the tile's k-block are one contiguous run of the slice (rows are stored in order); thread wt
    // takes entries wt, wt + 128, ...: at 1 % density that is two shared-memory stores per warp instruction slot
    // instead of one slot per nonzero of the longest row.
    const int grp = (warp - 2) >> 2;
    const int wt = (tid - 64) & (P_BM - 1);
    const size_t cap = (size_t)g.bm * g.bk;
    auto addr_of = [&](unsigned char* abuf, uint32_t w) -> uint16_t* {
      return (uint16_t*)(abuf + ((w >> 1) & 0x4000u) + ((w & 0x1FFFu) << 1));   // bit 15 = half (16 KiB apart), bits 0..12 = (offset inside the half) >> 1
    };
    const uint32_t lead_ready0 = map_to_cta(&a_ready[0], 0);
    // Cursor over this group's k-blocks, in the order the tensor core consumes them.  Row pointers are loaded
    // four group-steps ahead, the nonzeros two (raw registers, not touched until the step that uses them): no
    // global-memory latency sits between a buffer being released and being handed back.
    int c_wi = 0, c_kb = grp, c_rows = 0, c_sidx = 0;
    const uint16_t* c_ro = p.sl.rowidx;
    auto seat = [&]() {                // (idx, kb) -> pointers; the divisions run once per tile
      c_rows = 0; c_ro = p.sl.rowidx; c_sidx = 0;
      if (c_wi < nwork) {
        const PairTile t = tile_of(work_idx(c_wi));
        c_sidx = c_kb * g.mb + t.mbi;
        c_ro = p.sl.rowidx + (size_t)c_sidx * (g.bm + 1) + t.ml0;
        c_rows = t.rows;
      }
    };
    auto advance = [&]() {
      c_kb += P_NG;
      if (c_kb < nkb) { c_sidx += P_NG * g.mb; c_ro += (size_t)P_NG * g.mb * (g.bm + 1); }
      else {
        while (c_kb >= nkb && c_wi < nwork) { c_kb -= nkb; ++c_wi; }
        seat();
      }
    };
    while (c_kb >= nkb && c_wi < nwork) { c_kb -= nkb; ++c_wi; }
    seat();
    struct Ptr { int pf, sidx; };
    // rw: the slicing kernel's word per nonzero (xb_tc16_pack: bf16 value << 16 | half << 15 | position), hw: the
    // words this thread put into the buffer last time
    struct Raw { int sidx, first, last, n_old; uint32_t rw[P_NQ]; uint32_t hw[P_NQ]; };
    auto fetch_ptrs = [&](Ptr& P) {            // issue only: ONE load instruction, lanes 0..2 fetch the three pointers
      P.pf = 0; P.sidx = c_sidx;
      if (c_rows > 0 && lane < 3) P.pf = (int)__ldg(c_ro + (0 == lane ? 0 : (1 == lane ? c_rows : c_rows - 1)));
      advance();
    };
    auto fetch = [&](Raw& R, Ptr& P) {         // consumes the pointers, issues the nonzero loads and the next pointers
      const int pf = __shfl_sync(0xffffffffu, P.pf, 0), pl = __shfl_sync(0xffffffffu, P.pf, 1), pm = __shfl_sync(0xffffffffu, P.pf, 2);
      R.sidx = P.sidx; R.first = pf;
      R.last = (pl < pf) ? pm : pl;            // wrapped u16 counter of a full slice: the last row reads as empty
      const uint32_t* pw = p.sl.tcpk + R.sidx * cap;
#pragma unroll
      for (int i = 0; i < P_NQ; ++i) {
        if (R.first + i * P_BM >= R.last) break;           // uniform
        const int q = R.first + wt + i * P_BM;
        R.rw[i] = 0;
        if (q < R.last) R.rw[i] = __ldg(pw + q);
      }
      fetch_ptrs(P);
    };
    const uint32_t gk_end = (uint32_t)nwork * (uint32_t)nkb;
    auto step = [&](uint32_t gk, Raw& R, Ptr& P) {
      if (gk >= gk_end) return;
      const uint32_t j = gk % P_NA;
      if (gk >= P_NA) mbar_wait(&a_free[j], ((gk / P_NA) - 1) & 1);
      unsigned char* abuf = smem + P_SMEM_A + j * P_A_BUF;
      // clear what the previous k-block left in the buffer (same register set: NA = 2 * NG); a dense one is wiped
      if (R.n_old > P_NQ * P_BM) {
        uint4* z = (uint4*)abuf;
#pragma unroll
        for (int i = 0; i < P_A_BUF / 16 / P_BM; ++i) z[wt + i * P_BM] = make_uint4(0, 0, 0, 0);
      }
      else {
#pragma unroll
        for (int i = 0; i < P_NQ; ++i) {
          if (i * P_BM >= R.n_old) break;                  // uniform
          if (wt + i * P_BM < R.n_old) *addr_of(abuf, R.hw[i]) = 0;
        }
      }
      asm volatile("bar.sync %0, %1;\n" ::"r"(1 + grp), "n"(P_BM) : "memory");   // another thread may write where this one cleared
      // this k-block's nonzeros
      const int n = R.last - R.first;
#pragma unroll
      for (int i = 0; i < P_NQ; ++i) {
        if (i * P_BM >= n) break;                          // uniform
        if (wt + i * P_BM < n) {
          const uint32_t w = R.rw[i];
          *addr_of(abuf, w) = (uint16_t)(w >> 16);
          R.hw[i] = w;
        }
      }
      R.n_old = n;
      if (n > P_NQ * P_BM) {         // denser than NQ * 128 nonzeros per tile and k-block: the rest straight from memory
        const uint32_t* pw = p.sl.tcpk + R.sidx * cap;
#pragma unroll 4
        for (int q = R.first + wt + P_NQ * P_BM; q < R.last; q += P_BM) { const uint32_t w = __ldg(pw + q); *addr_of(abuf, w) = (uint16_t)(w >> 16); }
      }
      fence_proxy_async();
      __syncwarp();
      if (0 == lane) mbar_arrive_cluster(lead_ready0 + j * 8);
      fetch(R, P);                   // after the hand-over: refill this set for the step after next
    };
    Ptr pa, pb; Raw ra, rb;
    ra.n_old = 0; rb.n_old = 0;
#pragma unroll
    for (int i = 0; i < P_NQ; ++i) { ra.hw[i] = 0; rb.hw[i] = 0; }
    fetch_ptrs(pa); fetch_ptrs(pb);            // k-blocks 0 and 1 of this group
    // The A buffers start out zero and are only ever patched.  Each group wipes the two buffers it owns while its
    // first loads are in flight (and while the TMA producer is already filling the B ring).
#pragma unroll
    for (int b = 0; b < 2; ++b) {
      uint4* z = (uint4*)(smem + P_SMEM_A + (grp + b * P_NG) * P_A_BUF);
#pragma unroll 4
      for (int i = 0; i < P_A_BUF / 16 / P_BM; ++i) z[wt + i * P_BM] = make_uint4(0, 0, 0, 0);
    }
    asm volatile("bar.sync %0, %1;\n" ::"r"(1 + grp), "n"(P_BM) : "memory");
    fetch(ra, pa); fetch(rb, pb);              // their nonzeros; pa / pb now hold the pointers of k-blocks 2 and 3
    for (uint32_t gk = (uint32_t)grp; gk < gk_end; gk += 2 * P_NG) {
      step(gk, ra, pa);
      step(gk + P_NG, rb, pb);
    }
  }
  else {
    // ---------------- epilogue: warp owns TMEM lanes 32*(warp % 4) .. +31 of this CTA ----------------
    const int quarter = warp & 3;
    const int row = quarter * 32 + lane;
    const uint32_t lead_empty0 = map_to_cta(&acc_empty[0], 0);
    uint32_t it = 0;
    for (int wi = 0; wi < nwork; ++wi, ++it) {
      PairTile t = tile_of(work_idx(wi));
      const int half = work_half(wi), ncw = half < 0 ? P_BN : P_BNH;
      if (half > 0) t.n0 += P_BNH;
      const uint32_t acc = it & 1;
      mbar_wait(&acc_full[acc], (it >> 1) & 1);
      tc_fence_after();
      const size_t crow = (size_t)(t.mbi * g.bm + t.ml0 + row - p.row_origin);
#pragma unroll 1
      for (int cb = 0; cb < ncw; cb += 32) {
        uint32_t v[32];
        tc_ld32(tmem_d + acc * P_BN + ((uint32_t)(quarter * 32) << 16) + (uint32_t)cb, v);
        if (row < t.rows) {
          if (p.transc) {
#pragma unroll
            for (int jj = 0; jj < 32; ++jj) {
              const int col = t.n0 + cb + jj;
              if (col < p.ncols) {
                float* dst = p.c + (size_t)col * p.ldc + crow;
                *dst = (0.f != p.beta) ? fmaf(p.beta, *dst, __uint_as_float(v[jj])) : __uint_as_float(v[jj]);
              }
            }
          }
        }
        if (!p.transc) {   // thread = row: 16-byte streaming stores (measured slower: a lane-transposed line-per-instruction variant, +6 %; 32-byte STG.256 stores, +4 %)
          if (row < t.rows) {
            float* dst = p.c + crow * p.ldc + t.n0 + cb;
#pragma unroll
            for (int jj = 0; jj < 32; jj += 4) {
              const int col = t.n0 + cb + jj;
              float4 o = make_float4(__uint_as_float(v[jj]), __uint_as_float(v[jj + 1]), __uint_as_float(v[jj + 2]), __uint_as_float(v[jj + 3]));
              if (col + 3 < p.ncols) {
                if (0.f != p.beta) {
                  const float4 cin = *(const float4*)(dst + jj);
                  o.x = fmaf(p.beta, cin.x, o.x); o.y = fmaf(p.beta, cin.y, o.y); o.z = fmaf(p.beta, cin.z, o.z); o.w = fmaf(p.beta, cin.w, o.w);
                }
                st_global_cs_f4(dst + jj, o);
              }
              else {
                const float e[4] = { o.x, o.y, o.z, o.w };
#pragma unroll
                for (int t2 = 0; t2 < 4; ++t2) if (col + t2 < p.ncols) dst[jj + t2] = (0.f != p.beta) ? fmaf(p.beta, dst[jj + t2], e[t2]) : e[t2];
              }
            }
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (0 == lane) mbar_arrive_cluster(lead_empty0 + acc * 8);
    }
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();      // the peer's shared memory and barriers stay alive until every MMA and remote arrive has landed
  if (1 == warp) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;\n" ::"r"(tmem_d), "r"(512) : "memory");
  }
}

bool make_tensor_map_2d_sw128(CUtensorMap* map, const void* base, int elem_bytes, unsigned long long cols, unsigned long long rows,
                              unsigned long long row_pitch_bytes, unsigned box_cols, unsigned box_rows, bool atom32);

// returns false when the panel does not qualify (caller falls back to the CUDA-core kernels)
bool launch_compute_tc16p(const ComputeArgs& a, cudaStream_t stream)
{
  if (0 == a.aux_valid) return false;   // these kernels rebuild A from the packed per-nonzero words the slicing pass writes
  if (!a.is_bf16) return false;
  if (!a.transc && (0 != ((uintptr_t)a.c & 15) || 0 != (a.ldc & 3))) return false;
  CUtensorMap map;
  if (a.transb) {
    if (!make_tensor_map_2d_sw128(&map, a.b, 2, (unsigned long long)a.g.k, (unsigned long long)a.ncols, (unsigned long long)a.ldb * 2, 64, P_BNH, false)) return false;
  }
  else if (!make_tensor_map_2d_sw128(&map, a.b, 2, (unsigned long long)a.ncols, (unsigned long long)a.g.k, (unsigned long long)a.ldb * 2, 64, P_KH, false)) return false;
  ensure_smem_optin((const void*)spmdm_compute_tc16p_kernel, P_SMEM_BYTES);
  const int pairs_max = device_sm_count() / 2 > 0 ? device_sm_count() / 2 : 1;
  const int tiles_per_mb = (a.g.bm + P_BM - 1) / P_BM;
  const int pair_m = (a.mb_count * tiles_per_mb + 1) / 2;
  const int total = pair_m * ((a.ncols + P_BN - 1) / P_BN);
  if (total <= 0) return true;
  const int pairs = total < pairs_max ? total : pairs_max;
  count_launch(1);
  note_compute_kernel("spmdm_compute_tc16p_kernel");
  XB_CUDA(launch_pdl(spmdm_compute_tc16p_kernel, dim3(2u * (unsigned)pairs), dim3(P_THREADS), P_SMEM_BYTES, stream, map, a));   // may be scheduled while the slicing kernel drains (pdl_wait in the kernel)
  return true;
}

}  // namespace xb
