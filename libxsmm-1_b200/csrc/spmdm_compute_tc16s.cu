// K4s: the CTA-pair tensor-core kernel of the bf16 spmdm compute step on the 2:4 STRUCTURED-SPARSE tensor-core path
// (tcgen05.mma.sp.cta_group::2.kind::f16), for matrices that are sparse but not sparse enough for the CUDA-core kernels.
//
//   C[256 rows, 256 cols] = beta*C + sum_kb compress(slices(kb, rows))[256 x 64 kept] * B[kb*128 .. +128, 256 cols]
//
// K4p (spmdm_compute_tc16p.cu) multiplies the densified A tile: at 1 % density 99 % of what the tensor core multiplies is
// zero, and the kernel sits at the floor of that formulation (137 GFLOP of dense work for 4096^3).  The sparse tensor-core
// instruction takes A as two kept elements of every four consecutive k plus a 4-bit nibble naming their positions, and
// runs K = 32 in the time the dense one runs K = 16 (measured: 181 against 173 clocks per M = 256, N = 256 instruction,
// tools/umma_probe/probe_sp_rate.cu).  A random matrix of a few per cent density almost is such a matrix: of the 4.2 M
// groups of 4096^2 at 1 % about 17 hold three or four nonzeros.  So:
//   * the slicing kernel (K1x) writes one more word per nonzero (SliceArena::tcsp): where it goes in the COMPRESSED A
//     tile, the 16-bit metadata word of its row's 16-k span, and whether it is an OVERFLOW entry (third / fourth nonzero
//     of its group);
//   * the workers of this kernel patch the compressed tile (128 rows x 64 kept bf16 = 16 KiB per 128-k block, half of
//     K4p's) and a 2 KiB image of the block's metadata in shared memory (tensor-memory lane L at byte 16 L); the issuing
//     thread copies the image into four tensor-memory columns with tcgen05.cp right in front of the block's four MMAs.
//     Layout and nibble semantics were pinned with tools/umma_probe/probe_sp.cu;
//   * the overflow entries are added by the epilogue thread that owns the row (value * B[k, :] onto the accumulator it
//     drains, slices in ascending k-block, entries in ascending k): deterministic, correct at ANY density (it just gets
//     slow when many groups overflow, which is why the host only picks this kernel for matrices its density estimate puts
//     below kSpMaxDensity).  A first version did this in a second kernel: 16-27 us for a handful of rows.
// One ring slot per k-block holds everything the tensor core needs for it (A tile, metadata images, this CTA's 128 k x 128
// columns of B): the issuing thread waits once and commits once per k-block -- with separate A and B rings (three waits,
// three commits per k-block) it could not keep the instruction queue fed at 181 clocks per instruction (87 -> 78 us).
// The accumulator is double buffered in tensor memory like K4p's (a first version with one accumulator and a separate
// metadata ring ran every SM through its store phase at the same time: 30 us of HBM-write-bound epilogues for 4096^3), so
// tensor memory is full; the metadata columns of a tile are the first 16 columns of the accumulator it does NOT use, once
// the epilogue of the previous tile has read them.  C leaves through TMA boxes when it is only written (the epilogue's
// scattered 16-byte stores held up the workers' loads and stores in the load / store unit: 97 -> 88 us).
// Roles per CTA (14 warps): warp 0 TMA producer, warp 1 MMA issuer (leader CTA only) and TMEM owner, warps 2-9 workers
// (four groups of two warps taking k-blocks in turn, one slot each: with the metadata going through tcgen05.cp a group need
// not cover the four tensor-memory lane quarters, and 64 waiters per slot wake faster than 128: 68.5 -> 65.9 us), warps 10-13 epilogue.  Same 1e-2 contract as K4p (observed 1e-6).
// LIBXSMM_B200_K4S_DEBUG (developer timing aid, results are wrong when set): 1 no worker work, 2 no B loads, 4 no C
// stores, 16 no tensor-core instructions.  What they show on C2 (78 us): without workers 70, without stores 73, without
// MMAs 61, the bare hand-shake skeleton 48 -- the ring of four slots is one slot short of hiding the round trip
// commit -> waiters wake -> patch -> remote arrive, and shared memory (208 of 227 KiB in the ring) has no room for a fifth.
#include "common.cuh"
#include "tc_common.cuh"
#include <cstdlib>

namespace xb {

constexpr int S_BM = 128;                       // rows per CTA
constexpr int S_BN = 256;                       // columns per pair tile
constexpr int S_BNH = 128;                      // columns of B staged per CTA
constexpr int S_KB = 128;                       // k per ring slot = one k-block of the slices
constexpr int S_NG = 4;                         // worker groups taking k-blocks in turn
constexpr int S_GW = 2;                         // warps per worker group (the metadata goes to tensor memory by tcgen05.cp: a group need not cover the four lane quarters)
constexpr int S_GT = S_GW * 32;                 // threads per worker group
constexpr int S_NA = S_NG;                      // ring slots: every worker group owns one (A tile, metadata image, B stage)
constexpr int S_NQ = 4;                         // nonzeros per thread and k-block kept in registers
constexpr int S_NE = 4;                         // epilogue warps (one per TMEM lane quarter)
constexpr int S_A_BUF = S_BM * 128;             // 16 KiB: 128 rows x 64 kept bf16
constexpr int S_META = S_BM * 16;               // 2 KiB: per TMEM lane four 32-bit metadata columns
constexpr int S_B_STAGE = S_KB * S_BNH * 2;     // 32 KiB: two column blocks of [128 k x 64 columns]
constexpr int S_THREADS = (2 + S_GW * S_NG + S_NE) * 32;
constexpr int S_SMEM_A = 0;
constexpr int S_SMEM_B = S_SMEM_A + S_NA * S_A_BUF;
constexpr int S_SMEM_META = S_SMEM_B + S_NA * S_B_STAGE;
constexpr int S_SMEM_STAGE = S_SMEM_META + 2 * S_NA * S_META;         // per epilogue warp a [32 rows x 32 columns] fp32 box for the TMA store of C
constexpr int S_STAGE = 32 * 128;
constexpr int S_SMEM_BAR = S_SMEM_STAGE + S_NE * S_STAGE;
constexpr int S_NOVF = 4;                       // overflow entries of a row an epilogue thread keeps in registers
static_assert(0 == (S_SMEM_STAGE & 1023), "SWIZZLE_128B boxes sit on 1 KiB boundaries");
static_assert(S_NE * (S_BN / 32) * S_STAGE <= S_SMEM_META, "the last tile's C boxes fit in the (then idle) A / B ring");
constexpr int S_SMEM_BYTES = S_SMEM_BAR + 256;
// Tensor memory: two accumulators of 256 columns fill it.  The metadata ring of a tile (4 columns per k-block buffer) lives
// in the first columns of the accumulator the tile does NOT accumulate into: that accumulator belongs to the epilogue of the
// previous tile, which drains those columns first and says so (meta_free); the next tile's first MMA overwrites them only
// after this tile's MMAs, issued before it, have read them.
constexpr float kSpMaxDensity = 0.022f;         // measured crossover with K4p on 4096^3 (tools/crossover_sp.py): 0.5 % 70 / 95 us, 1 % 74 / 97, 2 % 90 / 101, 3 % 117 / 103 --
                                                // the workers' patching (three shared-memory stores per nonzero) and the overflow entries grow with the density

struct SpTile { int mbi, ml0, rows, n0; };

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(S_THREADS, 1)
spmdm_compute_tc16s_kernel(const __grid_constant__ CUtensorMap tmB, const __grid_constant__ CUtensorMap tmC, const int c_tma, const ComputeArgs p)
{
  extern __shared__ __align__(1024) unsigned char smem[];
  uint64_t* bar = (uint64_t*)(smem + S_SMEM_BAR);
  uint64_t* a_ready = bar;                  // [NA] leader: the slot is complete -- both B halves landed (bytes) and the workers of both CTAs built A and its metadata
  uint64_t* a_free = a_ready + S_NA;        // [NA] both: the MMAs that read the slot have completed
  uint64_t* acc_full = a_free + S_NA;       // [2]  both: all MMAs of the tile have completed
  uint64_t* acc_empty = acc_full + 2;       // [2]  leader: the epilogue warps of both CTAs drained the accumulator
  uint64_t* meta_free = acc_empty + 2;      // [1]  leader: the epilogue warps of both CTAs have read the columns the next tile's metadata goes to
  uint32_t* tmem_slot = (uint32_t*)(meta_free + 1);

  const Geom& g = p.g;
  if (p.tc_twin > 0 || p.sp_guard) {    // the twin / guard decision reads the slices' counts
    pdl_wait();
    const unsigned long long total = xb_total_nnz(p.sl.slice_nnz, g.mb * g.kb);
    if (p.tc_twin > 0 && total < p.tc_min_nnz) return;      // uniform over the grid
    if (p.sp_guard && total > p.sp_max_nnz) return;         // too dense for the overflow path: the dense kernel enqueued behind this one multiplies
  }
  const int tid = (int)threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t rank = cluster_rank();
  const int pair = (int)blockIdx.x >> 1, npairs = (int)gridDim.x >> 1;
  const int tiles_per_mb = (g.bm + S_BM - 1) / S_BM;
  const int ctiles_m = p.mb_count * tiles_per_mb;
  const int pair_m = (ctiles_m + 1) >> 1;
  const int n_tiles = (p.ncols + S_BN - 1) / S_BN;
  const int total = pair_m * n_tiles;
  const int nkb = g.kb;
  const uint32_t sbase = smem_u32(smem);

  auto tile_of = [&](int idx) -> SpTile {
    SpTile t;
    const int ct = 2 * (idx % pair_m) + (int)rank;
    t.n0 = (idx / pair_m) * S_BN;
    t.mbi = p.mb_first + ct / tiles_per_mb;
    t.ml0 = (ct % tiles_per_mb) * S_BM;
    t.rows = 0;
    if (ct < ctiles_m) t.rows = max(0, min(S_BM, min(g.bm, g.m - t.mbi * g.bm) - t.ml0));
    return t;
  };

  // work list of this pair: q full tiles, then (when the rest is at most half as many tiles as pairs) one HALF tile
  const int wq = total / npairs, wrem = total - wq * npairs;
  const bool wsplit = wrem > 0 && 2 * wrem <= npairs;
  const int nwork = wq + ((wsplit ? (pair < 2 * wrem) : (pair < wrem)) ? 1 : 0);
  auto work_idx = [&](int i) -> int { return i < wq ? pair + i * npairs : wq * npairs + (wsplit ? (pair >> 1) : pair); };
  auto work_half = [&](int i) -> int { return (i < wq || !wsplit) ? -1 : (pair & 1); };

  if (0 == tid) {
#pragma unroll
    for (int i = 0; i < S_NA; ++i) { mbar_init(&a_ready[i], 2 * S_GW + 1); mbar_init(&a_free[i], 1); }   // the worker warps of the group in both CTAs + the leader's producer (with the byte count)
#pragma unroll
    for (int i = 0; i < 2; ++i) { mbar_init(&acc_full[i], 1); mbar_init(&acc_empty[i], 2 * S_NE); }
    mbar_init(meta_free, 2 * S_NE);
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
  // everything above (barriers, tensor memory, cluster hand-shake) ran while the slicing kernel was still finishing: from here
  // on its output is read
  if (p.tc_twin <= 0 && !p.sp_guard) pdl_wait();

  if (0 == warp) {
    // ---------------- TMA producer: this CTA's 128 columns of every B stage ----------------
    if (0 == lane) {
      tma_prefetch_desc(&tmB);
      uint32_t gk = 0;
      for (int wi = 0; wi < nwork; ++wi) {
        const int idx = work_idx(wi), half = work_half(wi);
        const int n0 = (idx / pair_m) * S_BN + (half < 0 ? (int)rank * S_BNH : half * S_BNH + (int)rank * (S_BNH / 2));
        for (int kbi = 0; kbi < nkb; ++kbi, ++gk) {
          const uint32_t j = gk % S_NA, f = gk / S_NA;
          if (f > 0) mbar_wait(&a_free[j], (f - 1) & 1);
          if (p.debug_flags & 2) { if (0 == rank) mbar_arrive(&a_ready[j]); continue; }     // timing aid: no B loads
          if (0 == rank) mbar_arrive_expect_tx(&a_ready[j], half < 0 ? 2 * S_B_STAGE : S_B_STAGE);
          const uint32_t lbar = map_to_cta(&a_ready[j], 0);
          unsigned char* dst = smem + S_SMEM_B + j * S_B_STAGE;
          tma_load_2d_pair(dst, &tmB, n0, kbi * S_KB, lbar);                       // 128 k-rows x 64 columns
          if (half < 0) tma_load_2d_pair(dst + S_KB * 128, &tmB, n0 + 64, kbi * S_KB, lbar);
        }
      }
    }
  }
  else if (1 == warp) {
    // ---------------- MMA issuer (leader CTA) ----------------
    if (0 == rank && 0 == lane) {
      // sparse A, D = F32, A = B = BF16, A K-major (compressed), B MN-major, N = 256, M = 256 (pair)
      const uint32_t idesc = (1u << 2) | (1u << 4) | (1u << 7) | (1u << 10) | (1u << 16) | ((uint32_t)(S_BN >> 3) << 17) | ((uint32_t)((2 * S_BM) >> 4) << 24);
      uint32_t gk = 0;
      for (int wi = 0; wi < nwork; ++wi) {
        const uint32_t acc = (uint32_t)wi & 1u;
        const uint32_t idesc_w = (work_half(wi) < 0) ? idesc : ((idesc & ~(0x3Fu << 17)) | ((uint32_t)(S_BNH >> 3) << 17));
        if (wi >= 2) mbar_wait(&acc_empty[acc], (((uint32_t)wi >> 1) - 1u) & 1u);
        if (wi >= 1) mbar_wait(meta_free, (uint32_t)(wi - 1) & 1u);    // the epilogue of the previous tile has read the columns this tile's metadata goes to
        tc_fence_after();
        const uint32_t tacc = tmem_d + acc * S_BN, tmeta = tmem_d + (acc ^ 1u) * S_BN;
        for (int kbi = 0; kbi < nkb; ++kbi, ++gk) {
          const uint32_t j = gk % S_NA;
          mbar_wait(&a_ready[j], (gk / S_NA) & 1);
          tc_fence_after();
          const uint32_t a_base = sbase + S_SMEM_A + j * S_A_BUF, b_base = sbase + S_SMEM_B + j * S_B_STAGE;
          // the slot's metadata image (128 lanes x 16 bytes, lane L at byte 16 L) into its four tensor-memory columns, in both
          // CTAs; executes in order with the MMAs that follow
          if (!(p.debug_flags & 16)) {
            const uint64_t dm = tc_smem_desc(sbase + S_SMEM_META + (2u * j + ((gk / S_NA) & 1u)) * S_META, 16, 128, 0);
            asm volatile("tcgen05.cp.cta_group::2.128x128b [%0], %1;\n" ::"r"(tmeta + 4u * j), "l"(dm) : "memory");
          }
#pragma unroll
          for (int ks = 0; ks < 4; ++ks) {         // K = 32 (16 kept elements = 32 bytes of the compressed row) per instruction
            // the metadata of atom ks lives in column ks of the slot's four: the address names the even column, the
            // descriptor's selector bit the odd one
            const uint64_t da = tc_smem_desc(a_base + ks * 32, 16, 1024, 2);
            const uint64_t db = tc_smem_desc(b_base + ks * 4096, (uint32_t)(S_KB * 128), 1024, 2);
            if (!(p.debug_flags & 16)) tc_mma_bf16_sp_pair(tacc, da, db, tmeta + 4u * j + (uint32_t)(ks & 2), idesc_w | (uint32_t)(ks & 1), (kbi > 0 || ks > 0) ? 1u : 0u);
          }
          tc_commit_pair(&a_free[j]);
        }
        tc_commit_pair(&acc_full[acc]);
      }
    }
  }
  else if (warp < 2 + S_GW * S_NG) {
    // ---------------- workers: group grp (128 threads) builds k-blocks grp, grp + NG, ... ----------------
    const int grp = (warp - 2) / S_GW;
    const int wt = (tid - 64) % S_GT;
    const size_t cap = (size_t)g.bm * g.bk;
    const uint32_t lead_ready0 = map_to_cta(&a_ready[0], 0);
    // byte offset of the metadata word of (row, 16-k span) in the image (a lambda: calling the helper directly changes the SASS)
    auto meta_off = [](uint32_t pos) -> uint32_t { return xb_sp_meta_off(pos); };
    int c_wi = 0, c_kb = grp, c_rows = 0, c_sidx = 0;
    const uint16_t* c_ro = p.sl.rowidx;
    auto seat = [&]() {
      c_rows = 0; c_ro = p.sl.rowidx; c_sidx = 0;
      if (c_wi < nwork) {
        const SpTile t = tile_of(work_idx(c_wi));
        c_sidx = c_kb * g.mb + t.mbi;
        c_ro = p.sl.rowidx + (size_t)c_sidx * (g.bm + 1) + t.ml0;
        c_rows = t.rows;
      }
    };
    auto advance = [&]() {
      c_kb += S_NG;
      if (c_kb < nkb) { c_sidx += S_NG * g.mb; c_ro += (size_t)S_NG * g.mb * (g.bm + 1); }
      else {
        while (c_kb >= nkb && c_wi < nwork) { c_kb -= nkb; ++c_wi; }
        seat();
      }
    };
    while (c_kb >= nkb && c_wi < nwork) { c_kb -= nkb; ++c_wi; }
    seat();
    struct Ptr { int pf, sidx; };
    // rw: xb_tc16_pack word (the bf16 value in its upper half), sw: the structured-sparse word.  Two sets: the loads of a
    // k-block are issued two of this group's steps before they are used.  hs / n_old: what this thread put into the group's
    // slot the last time.
    struct Raw { int sidx, first, last; uint32_t rw[S_NQ]; uint32_t sw[S_NQ]; };
    uint32_t hs[S_NQ]; int n_old = 0;
    auto fetch_ptrs = [&](Ptr& P) {
      P.pf = 0; P.sidx = c_sidx;
      if (c_rows > 0 && lane < 3) P.pf = (int)__ldg(c_ro + (0 == lane ? 0 : (1 == lane ? c_rows : c_rows - 1)));
      advance();
    };
    auto fetch = [&](Raw& R, Ptr& P) {
      const int pf = __shfl_sync(0xffffffffu, P.pf, 0), pl = __shfl_sync(0xffffffffu, P.pf, 1), pm = __shfl_sync(0xffffffffu, P.pf, 2);
      R.sidx = P.sidx; R.first = pf;
      R.last = (pl < pf) ? pm : pl;            // wrapped u16 counter of a full slice: the last row reads as empty
      const uint32_t* pw = p.sl.tcpk + R.sidx * cap;
      const uint32_t* ps = p.sl.tcsp + R.sidx * cap;
#pragma unroll
      for (int i = 0; i < S_NQ; ++i) {
        if (R.first + i * S_GT >= R.last) break;           // uniform
        const int q = R.first + wt + i * S_GT;
        R.rw[i] = 0; R.sw[i] = 0;
        if (q < R.last) { R.rw[i] = __ldg(pw + q); R.sw[i] = __ldg(ps + q); }
      }
      fetch_ptrs(P);
    };
    const uint32_t gk_end = (uint32_t)nwork * (uint32_t)nkb;
    auto step = [&](uint32_t gk, Raw& R, Ptr& P) {
      if (gk >= gk_end) return;
      const uint32_t j = gk % S_NA;
      unsigned char* abuf = smem + S_SMEM_A + j * S_A_BUF;
      unsigned char* mimg = smem + S_SMEM_META + (2u * j + ((gk / S_NA) & 1u)) * S_META;
      const int n = R.last - R.first;
      const bool idle = 0 != (p.debug_flags & 1);      // timing aid: hand the slot over untouched
      // ---- while the tensor core still reads the slot: the k-block's metadata image.  Two images per slot: the copy of the
      // other one into tensor memory may still be in flight.  Stale metadata needs no clearing: a nibble whose two kept
      // elements are zero contributes nothing wherever it points.
      if (!idle) {
#pragma unroll
        for (int i = 0; i < S_NQ; ++i) {
          if (i * S_GT >= n) break;                          // uniform
          if (wt + i * S_GT < n) *(uint16_t*)(mimg + meta_off(R.sw[i] & 0x1FFFu)) = (uint16_t)(R.sw[i] >> 16);
        }
        if (n > S_NQ * S_GT) {         // denser than NQ * 64 nonzeros per tile and k-block: the rest straight from memory
          const uint32_t* ps = p.sl.tcsp + R.sidx * cap;
#pragma unroll 2
          for (int q = R.first + wt + S_NQ * S_GT; q < R.last; q += S_GT) { const uint32_t s = __ldg(ps + q); *(uint16_t*)(mimg + meta_off(s & 0x1FFFu)) = (uint16_t)(s >> 16); }
        }
      }
      // ---- the slot is ours once the MMAs of the k-block that used it have completed ----
      if (gk >= S_NA) mbar_wait(&a_free[j], ((gk / S_NA) - 1) & 1);
      if (!idle) {
        // clear the kept elements the previous k-block left behind (a dense one is wiped)
        if (n_old > S_NQ * S_GT) {
          uint4* z = (uint4*)abuf;
#pragma unroll
          for (int i = 0; i < S_A_BUF / 16 / S_GT; ++i) z[wt + i * S_GT] = make_uint4(0, 0, 0, 0);
        }
        else {
#pragma unroll
          for (int i = 0; i < S_NQ; ++i) {
            if (i * S_GT >= n_old) break;                    // uniform
            if (wt + i * S_GT < n_old) *(uint16_t*)(abuf + ((hs[i] & 0x1FFFu) << 1)) = 0;
          }
        }
        asm volatile("bar.sync %0, %1;\n" ::"r"(1 + grp), "n"(S_GT) : "memory");   // another thread may write where this one cleared
#pragma unroll
        for (int i = 0; i < S_NQ; ++i) {
          if (i * S_GT >= n) break;                          // uniform
          if (wt + i * S_GT < n) {
            const uint32_t s = R.sw[i];
            if (0 == (s & 0x8000u)) *(uint16_t*)(abuf + ((s & 0x1FFFu) << 1)) = (uint16_t)(R.rw[i] >> 16);   // overflow entries: the row's epilogue thread
            hs[i] = s;
          }
        }
        n_old = n;
        if (n > S_NQ * S_GT) {
          const uint32_t* pw = p.sl.tcpk + R.sidx * cap;
          const uint32_t* ps = p.sl.tcsp + R.sidx * cap;
#pragma unroll 2
          for (int q = R.first + wt + S_NQ * S_GT; q < R.last; q += S_GT) {
            const uint32_t w = __ldg(pw + q), s = __ldg(ps + q);
            if (0 == (s & 0x8000u)) *(uint16_t*)(abuf + ((s & 0x1FFFu) << 1)) = (uint16_t)(w >> 16);
          }
        }
        fence_proxy_async();
      }
      __syncwarp();
      if (0 == lane) mbar_arrive_cluster(lead_ready0 + j * 8);
      fetch(R, P);                   // after the hand-over: the k-block of this group's step after next
    };
    Ptr pa, pb; Raw ra, rb;
#pragma unroll
    for (int i = 0; i < S_NQ; ++i) hs[i] = 0;
    fetch_ptrs(pa); fetch_ptrs(pb);            // this group's first two k-blocks
    // the A buffer starts out zero and is only ever patched; the metadata image starts out as "kept elements at 0, 1"
    {
      uint4* z = (uint4*)(smem + S_SMEM_A + grp * S_A_BUF);
#pragma unroll 4
      for (int i = 0; i < S_A_BUF / 16 / S_GT; ++i) z[wt + i * S_GT] = make_uint4(0, 0, 0, 0);
      for (int i = wt; i < 2 * S_META / 16; i += S_GT) ((uint4*)(smem + S_SMEM_META + 2 * grp * S_META))[i] = make_uint4(0x44444444u, 0x44444444u, 0x44444444u, 0x44444444u);   // both images of the slot
    }
    asm volatile("bar.sync %0, %1;\n" ::"r"(1 + grp), "n"(S_GT) : "memory");
    fetch(ra, pa); fetch(rb, pb);              // their nonzeros; pa / pb now hold the pointers of the two after
    for (uint32_t gk = (uint32_t)grp; gk < gk_end; gk += 2 * S_NG) {
      step(gk, ra, pa);
      step(gk + S_NG, rb, pb);
    }
  }
  else {
    // ---------------- epilogue: warp owns TMEM lanes 32*(warp % 4) .. +31 of this CTA and half of the tile's columns ----------------
    const int quarter = warp & 3;
    const int row = quarter * 32 + lane;
    const uint32_t lead_empty0 = map_to_cta(&acc_empty[0], 0), lead_meta = map_to_cta(meta_free, 0);
    unsigned char* stage = smem + S_SMEM_STAGE + (warp - (2 + S_GW * S_NG)) * S_STAGE;
    const size_t cap = (size_t)g.bm * g.bk;
    const uint16_t* Bp = (const uint16_t*)p.b;
    for (int wi = 0; wi < nwork; ++wi) {
      SpTile t = tile_of(work_idx(wi));
      const int half = work_half(wi), ncw = half < 0 ? S_BN : S_BNH;
      if (half > 0) t.n0 += S_BNH;
      const uint32_t acc = (uint32_t)wi & 1u;
      const int rl = t.ml0 + row;
      const bool rvalid = row < t.rows;
      // ---- overflow entries of this thread's row (third / fourth nonzero of a group of four consecutive k): the tensor core
      // does not see them; the row's owner adds value * B[k, :] to the accumulator it drains, slices in ascending k-block,
      // entries in ascending k -- one fixed order.  Only slices whose overflow count is not zero are looked at (~2 of the 32
      // of a row block at 1 %), and all of this runs while the tensor core still works on the tile.
      auto scan = [&](auto&& f) {
        for (int kb0 = 0; kb0 < nkb; kb0 += 32) {
          const int kbl = kb0 + lane;
          uint32_t flagged = __ballot_sync(0xffffffffu, kbl < nkb && 0 != __ldg(p.sl.slice_ovf + kbl * g.mb + t.mbi));
          for (; flagged; flagged &= flagged - 1u) {
            const int kb = kb0 + __ffs((int)flagged) - 1;
            const size_t s = (size_t)kb * g.mb + t.mbi;
            int first = 0, last = 0;
            if (rvalid) { first = (int)__ldg(p.sl.rowidx + s * (g.bm + 1) + rl); last = (int)__ldg(p.sl.rowidx + s * (g.bm + 1) + rl + 1); }
            for (int q = first; q < last; ++q) {              // last < first: wrapped counter of a full slice, the row reads as empty
              if (__ldg(p.sl.tcsp + s * cap + q) & 0x8000u) f(kb * g.bk + (int)__ldg(p.sl.colidx + s * cap + q), __ldg(p.sl.values + s * cap + q));
            }
          }
        }
      };
      auto add_row = [&](uint32_t (&v)[32], int cb, int k, float a) {   // v[0..31] += a * B[k, n0 + cb .. +31]
        const uint16_t* bp = Bp + (size_t)k * p.ldb + t.n0 + cb;
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          if (t.n0 + cb + 8 * u + 7 < p.ncols) {
            const uint4 b8 = __ldg((const uint4*)bp + u);
            const uint32_t bw[4] = { b8.x, b8.y, b8.z, b8.w };
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              v[8 * u + 2 * e] = __float_as_uint(fmaf(a, __uint_as_float(bw[e] << 16), __uint_as_float(v[8 * u + 2 * e])));
              v[8 * u + 2 * e + 1] = __float_as_uint(fmaf(a, __uint_as_float(bw[e] & 0xFFFF0000u), __uint_as_float(v[8 * u + 2 * e + 1])));
            }
          }
          else {
#pragma unroll
            for (int e = 0; e < 8; ++e) if (t.n0 + cb + 8 * u + e < p.ncols) v[8 * u + e] = __float_as_uint(fmaf(a, __uint_as_float((uint32_t)__ldg(bp + 8 * u + e) << 16), __uint_as_float(v[8 * u + e])));
          }
        }
      };
      // The slicing kernel lists the overflow entries of a slice (the first kSpOvfCap, in no particular order): a thread reads
      // the lists of the flagged slices (same address for all lanes), keeps the entries of its row -- sorted by k, slices come
      // in ascending k-block -- and falls back to walking the row pointers (scan) when a slice has more entries than the list
      // holds or the row more than S_NOVF.
      int ne = 0, ok[S_NOVF]; float ov[S_NOVF];
#pragma unroll
      for (int i = 0; i < S_NOVF; ++i) { ok[i] = 0x7FFFFFFF; ov[i] = 0.f; }
      for (int kb0 = 0; kb0 < nkb; kb0 += 32) {
        const int kbl = kb0 + lane;
        const uint32_t cnt = (kbl < nkb) ? __ldg(p.sl.slice_ovf + kbl * g.mb + t.mbi) : 0u;
        uint32_t flagged = __ballot_sync(0xffffffffu, 0 != cnt);
        for (; flagged; flagged &= flagged - 1u) {
          const int src = __ffs((int)flagged) - 1, kb = kb0 + src;
          const uint32_t c = __shfl_sync(0xffffffffu, cnt, src);
          if (c > (uint32_t)kSpOvfCap) { ne = S_NOVF + 1; continue; }
          const uint2* lst = p.sl.ovf_list + ((size_t)kb * g.mb + t.mbi) * kSpOvfCap;
          for (uint32_t e = 0; e < c; ++e) {
            const uint2 w = __ldg(lst + e);
            if (rvalid && (int)(w.x & 0xFFFFu) == rl) {
              const int k = kb * g.bk + (int)(w.x >> 16);
              if (ne < S_NOVF) {       // insert by ascending k (entries of one slice come in any order)
                int ck = k; float cv = __uint_as_float(w.y);
#pragma unroll
                for (int i = 0; i < S_NOVF; ++i) {
                  if (ck < ok[i]) { const int tk = ok[i]; const float tv = ov[i]; ok[i] = ck; ov[i] = cv; ck = tk; cv = tv; }
                }
              }
              ++ne;
            }
          }
        }
      }
      const bool many = 0 != __any_sync(0xffffffffu, ne > S_NOVF);     // warp-uniform: scan() votes
      // C box by TMA: every row of this warp belongs to the tile, C is not read, rows are 16-byte aligned
      const bool use_tma = (0 != c_tma) && (t.rows >= quarter * 32 + 32);
      mbar_wait(&acc_full[acc], ((uint32_t)wi >> 1) & 1u);
      tc_fence_after();
      const size_t crow = (size_t)(t.mbi * g.bm + t.ml0 + row - p.row_origin);
#pragma unroll 1
      for (int cb = 0; cb < ncw; cb += 32) {
        uint32_t v[32];
        tc_ld32(tmem_d + acc * S_BN + ((uint32_t)(quarter * 32) << 16) + (uint32_t)cb, v);
        if (0 == cb) {         // columns 0..31 of this accumulator are read: the next tile's metadata may go there
          tc_fence_before();
          __syncwarp();
          if (0 == lane) mbar_arrive_cluster(lead_meta);
        }
        if (many) scan([&](int k, float a) { add_row(v, cb, k, a); });   // rows with many overflow entries (a dense matrix forced onto this kernel): the whole warp walks the slices again
        else if (ne > 0) {     // rare
#pragma unroll
          for (int i = 0; i < S_NOVF; ++i) if (i < ne) add_row(v, cb, ok[i], ov[i]);
        }
        if (p.debug_flags & 4) continue;
        if (use_tma) {
          // thread = row: eight 16-byte units of the row's 128 bytes, swizzled like the tensor map (unit ^ row % 8): no bank
          // conflicts, and the store engine, not the load / store unit the workers depend on, moves the box.
          // One staging box per warp: a chunk waits until the store engine has read the previous one out (about a microsecond,
          // hidden behind the next tile's k loop) -- except in the pair's LAST tile, whose epilogue nothing overlaps: once its
          // MMAs have completed the ring is idle, and every chunk gets a box of its own there (measured: 4.7 us of tail for a
          // half tile, 9.3 us for a full one, with the single box).
          unsigned char* sbox = stage;
          if (wi == nwork - 1) sbox = smem + S_SMEM_A + ((warp - (2 + S_GW * S_NG)) * (S_BN / 32) + (cb >> 5)) * S_STAGE;
          else {
            if (0 == lane) asm volatile("cp.async.bulk.wait_group.read 0;\n" ::: "memory");
            __syncwarp();
          }
#pragma unroll
          for (int u = 0; u < 8; ++u) *(uint4*)(sbox + lane * 128 + ((u ^ (lane & 7)) << 4)) = make_uint4(v[4 * u], v[4 * u + 1], v[4 * u + 2], v[4 * u + 3]);
          fence_proxy_async();
          __syncwarp();
          if (0 == lane) {
            asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%1, %2}], [%3];\n"
                         ::"l"(&tmC), "r"(t.n0 + cb), "r"((int)(crow - (size_t)lane)), "r"(smem_u32(sbox)) : "memory");
            asm volatile("cp.async.bulk.commit_group;\n" ::: "memory");
          }
        }
        else if (rvalid) {
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
          else {
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
    if (0 == lane) asm volatile("cp.async.bulk.wait_group.read 0;\n" ::: "memory");    // shared memory stays alive until the store engine has read every box
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

// returns false when the panel does not qualify (caller falls back to K4p)
bool launch_compute_tc16s(const ComputeArgs& a, cudaStream_t stream)
{
  const char* env = getenv("LIBXSMM_B200_TC16_SPARSE");      // "0": never, "1": whenever the slices carry the words, else: by density
  if (env && '0' == *env) return false;
  if (0 == a.aux_valid || 0 == a.sp_valid || 0 == a.sl.tcsp || 0 == a.sl.slice_ovf || 0 == a.sl.ovf_list) return false;
  if (!a.is_bf16 || a.transb) return false;
  const bool forced = env && '1' == *env;
  if (!forced && !(a.density_hint >= 0.f && a.density_hint <= kSpMaxDensity)) return false;
  if (!a.transc && (0 != ((uintptr_t)a.c & 15) || 0 != (a.ldc & 3))) return false;
  CUtensorMap map;
  if (!make_tensor_map_2d_sw128(&map, a.b, 2, (unsigned long long)a.ncols, (unsigned long long)a.g.k, (unsigned long long)a.ldb * 2, 64, S_KB, false)) return false;
  ensure_smem_optin((const void*)spmdm_compute_tc16s_kernel, S_SMEM_BYTES);
  const int pairs_max = device_sm_count() / 2 > 0 ? device_sm_count() / 2 : 1;
  const int tiles_per_mb = (a.g.bm + S_BM - 1) / S_BM;
  const int pair_m = (a.mb_count * tiles_per_mb + 1) / 2;
  const int total = pair_m * ((a.ncols + S_BN - 1) / S_BN);
  if (total <= 0) return true;
  const int pairs = total < pairs_max ? total : pairs_max;
  // C leaves through TMA boxes of 32 x 32 when it is only written (beta = 0) and stored row-major
  CUtensorMap cmap = map;
  int c_tma = 0;
  if (!a.transc && 0.f == a.beta) {
    const long long crows = (long long)a.g.m - a.row_origin;
    if (crows > 0 && make_tensor_map_2d_sw128(&cmap, a.c, 4, (unsigned long long)a.ncols, (unsigned long long)crows, (unsigned long long)a.ldc * 4, 32, 32, false)) c_tma = 1;
    else cmap = map;
  }
  count_launch(1);
  note_compute_kernel("spmdm_compute_tc16s_kernel");
  ComputeArgs a2 = a;
  if (forced) a2.sp_guard = 0;
  if (const char* dbg = getenv("LIBXSMM_B200_K4S_DEBUG")) a2.debug_flags = atoi(dbg);   // developer timing aid: results are wrong when set
  // programmatic dependent launch: the CTAs may be scheduled, and run their prologue, while the kernel in front of this one
  // (normally the slicing kernel) is still draining
  XB_CUDA(launch_pdl(spmdm_compute_tc16s_kernel, dim3(2u * (unsigned)pairs), dim3(S_THREADS), S_SMEM_BYTES, stream, map, cmap, c_tma, a2));
  return true;
}

}  // namespace xb
