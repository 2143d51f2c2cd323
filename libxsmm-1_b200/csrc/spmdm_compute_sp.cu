// K2s: the order-preserving sliced SpMM for the SPARSE regime, second generation (sm_100a).
//
//   C[tile rows, tile cols] = beta*C + sum_kb slice(kb, mb)[tile rows, :] * B[kb*128 .. +128, tile cols]
//
// Same arithmetic as K2 (spmdm_compute_tma.cu): per output element the reference's rounding sequence -- start
// from beta*C, one fused multiply-add per nonzero in ascending (kb, column) order (reference
// src/template/libxsmm_spmdm_compute_fp32_thread.tpl.c:309-370, ..._bfloat16_thread.tpl.c:309-370) -- so the
// result is bit-identical to the reference's full-width blocks.  What changed is everything around the fma:
//
//  * B tiles (128 k x BN columns, 64 KiB) arrive by TMA in a 3-deep ring, fed by a dedicated producer warp, so no
//    consumer ever waits inside the producer's empty-slot wait; a slot is refilled when all 16 consumer warps have
//    released it.  Each CTA fetches its own tiles: sharing them over a thread-block cluster by TMA multicast measured
//    slower (4096^3 bf16 at 1 %, B tile loads alone: 106 us per CTA, 161 us for pairs, 178 us for quads).
//  * bf16: the nonzero travels as ONE word (bf16 value << 16 | column * 512), one shuffle per nonzero, and the
//    multiply-add is the mixed-precision instruction fma.rn.f32.bf16 (SASS FHFMA.BF16 with .H0/.H1 operand
//    selectors): bf16 x bf16 is exact in fp32, the sum is rounded once, so it equals fmaf(widen(a), widen(b), c)
//    bit for bit and the 8 unpack operations per 16-byte shared-memory read disappear.
//  * the next nonzero's word is shuffled while the current one is multiplied; row pointers are fetched two
//    k-blocks ahead and the first 32 nonzeros one k-block ahead; denser rows walk their range in chunks of 32 with
//    the following chunk in flight.
//  * only a completely full 512 x 128 slice can wrap its u16 row pointers (reference quirk, template :72), and
//    only its last pointer does: the fix-up is confined to the one warp that owns row 511.
//
// Only transb = transc = 'N', 16-byte aligned panels and the reference's full-width column blocks come here.
#include "common.cuh"
#include "ptx.cuh"
#include <cstdlib>

namespace xb {

bool make_tensor_map_2d(CUtensorMap* map, const void* base, int elem_bytes, unsigned long long cols, unsigned long long rows,
                        unsigned long long row_pitch_bytes, unsigned box_cols, unsigned box_rows);

namespace {

constexpr int SP_CW = 16;                // consumer warps per CTA
constexpr int SP_R = 8;                  // rows per warp
constexpr int SP_TM = SP_CW * SP_R;      // rows per CTA
constexpr int SP_ROWB = 512;             // bytes per tile row (256 bf16 or 128 fp32 columns)
constexpr int SP_STAGEB = 128 * SP_ROWB; // 64 KiB
constexpr int SP_STAGES = 3;
constexpr int SP_THREADS = (SP_CW + 4) * 32;   // 16 consumer warps + one producer warp group (registers are handed out per 4 warps: 640 x 96 at launch;
                                               // the producer group gives its share back with setmaxnreg, the consumers take it)
constexpr int SP_WSCRATCH = 384;               // bytes of per-warp list space: 33 x {1, 2} words of nonzeros (+ pad), 16 row offsets
constexpr int SP_SMEM = SP_STAGES * SP_STAGEB + 64 + SP_CW * SP_WSCRATCH;

__device__ __forceinline__ void mbar_arrive_u32(uint32_t bar) { asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];\n" ::"r"(bar) : "memory"); }
__device__ __forceinline__ void mbar_wait_u32(uint32_t bar, uint32_t parity)
{
  asm volatile(
    "{\n\t.reg .pred p;\n"
    "SP_WAIT:\n\t"
    "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, %2;\n\t"
    "@p bra.uni SP_DONE;\n\t"
    "bra.uni SP_WAIT;\n"
    "SP_DONE:\n\t}\n"
    ::"r"(bar), "r"(parity), "r"(0x989680) : "memory");
}
// One nonzero of the warp's rows as it is kept in registers between its (prefetched) load and the moment it is put on the
// warp's shared-memory list.  A list entry is 8 bytes {address of the B tile row in shared memory, w}: for bf16 slices w
// holds the value in its high half (the widened fp32 value has 16 zero bits below it), for fp32 slices w is the value.
struct Nz {
  uint32_t col, val;      // raw: nothing touches the loaded registers before put(), so the loads stay in flight during the walk
  __device__ __forceinline__ void clear() { col = 0; val = 0; }
  __device__ __forceinline__ void load(const uint16_t* cp, const float* vp) { col = __ldg(cp); val = __float_as_uint(__ldg(vp)); }
  __device__ __forceinline__ void put(uint32_t entry, uint32_t stage) const { asm volatile("st.shared.v2.b32 [%0], {%1, %2};\n" ::"r"(entry), "r"(stage + (col << 9)), "r"(val) : "memory"); }
};

// Walks the list entries [lp, hip) of ONE output row: acc += value * B[tile row][this lane's columns], in list order.
// On entry {o, w} is the entry at lp (already loaded); on exit lp == hip and {o, w} is the entry at hip (the list has a spare
// slot): the next entry is fetched while the current one is multiplied.  Written in PTX so that the loop is exactly
// this instruction sequence; every branch is warp-uniform by construction (the bounds come from warp-wide lists).
template <bool BF16> struct RowWalk;
template <> struct RowWalk<true> {
  static __device__ __forceinline__ void run(float (&a)[8], uint32_t& lp, uint32_t hip, uint32_t& o, uint32_t& w, uint32_t lane_off)
  {
    asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      ".reg .b32 ad, b0, b1, b2, b3;\n\t"
      ".reg .b16 wl, wh, l0, h0, l1, h1, l2, h2, l3, h3;\n\t"
      "setp.ge.u32 p, %8, %11;\n\t"
      "@p bra.uni ROW_DONE;\n"
      "ROW_LOOP:\n\t"
      "add.u32 ad, %9, %12;\n\t"
      "ld.shared.v4.b32 {b0, b1, b2, b3}, [ad];\n\t"
      "mov.b32 {wl, wh}, %10;\n\t"
      "ld.shared.v2.b32 {%9, %10}, [%8+8];\n\t"
      "add.u32 %8, %8, 8;\n\t"
      "mov.b32 {l0, h0}, b0;\n\tmov.b32 {l1, h1}, b1;\n\tmov.b32 {l2, h2}, b2;\n\tmov.b32 {l3, h3}, b3;\n\t"
      "fma.rn.f32.bf16 %0, wh, l0, %0;\n\tfma.rn.f32.bf16 %1, wh, h0, %1;\n\t"
      "fma.rn.f32.bf16 %2, wh, l1, %2;\n\tfma.rn.f32.bf16 %3, wh, h1, %3;\n\t"
      "fma.rn.f32.bf16 %4, wh, l2, %4;\n\tfma.rn.f32.bf16 %5, wh, h2, %5;\n\t"
      "fma.rn.f32.bf16 %6, wh, l3, %6;\n\tfma.rn.f32.bf16 %7, wh, h3, %7;\n\t"
      "setp.lt.u32 p, %8, %11;\n\t"
      "@p bra.uni ROW_LOOP;\n"
      "ROW_DONE:\n\t"
      "}\n"
      : "+f"(a[0]), "+f"(a[1]), "+f"(a[2]), "+f"(a[3]), "+f"(a[4]), "+f"(a[5]), "+f"(a[6]), "+f"(a[7]), "+r"(lp), "+r"(o), "+r"(w)
      : "r"(hip), "r"(lane_off) : "memory");
  }
};
template <> struct RowWalk<false> {
  static __device__ __forceinline__ void run(float (&a)[4], uint32_t& lp, uint32_t hip, uint32_t& o, uint32_t& w, uint32_t lane_off)
  {
    asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      ".reg .b32 ad;\n\t"
      ".reg .f32 v, b0, b1, b2, b3;\n\t"
      "setp.ge.u32 p, %4, %7;\n\t"
      "@p bra.uni ROW_DONE;\n"
      "ROW_LOOP:\n\t"
      "add.u32 ad, %5, %8;\n\t"
      "ld.shared.v4.f32 {b0, b1, b2, b3}, [ad];\n\t"
      "mov.b32 v, %6;\n\t"
      "ld.shared.v2.b32 {%5, %6}, [%4+8];\n\t"
      "add.u32 %4, %4, 8;\n\t"
      "fma.rn.f32 %0, v, b0, %0;\n\tfma.rn.f32 %1, v, b1, %1;\n\tfma.rn.f32 %2, v, b2, %2;\n\tfma.rn.f32 %3, v, b3, %3;\n\t"
      "setp.lt.u32 p, %4, %7;\n\t"
      "@p bra.uni ROW_LOOP;\n"
      "ROW_DONE:\n\t"
      "}\n"
      : "+f"(a[0]), "+f"(a[1]), "+f"(a[2]), "+f"(a[3]), "+r"(lp), "+r"(o), "+r"(w)
      : "r"(hip), "r"(lane_off) : "memory");
  }
};

template <bool BF16>
__global__ void __launch_bounds__(SP_THREADS, 1)
spmdm_compute_sp_kernel(const __grid_constant__ CUtensorMap tmB, const ComputeArgs p)
{
  constexpr int VEC = BF16 ? 8 : 4;
  constexpr int BN = 32 * VEC;
  constexpr int R = SP_R;
  extern __shared__ __align__(128) unsigned char smem[];
  uint64_t* full = (uint64_t*)(smem + (size_t)SP_STAGES * SP_STAGEB);
  uint64_t* empty = full + SP_STAGES;

  const Geom& g = p.g;
  pdl_wait();     // launched with programmatic stream serialization: the CTAs of the first wave are in place when the slicing kernel ends
  if (p.tc_twin > 0 && xb_total_nnz(p.sl.slice_nnz, g.mb * g.kb) >= p.tc_min_nnz) return;   // the tensor-core twin does this multiply (uniform over the grid)
  const int tid = (int)threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int n0 = (int)blockIdx.y * BN;

  if (0 == tid) {
#pragma unroll
    for (int s = 0; s < SP_STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], SP_CW); }
    mbar_fence_init();
  }
  __syncthreads();

  if (warp >= SP_CW) {
    // ---------------- producer warp group: one lane streams the B tiles ----------------
    asm volatile("setmaxnreg.dec.sync.aligned.u32 24;\n");
    if (SP_CW == warp && 0 == lane) {
      tma_prefetch_desc(&tmB);
      for (int t = 0; t < g.kb && !(p.debug_flags & 2); ++t) {
        const int s = t % SP_STAGES, f = t / SP_STAGES;
        if (f > 0) mbar_wait(&empty[s], (f - 1) & 1);          // every consumer warp is done with the slot
        mbar_arrive_expect_tx(&full[s], SP_STAGEB);
        tma_load_2d(smem + (size_t)s * SP_STAGEB, &tmB, n0, t * g.bk, &full[s]);
      }
    }
    __syncwarp();
  }
  else {
    // ---------------- consumers ----------------
    asm volatile("setmaxnreg.inc.sync.aligned.u32 112;\n");   // 16 x 512 <= the 72 x 128 registers the producer group released (the pool is per CTA)
    const uint32_t smem0 = smem_u32(smem);
    const uint32_t wlist = smem0 + (uint32_t)(SP_STAGES * SP_STAGEB + 64 + warp * SP_WSCRATCH);   // 33 entries of 8 bytes (one spare)
    const uint32_t wrel = wlist + 284;   // entries 1..8 start 16-byte aligned (two 16-byte loads fetch all row ends)                                                               // R + 1 list addresses: row i = [wrel[i], wrel[i+1])
    uint32_t lane_off = (uint32_t)lane * 16u;
    asm volatile("" : "+r"(lane_off));
    const int tiles_per_mb = (g.bm + SP_TM - 1) / SP_TM;
    const int rt = (int)blockIdx.x;
    const int mbi = p.mb_first + rt / tiles_per_mb;
    const int ml0 = (rt % tiles_per_mb) * SP_TM;
    const int rows_in_block = min(g.bm, g.m - mbi * g.bm);
    const int mycol = n0 + lane * VEC;
    const int wrow0 = ml0 + warp * R;
    const int nvalid = max(0, min(R, rows_in_block - wrow0));
    const size_t crow0 = (size_t)(mbi * g.bm + wrow0 - p.row_origin);
    const size_t cap = (size_t)g.bm * g.bk;
    const bool colfull = (mycol + VEC <= p.ncols);

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

    // slice s = kb*mb + mbi: 32-bit element offsets into the arena arrays (the host sends arenas of 2^31 or more elements to
    // K2), advanced by one "kb" stride per iteration
    const uint32_t rp_stride = (uint32_t)g.mb * (uint32_t)(g.bm + 1);
    const uint32_t nz_stride = (uint32_t)g.mb * (uint32_t)cap;
    const bool rp_lane = (lane <= R) && (nvalid > 0);
    const bool wrap_warp = (512 == g.bm) && (wrow0 + R == 512);   // the only row pointer that can wrap is rowidx[512] of a full 512 x 128 slice
    uint32_t rpo = (uint32_t)mbi * (uint32_t)(g.bm + 1) + (uint32_t)(wrow0 + min(lane, nvalid));   // row pointers of k-block kb+2 (lanes past the last valid row repeat its end: empty rows)
    uint32_t nzo = (uint32_t)mbi * (uint32_t)cap + (uint32_t)lane;                                   // nonzeros of k-block kb+1
    const uint16_t* const rowidx = p.sl.rowidx;
    const uint16_t* const colidx = p.sl.colidx;
    const float* const values = p.sl.values;

    auto fix_wrap = [&](int rp) -> int {
      if (wrap_warp) { const int prev = __shfl_up_sync(0xffffffffu, rp, 1); if (R == lane && rp < prev) rp = prev; }
      return rp;
    };
    int rp_cur = fix_wrap(rp_lane ? (int)__ldg(rowidx + rpo) : 0);
    rpo += rp_stride;
    int rp_nxt = (rp_lane && 1 < g.kb) ? (int)__ldg(rowidx + rpo) : 0;
    rpo += rp_stride;
    int first = __shfl_sync(0xffffffffu, rp_cur, 0);
    int total = __shfl_sync(0xffffffffu, rp_cur, R) - first;
    Nz nz_c;                               // lane q: nonzero (first + q) of the warp's rows, current k-block
    nz_c.clear();
    if (lane < total) { const uint32_t ix = nzo + (uint32_t)first; nz_c.load(colidx + ix, values + ix); }
    uint32_t nzo_cur = nzo;                      // this k-block's offset (lane included), for the chunks after the first
    nzo += nz_stride;

    // ring state, kept incrementally (no division by the ring depth in the loop); the shared-memory addresses are made opaque
    // so that the compiler keeps them in registers instead of re-deriving them from the thread id in every iteration
    uint32_t stage = smem0, fullb = smem_u32(&full[0]), phase = 0, slot = 0;
    uint32_t wl = wlist, wr = wrel, ulane = (uint32_t)lane;
    asm volatile("" : "+r"(stage), "+r"(fullb), "+r"(wl), "+r"(wr), "+r"(ulane));
    const int kbn = g.kb;

    for (int kb = 0; kb < kbn; ++kb) {
      // ---- prefetch: row pointers of kb+2, first 32 nonzeros of kb+1 -------------------------------------------
      const int rp_nn = (rp_lane && kb + 2 < kbn) ? (int)__ldg(rowidx + rpo) : 0;
      rpo += rp_stride;
      rp_nxt = fix_wrap(rp_nxt);
      const int first_n = __shfl_sync(0xffffffffu, rp_nxt, 0);
      const int total_n = __shfl_sync(0xffffffffu, rp_nxt, R) - first_n;   // 0 past the last k-block
      Nz nz_n;
      nz_n.clear();
      if (lane < total_n) { const uint32_t ix = nzo + (uint32_t)first_n; nz_n.load(colidx + ix, values + ix); }
      const int relv = rp_cur - first;             // lane i <= R: offset of row i's first nonzero inside the warp's range
      // ---- wait for the B tile of this k-block (every warp, also one without nonzeros: the ring's phases are counted) ----
      if (!(p.debug_flags & 2)) mbar_wait_u32(fullb, phase);
      // ---- walk the warp's nonzeros: they and the row boundaries go to the warp's shared-memory list, which the row
      //      walks read with broadcast loads.  Sparse regime: one list of at most 32 entries, everything already here.
      //      Denser rows: chunks of 32, the following chunk in flight, row boundaries clipped to the chunk. ----
      if (total > 0 && !(p.debug_flags & 1)) {
        if (total <= 32) {
          __syncwarp();                                  // everybody is done reading the previous list
          nz_c.put(wl + 8u * ulane, stage);
          if (ulane <= R) asm volatile("st.shared.b32 [%0], %1;\n" ::"r"(wr + 4u * ulane), "r"(wl + 8u * (uint32_t)relv) : "memory");
          __syncwarp();
          uint32_t lp = wl, o, w, h[R];
          asm volatile("ld.shared.v2.b32 {%0, %1}, [%2];\n" : "=r"(o), "=r"(w) : "r"(lp) : "memory");
          asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4+4];\n" : "=r"(h[0]), "=r"(h[1]), "=r"(h[2]), "=r"(h[3]) : "r"(wr) : "memory");
          asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4+20];\n" : "=r"(h[4]), "=r"(h[5]), "=r"(h[6]), "=r"(h[7]) : "r"(wr) : "memory");
#pragma unroll
          for (int i = 0; i < R; ++i) RowWalk<BF16>::run(acc[i], lp, h[i], o, w, lane_off);
        }
        else {
#pragma unroll 1
          for (int p0 = 0; p0 < total; p0 += 32) {
            Nz nz_x;
            nz_x.clear();
            if (p0 + 32 + lane < total) { const uint32_t ix = nzo_cur + (uint32_t)(first + p0 + 32); nz_x.load(colidx + ix, values + ix); }
            __syncwarp();
            nz_c.put(wl + 8u * ulane, stage);
            if (ulane <= R) asm volatile("st.shared.b32 [%0], %1;\n" ::"r"(wr + 4u * ulane), "r"(wl + 8u * (uint32_t)min(max(relv - p0, 0), 32)) : "memory");
            __syncwarp();
            uint32_t lp = wl, o, w, h[R];
            asm volatile("ld.shared.v2.b32 {%0, %1}, [%2];\n" : "=r"(o), "=r"(w) : "r"(lp) : "memory");
            asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4+4];\n" : "=r"(h[0]), "=r"(h[1]), "=r"(h[2]), "=r"(h[3]) : "r"(wr) : "memory");
            asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4+20];\n" : "=r"(h[4]), "=r"(h[5]), "=r"(h[6]), "=r"(h[7]) : "r"(wr) : "memory");
#pragma unroll
            for (int i = 0; i < R; ++i) RowWalk<BF16>::run(acc[i], lp, h[i], o, w, lane_off);
            nz_c = nz_x;
          }
        }
      }
      // ---- release the slot to the producer (not needed for the last tiles: nobody refills) ----
      if (kb + SP_STAGES < kbn && !(p.debug_flags & 2)) {
        __syncwarp();
        if (0 == ulane) mbar_arrive_u32(fullb + 8u * SP_STAGES);
      }
      stage += SP_STAGEB; fullb += 8u;
      if (++slot == SP_STAGES) { slot = 0; stage -= SP_STAGES * SP_STAGEB; fullb -= 8u * SP_STAGES; phase ^= 1u; }
      nzo_cur = nzo; nzo += nz_stride;
      rp_cur = rp_nxt; rp_nxt = rp_nn; nz_c = nz_n; first = first_n; total = total_n;
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
}

template <bool BF16>
bool launch_sp(const ComputeArgs& a, cudaStream_t stream)
{
  constexpr int ESZ = BF16 ? 2 : 4;
  constexpr int BN = SP_ROWB / ESZ;
  CUtensorMap map;
  if (!make_tensor_map_2d(&map, a.b, ESZ, (unsigned long long)a.ncols, (unsigned long long)a.g.k,
                          (unsigned long long)a.ldb * ESZ, BN, 128)) return false;
  auto kern = spmdm_compute_sp_kernel<BF16>;
  ensure_smem_optin((const void*)kern, SP_SMEM);
  const int tiles_per_mb = (a.g.bm + SP_TM - 1) / SP_TM;
  const dim3 grid((unsigned)(a.mb_count * tiles_per_mb), (unsigned)((a.ncols + BN - 1) / BN), 1);
  count_launch(1);
  note_compute_kernel("spmdm_compute_sp_kernel");
  XB_CUDA(launch_pdl(kern, grid, dim3(SP_THREADS), (size_t)SP_SMEM, stream, map, a));
  return true;
}

}  // namespace

// returns false when the panel does not qualify (caller then uses K2 or the generic kernel)
bool launch_compute_sp(const ComputeArgs& a_in, cudaStream_t stream)
{
  if (a_in.transb || a_in.transc) return false;
  if (0 != ((uintptr_t)a_in.c & 15) || 0 != (a_in.ldc & 3)) return false;
  if (a_in.ncols <= 32) return false;
  if ((unsigned long long)a_in.g.mb * a_in.g.kb * a_in.g.bm * a_in.g.bk >= (1ull << 31)) return false;   // the kernel indexes the slice arena with 32-bit element offsets
  static const int dbg = [] { const char* e = getenv("LIBXSMM_B200_K2S_DEBUG"); return (e && *e) ? atoi(e) : 0; }();
  ComputeArgs a = a_in;
  a.debug_flags = dbg;
  return a.is_bf16 ? launch_sp<true>(a, stream) : launch_sp<false>(a, stream);
}

}  // namespace xb
