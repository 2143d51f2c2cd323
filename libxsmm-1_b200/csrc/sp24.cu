// Fixed 2:4-sparse bf16 and FP8 operators (libxsmm_b200_sp24_*).  A matrix with at most two kept elements in every aligned
// group of four along k is exactly the operand of the structured-sparse tensor-core instruction, so the compressed tile K4s
// (spmdm_compute_tc16s.cu) rebuilds in shared memory on every call can be written to HBM once, at create:
//   * values: [M_pad][K_pad / 2] bf16, plain row-major.  A TMA box of {64 kept, 128 rows} with SWIZZLE_128B puts it in shared
//     memory at the positions xb_sp_pos gives (row * 128 bytes, 16-byte unit XOR row % 8): K4s's compressed tile;
//   * metadata: per (128-row tile, 128-k block) the 2 KiB image K4s's workers write (common.cuh: xb_sp_meta_off), which the
//     issuing thread hands to tcgen05.cp unchanged.
// Padding (rows >= M, k >= K) holds zero values under the nibble of an empty group.
// The multiply is K4s's skeleton -- CTA pair, persistent over 256 x 256 output tiles, one ring slot per 128-k block, the
// accumulator double buffered in tensor memory, the metadata columns in the idle accumulator -- with the slot's A tile and
// metadata image fetched by TMA next to B: no worker warps, no overflow pass, and a slot completes on bytes alone.
// Roles per CTA (6 warps): warp 0 TMA producer, warp 1 MMA issuer (leader CTA) and TMEM owner, warps 2-5 epilogue.
// TB (transb = 'T', B stored N x K) is a K-major B operand: another box and the descriptor's major bit, a template parameter
// because K4s's run-time flag for it cost 10 us (DESIGN.md section 8).
// F8 (FP8 operators, e4m3 / e5m2, tcgen05.mma.sp kind::f8f6f4, K = 64 per instruction) keeps every byte count of a ring slot
// and takes twice the k: a slot holds 256 k -- A 128 rows x 128 kept bytes (the same 128-byte swizzle rows), B 256 k x 128
// columns (32 KiB) -- and a 4 KiB metadata image, lane = row, two tensor-memory columns per instruction
// (tools/umma_probe/probe_sp8.cu): [column half][128 lanes][16 bytes], copied with two tcgen05.cp.  An MN-major ('N') 8-bit B
// of 128 columns is two 64-byte SWIZZLE_64B blocks, so that the half tile's 64 columns per CTA are one block as in bf16.
// The epilogue scales the accumulator by alpha (the per-tensor scales of A and B) before beta C is added.
// OB (the *_bf16out entries) changes the epilogue only: v = alpha acc (F8), + bias[m] (one fp32 addition, none for a NULL
// bias), fmaf(beta, C_old, v), rounded to bf16 to nearest even in pairs.  Its TMA store stages two 32-column chunks as one box
// of 32 rows x 64 bf16 (128-byte rows, SWIZZLE_128B): the fp32 box's size and staging layout, half as many boxes per tile.
#include "common.cuh"
#include "tc_common.cuh"

namespace xb {

constexpr int F_BM = 128;                       // rows per CTA
constexpr int F_BN = 256;                       // columns per pair tile
constexpr int F_BNH = 128;                      // columns of B staged per CTA
constexpr int F_NA = 4;                         // ring slots (a fifth does not fit: 5 x 50 KiB > 227 KiB)
constexpr int F_NE = 4;                         // epilogue warps (one per TMEM lane quarter)
constexpr int F_A_BUF = F_BM * 128;             // 16 KiB: 128 rows x 128 bytes of kept elements
constexpr int F_B_STAGE = 32768;                // 32 KiB: 128 k x 128 bf16 columns, or 256 k x 128 FP8 columns
constexpr int F_THREADS = (2 + F_NE) * 32;
constexpr int F_STAGE = 32 * 128;

template <bool F8> struct Sp24Geo {
  static constexpr int KB = F8 ? 256 : 128;                   // k per ring slot
  static constexpr int META = F_BM * (F8 ? 32 : 16);          // metadata image: per TMEM lane eight (F8) or four 32-bit columns
  static constexpr int SMEM_A = 0;
  static constexpr int SMEM_B = SMEM_A + F_NA * F_A_BUF;
  static constexpr int SMEM_META = SMEM_B + F_NA * F_B_STAGE;
  static constexpr int SMEM_STAGE = SMEM_META + F_NA * META;  // per epilogue warp a [32 rows x 32 columns] fp32 box for the TMA store of C
  static constexpr int SMEM_BAR = SMEM_STAGE + F_NE * F_STAGE;
  static constexpr int SMEM_BYTES = SMEM_BAR + 256;
  static_assert(KB * F_BNH * (F8 ? 1 : 2) == F_B_STAGE, "B stage");
  static_assert(0 == (SMEM_STAGE & 1023), "SWIZZLE_128B boxes sit on 1 KiB boundaries");
  static_assert(F_NE * (F_BN / 32) * F_STAGE <= SMEM_META, "the last tile's C boxes fit in the (then idle) A / B ring");
  static_assert(SMEM_BYTES <= 227 * 1024, "shared memory");
  static_assert(F_NA * META / F_BM / 4 <= 32, "the metadata columns are read by the epilogue's first chunk before meta_free");
};

struct Sp24Args {
  float* c;
  long long ldc;
  int M, N, nkb, ctiles_m;
  float beta;
  int transc;
  int c_vec;            // C and ldc allow 16-byte stores (transc = 'N')
};
struct Sp24F8Args : Sp24Args {
  float alpha;
  uint32_t idesc_fmt;   // instruction-descriptor bits of the A and B formats
};
// bf16 C (OB): c holds the address of the bf16 C, c_vec means 16-byte stores of 8 elements
template <typename Base> struct Sp24OutArgs : Base {
  const unsigned short* bias;   // NULL or M bf16 values, indexed by A's row
};
template <bool F8, bool OB> using Sp24KArgs =
  typename std::conditional<OB, Sp24OutArgs<typename std::conditional<F8, Sp24F8Args, Sp24Args>::type>,
                            typename std::conditional<F8, Sp24F8Args, Sp24Args>::type>::type;

// two fp32 values rounded to bf16 (nearest even; NaN stays NaN, overflow gives +-Inf): lo in bits 0..15, hi in 16..31
__device__ __forceinline__ uint32_t bf16x2_rn(float lo, float hi)
{
  uint32_t r;
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;\n" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}
__device__ __forceinline__ float bf16_value(unsigned short h) { return __uint_as_float((uint32_t)h << 16); }

template <bool TB, bool F8, bool OB>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(F_THREADS, 1)
sp24_compute_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmE, const __grid_constant__ CUtensorMap tmB,
                    const __grid_constant__ CUtensorMap tmC, const int c_tma, const Sp24KArgs<F8, OB> p)
{
  using G = Sp24Geo<F8>;
  constexpr int F_KB = G::KB, F_META = G::META;
  constexpr int F_SMEM_A = G::SMEM_A, F_SMEM_B = G::SMEM_B, F_SMEM_META = G::SMEM_META, F_SMEM_STAGE = G::SMEM_STAGE, F_SMEM_BAR = G::SMEM_BAR;
  extern __shared__ __align__(1024) unsigned char smem[];
  uint64_t* bar = (uint64_t*)(smem + F_SMEM_BAR);
  uint64_t* a_ready = bar;                  // [NA] leader: A, metadata and B of both CTAs landed (bytes)
  uint64_t* a_free = a_ready + F_NA;        // [NA] both: the MMAs that read the slot have completed
  uint64_t* acc_full = a_free + F_NA;       // [2]  both: all MMAs of the tile have completed
  uint64_t* acc_empty = acc_full + 2;       // [2]  leader: the epilogue warps of both CTAs drained the accumulator
  uint64_t* meta_free = acc_empty + 2;      // [1]  leader: the epilogue warps of both CTAs have read the columns the next tile's metadata goes to
  uint32_t* tmem_slot = (uint32_t*)(meta_free + 1);

  const int tid = (int)threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t rank = cluster_rank();
  const int pair = (int)blockIdx.x >> 1, npairs = (int)gridDim.x >> 1;
  const int pair_m = (p.ctiles_m + 1) >> 1;
  const int n_tiles = (p.N + F_BN - 1) / F_BN;
  const int total = pair_m * n_tiles;
  const int nkb = p.nkb;
  const uint32_t sbase = smem_u32(smem);

  // work list of this pair (as K4s): q full tiles, then (when the rest is at most half as many tiles as pairs) one HALF tile
  const int wq = total / npairs, wrem = total - wq * npairs;
  const bool wsplit = wrem > 0 && 2 * wrem <= npairs;
  const int nwork = wq + ((wsplit ? (pair < 2 * wrem) : (pair < wrem)) ? 1 : 0);
  auto work_idx = [&](int i) -> int { return i < wq ? pair + i * npairs : wq * npairs + (wsplit ? (pair >> 1) : pair); };
  auto work_half = [&](int i) -> int { return (i < wq || !wsplit) ? -1 : (pair & 1); };

  if (0 == tid) {
#pragma unroll
    for (int i = 0; i < F_NA; ++i) { mbar_init(&a_ready[i], 1); mbar_init(&a_free[i], 1); }   // the leader's producer (with the byte count)
#pragma unroll
    for (int i = 0; i < 2; ++i) { mbar_init(&acc_full[i], 1); mbar_init(&acc_empty[i], 2 * F_NE); }
    mbar_init(meta_free, 2 * F_NE);
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

  if (0 == warp) {
    // ---------------- TMA producer: this CTA's A tile, metadata image and 128 columns of B per slot ----------------
    if (0 == lane) {
      tma_prefetch_desc(&tmA); tma_prefetch_desc(&tmE); tma_prefetch_desc(&tmB);
      uint32_t gk = 0;
      for (int wi = 0; wi < nwork; ++wi) {
        const int idx = work_idx(wi), half = work_half(wi);
        const int n0 = (idx / pair_m) * F_BN + (half < 0 ? (int)rank * F_BNH : half * F_BNH + (int)rank * (F_BNH / 2));
        // the odd CTA of a pair past the last row tile reads the last tile again: its rows are never stored
        const int mt = min(2 * (idx % pair_m) + (int)rank, p.ctiles_m - 1);
        for (int kbi = 0; kbi < nkb; ++kbi, ++gk) {
          const uint32_t j = gk % F_NA, f = gk / F_NA;
          if (f > 0) mbar_wait(&a_free[j], (f - 1) & 1);
          if (0 == rank) mbar_arrive_expect_tx(&a_ready[j], 2 * (F_A_BUF + F_META) + (half < 0 ? 2 * F_B_STAGE : F_B_STAGE));
          const uint32_t lbar = map_to_cta(&a_ready[j], 0);
          tma_load_2d_pair(smem + F_SMEM_A + j * F_A_BUF, &tmA, kbi * (F_KB / 2), mt * F_BM, lbar);
          tma_load_2d_pair(smem + F_SMEM_META + j * F_META, &tmE, 0, (mt * nkb + kbi) * (F_META / 128), lbar);
          unsigned char* dst = smem + F_SMEM_B + j * F_B_STAGE;
          if (TB) {      // K-major: [k half][128 n rows x 128 bytes of k], boxes of 64 n rows
            for (int kh = 0; kh < 2; ++kh) {
              tma_load_2d_pair(dst + kh * (F_B_STAGE / 2), &tmB, kbi * F_KB + kh * (F_KB / 2), n0, lbar);
              if (half < 0) tma_load_2d_pair(dst + kh * (F_B_STAGE / 2) + 64 * 128, &tmB, kbi * F_KB + kh * (F_KB / 2), n0 + 64, lbar);
            }
          }
          else {         // MN-major: [column block][k rows x 64 columns]
            tma_load_2d_pair(dst, &tmB, n0, kbi * F_KB, lbar);
            if (half < 0) tma_load_2d_pair(dst + F_B_STAGE / 2, &tmB, n0 + 64, kbi * F_KB, lbar);
          }
        }
      }
    }
  }
  else if (1 == warp) {
    // ---------------- MMA issuer (leader CTA) ----------------
    if (0 == rank && 0 == lane) {
      // sparse A, D = F32, A = B = BF16 (F8: the formats of A and B), A K-major (compressed), B MN-major ('N') or K-major ('T'),
      // N = 256, M = 256 (pair)
      uint32_t idesc_ab = (1u << 7) | (1u << 10);
      if constexpr (F8) idesc_ab = p.idesc_fmt;
      const uint32_t idesc = (1u << 2) | (1u << 4) | idesc_ab | (TB ? 0u : (1u << 16)) | ((uint32_t)(F_BN >> 3) << 17) | ((uint32_t)((2 * F_BM) >> 4) << 24);
      uint32_t gk = 0;
      for (int wi = 0; wi < nwork; ++wi) {
        const uint32_t acc = (uint32_t)wi & 1u;
        const uint32_t idesc_w = (work_half(wi) < 0) ? idesc : ((idesc & ~(0x3Fu << 17)) | ((uint32_t)(F_BNH >> 3) << 17));
        if (wi >= 2) mbar_wait(&acc_empty[acc], (((uint32_t)wi >> 1) - 1u) & 1u);
        if (wi >= 1) mbar_wait(meta_free, (uint32_t)(wi - 1) & 1u);    // the epilogue of the previous tile has read the columns this tile's metadata goes to
        tc_fence_after();
        const uint32_t tacc = tmem_d + acc * F_BN, tmeta = tmem_d + (acc ^ 1u) * F_BN;
        for (int kbi = 0; kbi < nkb; ++kbi, ++gk) {
          const uint32_t j = gk % F_NA;
          mbar_wait(&a_ready[j], (gk / F_NA) & 1);
          tc_fence_after();
          const uint32_t a_base = sbase + F_SMEM_A + j * F_A_BUF, b_base = sbase + F_SMEM_B + j * F_B_STAGE;
          if constexpr (F8) {      // eight columns per slot: two copies of four
#pragma unroll
            for (int h = 0; h < 2; ++h) {
              const uint64_t dm = tc_smem_desc(sbase + F_SMEM_META + j * F_META + h * (F_META / 2), 16, 128, 0);
              asm volatile("tcgen05.cp.cta_group::2.128x128b [%0], %1;\n" ::"r"(tmeta + 8u * j + 4u * (uint32_t)h), "l"(dm) : "memory");
            }
          }
          else {
            const uint64_t dm = tc_smem_desc(sbase + F_SMEM_META + j * F_META, 16, 128, 0);
            asm volatile("tcgen05.cp.cta_group::2.128x128b [%0], %1;\n" ::"r"(tmeta + 4u * j), "l"(dm) : "memory");
          }
#pragma unroll
          for (int ks = 0; ks < 4; ++ks) {         // K = 32 bf16 / 64 FP8 (32 bytes of the compressed row) per instruction
            const uint64_t da = tc_smem_desc(a_base + ks * 32, 16, 1024, 2);
            if constexpr (F8) {    // 'N': [64-column block][256 k rows x 64 bytes], SWIZZLE_64B
              const uint64_t db = TB ? tc_smem_desc(b_base + (ks >> 1) * (F_B_STAGE / 2) + (ks & 1) * 64, 16, 1024, 2)
                                     : tc_smem_desc(b_base + ks * 4096, (uint32_t)(F_B_STAGE / 2), 512, 4);
              tc_mma_f8_sp_pair(tacc, da, db, tmeta + 8u * j + 2u * (uint32_t)ks, idesc_w, (kbi > 0 || ks > 0) ? 1u : 0u);
            }
            else {
              const uint64_t db = TB ? tc_smem_desc(b_base + (ks >> 1) * (F_B_STAGE / 2) + (ks & 1) * 64, 16, 1024, 2)
                                     : tc_smem_desc(b_base + ks * 4096, (uint32_t)(F_KB * 128), 1024, 2);
              tc_mma_bf16_sp_pair(tacc, da, db, tmeta + 4u * j + (uint32_t)(ks & 2), idesc_w | (uint32_t)(ks & 1), (kbi > 0 || ks > 0) ? 1u : 0u);
            }
          }
          tc_commit_pair(&a_free[j]);
        }
        tc_commit_pair(&acc_full[acc]);
      }
    }
  }
  else {
    // ---------------- epilogue: warp owns TMEM lanes 32*(warp % 4) .. +31 of this CTA and half of the tile's columns ----------------
    const int quarter = warp & 3;
    const int row = quarter * 32 + lane;
    const uint32_t lead_empty0 = map_to_cta(&acc_empty[0], 0), lead_meta = map_to_cta(meta_free, 0);
    unsigned char* stage = smem + F_SMEM_STAGE + (warp - 2) * F_STAGE;
    for (int wi = 0; wi < nwork; ++wi) {
      const int idx = work_idx(wi), half = work_half(wi), ncw = half < 0 ? F_BN : F_BNH;
      const int ct = 2 * (idx % pair_m) + (int)rank;
      const int n0 = (idx / pair_m) * F_BN + (half > 0 ? F_BNH : 0);
      const int rows = ct < p.ctiles_m ? min(F_BM, p.M - ct * F_BM) : 0;
      const bool rvalid = row < rows;
      const bool use_tma = (0 != c_tma) && (rows >= quarter * 32 + 32);    // every row of this warp belongs to the tile
      const uint32_t acc = (uint32_t)wi & 1u;
      mbar_wait(&acc_full[acc], ((uint32_t)wi >> 1) & 1u);
      tc_fence_after();
      const size_t crow = (size_t)ct * F_BM + (size_t)row;
      float bias_v = 0.f;      // OB: the row is fixed for the tile, so its bias is loaded once
      if constexpr (OB) {
        if (0 != p.bias && rvalid) bias_v = bf16_value(__ldg(p.bias + crow));
      }
#pragma unroll 1
      for (int cb = 0; cb < ncw; cb += 32) {
        uint32_t v[32];
        tc_ld32(tmem_d + acc * F_BN + ((uint32_t)(quarter * 32) << 16) + (uint32_t)cb, v);
        if constexpr (F8) {
#pragma unroll
          for (int jj = 0; jj < 32; ++jj) v[jj] = __float_as_uint(p.alpha * __uint_as_float(v[jj]));
        }
        if constexpr (OB) {    // a separate rounded addition (never contracted with alpha's multiply); none without a bias, so -0 stays
          if (0 != p.bias) {
#pragma unroll
            for (int jj = 0; jj < 32; ++jj) v[jj] = __float_as_uint(__fadd_rn(__uint_as_float(v[jj]), bias_v));
          }
        }
        if (0 == cb) {         // columns 0..31 of this accumulator are read: the next tile's metadata may go there
          tc_fence_before();
          __syncwarp();
          if (0 == lane) mbar_arrive_cluster(lead_meta);
        }
        if constexpr (OB) {
          unsigned short* const cc = (unsigned short*)p.c;
          if (use_tma) {
            // beta = 0: chunk pairs (cb, cb + 32) share one box of 32 rows x 64 bf16; chunk h fills 16-byte units 4h .. 4h + 3
            // of each 128-byte row (XOR row % 8, SWIZZLE_128B), the second chunk stores the box
            const int h = (cb >> 5) & 1;
            unsigned char* sbox = stage;
            if (wi == nwork - 1) sbox = smem + F_SMEM_A + ((warp - 2) * (F_BN / 64) + (cb >> 6)) * F_STAGE;
            else if (0 == h) {
              if (0 == lane) asm volatile("cp.async.bulk.wait_group.read 0;\n" ::: "memory");
              __syncwarp();
            }
#pragma unroll
            for (int u = 0; u < 4; ++u)
              *(uint4*)(sbox + lane * 128 + (((4 * h + u) ^ (lane & 7)) << 4)) =
                make_uint4(bf16x2_rn(__uint_as_float(v[8 * u]), __uint_as_float(v[8 * u + 1])), bf16x2_rn(__uint_as_float(v[8 * u + 2]), __uint_as_float(v[8 * u + 3])),
                           bf16x2_rn(__uint_as_float(v[8 * u + 4]), __uint_as_float(v[8 * u + 5])), bf16x2_rn(__uint_as_float(v[8 * u + 6]), __uint_as_float(v[8 * u + 7])));
            if (h) {
              fence_proxy_async();
              __syncwarp();
              if (0 == lane) {
                asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%1, %2}], [%3];\n"
                             ::"l"(&tmC), "r"(n0 + cb - 32), "r"((int)(crow - (size_t)lane)), "r"(smem_u32(sbox)) : "memory");
                asm volatile("cp.async.bulk.commit_group;\n" ::: "memory");
              }
            }
          }
          else if (rvalid) {
            if (p.transc) {    // lanes hold consecutive m: per column the warp writes 64 contiguous bytes
              if (0.f != p.beta) {
#pragma unroll
                for (int jj = 0; jj < 32; ++jj) {
                  const int col = n0 + cb + jj;
                  if (col < p.N) v[jj] = __float_as_uint(fmaf(p.beta, bf16_value(cc[(size_t)col * p.ldc + crow]), __uint_as_float(v[jj])));
                }
              }
#pragma unroll
              for (int jj = 0; jj < 32; jj += 2) {
                const uint32_t w = bf16x2_rn(__uint_as_float(v[jj]), __uint_as_float(v[jj + 1]));
                const int col = n0 + cb + jj;
                if (col < p.N) cc[(size_t)col * p.ldc + crow] = (unsigned short)w;
                if (col + 1 < p.N) cc[(size_t)(col + 1) * p.ldc + crow] = (unsigned short)(w >> 16);
              }
            }
            else {             // 16-byte units of 8 bf16 where C allows them, element stores at the ragged end
              unsigned short* dst = cc + crow * p.ldc + n0 + cb;
#pragma unroll
              for (int jj = 0; jj < 32; jj += 8) {
                const int col = n0 + cb + jj;
                const bool vec = p.c_vec && col + 7 < p.N;
                if (0.f != p.beta) {
                  if (vec) {
                    const uint4 cin = *(const uint4*)(dst + jj);
                    const uint32_t cw[4] = { cin.x, cin.y, cin.z, cin.w };
#pragma unroll
                    for (int t2 = 0; t2 < 8; ++t2)
                      v[jj + t2] = __float_as_uint(fmaf(p.beta, bf16_value((unsigned short)(cw[t2 >> 1] >> (16 * (t2 & 1)))), __uint_as_float(v[jj + t2])));
                  }
                  else {
#pragma unroll
                    for (int t2 = 0; t2 < 8; ++t2)
                      if (col + t2 < p.N) v[jj + t2] = __float_as_uint(fmaf(p.beta, bf16_value(dst[jj + t2]), __uint_as_float(v[jj + t2])));
                  }
                }
                uint32_t w[4];
#pragma unroll
                for (int t2 = 0; t2 < 4; ++t2) w[t2] = bf16x2_rn(__uint_as_float(v[jj + 2 * t2]), __uint_as_float(v[jj + 2 * t2 + 1]));
                if (vec) st_global_cs_f4((float*)(dst + jj), make_float4(__uint_as_float(w[0]), __uint_as_float(w[1]), __uint_as_float(w[2]), __uint_as_float(w[3])));
                else {
#pragma unroll
                  for (int t2 = 0; t2 < 8; ++t2) if (col + t2 < p.N) dst[jj + t2] = (unsigned short)(w[t2 >> 1] >> (16 * (t2 & 1)));
                }
              }
            }
          }
        }
        else if (use_tma) {
          // as K4s: one box per warp, except in the pair's last tile, whose chunks each get a box in the idle ring
          unsigned char* sbox = stage;
          if (wi == nwork - 1) sbox = smem + F_SMEM_A + ((warp - 2) * (F_BN / 32) + (cb >> 5)) * F_STAGE;
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
                         ::"l"(&tmC), "r"(n0 + cb), "r"((int)(crow - (size_t)lane)), "r"(smem_u32(sbox)) : "memory");
            asm volatile("cp.async.bulk.commit_group;\n" ::: "memory");
          }
        }
        else if (rvalid) {
          if (p.transc) {
#pragma unroll
            for (int jj = 0; jj < 32; ++jj) {
              const int col = n0 + cb + jj;
              if (col < p.N) {
                float* dst = p.c + (size_t)col * p.ldc + crow;
                *dst = (0.f != p.beta) ? fmaf(p.beta, *dst, __uint_as_float(v[jj])) : __uint_as_float(v[jj]);
              }
            }
          }
          else {
            float* dst = p.c + crow * p.ldc + n0 + cb;
#pragma unroll
            for (int jj = 0; jj < 32; jj += 4) {
              const int col = n0 + cb + jj;
              float4 o = make_float4(__uint_as_float(v[jj]), __uint_as_float(v[jj + 1]), __uint_as_float(v[jj + 2]), __uint_as_float(v[jj + 3]));
              if (p.c_vec && col + 3 < p.N) {
                if (0.f != p.beta) {
                  const float4 cin = *(const float4*)(dst + jj);
                  o.x = fmaf(p.beta, cin.x, o.x); o.y = fmaf(p.beta, cin.y, o.y); o.z = fmaf(p.beta, cin.z, o.z); o.w = fmaf(p.beta, cin.w, o.w);
                }
                st_global_cs_f4(dst + jj, o);
              }
              else {
                const float e[4] = { o.x, o.y, o.z, o.w };
#pragma unroll
                for (int t2 = 0; t2 < 4; ++t2) if (col + t2 < p.N) dst[jj + t2] = (0.f != p.beta) ? fmaf(p.beta, dst[jj + t2], e[t2]) : e[t2];
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

// ---- create: compression -------------------------------------------------------------------------------------------------
// One thread per (row, 16-k span) of the padded image: the span's four groups give eight kept slots (16 bytes of the values
// image for bf16, 8 for FP8) and one 16-bit metadata word.  A group keeping three or four elements is counted; `first` keeps
// the smallest (row << 32 | group).  An element is kept when its bits without the sign lie in [1, keep_max]: ordered nonzeros,
// +-0 and NaN dropped (bf16 0x7F80, e4m3 0x7E, e5m2 0x7C: Inf kept).
template <typename T>
__global__ void __launch_bounds__(256)
sp24_compress_kernel(const T* __restrict__ a, long long lda, int M, int K, int K_pad, int nkb, uint32_t keep_max,
                     T* __restrict__ vals, unsigned char* __restrict__ meta, unsigned int* bad, unsigned long long* first)
{
  constexpr bool F8 = 1 == sizeof(T);
  constexpr uint32_t mag = F8 ? 0x7Fu : 0x7FFFu;
  const int spans = K_pad / 16;
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int row = (int)(t / spans), span = (int)(t % spans);
  if (row >= ((M + 127) & ~127)) return;
  uint32_t e[16];
#pragma unroll
  for (int i = 0; i < 16; ++i) {
    const int k = span * 16 + i;
    e[i] = (row < M && k < K) ? (uint32_t)__ldg(a + (size_t)row * lda + k) : 0u;
  }
  uint32_t kept[4] = { 0, 0, 0, 0 }, meta16 = 0;
#pragma unroll
  for (int gi = 0; gi < 4; ++gi) {
    uint32_t gm = 0;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const uint32_t h = e[4 * gi + q] & mag;
      if (h >= 1u && h <= keep_max) gm |= 1u << q;        // ordered nonzero, as the spmdm slicing kernels
    }
    if (__popc(gm) > 2) {
      atomicAdd(bad, 1u);
      atomicMin(first, ((unsigned long long)row << 32) | (unsigned long long)(span * 4 + gi));
    }
    meta16 |= xb_sp_nibble(gm) << (4 * gi);
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const uint32_t slot = xb_sp_slot(gm, (uint32_t)q);
      if (((gm >> q) & 1u) && slot < 2u) kept[gi] |= e[4 * gi + q] << (8 * sizeof(T) * slot);
    }
  }
  // kept slot 2 gi + s of the span = element hs * 8 + 2 gi + s of the row's kept elements in the k-block: row-major in the image
  const uint32_t rm = (uint32_t)row & 127u, kb = (uint32_t)span / (uint32_t)(F8 ? 16 : 8);
  unsigned char* img = meta + ((size_t)(row >> 7) * nkb + kb) * Sp24Geo<F8>::META;
  if constexpr (F8) {
    // FP8 image: [column half][lane = row][16 bytes]; the span's four groups are half (span & 1) of column (span & 15) / 2
    *(uint2*)(vals + (size_t)row * (K_pad / 2) + (size_t)span * 8) = make_uint2(kept[0] | (kept[1] << 16), kept[2] | (kept[3] << 16));
    const uint32_t s = (uint32_t)span & 15u, c = s >> 1;
    *(uint16_t*)(img + (c >> 2) * 2048u + rm * 16u + (c & 3u) * 4u + (s & 1u) * 2u) = (uint16_t)meta16;
  }
  else {
    *(uint4*)(vals + (size_t)row * (K_pad / 2) + (size_t)span * 8) = make_uint4(kept[0], kept[1], kept[2], kept[3]);
    *(uint16_t*)(img + xb_sp_meta_off(xb_sp_pos(rm, ((uint32_t)span & 7u) * 8u))) = (uint16_t)meta16;
  }
}

bool make_tensor_map_2d(CUtensorMap* map, const void* base, int elem_bytes, unsigned long long cols, unsigned long long rows,
                        unsigned long long row_pitch_bytes, unsigned box_cols, unsigned box_rows);
bool make_tensor_map_2d_sw128(CUtensorMap* map, const void* base, int elem_bytes, unsigned long long cols, unsigned long long rows,
                              unsigned long long row_pitch_bytes, unsigned box_cols, unsigned box_rows, bool atom32);
bool make_tensor_map_2d_u8(CUtensorMap* map, const void* base, unsigned long long cols, unsigned long long rows,
                           unsigned long long row_pitch_bytes, unsigned box_cols, unsigned box_rows, int swizzle_bytes);

struct Sp24Op {
  CUtensorMap tmA, tmE;
  int M, K, K_pad, M_pad, device;
  int format;           // -1: bf16, 0: e4m3, 1: e5m2
  void* mem;            // values image, then the metadata images
};

// format: -1 bf16 (a holds uint16_t), 0 / 1 FP8 e4m3 / e5m2 (a holds bytes)
Sp24Op* sp24_create(int M, int K, int lda, const void* a, bool a_on_device, int format)
{
  const bool f8 = format >= 0;
  const char* const who = f8 ? "sp24_create_fp8" : "sp24_create_bfloat16";
  const int esz = f8 ? 1 : 2, kbk = f8 ? Sp24Geo<true>::KB : Sp24Geo<false>::KB, meta_bytes = f8 ? Sp24Geo<true>::META : Sp24Geo<false>::META;
  int dev = 0;
  XB_CUDA(cudaGetDevice(&dev));
  const int M_pad = (M + 127) & ~127, K_pad = (K + kbk - 1) / kbk * kbk, nkb = K_pad / kbk;
  const size_t vbytes = (size_t)M_pad * (K_pad / 2) * esz, mbytes = (size_t)(M_pad / 128) * nkb * meta_bytes;     // values: M_pad x K_pad / 2 kept elements
  void* mem = 0; void* tmp = 0; unsigned long long* cnt = 0;
  Sp24Op* op = 0;
  bool ok = cudaSuccess == cudaMalloc(&mem, vbytes + mbytes) && cudaSuccess == cudaMalloc((void**)&cnt, 16);
  long long lda_d = lda;
  const void* src = a;
  if (ok && !a_on_device) {              // a host A is uploaded (packed) first, so there is one code path
    ok = cudaSuccess == cudaMalloc(&tmp, (size_t)M * K * esz) &&
         cudaSuccess == cudaMemcpy2D(tmp, (size_t)K * esz, a, (size_t)lda * esz, (size_t)K * esz, (size_t)M, cudaMemcpyHostToDevice);
    src = tmp; lda_d = K;
  }
  if (ok) {
    const unsigned long long init[2] = { 0ull, ~0ull };     // {violations, first}
    ok = cudaSuccess == cudaMemcpy(cnt, init, 16, cudaMemcpyHostToDevice);
  }
  if (ok) {
    const long long threads = (long long)M_pad * (K_pad / 16);
    const unsigned grid = (unsigned)((threads + 255) / 256);
    count_launch(1);
    if (f8) sp24_compress_kernel<uint8_t><<<grid, 256>>>((const uint8_t*)src, lda_d, M, K, K_pad, nkb, 0 == format ? 0x7Eu : 0x7Cu, (uint8_t*)mem,
                                                         (unsigned char*)mem + vbytes, (unsigned int*)cnt, cnt + 1);
    else sp24_compress_kernel<uint16_t><<<grid, 256>>>((const uint16_t*)src, lda_d, M, K, K_pad, nkb, 0x7F80u, (uint16_t*)mem,
                                                      (unsigned char*)mem + vbytes, (unsigned int*)cnt, cnt + 1);
    unsigned long long res[2] = { 0, 0 };
    ok = cudaSuccess == cudaGetLastError() && cudaSuccess == cudaMemcpy(res, cnt, 16, cudaMemcpyDeviceToHost);
    if (ok && 0 != (unsigned int)res[0]) {
      const int r = (int)(res[1] >> 32), g = (int)(res[1] & 0xFFFFFFFFu);
      set_error(-96, "%s: A is not 2:4: row %d, group %d (k = %d .. %d) keeps more than two elements (%u such groups)",
                who, r, g, 4 * g, min(4 * g + 3, K - 1), (unsigned int)res[0]);
      cudaFree(tmp); cudaFree(cnt); cudaFree(mem);
      return 0;
    }
  }
  if (ok) {
    op = new Sp24Op();
    op->M = M; op->K = K; op->K_pad = K_pad; op->M_pad = M_pad; op->device = dev; op->format = format; op->mem = mem;
    ok = (f8 ? make_tensor_map_2d_u8(&op->tmA, mem, (unsigned long long)K_pad / 2, (unsigned long long)M_pad, (unsigned long long)K_pad / 2, 128, F_BM, 128)
             : make_tensor_map_2d_sw128(&op->tmA, mem, 2, (unsigned long long)K_pad / 2, (unsigned long long)M_pad, (unsigned long long)K_pad, 64, F_BM, false)) &&
         make_tensor_map_2d(&op->tmE, (unsigned char*)mem + vbytes, 4, 32, (unsigned long long)(mbytes / 128), 128, 32, meta_bytes / 128);
  }
  if (!ok) {
    const cudaError_t e = cudaGetLastError();
    set_error(cudaSuccess != e ? (int)e : -95, "%s: %s", who, cudaSuccess != e ? cudaGetErrorString(e) : "tensor map of the compressed A");
    delete op; op = 0;
    cudaFree(mem);
  }
  cudaFree(tmp); cudaFree(cnt);
  return op;
}

int sp24_device(const Sp24Op* op) { return op->device; }
int sp24_rows(const Sp24Op* op) { return op->M; }
int sp24_cols(const Sp24Op* op) { return op->K; }
int sp24_format(const Sp24Op* op) { return op->format; }

void sp24_destroy(Sp24Op* op)
{
  if (0 == op) return;
  cudaFree(op->mem);
  delete op;
}

template <bool TB, bool F8, bool OB, typename Args>
static void launch_sp24(const Sp24Op* op, const CUtensorMap& mB, const CUtensorMap& mC, int c_tma, const Args& p, int pairs, cudaStream_t stream)
{
  ensure_smem_optin((const void*)sp24_compute_kernel<TB, F8, OB>, Sp24Geo<F8>::SMEM_BYTES);
  count_launch(1);
  note_compute_kernel(OB ? (F8 ? "sp24_compute_kernel_fp8_bf16out" : "sp24_compute_kernel_bf16out") : (F8 ? "sp24_compute_kernel_fp8" : "sp24_compute_kernel"));
  sp24_compute_kernel<TB, F8, OB><<<dim3(2u * (unsigned)pairs), dim3(F_THREADS), Sp24Geo<F8>::SMEM_BYTES, stream>>>(op->tmA, op->tmE, mB, mC, c_tma, p);
  XB_CUDA(cudaGetLastError());
}

// the part of the launch both kinds share: C's tensor map and the fields of Sp24Args (c_esz: 4 fp32 C, 2 bf16 C).
// false: B's map was refused (-97 set)
static bool sp24_prepare(const Sp24Op* op, bool okb, bool transc, int N, int ldb, float beta, void* d_c, int ldc, int c_esz, int kb,
                         CUtensorMap& mB, CUtensorMap& mC, int& c_tma, Sp24Args& p, int& pairs)
{
  if (!okb) { set_error(-97, "sp24_execute: B (N=%d, ldb=%d) cannot be described by a tensor map", N, ldb); return false; }
  // C leaves through TMA boxes of 32 rows x 128 bytes when it is only written and stored row-major, with whole 16-byte units
  // per row (a store box is clipped at the last column only to 16 bytes, DESIGN.md section 2)
  const bool c_vec = !transc && 0 == ((uintptr_t)d_c & 15) && 0 == (((long long)ldc * c_esz) & 15);
  c_tma = 0;
  mC = mB;
  if (c_vec && 0.f == beta && 0 == (((long long)N * c_esz) & 15) &&
      make_tensor_map_2d_sw128(&mC, d_c, c_esz, (unsigned long long)N, (unsigned long long)op->M, (unsigned long long)ldc * c_esz, 128 / c_esz, 32, false)) c_tma = 1;
  else mC = mB;
  p.c = (float*)d_c; p.ldc = ldc; p.M = op->M; p.N = N; p.nkb = op->K_pad / kb; p.ctiles_m = op->M_pad / F_BM; p.beta = beta;
  p.transc = transc ? 1 : 0; p.c_vec = c_vec ? 1 : 0;
  const int pairs_max = device_sm_count() / 2 > 0 ? device_sm_count() / 2 : 1;
  const int total = ((p.ctiles_m + 1) / 2) * ((N + F_BN - 1) / F_BN);
  pairs = total < pairs_max ? total : pairs_max;
  return true;
}

static bool sp24_map_b_bf16(CUtensorMap& mB, const Sp24Op* op, bool transb, int N, const uint16_t* d_b, int ldb)
{
  return transb ? make_tensor_map_2d_sw128(&mB, d_b, 2, (unsigned long long)op->K, (unsigned long long)N, (unsigned long long)ldb * 2, 64, 64, false)
                : make_tensor_map_2d_sw128(&mB, d_b, 2, (unsigned long long)N, (unsigned long long)op->K, (unsigned long long)ldb * 2, 64, Sp24Geo<false>::KB, false);
}

// FP8: B is read as bytes, 'T' in 128-byte boxes of k (SWIZZLE_128B), 'N' in 64-column boxes (SWIZZLE_64B)
static bool sp24_map_b_fp8(CUtensorMap& mB, const Sp24Op* op, bool transb, int N, const unsigned char* d_b, int ldb)
{
  return transb ? make_tensor_map_2d_u8(&mB, d_b, (unsigned long long)op->K, (unsigned long long)N, (unsigned long long)ldb, 128, 64, 128)
                : make_tensor_map_2d_u8(&mB, d_b, (unsigned long long)N, (unsigned long long)op->K, (unsigned long long)ldb, 64, Sp24Geo<true>::KB, 64);
}

// arguments checked by the caller (capi.cu); N > 0
void sp24_execute(const Sp24Op* op, bool transb, bool transc, int N, const uint16_t* d_b, int ldb, float beta, float* d_c, int ldc, cudaStream_t stream)
{
  CUtensorMap mB, mC;
  const bool okb = sp24_map_b_bf16(mB, op, transb, N, d_b, ldb);
  Sp24Args p;
  int c_tma = 0, pairs = 0;
  if (!sp24_prepare(op, okb, transc, N, ldb, beta, d_c, ldc, 4, Sp24Geo<false>::KB, mB, mC, c_tma, p, pairs)) return;
  if (transb) launch_sp24<true, false, false>(op, mB, mC, c_tma, p, pairs, stream);
  else launch_sp24<false, false, false>(op, mB, mC, c_tma, p, pairs, stream);
}

void sp24_execute_fp8(const Sp24Op* op, bool transb, bool transc, int N, const unsigned char* d_b, int b_format, int ldb, float alpha, float beta,
                      float* d_c, int ldc, cudaStream_t stream)
{
  constexpr int KB = Sp24Geo<true>::KB;
  CUtensorMap mB, mC;
  const bool okb = sp24_map_b_fp8(mB, op, transb, N, d_b, ldb);
  Sp24F8Args p;
  int c_tma = 0, pairs = 0;
  if (!sp24_prepare(op, okb, transc, N, ldb, beta, d_c, ldc, 4, KB, mB, mC, c_tma, p, pairs)) return;
  p.alpha = alpha;
  p.idesc_fmt = ((uint32_t)op->format << 7) | ((uint32_t)b_format << 10);
  if (transb) launch_sp24<true, true, false>(op, mB, mC, c_tma, p, pairs, stream);
  else launch_sp24<false, true, false>(op, mB, mC, c_tma, p, pairs, stream);
}

// bf16 C with an optional per-row bias (d_bias: NULL or M bf16 values); arguments checked by capi.cu; N > 0
void sp24_execute_bf16out(const Sp24Op* op, bool transb, bool transc, int N, const uint16_t* d_b, int ldb, const uint16_t* d_bias, float beta,
                          uint16_t* d_c, int ldc, cudaStream_t stream)
{
  CUtensorMap mB, mC;
  const bool okb = sp24_map_b_bf16(mB, op, transb, N, d_b, ldb);
  Sp24OutArgs<Sp24Args> p;
  int c_tma = 0, pairs = 0;
  if (!sp24_prepare(op, okb, transc, N, ldb, beta, d_c, ldc, 2, Sp24Geo<false>::KB, mB, mC, c_tma, p, pairs)) return;
  p.bias = d_bias;
  if (transb) launch_sp24<true, false, true>(op, mB, mC, c_tma, p, pairs, stream);
  else launch_sp24<false, false, true>(op, mB, mC, c_tma, p, pairs, stream);
}

void sp24_execute_fp8_bf16out(const Sp24Op* op, bool transb, bool transc, int N, const unsigned char* d_b, int b_format, int ldb, float alpha,
                              const uint16_t* d_bias, float beta, uint16_t* d_c, int ldc, cudaStream_t stream)
{
  constexpr int KB = Sp24Geo<true>::KB;
  CUtensorMap mB, mC;
  const bool okb = sp24_map_b_fp8(mB, op, transb, N, d_b, ldb);
  Sp24OutArgs<Sp24F8Args> p;
  int c_tma = 0, pairs = 0;
  if (!sp24_prepare(op, okb, transc, N, ldb, beta, d_c, ldc, 2, KB, mB, mC, c_tma, p, pairs)) return;
  p.alpha = alpha;
  p.idesc_fmt = ((uint32_t)op->format << 7) | ((uint32_t)b_format << 10);
  p.bias = d_bias;
  if (transb) launch_sp24<true, true, true>(op, mB, mC, c_tma, p, pairs, stream);
  else launch_sp24<false, true, true>(op, mB, mC, c_tma, p, pairs, stream);
}

}  // namespace xb
