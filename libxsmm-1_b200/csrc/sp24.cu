// Fixed 2:4-sparse bf16 operators (libxsmm_b200_sp24_*).  A matrix with at most two kept elements in every aligned
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
#include "common.cuh"
#include "tc_common.cuh"

namespace xb {

constexpr int F_BM = 128;                       // rows per CTA
constexpr int F_BN = 256;                       // columns per pair tile
constexpr int F_BNH = 128;                      // columns of B staged per CTA
constexpr int F_KB = 128;                       // k per ring slot
constexpr int F_NA = 4;                         // ring slots (a fifth does not fit: 5 x 50 KiB > 227 KiB)
constexpr int F_NE = 4;                         // epilogue warps (one per TMEM lane quarter)
constexpr int F_A_BUF = F_BM * 128;             // 16 KiB: 128 rows x 64 kept bf16
constexpr int F_META = F_BM * 16;               // 2 KiB: per TMEM lane four 32-bit metadata columns
constexpr int F_B_STAGE = F_KB * F_BNH * 2;     // 32 KiB
constexpr int F_THREADS = (2 + F_NE) * 32;
constexpr int F_SMEM_A = 0;
constexpr int F_SMEM_B = F_SMEM_A + F_NA * F_A_BUF;
constexpr int F_SMEM_META = F_SMEM_B + F_NA * F_B_STAGE;
constexpr int F_SMEM_STAGE = F_SMEM_META + F_NA * F_META;            // per epilogue warp a [32 rows x 32 columns] fp32 box for the TMA store of C
constexpr int F_STAGE = 32 * 128;
constexpr int F_SMEM_BAR = F_SMEM_STAGE + F_NE * F_STAGE;
constexpr int F_SMEM_BYTES = F_SMEM_BAR + 256;
static_assert(0 == (F_SMEM_STAGE & 1023), "SWIZZLE_128B boxes sit on 1 KiB boundaries");
static_assert(F_NE * (F_BN / 32) * F_STAGE <= F_SMEM_META, "the last tile's C boxes fit in the (then idle) A / B ring");
static_assert(F_SMEM_BYTES <= 227 * 1024, "shared memory");

struct Sp24Args {
  float* c;
  long long ldc;
  int M, N, nkb, ctiles_m;
  float beta;
  int transc;
  int c_vec;            // C and ldc allow 16-byte stores (transc = 'N')
};

template <bool TB>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(F_THREADS, 1)
sp24_compute_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmE, const __grid_constant__ CUtensorMap tmB,
                    const __grid_constant__ CUtensorMap tmC, const int c_tma, const Sp24Args p)
{
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
          if (TB) {      // K-major: [k half][128 n rows x 64 k], boxes of 64 n rows
            for (int kh = 0; kh < 2; ++kh) {
              tma_load_2d_pair(dst + kh * (F_B_STAGE / 2), &tmB, kbi * F_KB + kh * 64, n0, lbar);
              if (half < 0) tma_load_2d_pair(dst + kh * (F_B_STAGE / 2) + 64 * 128, &tmB, kbi * F_KB + kh * 64, n0 + 64, lbar);
            }
          }
          else {         // MN-major: [column block][128 k rows x 64 columns]
            tma_load_2d_pair(dst, &tmB, n0, kbi * F_KB, lbar);
            if (half < 0) tma_load_2d_pair(dst + F_KB * 128, &tmB, n0 + 64, kbi * F_KB, lbar);
          }
        }
      }
    }
  }
  else if (1 == warp) {
    // ---------------- MMA issuer (leader CTA) ----------------
    if (0 == rank && 0 == lane) {
      // sparse A, D = F32, A = B = BF16, A K-major (compressed), B MN-major ('N') or K-major ('T'), N = 256, M = 256 (pair)
      const uint32_t idesc = (1u << 2) | (1u << 4) | (1u << 7) | (1u << 10) | (TB ? 0u : (1u << 16)) | ((uint32_t)(F_BN >> 3) << 17) | ((uint32_t)((2 * F_BM) >> 4) << 24);
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
          const uint64_t dm = tc_smem_desc(sbase + F_SMEM_META + j * F_META, 16, 128, 0);
          asm volatile("tcgen05.cp.cta_group::2.128x128b [%0], %1;\n" ::"r"(tmeta + 4u * j), "l"(dm) : "memory");
#pragma unroll
          for (int ks = 0; ks < 4; ++ks) {         // K = 32 (16 kept elements = 32 bytes of the compressed row) per instruction
            const uint64_t da = tc_smem_desc(a_base + ks * 32, 16, 1024, 2);
            const uint64_t db = TB ? tc_smem_desc(b_base + (ks >> 1) * (F_B_STAGE / 2) + (ks & 1) * 64, 16, 1024, 2)
                                   : tc_smem_desc(b_base + ks * 4096, (uint32_t)(F_KB * 128), 1024, 2);
            tc_mma_bf16_sp_pair(tacc, da, db, tmeta + 4u * j + (uint32_t)(ks & 2), idesc_w | (uint32_t)(ks & 1), (kbi > 0 || ks > 0) ? 1u : 0u);
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
#pragma unroll 1
      for (int cb = 0; cb < ncw; cb += 32) {
        uint32_t v[32];
        tc_ld32(tmem_d + acc * F_BN + ((uint32_t)(quarter * 32) << 16) + (uint32_t)cb, v);
        if (0 == cb) {         // columns 0..31 of this accumulator are read: the next tile's metadata may go there
          tc_fence_before();
          __syncwarp();
          if (0 == lane) mbar_arrive_cluster(lead_meta);
        }
        if (use_tma) {
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
// image) and one 16-bit metadata word.  A group keeping three or four elements is counted; `first` keeps the smallest
// (row << 32 | group).
__global__ void __launch_bounds__(256)
sp24_compress_kernel(const uint16_t* __restrict__ a, long long lda, int M, int K, int K_pad, int nkb,
                     uint16_t* __restrict__ vals, unsigned char* __restrict__ meta, unsigned int* bad, unsigned long long* first)
{
  const int spans = K_pad / 16;
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int row = (int)(t / spans), span = (int)(t % spans);
  if (row >= ((M + 127) & ~127)) return;
  uint16_t e[16];
#pragma unroll
  for (int i = 0; i < 16; ++i) {
    const int k = span * 16 + i;
    e[i] = (row < M && k < K) ? __ldg(a + (size_t)row * lda + k) : (uint16_t)0;
  }
  uint32_t kept[4] = { 0, 0, 0, 0 }, meta16 = 0;
#pragma unroll
  for (int gi = 0; gi < 4; ++gi) {
    uint32_t gm = 0;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const uint32_t h = e[4 * gi + q] & 0x7FFFu;
      if (h >= 1u && h <= 0x7F80u) gm |= 1u << q;        // ordered nonzero: +-0 and NaN dropped, as the spmdm slicing kernels
    }
    if (__popc(gm) > 2) {
      atomicAdd(bad, 1u);
      atomicMin(first, ((unsigned long long)row << 32) | (unsigned long long)(span * 4 + gi));
    }
    meta16 |= xb_sp_nibble(gm) << (4 * gi);
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const uint32_t slot = xb_sp_slot(gm, (uint32_t)q);
      if (((gm >> q) & 1u) && slot < 2u) kept[gi] |= (uint32_t)e[4 * gi + q] << (16 * slot);
    }
  }
  // kept slot 2 gi + s of the span = element hs * 8 + 2 gi + s of the row's 64 in the k-block: row-major in the image
  *(uint4*)(vals + (size_t)row * (K_pad / 2) + (size_t)span * 8) = make_uint4(kept[0], kept[1], kept[2], kept[3]);
  const uint32_t rm = (uint32_t)row & 127u, kb = (uint32_t)span >> 3;
  *(uint16_t*)(meta + ((size_t)(row >> 7) * nkb + kb) * F_META + xb_sp_meta_off(xb_sp_pos(rm, ((uint32_t)span & 7u) * 8u))) = (uint16_t)meta16;
}

bool make_tensor_map_2d(CUtensorMap* map, const void* base, int elem_bytes, unsigned long long cols, unsigned long long rows,
                        unsigned long long row_pitch_bytes, unsigned box_cols, unsigned box_rows);
bool make_tensor_map_2d_sw128(CUtensorMap* map, const void* base, int elem_bytes, unsigned long long cols, unsigned long long rows,
                              unsigned long long row_pitch_bytes, unsigned box_cols, unsigned box_rows, bool atom32);

struct Sp24Op {
  CUtensorMap tmA, tmE;
  int M, K, K_pad, M_pad, device;
  void* mem;            // values image, then the metadata images
};

Sp24Op* sp24_create(int M, int K, int lda, const uint16_t* a, bool a_on_device)
{
  int dev = 0;
  XB_CUDA(cudaGetDevice(&dev));
  const int M_pad = (M + 127) & ~127, K_pad = (K + 127) & ~127, nkb = K_pad / 128;
  const size_t vbytes = (size_t)M_pad * K_pad, mbytes = (size_t)(M_pad / 128) * nkb * F_META;     // values: M_pad x K_pad / 2 bf16
  void* mem = 0; void* tmp = 0; unsigned long long* cnt = 0;
  Sp24Op* op = 0;
  bool ok = cudaSuccess == cudaMalloc(&mem, vbytes + mbytes) && cudaSuccess == cudaMalloc((void**)&cnt, 16);
  long long lda_d = lda;
  const uint16_t* src = a;
  if (ok && !a_on_device) {              // a host A is uploaded (packed) first, so there is one code path
    ok = cudaSuccess == cudaMalloc(&tmp, (size_t)M * K * 2) &&
         cudaSuccess == cudaMemcpy2D(tmp, (size_t)K * 2, a, (size_t)lda * 2, (size_t)K * 2, (size_t)M, cudaMemcpyHostToDevice);
    src = (const uint16_t*)tmp; lda_d = K;
  }
  if (ok) {
    const unsigned long long init[2] = { 0ull, ~0ull };     // {violations, first}
    ok = cudaSuccess == cudaMemcpy(cnt, init, 16, cudaMemcpyHostToDevice);
  }
  if (ok) {
    const long long threads = (long long)M_pad * (K_pad / 16);
    count_launch(1);
    sp24_compress_kernel<<<(unsigned)((threads + 255) / 256), 256>>>(src, lda_d, M, K, K_pad, nkb, (uint16_t*)mem, (unsigned char*)mem + vbytes,
                                                                     (unsigned int*)cnt, cnt + 1);
    unsigned long long res[2] = { 0, 0 };
    ok = cudaSuccess == cudaGetLastError() && cudaSuccess == cudaMemcpy(res, cnt, 16, cudaMemcpyDeviceToHost);
    if (ok && 0 != (unsigned int)res[0]) {
      const int r = (int)(res[1] >> 32), g = (int)(res[1] & 0xFFFFFFFFu);
      set_error(-96, "sp24_create_bfloat16: A is not 2:4: row %d, group %d (k = %d .. %d) keeps more than two elements (%u such groups)",
                r, g, 4 * g, min(4 * g + 3, K - 1), (unsigned int)res[0]);
      cudaFree(tmp); cudaFree(cnt); cudaFree(mem);
      return 0;
    }
  }
  if (ok) {
    op = new Sp24Op();
    op->M = M; op->K = K; op->K_pad = K_pad; op->M_pad = M_pad; op->device = dev; op->mem = mem;
    ok = make_tensor_map_2d_sw128(&op->tmA, mem, 2, (unsigned long long)K_pad / 2, (unsigned long long)M_pad, (unsigned long long)K_pad, 64, F_BM, false) &&
         make_tensor_map_2d(&op->tmE, (unsigned char*)mem + vbytes, 4, 32, (unsigned long long)(mbytes / 128), 128, 32, F_META / 128);
  }
  if (!ok) {
    const cudaError_t e = cudaGetLastError();
    set_error(cudaSuccess != e ? (int)e : -95, "sp24_create_bfloat16: %s", cudaSuccess != e ? cudaGetErrorString(e) : "tensor map of the compressed A");
    delete op; op = 0;
    cudaFree(mem);
  }
  cudaFree(tmp); cudaFree(cnt);
  return op;
}

int sp24_device(const Sp24Op* op) { return op->device; }
int sp24_rows(const Sp24Op* op) { return op->M; }
int sp24_cols(const Sp24Op* op) { return op->K; }

void sp24_destroy(Sp24Op* op)
{
  if (0 == op) return;
  cudaFree(op->mem);
  delete op;
}

template <bool TB>
static void launch_sp24(const Sp24Op* op, const CUtensorMap& mB, const CUtensorMap& mC, int c_tma, const Sp24Args& p, int pairs, cudaStream_t stream)
{
  ensure_smem_optin((const void*)sp24_compute_kernel<TB>, F_SMEM_BYTES);
  count_launch(1);
  note_compute_kernel("sp24_compute_kernel");
  sp24_compute_kernel<TB><<<dim3(2u * (unsigned)pairs), dim3(F_THREADS), F_SMEM_BYTES, stream>>>(op->tmA, op->tmE, mB, mC, c_tma, p);
  XB_CUDA(cudaGetLastError());
}

// arguments checked by the caller (capi.cu); N > 0
void sp24_execute(const Sp24Op* op, bool transb, bool transc, int N, const uint16_t* d_b, int ldb, float beta, float* d_c, int ldc, cudaStream_t stream)
{
  CUtensorMap mB, mC;
  const bool okb = transb ? make_tensor_map_2d_sw128(&mB, d_b, 2, (unsigned long long)op->K, (unsigned long long)N, (unsigned long long)ldb * 2, 64, 64, false)
                          : make_tensor_map_2d_sw128(&mB, d_b, 2, (unsigned long long)N, (unsigned long long)op->K, (unsigned long long)ldb * 2, 64, F_KB, false);
  if (!okb) { set_error(-97, "sp24_execute: B (N=%d, ldb=%d) cannot be described by a tensor map", N, ldb); return; }
  // C leaves through TMA boxes of 32 x 32 when it is only written and stored row-major, with whole 16-byte units per row
  // (a store box is clipped at the last column only to 16 bytes, DESIGN.md section 2)
  const bool c_vec = !transc && 0 == ((uintptr_t)d_c & 15) && 0 == (ldc & 3);
  int c_tma = 0;
  mC = mB;
  if (c_vec && 0.f == beta && 0 == (N & 3) && make_tensor_map_2d_sw128(&mC, d_c, 4, (unsigned long long)N, (unsigned long long)op->M, (unsigned long long)ldc * 4, 32, 32, false)) c_tma = 1;
  else mC = mB;
  Sp24Args p;
  p.c = d_c; p.ldc = ldc; p.M = op->M; p.N = N; p.nkb = op->K_pad / F_KB; p.ctiles_m = op->M_pad / F_BM; p.beta = beta;
  p.transc = transc ? 1 : 0; p.c_vec = c_vec ? 1 : 0;
  const int pairs_max = device_sm_count() / 2 > 0 ? device_sm_count() / 2 : 1;
  const int total = ((p.ctiles_m + 1) / 2) * ((N + F_BN - 1) / F_BN);
  const int pairs = total < pairs_max ? total : pairs_max;
  if (transb) launch_sp24<true>(op, mB, mC, c_tma, p, pairs, stream);
  else launch_sp24<false>(op, mB, mC, c_tma, p, pairs, stream);
}

}  // namespace xb
