// Developer probe: tcgen05.mma.sp kind::f8f6f4 (2:4 structured-sparse 8-bit A), single CTA, M = 128, N = 256, four K = 64
// atoms (256 logical k, 128 kept bytes per A row).
// A: compressed, K-major SWIZZLE_128B (one 128-byte swizzle row per A row); B in one of three layouts:
//   bmode 0: K-major SWIZZLE_128B ('T': B stored N x K), [k half][256 n rows][128 bytes];
//   bmode 1: MN-major SWIZZLE_64B ('N': B stored K x N), [64-column block][256 k rows][64 bytes];
//   bmode 2: MN-major SWIZZLE_128B, [128-column block][256 k rows][128 bytes].
// Metadata: eight TMEM columns, written with tcgen05.st or copied from a shared-memory image with two tcgen05.cp.128x128b.
// Phase 1 checks the hypothesised metadata layout (CUTLASS cute/atom/mma_traits_sm100.hpp, tmem_e_frg for 8-bit types,
// read not included: lane = row, bit k of the row's 64 per instruction, two columns per K = 64 atom) on random 2:4 patterns
// with exact small dyadic values, for every B layout and every pair of formats (e4m3 / e5m2); phase 2 maps every
// (lane, column, nibble) to the (row, group) it steers by multiplying with an identity B; phase 3 reads what each of the 16
// nibble values selects.  Result (profiles/sp24_fp8_probe.log): the hypothesis holds for every B layout and format pair,
// the nibbles mean what they mean for bf16, and the instruction descriptor's sparse selector bits must stay 0 for this kind
// (1 was tried once and is an illegal instruction), so the probe no longer sets them.
#include <cuda_runtime.h>
#include <cstdio>
#include <cstdint>
#include <cstring>
#include <cstdlib>
#include <vector>
#include <cmath>
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ uint64_t mkdesc(uint32_t saddr, uint32_t lbo, uint32_t sbo, uint32_t layout)
{
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3FFF);
  d |= (uint64_t)((lbo >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)layout << 61;
  return d;
}
constexpr int M = 128, N = 256, K = 256, KC = 128;
constexpr int MCOL = 256;   // metadata columns start here (accumulator: columns 0..255)
constexpr int SA = 0, SB = 16384, SIMG = 16384 + 65536, SMEM = SIMG + 4096 + 1024;
__device__ __forceinline__ void ld32(uint32_t taddr, uint32_t (&r)[32])
{
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n"
    : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
      "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
    : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;\n" ::: "memory");
}
__device__ __forceinline__ void st_meta(uint32_t taddr, const uint32_t (&w)[8])
{
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};\n"
               ::"r"(taddr), "r"(w[0]), "r"(w[1]), "r"(w[2]), "r"(w[3]), "r"(w[4]), "r"(w[5]), "r"(w[6]), "r"(w[7]) : "memory");
  asm volatile("tcgen05.wait::st.sync.aligned;\n" ::: "memory");
}
__host__ __device__ inline uint32_t b_off(int bmode, int k, int n)    // byte offset of logical B[k][n] in the staged tile
{
  if (0 == bmode) return (uint32_t)((k >> 7) * 32768 + (n >> 3) * 1024 + (n & 7) * 128 + (((((k & 127) >> 4) ^ (n & 7)) & 7) << 4) + (k & 15));
  if (1 == bmode) { const uint32_t o = (uint32_t)(k * 64 + (n & 63)); return (uint32_t)((n >> 6) * 16384) + (o ^ ((o >> 3) & 0x30u)); }
  const uint32_t o = (uint32_t)(k * 128 + (n & 127)); return (uint32_t)((n >> 7) * 32768) + (o ^ ((o >> 3) & 0x70u));
}
// mode 0: one multiply with the metadata words given per lane (meta[lane*8 + c]); D written out.
// mode 1: discovery: experiment e = (lane L, column c, nibble q) sets that nibble to 0xE; res[e] = 1 + row*64 + group that changed
// (0: none), cnt[e] = how many (row, group) cells changed.  mode 2: lane 0, column 0, nibble 0 takes every value v;
// pat[v*4 + i] = D[r0][4*g0 + i] for the (r0, g0) that experiment (0, 0, 0) found.
struct P { uint32_t idesc; int mode; int bmode; int meta_by_cp; uint32_t r0g0; };
__global__ void __launch_bounds__(128, 1) probe(const uint8_t* Ac, const uint8_t* B, const uint32_t* meta, float* D, float* base,
                                                uint32_t* res, uint32_t* cnt, float* pat, P p)
{
  extern __shared__ __align__(1024) unsigned char smem[];
  __shared__ uint64_t bar;
  __shared__ uint32_t slot;
  const int tid = threadIdx.x, warp = tid >> 5;
  unsigned char* sa = smem + SA; unsigned char* sb = smem + SB; unsigned char* simg = smem + SIMG;
  for (int i = tid; i < M * KC; i += 128) {
    const int m = i / KC, j = i % KC;
    sa[(m >> 3) * 1024 + (m & 7) * 128 + ((((j >> 4) ^ (m & 7)) & 7) << 4) + (j & 15)] = Ac[i];
  }
  for (int i = tid; i < K * N; i += 128) sb[b_off(p.bmode, i / N, i % N)] = B[i];
  if (0 == tid) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;\n" ::"r"(smem_u32(&bar)) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
  }
  if (0 == warp) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;\n" ::"r"(smem_u32(&slot)), "r"(512) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n" ::: "memory");
  }
  asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
  asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
  const uint32_t tm = slot;
  const uint32_t my_t = tm + ((uint32_t)(warp * 32) << 16);
  uint32_t phase = 0;
  auto multiply = [&](const uint32_t (&w)[8]) {
    if (p.meta_by_cp) {     // image: [column half][lane][16 bytes]
      *(uint4*)(simg + tid * 16) = make_uint4(w[0], w[1], w[2], w[3]);
      *(uint4*)(simg + 2048 + tid * 16) = make_uint4(w[4], w[5], w[6], w[7]);
      asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
    }
    else st_meta(my_t + MCOL, w);
    asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
    __syncthreads();
    if (0 == tid) {
      asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
      if (p.meta_by_cp) {
        for (int h = 0; h < 2; ++h) {
          const uint64_t dm = mkdesc(smem_u32(simg) + 2048 * h, 16, 128, 0);
          asm volatile("tcgen05.cp.cta_group::1.128x128b [%0], %1;\n" ::"r"(tm + MCOL + 4 * h), "l"(dm) : "memory");
        }
      }
      for (int ks = 0; ks < 4; ++ks) {   // K = 64 logical (32 kept bytes) per MMA
        const uint64_t da = mkdesc(smem_u32(sa) + ks * 32, 16, 1024, 2);
        const uint64_t db = 0 == p.bmode ? mkdesc(smem_u32(sb) + (ks >> 1) * 32768 + (ks & 1) * 64, 16, 1024, 2)
                          : 1 == p.bmode ? mkdesc(smem_u32(sb) + ks * 4096, 16384, 512, 4)
                                         : mkdesc(smem_u32(sb) + ks * 8192, 32768, 1024, 2);
        const uint32_t acc = ks > 0 ? 1u : 0u, te = tm + MCOL + 2 * ks;
        asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.b32 q, %5, 0;\n\ttcgen05.mma.sp.cta_group::1.kind::f8f6f4 [%0], %1, %2, [%3], %4, q;\n\t}\n"
                     ::"r"(tm), "l"(da), "l"(db), "r"(te), "r"(p.idesc), "r"(acc) : "memory");
      }
      asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n" ::"r"(smem_u32(&bar)) : "memory");
    }
    uint32_t ok = 0;
    while (!ok) asm volatile("{\n\t.reg .pred q;\n\tmbarrier.try_wait.parity.shared::cta.b64 q, [%1], %2;\n\tselp.u32 %0, 1, 0, q;\n\t}\n" : "=r"(ok) : "r"(smem_u32(&bar)), "r"(phase) : "memory");
    phase ^= 1;
    asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
  };
  uint32_t w[8];
  if (0 == p.mode) {
    for (int c = 0; c < 8; ++c) w[c] = meta[tid * 8 + c];
    multiply(w);
    for (int cb = 0; cb < N; cb += 32) {
      uint32_t r[32];
      ld32(my_t + cb, r);
      for (int j = 0; j < 32; ++j) D[tid * N + cb + j] = __uint_as_float(r[j]);
    }
  }
  else {
    // baseline: every nibble 0x4; B = identity, every kept element 1 (mode 1) or slot 0 = 1, slot 1 = 2 (mode 2)
    const int n_exp = (1 == p.mode) ? 128 * 8 * 8 : 16;
    for (int c = 0; c < 8; ++c) w[c] = 0x44444444u;
    multiply(w);
    for (int cb = 0; cb < N; cb += 32) { uint32_t r[32]; ld32(my_t + cb, r); for (int j = 0; j < 32; ++j) base[tid * N + cb + j] = __uint_as_float(r[j]); }
    asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
    __syncthreads();
    for (int e = 0; e < n_exp; ++e) {
      for (int c = 0; c < 8; ++c) w[c] = 0x44444444u;
      int L, c, q; uint32_t v;
      if (1 == p.mode) { L = e >> 6; c = (e >> 3) & 7; q = e & 7; v = 0xEu; }
      else { L = 0; c = 0; q = 0; v = (uint32_t)e; }
      if (tid == L) w[c] = (w[c] & ~(0xFu << (4 * q))) | (v << (4 * q));
      multiply(w);
      uint32_t changed = 0, first = 0;
      for (int cb = 0; cb < N; cb += 32) {
        uint32_t r[32];
        ld32(my_t + cb, r);
        if (1 == p.mode) {
          for (int gl = 0; gl < 8; ++gl) {
            const int g = (cb >> 2) + gl;
            bool same = true;
            for (int i = 0; i < 4; ++i) same = same && __uint_as_float(r[4 * gl + i]) == base[tid * N + 4 * g + i];
            if (!same) { if (0 == changed) first = 1u + (uint32_t)tid * 64u + (uint32_t)g; ++changed; }
          }
        }
        else {
          const uint32_t r0 = (p.r0g0 - 1) >> 6, g0 = (p.r0g0 - 1) & 63;
          if ((uint32_t)tid == r0 && (uint32_t)cb == (g0 >> 3) * 32) for (int i = 0; i < 4; ++i) pat[e * 4 + i] = __uint_as_float(r[4 * (g0 & 7) + i]);
        }
      }
      if (1 == p.mode && changed) { atomicAdd(&cnt[e], changed); res[e] = first; }
      asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
      __syncthreads();
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
  __syncthreads();
  if (0 == warp) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;\n" ::"r"(tm), "r"(512) : "memory");
}
// normal, exactly representable values only
static uint8_t enc(float v, int fmt)
{
  if (0.f == v) return 0;
  const int mb = fmt ? 2 : 3, bias = fmt ? 15 : 7;
  int e; const float m = frexpf(fabsf(v), &e);   // |v| = m * 2^e, m in [0.5, 1)
  const int ex = e - 1 + bias, man = (int)lrintf((m * 2.f - 1.f) * (float)(1 << mb));
  return (uint8_t)((v < 0 ? 0x80 : 0) | (ex << mb) | man);
}
static uint32_t nib(uint32_t gm) { return (((gm & 8u) ? 0x498E4DCEu : 0x498E4444u) >> ((gm & 7u) * 4u)) & 15u; }
int main()
{
  cudaDeviceProp prop; cudaGetDeviceProperties(&prop, 0);
  printf("device: %s (sm_%d%d)\n", prop.name, prop.major, prop.minor);
  std::vector<uint8_t> Ac(M * KC), B(K * N);
  std::vector<float> Ad(M * K, 0.f), Bf(K * N), D(M * N), E(M * N);
  std::vector<uint32_t> meta(M * 8, 0);
  uint8_t *dA, *dB; float *dD, *dBase, *dPat; uint32_t *dMeta, *dRes, *dCnt;
  cudaMalloc(&dA, Ac.size()); cudaMalloc(&dB, B.size()); cudaMalloc(&dD, D.size() * 4); cudaMalloc(&dBase, D.size() * 4);
  cudaMalloc(&dMeta, meta.size() * 4); cudaMalloc(&dRes, 8192 * 4); cudaMalloc(&dCnt, 8192 * 4); cudaMalloc(&dPat, 64 * 4);
  cudaFuncSetAttribute(probe, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM);
  auto idesc_of = [&](int fa, int fb, int bmode) {
    return (1u << 2) | (1u << 4) | ((uint32_t)fa << 7) | ((uint32_t)fb << 10) | (bmode ? (1u << 16) : 0u) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
  };
  // phase 1: random 2:4 patterns of {+-0.5, +-1, +-1.5, +-2, +-3}; hypothesis: lane = row, column = k / 32, bits 4 * (k % 32 / 4)
  const float vals[10] = { 0.5f, -0.5f, 1.f, -1.f, 1.5f, -1.5f, 2.f, -2.f, 3.f, -3.f };
  uint32_t rng = 12345u;
  auto rnd = [&]() { rng = rng * 1664525u + 1013904223u; return rng >> 8; };
  struct Case { int bmode, fa, fb, cp; };
  std::vector<Case> cases;
  for (int bm = 0; bm < 3; ++bm) for (int fa = 0; fa < 2; ++fa) for (int fb = 0; fb < 2; ++fb) cases.push_back({ bm, fa, fb, 0 });
  cases.push_back({ 0, 0, 0, 1 }); cases.push_back({ 1, 1, 0, 1 });
  for (const Case& cs : cases) {
    std::fill(Ad.begin(), Ad.end(), 0.f); std::fill(meta.begin(), meta.end(), 0u); std::fill(Ac.begin(), Ac.end(), (uint8_t)0);
    for (int m = 0; m < M; ++m) for (int g = 0; g < K / 4; ++g) {
      uint32_t gm;
      do gm = rnd() & 15u; while (__builtin_popcount(gm) > 2);
      int s = 0;
      for (int q = 0; q < 4; ++q) if ((gm >> q) & 1u) {
        const int slot = 0 == (gm & (gm - 1u)) ? (q & 1) : s++;
        const float v = vals[rnd() % 10];
        Ac[m * KC + 2 * g + slot] = enc(v, cs.fa); Ad[m * K + 4 * g + q] = v;
      }
      meta[m * 8 + g / 8] |= nib(gm) << (4 * (g % 8));
    }
    for (int i = 0; i < K * N; ++i) { Bf[i] = vals[rnd() % 10]; B[i] = enc(Bf[i], cs.fb); }
    for (int m = 0; m < M; ++m) for (int n = 0; n < N; ++n) { double s = 0; for (int k = 0; k < K; ++k) s += (double)Ad[m * K + k] * Bf[k * N + n]; E[m * N + n] = (float)s; }
    cudaMemcpy(dA, Ac.data(), Ac.size(), cudaMemcpyHostToDevice); cudaMemcpy(dB, B.data(), B.size(), cudaMemcpyHostToDevice);
    cudaMemcpy(dMeta, meta.data(), meta.size() * 4, cudaMemcpyHostToDevice);
    cudaMemset(dD, 0xFF, D.size() * 4);
    P p = { idesc_of(cs.fa, cs.fb, cs.bmode), 0, cs.bmode, cs.cp, 0 };
    probe<<<1, 128, SMEM>>>(dA, dB, dMeta, dD, dBase, dRes, dCnt, dPat, p);
    cudaError_t e = cudaDeviceSynchronize();
    if (e != cudaSuccess) { printf("phase 1 (bmode %d, A fmt %d, B fmt %d, cp %d): %s\n", cs.bmode, cs.fa, cs.fb, cs.cp, cudaGetErrorString(e)); return 1; }
    cudaMemcpy(D.data(), dD, D.size() * 4, cudaMemcpyDeviceToHost);
    int bad = 0; double maxerr = 0;
    for (int i = 0; i < M * N; ++i) { const double d = fabs((double)D[i] - E[i]); if (!(d == 0)) ++bad; if (d > maxerr || d != d) maxerr = d; }
    printf("phase 1 %s B (%s), A %s, B %s, metadata by %s: %d of %d differ from the exact product (max |err| %g)  D[0][0..3] = %g %g %g %g, exact %g %g %g %g\n",
           0 == cs.bmode ? "K-major SW128" : 1 == cs.bmode ? "MN-major SW64" : "MN-major SW128", cs.bmode ? "'N'" : "'T'",
           cs.fa ? "e5m2" : "e4m3", cs.fb ? "e5m2" : "e4m3", cs.cp ? "tcgen05.cp" : "tcgen05.st",
           bad, M * N, maxerr, D[0], D[1], D[2], D[3], E[0], E[1], E[2], E[3]);
    fflush(stdout);
  }
  // phase 2: identity B ('T' layout), every kept element 1.0
  for (int m = 0; m < M; ++m) for (int j = 0; j < KC; ++j) Ac[m * KC + j] = enc(1.f, 0);
  for (int k = 0; k < K; ++k) for (int n = 0; n < N; ++n) B[k * N + n] = enc(k == n ? 1.f : 0.f, 0);
  cudaMemcpy(dA, Ac.data(), Ac.size(), cudaMemcpyHostToDevice); cudaMemcpy(dB, B.data(), B.size(), cudaMemcpyHostToDevice);
  cudaMemset(dRes, 0, 8192 * 4); cudaMemset(dCnt, 0, 8192 * 4); cudaMemset(dPat, 0, 64 * 4);
  P p = { idesc_of(0, 0, 0), 1, 0, 0, 0 };
  probe<<<1, 128, SMEM>>>(dA, dB, dMeta, dD, dBase, dRes, dCnt, dPat, p);
  cudaError_t e = cudaDeviceSynchronize();
  if (e != cudaSuccess) { printf("phase 2: %s\n", cudaGetErrorString(e)); return 1; }
  std::vector<uint32_t> res(8192), cnt(8192);
  cudaMemcpy(res.data(), dRes, 8192 * 4, cudaMemcpyDeviceToHost); cudaMemcpy(cnt.data(), dCnt, 8192 * 4, cudaMemcpyDeviceToHost);
  int agree = 0, none = 0, multi = 0;
  for (int e2 = 0; e2 < 8192; ++e2) {
    const int L = e2 >> 6, c = (e2 >> 3) & 7, q = e2 & 7;
    if (0 == res[e2]) { ++none; continue; }
    if (cnt[e2] > 1) ++multi;
    const int row = (int)(res[e2] - 1) >> 6, g = (int)(res[e2] - 1) & 63;
    if (row == L && g == 8 * c + q) ++agree;
  }
  printf("phase 2: %d of 8192 nibbles (128 lanes x 8 columns x 8) agree with lane = row, column = group / 8, nibble = group %% 8; %d steer nothing, %d steer several cells\n", agree, none, multi);
  for (int e2 = 0; e2 < 8192; e2 += 1031)
    printf("  lane %3d col %d nib %d -> row %3d group %2d (cells %u)\n", e2 >> 6, (e2 >> 3) & 7, e2 & 7,
           res[e2] ? (int)((res[e2] - 1) >> 6) : -1, res[e2] ? (int)((res[e2] - 1) & 63) : -1, cnt[e2]);
  // phase 3: nibble semantics, kept slot 0 = 1, slot 1 = 2
  if (res[0]) {
    for (int m = 0; m < M; ++m) for (int j = 0; j < KC; ++j) Ac[m * KC + j] = enc((j & 1) ? 2.f : 1.f, 0);
    cudaMemcpy(dA, Ac.data(), Ac.size(), cudaMemcpyHostToDevice);
    P p2 = { idesc_of(0, 0, 0), 2, 0, 0, res[0] };
    probe<<<1, 128, SMEM>>>(dA, dB, dMeta, dD, dBase, dRes, dCnt, dPat, p2);
    cudaDeviceSynchronize();
    float pat[64]; cudaMemcpy(pat, dPat, sizeof pat, cudaMemcpyDeviceToHost);
    for (int v = 0; v < 16; ++v) printf("  nibble 0x%X -> group reads %g %g %g %g (kept slot 0 = 1, slot 1 = 2)\n", v, pat[4 * v], pat[4 * v + 1], pat[4 * v + 2], pat[4 * v + 3]);
  }
  return 0;
}
