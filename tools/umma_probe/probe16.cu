// Developer probe: 128x128x64 BF16 tcgen05.mma chain; A K-major SWIZZLE_128B, B MN-major SWIZZLE_128B (the [k][n] tile a TMA
// box of 64 columns lands), to pin LBO / SBO / k-step for the bf16 tensor-core kernels (spmdm_compute_tc16p.cu).
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cstdio>
#include <cstdint>
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
struct P { uint32_t b_lbo, b_sbo, b_kstep, idesc; int fill_mode; };
__global__ void __launch_bounds__(128, 1) probe(const uint16_t* A, const uint16_t* B, float* D, P p)
{
  extern __shared__ __align__(1024) unsigned char smem[];
  __shared__ uint64_t bar;
  __shared__ uint32_t slot;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  unsigned char* sa = smem; unsigned char* sb = smem + 16384;
  for (int i = tid; i < 32768 / 4; i += 128) ((uint32_t*)smem)[i] = 0;
  __syncthreads();
  for (int i = tid; i < 128 * 64; i += 128) {   // A[m][k], K-major SW128: rows of 64 bf16
    const int m = i / 64, k = i % 64;
    const uint32_t off = (m >> 3) * 1024 + (m & 7) * 128 + ((((k >> 3) ^ (m & 7)) & 7) << 4) + ((k & 7) << 1);
    *(uint16_t*)(sa + off) = A[m * 64 + k];
  }
  for (int i = tid; i < 64 * 128; i += 128) {   // B[k][n], MN-major SW128: [n block of 64][k][128 B]
    const int k = i / 128, n = i % 128;
    const uint32_t off = (n >> 6) * 8192 + k * 128 + (((((n & 63) >> 3) ^ (k & 7)) & 7) << 4) + ((n & 7) << 1);
    *(uint16_t*)(sb + off) = B[k * 128 + n];
  }
  if (0 == tid) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;\n" ::"r"(smem_u32(&bar)) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
  }
  if (0 == warp) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;\n" ::"r"(smem_u32(&slot)), "r"(128) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n" ::: "memory");
  }
  asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
  asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
  const uint32_t tm = slot;
  if (0 == tid) {
    for (int ks = 0; ks < 4; ++ks) {   // K = 16 per MMA
      const uint64_t da = mkdesc(smem_u32(sa) + ks * 32, 16, 1024, 2);
      const uint64_t db = mkdesc(smem_u32(sb) + ks * p.b_kstep, p.b_lbo, p.b_sbo, 2);
      const uint32_t acc = ks > 0 ? 1u : 0u;
      asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.b32 q, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, q;\n\t}\n"
                   ::"r"(tm), "l"(da), "l"(db), "r"(p.idesc), "r"(acc) : "memory");
    }
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n" ::"r"(smem_u32(&bar)) : "memory");
  }
  {
    uint32_t ok = 0;
    while (!ok) asm volatile("{\n\t.reg .pred q;\n\tmbarrier.try_wait.parity.shared::cta.b64 q, [%1], %2;\n\tselp.u32 %0, 1, 0, q;\n\t}\n" : "=r"(ok) : "r"(smem_u32(&bar)), "r"(0) : "memory");
  }
  asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
  for (int cb = 0; cb < 128; cb += 32) {
    uint32_t r[32];
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
        "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(tm + ((uint32_t)(warp * 32) << 16) + cb));
    asm volatile("tcgen05.wait::ld.sync.aligned;\n" ::: "memory");
    for (int j = 0; j < 32; ++j) D[(warp * 32 + lane) * 128 + cb + j] = __uint_as_float(r[j]);
  }
  asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
  __syncthreads();
  if (0 == warp) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;\n" ::"r"(tm), "r"(128) : "memory");
}
static uint16_t f2bf(float f) { uint32_t u; memcpy(&u, &f, 4); return (uint16_t)(u >> 16); }
int main()
{
  std::vector<uint16_t> A(128 * 64), B(64 * 128);
  std::vector<float> Af(128 * 64), Bf(64 * 128), D(128 * 128), E(128 * 128, 0.f);
  for (int i = 0; i < 128 * 64; ++i) { Af[i] = (float)((i * 7 + 3) % 11 - 5); A[i] = f2bf(Af[i]); }
  for (int i = 0; i < 64 * 128; ++i) { Bf[i] = (float)((i * 5 + 1) % 13 - 6); B[i] = f2bf(Bf[i]); }
  for (int m = 0; m < 128; ++m) for (int n = 0; n < 128; ++n) { float s = 0; for (int k = 0; k < 64; ++k) s += Af[m * 64 + k] * Bf[k * 128 + n]; E[m * 128 + n] = s; }
  uint16_t *dA, *dB; float* dD;
  cudaMalloc(&dA, A.size() * 2); cudaMalloc(&dB, B.size() * 2); cudaMalloc(&dD, D.size() * 4);
  cudaMemcpy(dA, A.data(), A.size() * 2, cudaMemcpyHostToDevice); cudaMemcpy(dB, B.data(), B.size() * 2, cudaMemcpyHostToDevice);
  cudaFuncSetAttribute(probe, cudaFuncAttributeMaxDynamicSharedMemorySize, 32768 + 1024);
  const uint32_t base = (1u << 4) | (1u << 7) | (1u << 10) | (16u << 17) | (8u << 24) | (1u << 16);
  struct { const char* name; P p; } cases[] = {
    { "B MN SW128 lbo=8192 sbo=1024 kstep=2048", { 8192, 1024, 2048, base, 0 } },
    { "B MN SW128 lbo=1024 sbo=8192 kstep=2048", { 1024, 8192, 2048, base, 0 } },
  };
  for (auto& c : cases) {
    cudaMemset(dD, 0xFF, D.size() * 4);
    probe<<<1, 128, 32768 + 1024>>>(dA, dB, dD, c.p);
    cudaError_t e = cudaDeviceSynchronize();
    if (e != cudaSuccess) { printf("%s: %s\n", c.name, cudaGetErrorString(e)); break; }
    cudaMemcpy(D.data(), dD, D.size() * 4, cudaMemcpyDeviceToHost);
    double maxerr = 0; int bad = 0;
    for (int i = 0; i < 128 * 128; ++i) { double d = fabs((double)D[i] - E[i]); if (!(d <= 1e-3)) ++bad; if (d > maxerr) maxerr = d; }
    printf("%s: bad=%d maxerr=%g  D[0..3]=%g %g %g %g  E=%g %g %g %g\n", c.name, bad, maxerr, D[0], D[1], D[2], D[3], E[0], E[1], E[2], E[3]);
  }
  return 0;
}
