// Developer probe: sustained DFMA and FFMA throughput of the whole device (the FMA floors of tools/time_rm_soa.py).
//     nvcc -gencode arch=compute_100a,code=sm_100a -O3 -o fma_peak tools/fma_peak.cu && ./fma_peak
// Every thread runs kChains independent chains of fused multiply-adds (enough to hide the pipe latency), the grid fills every
// SM several times over; the best of several timed launches is reported as one JSON line per precision.
#include <cuda_runtime.h>
#include <cstdio>

constexpr int kChains = 8;

template <typename T>
__global__ void __launch_bounds__(256) fma_loop(T* out, T a, T b, int iters)
{
  T x[kChains];
#pragma unroll
  for (int i = 0; i < kChains; ++i) x[i] = (T)(threadIdx.x + i) * (T)1e-3;
  for (int it = 0; it < iters; ++it) {
#pragma unroll
    for (int u = 0; u < 16; ++u)
#pragma unroll
      for (int i = 0; i < kChains; ++i) x[i] = fma(x[i], a, b);
  }
  T s = 0;
#pragma unroll
  for (int i = 0; i < kChains; ++i) s += x[i];
  if (s == (T)-1) out[blockIdx.x * blockDim.x + threadIdx.x] = s;       // never true; keeps the chains alive
}

template <typename T>
static void run(const char* name, int sms)
{
  const int threads = 256, blocks = sms * 8, iters = sizeof(T) == 8 ? 2048 : 8192;
  T* out = 0;
  cudaMalloc(&out, (size_t)blocks * threads * sizeof(T));
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0); cudaEventCreate(&e1);
  fma_loop<T><<<blocks, threads>>>(out, (T)0.999999, (T)1e-7, iters);   // warm-up
  float best = 1e30f;
  for (int r = 0; r < 10; ++r) {
    cudaEventRecord(e0);
    fma_loop<T><<<blocks, threads>>>(out, (T)0.999999, (T)1e-7, iters);
    cudaEventRecord(e1);
    cudaEventSynchronize(e1);
    float ms = 0;
    cudaEventElapsedTime(&ms, e0, e1);
    if (ms < best) best = ms;
  }
  const double flops = 2.0 * kChains * 16 * (double)iters * threads * blocks;
  printf("{\"probe\": \"%s\", \"tflops\": %.3f, \"best_ms\": %.4f, \"flops\": %.6g, \"blocks\": %d, \"threads\": %d}\n", name,
         flops / (best * 1e-3) / 1e12, best, flops, blocks, threads);
  cudaEventDestroy(e0); cudaEventDestroy(e1);
  cudaFree(out);
}

int main()
{
  cudaDeviceProp p;
  if (cudaSuccess != cudaGetDeviceProperties(&p, 0)) { fprintf(stderr, "no CUDA device\n"); return 1; }
  printf("{\"device\": \"%s\", \"sms\": %d}\n", p.name, p.multiProcessorCount);
  run<double>("dfma", p.multiProcessorCount);
  run<float>("ffma", p.multiProcessorCount);
  const cudaError_t e = cudaGetLastError();
  if (cudaSuccess != e) { fprintf(stderr, "%s\n", cudaGetErrorString(e)); return 1; }
  return 0;
}
