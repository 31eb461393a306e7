// Probe: cost of double-precision exp / log1p (the correctly rounded fp32 exp the trainers share with the oracle) next to
// expf / log1pf and a plain DFMA chain on this GPU. One warp per "triple", like the BPR kernels: 2,048 warps x REPS calls.
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -o scripts/bin/fp64_probe scripts/fp64_probe.cu
#include <cuda_runtime.h>
#include <stdio.h>
#define CK(x) do { cudaError_t e = (x); if (e != cudaSuccess) { printf("CUDA error %s line %d\n", cudaGetErrorString(e), __LINE__); return 1; } } while (0)
template <int MODE> __global__ void probe(const float* in, float* out, int reps) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  float x = in[t & 1023];
  float acc = 0.f;
  double dacc = 1.0;
  for (int r = 0; r < reps; ++r) {
    if (MODE == 0) { acc += log1pf(expf(-fabsf(x))); x += 1e-3f; }
    if (MODE == 1) { acc += (float)log1p((double)(float)exp((double)(-fabsf(x)))); x += 1e-3f; }
    if (MODE == 2) { acc += (float)exp((double)(-fabsf(x))); x += 1e-3f; }
    if (MODE == 3) { dacc = fma(dacc, 1.0000001, 1e-9); }
  }
  out[t] = acc + (float)dacc;
}
template <int MODE> static float run(const float* in, float* out, int reps, int blocks) {
  cudaEvent_t a, b; cudaEventCreate(&a); cudaEventCreate(&b);
  probe<MODE><<<blocks, 512>>>(in, out, reps);
  cudaDeviceSynchronize();
  cudaEventRecord(a);
  probe<MODE><<<blocks, 512>>>(in, out, reps);
  cudaEventRecord(b); cudaEventSynchronize(b);
  float ms = 0; cudaEventElapsedTime(&ms, a, b);
  return ms * 1000.f;
}
int main() {
  float *in, *out; CK(cudaMalloc(&in, 4096)); CK(cudaMalloc(&out, 148 * 16 * 32 * 4 * 4));
  float h[1024]; for (int i = 0; i < 1024; ++i) h[i] = 0.01f * i - 3.f;
  CK(cudaMemcpy(in, h, 4096, cudaMemcpyHostToDevice));
  const int reps = 64, blocks = 148;     // 148 CTAs x 16 warps = 2,368 warps (the BPR-MF trainer's grid)
  printf("per call, 2,368 warps each evaluating the function once (all 32 lanes):\n");
  printf("  log1pf(expf(x))               %8.3f us\n", run<0>(in, out, reps, blocks) / reps);
  printf("  (float)log1p((float)exp(dbl)) %8.3f us\n", run<1>(in, out, reps, blocks) / reps);
  printf("  (float)exp(dbl)               %8.3f us\n", run<2>(in, out, reps, blocks) / reps);
  printf("  one dependent DFMA            %8.4f us\n", run<3>(in, out, 4096, blocks) / 4096);
  CK(cudaGetLastError());
  return 0;
}
