// Microbenchmark: FP64 throughput of this card on the CUDA-core pipe (DFMA) and the tensor-core pipe (DMMA), the two
// choices for the float64 chain (bb_chain_f64.cu).  Every SM runs 4 CTAs of 256 threads, each thread (warp) keeps 8
// independent accumulators (fragments) in flight; the rate is FLOP over CUDA-event time of the whole grid.
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -o tools/bin/fp64_rate_bench tools/fp64_rate_bench.cu
#include <cstdio>
#include <cuda_runtime.h>

constexpr int ACC = 8;

__global__ void __launch_bounds__(256) dfma_kernel(double* out, int iters, double a, double b) {
  double x[ACC];
#pragma unroll
  for (int j = 0; j < ACC; ++j) x[j] = threadIdx.x * 1e-3 + j;
  for (int i = 0; i < iters; ++i)
#pragma unroll
    for (int j = 0; j < ACC; ++j) x[j] = fma(x[j], a, b);
  double s = 0.0;
#pragma unroll
  for (int j = 0; j < ACC; ++j) s += x[j];
  if (s == 12345.678) out[threadIdx.x] = s;  // keeps the chain alive
}

// mma.sync m8n8k4 f64: one DMMA.8x8x4 (512 FLOP per warp)
__global__ void __launch_bounds__(256) dmma884_kernel(double* out, int iters) {
  double a = 1.0 + threadIdx.x * 1e-6, b = 1.0 - threadIdx.x * 1e-6;
  double c[ACC][2];
#pragma unroll
  for (int j = 0; j < ACC; ++j) c[j][0] = c[j][1] = 0.0;
  for (int i = 0; i < iters; ++i)
#pragma unroll
    for (int j = 0; j < ACC; ++j)
      asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                   : "+d"(c[j][0]), "+d"(c[j][1]) : "d"(a), "d"(b));
  double s = 0.0;
#pragma unroll
  for (int j = 0; j < ACC; ++j) s += c[j][0] + c[j][1];
  if (s == 12345.678) out[threadIdx.x] = s;
}

// mma.sync m16n8k16 f64: 4096 FLOP per warp (8 x DMMA.8x8x4 in SASS on sm_100a)
__global__ void __launch_bounds__(256) dmma16816_kernel(double* out, int iters) {
  double a[8], b[4], c[ACC / 2][4];
#pragma unroll
  for (int j = 0; j < 8; ++j) a[j] = 1.0 + (threadIdx.x + j) * 1e-6;
#pragma unroll
  for (int j = 0; j < 4; ++j) b[j] = 1.0 - (threadIdx.x + j) * 1e-6;
#pragma unroll
  for (int j = 0; j < ACC / 2; ++j) c[j][0] = c[j][1] = c[j][2] = c[j][3] = 0.0;
  for (int i = 0; i < iters; ++i)
#pragma unroll
    for (int j = 0; j < ACC / 2; ++j)
      asm volatile("mma.sync.aligned.m16n8k16.row.col.f64.f64.f64.f64 {%0,%1,%2,%3}, {%4,%5,%6,%7,%8,%9,%10,%11}, "
                   "{%12,%13,%14,%15}, {%0,%1,%2,%3};"
                   : "+d"(c[j][0]), "+d"(c[j][1]), "+d"(c[j][2]), "+d"(c[j][3])
                   : "d"(a[0]), "d"(a[1]), "d"(a[2]), "d"(a[3]), "d"(a[4]), "d"(a[5]), "d"(a[6]), "d"(a[7]), "d"(b[0]),
                     "d"(b[1]), "d"(b[2]), "d"(b[3]));
  double s = 0.0;
#pragma unroll
  for (int j = 0; j < ACC / 2; ++j) s += c[j][0] + c[j][1] + c[j][2] + c[j][3];
  if (s == 12345.678) out[threadIdx.x] = s;
}

int main() {
  cudaDeviceProp p;
  cudaGetDeviceProperties(&p, 0);
  int clk_khz = 0;
  cudaDeviceGetAttribute(&clk_khz, cudaDevAttrClockRate, 0);
  printf("device %s, %d SMs, max SM clock %.0f MHz\n", p.name, p.multiProcessorCount, clk_khz / 1e3);
  double* out;
  cudaMalloc(&out, 4096 * sizeof(double));
  const int grid = p.multiProcessorCount * 4, block = 256;
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0);
  cudaEventCreate(&e1);
  struct Run {
    const char* name;
    int iters;
    double flop_per_iter_per_thread;  // per thread of the grid
  };
  for (int which = 0; which < 3; ++which) {
    const Run runs[3] = {{"DFMA (fma.rn.f64)", 1 << 16, 2.0 * ACC},
                         {"DMMA mma.sync m8n8k4", 1 << 14, 512.0 * ACC / 32},
                         {"DMMA mma.sync m16n8k16", 1 << 12, 4096.0 * (ACC / 2) / 32}};
    const Run& r = runs[which];
    float best = 1e30f;
    for (int rep = 0; rep < 4; ++rep) {  // first pass warms up
      cudaEventRecord(e0);
      if (which == 0) dfma_kernel<<<grid, block>>>(out, r.iters, 1.0000001, 1e-9);
      else if (which == 1) dmma884_kernel<<<grid, block>>>(out, r.iters);
      else dmma16816_kernel<<<grid, block>>>(out, r.iters);
      cudaEventRecord(e1);
      cudaEventSynchronize(e1);
      float ms = 0.f;
      cudaEventElapsedTime(&ms, e0, e1);
      if (rep > 0 && ms < best) best = ms;
    }
    const cudaError_t err = cudaGetLastError();
    const double flop = (double)grid * block * r.iters * r.flop_per_iter_per_thread;
    printf("%-24s %8.3f ms  %7.2f TFLOP/s  (%s)\n", r.name, best, flop / (best * 1e-3) / 1e12, cudaGetErrorString(err));
  }
  cudaFree(out);
  return 0;
}
