// Stand-alone probe of the observation store phase (debugging aid, not product code).
// mode 0: linear stores; 1: six interleaved channel planes; 2: planes + mask bytes from smem + LUT expansion (as the round-1 k_render)
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>
#include <stdint.h>

template <int MODE>
__global__ void __launch_bounds__(256, 4) k(float* ring, size_t env_stride_f, int head_off_f) {
  extern __shared__ __align__(16) uint8_t smem[];
  constexpr int O = 96, C = 6;
  float4* lut = (float4*)(smem + 9216);
  if (threadIdx.x < 16)
    lut[threadIdx.x] = make_float4((threadIdx.x & 1) ? 1.f : 0.f, (threadIdx.x & 2) ? 1.f : 0.f, (threadIdx.x & 4) ? 1.f : 0.f, (threadIdx.x & 8) ? 1.f : 0.f);
  for (int i = threadIdx.x; i < 9216 / 4; i += 256) ((uint32_t*)smem)[i] = (i * 2654435761u) & 0x3f3f3f3fu & ((i & 7) ? 0x02020202u : 0xffffffffu);
  __syncthreads();
  float* fb = ring + (size_t)blockIdx.x * env_stride_f + head_off_f;
  if (MODE == 0) {
    float4 v = lut[5];
    for (int q = threadIdx.x; q < C * O * O / 4; q += 256)
      asm volatile("st.global.cs.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(fb + 4 * q), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
  } else {
    for (int q = threadIdx.x; q < O * O / 4; q += 256) {
      const uint32_t m4 = ((const uint32_t*)smem)[q];
#pragma unroll
      for (int c = 0; c < C; ++c) {
        float4 v;
        if (MODE == 1) v = make_float4(__uint_as_float(m4), 0.f, 1.f, 0.f);
        else { const uint32_t t = (m4 >> c) & 0x01010101u; v = lut[(t * 0x01020408u) >> 24]; }
        asm volatile("st.global.cs.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(fb + c * (O * O) + 4 * q), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
      }
    }
  }
}

int main(int argc, char** argv) {
  int N = 4096, L = 64;
  int mode = argc > 1 ? atoi(argv[1]) : 0, smem = argc > 2 ? atoi(argv[2]) : 55000;
  size_t frame = 221184, stride = (size_t)L * frame;
  float* ring;
  if (cudaMalloc(&ring, (size_t)N * stride) != cudaSuccess) { printf("alloc failed\n"); return 1; }
  auto launch = [&](int i) {
    int off = (i % L) * (frame / 4);
    if (mode == 0) k<0><<<N, 256, smem>>>(ring, stride / 4, off);
    else if (mode == 1) k<1><<<N, 256, smem>>>(ring, stride / 4, off);
    else k<2><<<N, 256, smem>>>(ring, stride / 4, off);
  };
  cudaFuncSetAttribute(k<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
  cudaFuncSetAttribute(k<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
  cudaFuncSetAttribute(k<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
  cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);
  for (int i = 0; i < 5; ++i) launch(i);
  cudaDeviceSynchronize();
  cudaEventRecord(e0);
  int iters = 40;
  for (int i = 0; i < iters; ++i) launch(i + 5);
  cudaEventRecord(e1); cudaDeviceSynchronize();
  float ms; cudaEventElapsedTime(&ms, e0, e1);
  printf("mode %d smem %6d: %.1f us/launch -> %.0f GB/s (%s)\n", mode, smem, ms / iters * 1e3,
         (double)N * frame / (ms / iters * 1e-3) / 1e9, cudaGetErrorString(cudaGetLastError()));
  return 0;
}
