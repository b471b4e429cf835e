// Micro-benchmark: issue rate / execution time of tcgen05.mma kind::f16 (bf16, M=128, K=16) with both operands in
// shared memory, as a function of N and of the operand layout (no swizzle with the overlapping LBO = 16 B trick of
// conv_stem_tz.cu, plain no-swizzle, 128B swizzle).  One CTA per SM, one issuing thread,
// `reps` UMMAs into the same accumulator, one commit; cycles from clock64.
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -I mslesions3d_b200/csrc scripts/ubench/umma_rate.cu -o gpurun_out/umma_rate
#include "common.cuh"
#include <cstdio>
using namespace ssd3d;

__device__ __forceinline__ uint64_t desc_nosw(uint32_t addr, uint32_t lbo, uint32_t sbo) {
  uint64_t d = 0;
  d |= (uint64_t)((addr & 0x3FFFFu) >> 4);
  d |= (uint64_t)(lbo >> 4) << 16;
  d |= (uint64_t)(sbo >> 4) << 32;
  d |= (uint64_t)1 << 46;
  return d;
}

__global__ void __launch_bounds__(64, 1) k(int mode, int N, int reps, int nslice, long long* out) {
  extern __shared__ uint8_t raw[];
  uint8_t* smem = raw + ((1024u - (smem_u32(raw) & 1023u)) & 1023u);
  __shared__ uint64_t bar;
  __shared__ uint32_t slot;
  for (int i = threadIdx.x; i < 160 * 1024 / 16; i += 64) reinterpret_cast<uint4*>(smem)[i] = make_uint4(0, 0, 0, 0);
  if (threadIdx.x == 0) { mbar_init(&bar, 1); fence_barrier_init(); }
  if (threadIdx.x < 32) { tmem_alloc(&slot, 512); tmem_relinquish(); }
  fence_proxy_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tb = slot;
  if (threadIdx.x == 0) {
    const uint32_t idesc = umma_idesc_bf16(128, N);
    const uint32_t a = smem_u32(smem), b = smem_u32(smem + 80 * 1024);
    uint64_t da, db;
    if (mode == 0) { da = desc_nosw(a, 16, 144); db = desc_nosw(b, 128, 256); }          // overlapped LBO
    else if (mode == 1) { da = desc_nosw(a, 128, 256); db = desc_nosw(b, 128, 256); }    // plain no-swizzle
    else { da = umma_desc_k_sw128(a); db = umma_desc_k_sw128(b); }                       // 128B swizzle (K=64 tile)
    const uint64_t step = (uint64_t)(nslice > 1 ? 2 : 0);     // lean loop: constant descriptors (+32 B when nslice > 1)
    const long long t0 = clock64();
#pragma unroll 1
    for (int r = 0; r < reps; r += 8) {
#pragma unroll
      for (int q = 0; q < 8; ++q) umma_bf16_ss(tb, da + step * (q & 3), db + step * (q & 3), idesc, 1u);
    }
    umma_commit(&bar);
    const long long t1 = clock64();
    mbar_wait(&bar, 0);
    const long long t2 = clock64();
    if (blockIdx.x == 0) { out[0] = t1 - t0; out[1] = t2 - t0; }
  }
  tc_fence_before();
  __syncthreads();
  if (threadIdx.x < 32) { tc_fence_after(); tmem_dealloc(tb, 512); }
}

int main() {
  long long* d;
  cudaMalloc(&d, 16);
  cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, 170 * 1024);
  const int reps = 2000;
  for (int mode = 0; mode < 3; ++mode)
    for (int N : {64, 128, 256})
      for (int nslice : {1, 4}) {
        long long h[2];
        for (int w = 0; w < 2; ++w) {
          k<<<148, 64, 170 * 1024>>>(mode, N, reps, nslice, d);
          cudaError_t e = cudaDeviceSynchronize();
          if (e != cudaSuccess) { printf("error %s\n", cudaGetErrorString(e)); return 1; }
        }
        cudaMemcpy(h, d, 16, cudaMemcpyDeviceToHost);
        printf("mode %d (%s) N %3d slices %d: issue %.1f clk/UMMA, complete %.1f clk/UMMA\n", mode,
               mode == 0 ? "nosw LBO16" : (mode == 1 ? "nosw plain" : "sw128"), N, nslice, (double)h[0] / reps,
               (double)h[1] / reps);
      }
  return 0;
}
