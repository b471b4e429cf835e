// Shared device helpers for the sm_100a SSD3D kernels: bf16 packing, NaN-propagating ReLU,
// and thin inline-PTX wrappers for mbarrier / TMA / tcgen05 (TMEM + UMMA).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cuda.h>
#include <stdint.h>

#include "../../include/ssd3d_b200.h"

#define SSD3D_CHECK_LAUNCH()                         \
  do {                                               \
    cudaError_t e__ = cudaGetLastError();            \
    if (e__ != cudaSuccess) return (int)e__;         \
  } while (0)

#include <utility>

namespace ssd3d {

// ---------------------------------------------------------------------------------------------
// Programmatic dependent launch: consecutive kernels of the step are launched with programmatic stream
// serialization, so the next kernel's CTAs are scheduled (and run their prologue: barrier init, TMEM
// allocation, constant loads) while the previous kernel drains.  pdl_wait() blocks until every
// prerequisite grid has completed and its writes are visible: it must precede the first access to memory
// another kernel produces or still reads.  pdl_launch_dependents() lets the next kernel start launching.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// SMs a persistent kernel spreads over: the device's SM count, read once.
inline int persistent_sms() {
  static int n = 0;
  if (n == 0) {
    int dev = 0, sms = 0;
    cudaGetDevice(&dev);
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms <= 0) sms = 148;
    n = sms;
  }
  return n;
}

template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                              Args&&... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kernel, std::forward<Args>(args)...);
}

#define SSD3D_LAUNCH_PDL(kernel, grid, block, smem, st, ...)                                 \
  do {                                                                                       \
    cudaError_t e__ = ssd3d::launch_pdl(kernel, grid, block, smem, st, __VA_ARGS__);         \
    if (e__ != cudaSuccess) return (int)e__;                                                 \
  } while (0)

// ---------------------------------------------------------------------------------------------
// numerics
// ---------------------------------------------------------------------------------------------
// torch.relu semantics: NaN propagates (fmaxf(NaN, 0) would return 0).  mobilenet.py:30,44-45
__device__ __forceinline__ float relu_nan(float v) { return (v < 0.0f) ? 0.0f : v; }
// Activation floor: 0 = ReLU, -inf = identity (raw conv output for training-mode BatchNorm).  NaN propagates.
__device__ __forceinline__ float clamp_floor(float v, float floor) { return (v < floor) ? floor : v; }
#define SSD3D_FLOOR(relu) ((relu) ? 0.0f : -__builtin_huge_valf())

__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  __nv_bfloat162 p = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&p);
}
__device__ __forceinline__ float bf16_lo(uint32_t u) { return __uint_as_float(u << 16); }
__device__ __forceinline__ float bf16_hi(uint32_t u) { return __uint_as_float(u & 0xffff0000u); }

// ---------------------------------------------------------------------------------------------
// shared-memory addresses, mbarrier
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// Bounded wait: a protocol bug must surface as a trapped kernel (an error code on the host), never
// as a hung GPU.  The deadline is ~2 s of SM clock, checked on every poll (try_wait itself sleeps in hardware).
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  const long long t0 = clock64();
  while (!mbar_try_wait(bar, parity)) {
    if ((clock64() - t0) > 4000000000LL) __trap();
  }
}

// ---------------------------------------------------------------------------------------------
// TMA (cp.async.bulk.tensor) loads, completing on an mbarrier
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_5d(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1,
                                            int c2, int c3, int c4) {
  asm volatile(
      "cp.async.bulk.tensor.5d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6, "
      "%7}], [%2];" ::"r"(smem_u32(smem_dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
      : "memory");
}

// ---------------------------------------------------------------------------------------------
// tcgen05: TMEM allocation, UMMA issue/commit, TMEM loads
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_result, uint32_t ncols) {  // whole warp, .sync.aligned
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_result)),
               "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {  // whole warp
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// tcgen05.commit: the mbarrier gets one arrival once every UMMA issued so far by this thread has retired
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}

// D[tmem] (+)= A[smem] * B[smem]^T, bf16 inputs, fp32 accumulate.  One thread issues.
__device__ __forceinline__ void umma_bf16_ss(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                             uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}

// Shared-memory matrix descriptor, K-major operand, 128-byte swizzle (cute::UMMA::SmemDescriptor,
// mma_sm100_desc.hpp): rows are 128 B (64 bf16 of K), 8-row groups are SBO = 1024 B apart, the
// leading-dimension offset is unused for swizzled K-major, version = 1 (Blackwell), layout type 2.
__device__ __forceinline__ uint64_t umma_desc_k_sw128(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFFu) >> 4);         // start address        bits [0,14)
  d |= (uint64_t)1 << 16;                               // LBO (ignored)        bits [16,30)
  d |= (uint64_t)(1024u >> 4) << 32;                    // SBO = 1024 B         bits [32,46)
  d |= (uint64_t)1 << 46;                               // descriptor version   bits [46,48)
  d |= (uint64_t)2 << 61;                               // SWIZZLE_128B         bits [61,64)
  return d;
}

// Instruction descriptor for kind::f16: bf16 x bf16 -> fp32, both operands K-major
// (cute::UMMA::InstrDescriptor bit layout).
__device__ __host__ constexpr uint32_t umma_idesc_bf16(int M, int N) {
  return (1u << 4)                    // c_format = F32
         | (1u << 7)                  // a_format = BF16
         | (1u << 10)                 // b_format = BF16
         | ((uint32_t)(N >> 3) << 17) // n_dim
         | ((uint32_t)(M >> 4) << 24);// m_dim
}

// TMEM -> registers: 32 lanes x 32-bit, 16 consecutive columns per thread (thread i <-> lane base+i)
__device__ __forceinline__ void tmem_ld_32x32b_x16(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, "
      "%15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(pred));
  return pred != 0;
}

}  // namespace ssd3d
