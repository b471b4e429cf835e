// Depthwise 3x3x3 conv + BN + ReLU with TMA halo tiles (mobilenet.py:38,44), channels-last-3d bf16.
//
// One CTA owns an output tile (TD x TH x TW voxels) of a 32-channel chunk.  The input halo box
// ((S*(TD-1)+3) x (S*(TH-1)+3) x TWI voxels x 32 channels) arrives with ONE 5-D cp.async.bulk.tensor: the TMA
// unit zero-fills whatever lies outside the volume, which is exactly the conv's padding, and every input byte
// crosses L2->SM once per tile instead of once per tap.  CTAs are persistent and double buffered: the box of
// tile i+1 is in flight while tile i is computed from shared memory.
//
// The direct kernel (conv_direct.cu) turned out to be instruction-issue bound (ncu: 61 % issue slots busy at 25 %
// occupancy, 112 instructions per output element: bf16 unpacking of the weights, bounds predicates, 64-bit
// address arithmetic), not memory bound.  Here a thread owns 4 channels and keeps all 27 x 4 weights in
// registers as fp32 pairs for the whole kernel (its channel chunk never changes), accumulates with the packed
// FFMA2 (fma.rn.f32x2: two IEEE fp32 FMAs per instruction, so results are bit-identical to the scalar kernel),
// needs no bounds checks (TMA zero fill) and addresses shared memory with compile-time offsets: ~12
// instructions per output element.  A thread produces WT outputs along W with a sliding register window.
//
// Roofline: HBM (SURVEY.md 8d): bytes = 2*N*C*(Vin+Vout) + 54*C.  The halo re-reads (1.3x for stride 2) are
// L2 hits.
#include "common.cuh"
#include "tma_host.h"
#include "../../include/ssd3d_b200.h"

namespace ssd3d {

constexpr int DW_CB = 32;   // channels per tile (64 bytes per voxel)

struct DwTmaParams {
  int N, C, D, H, W, Do, Ho, Wo;
  int tiles_w, tiles_h, tiles_d, chunks;
  int spatial_tiles;          // tiles_w * tiles_h * tiles_d * N
  const __nv_bfloat16* w;     // (27, C)
  const float* scale;
  const float* shift;
  __nv_bfloat16* y;
  float floor;
};

typedef unsigned long long f32x2;   // two fp32 lanes {lo, hi} in one 64-bit register pair

__device__ __forceinline__ f32x2 pack_f32x2(float lo, float hi) {
  f32x2 r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "r"(__float_as_uint(lo)), "r"(__float_as_uint(hi)));
  return r;
}
// two bf16 packed in a 32-bit word -> two fp32
__device__ __forceinline__ f32x2 bf16x2_to_f32x2(uint32_t u) {
  f32x2 r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "r"(u << 16), "r"(u & 0xffff0000u));
  return r;
}
__device__ __forceinline__ void ffma2(f32x2& acc, f32x2 a, f32x2 b) {
  asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(acc) : "l"(a), "l"(b));
}
__device__ __forceinline__ void unpack_f32x2(f32x2 v, float& lo, float& hi) {
  uint32_t a, b;
  asm("mov.b64 {%0, %1}, %2;" : "=r"(a), "=r"(b) : "l"(v));
  lo = __uint_as_float(a);
  hi = __uint_as_float(b);
}

template <int S, int WT, int TD, int TH, int TW>
struct DwTile {
  static constexpr int TDI = S * (TD - 1) + 3;
  static constexpr int THI = S * (TH - 1) + 3;
  static constexpr int TWI0 = S * (TW - 1) + 3;
  static constexpr int TWI = (TWI0 & 1) ? TWI0 : TWI0 + 1;     // odd row pitch (in 64-byte voxels)
  static constexpr int BYTES = TDI * THI * TWI * DW_CB * 2;
  static constexpr int PITCH = (BYTES + 127) & ~127;
  static constexpr int WQ = TW / WT;
  static constexpr int ITEMS = TD * TH * WQ * 8;               // (4-channel vector, h, w group, d)
  static constexpr size_t SMEM = 128 + 2 * (size_t)PITCH + 16;
};

template <int S, int WT, int TD, int TH, int TW>
__global__ void __launch_bounds__(256, 1) dw_tma_kernel(const __grid_constant__ CUtensorMap tm, const DwTmaParams p) {
  using T = DwTile<S, WT, TD, TH, TW>;
  constexpr int NI = (WT - 1) * S + 3;
  extern __shared__ uint8_t dw_raw[];
  const uint32_t raw = smem_u32(dw_raw);
  uint8_t* smem = dw_raw + ((128u - (raw & 127u)) & 127u);
  uint8_t* tiles = smem;
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + 2 * T::PITCH);
  const int tid = threadIdx.x;
  if (tid == 0) {
    tma_prefetch_desc(&tm);
    mbar_init(&full[0], 1);
    mbar_init(&full[1], 1);
    fence_barrier_init();
  }
  __syncthreads();
  pdl_wait();
  pdl_launch_dependents();

  // This CTA's channel chunk is fixed; it walks the spatial tiles blockIdx.x / chunks, + gridDim.x / chunks, ...
  const int chunk = blockIdx.x % p.chunks;
  const int cbase = chunk * DW_CB;
  const int first = blockIdx.x / p.chunks;
  const int step = gridDim.x / p.chunks;          // the host makes gridDim.x a multiple of chunks

  auto decode = [&](int tile, int& ow0, int& oh0, int& od0, int& n) {
    int t = tile;
    ow0 = (t % p.tiles_w) * TW; t /= p.tiles_w;
    oh0 = (t % p.tiles_h) * TH; t /= p.tiles_h;
    od0 = (t % p.tiles_d) * TD;
    n = t / p.tiles_d;
  };
  auto issue = [&](int tile, int buf) {
    int ow0, oh0, od0, n;
    decode(tile, ow0, oh0, od0, n);
    mbar_arrive_expect_tx(&full[buf], (uint32_t)T::BYTES);
    tma_load_5d(tiles + (size_t)buf * T::PITCH, &tm, &full[buf], cbase, ow0 * S - 1, oh0 * S - 1, od0 * S - 1, n);
  };
  if (tid == 0 && first < p.spatial_tiles) issue(first, 0);

  // ---- per-thread constants: 4 channels, their 27 weights (fp32 pairs), BN scale / shift ----
  const int cv = tid & 7;                         // 4-channel vector inside the chunk
  const int c0 = cbase + cv * 4;
  f32x2 wreg[27][2];
#pragma unroll
  for (int t = 0; t < 27; ++t) {
    const uint2 u = __ldg(reinterpret_cast<const uint2*>(p.w + (size_t)t * p.C + c0));
    wreg[t][0] = bf16x2_to_f32x2(u.x);
    wreg[t][1] = bf16x2_to_f32x2(u.y);
  }
  const float4 sc = __ldg(reinterpret_cast<const float4*>(p.scale + c0));
  const float4 sh = __ldg(reinterpret_cast<const float4*>(p.shift + c0));

  int it = 0;
  for (int tile = first; tile < p.spatial_tiles; tile += step, ++it) {
    const int buf = it & 1;
    const int next = tile + step;
    if (tid == 0 && next < p.spatial_tiles) issue(next, buf ^ 1);   // released by the trailing barrier of it-1
    int ow0, oh0, od0, n;
    decode(tile, ow0, oh0, od0, n);
    mbar_wait(&full[buf], (uint32_t)((it >> 1) & 1));
    const uint8_t* in = tiles + (size_t)buf * T::PITCH;

#pragma unroll 1
    for (int item = tid; item < T::ITEMS; item += 256) {
      int r = item >> 3;
      const int h = r % TH; r /= TH;
      const int wq = r % T::WQ;
      const int d = r / T::WQ;
      const int od = od0 + d, oh = oh0 + h, owb = ow0 + wq * WT;
      if (od >= p.Do || oh >= p.Ho || owb >= p.Wo) continue;
      f32x2 acc[WT][2];
#pragma unroll
      for (int i = 0; i < WT; ++i) { acc[i][0] = 0ull; acc[i][1] = 0ull; }
      const uint8_t* base = in + ((size_t)(((d * S) * T::THI + h * S) * T::TWI + wq * WT * S) * DW_CB + cv * 4) * 2;
#pragma unroll
      for (int kd = 0; kd < 3; ++kd) {
#pragma unroll
        for (int kh = 0; kh < 3; ++kh) {
          const uint8_t* row = base + (size_t)((kd * T::THI + kh) * T::TWI) * DW_CB * 2;
          f32x2 x[NI][2];
#pragma unroll
          for (int i = 0; i < NI; ++i) {
            const uint2 u = *reinterpret_cast<const uint2*>(row + i * DW_CB * 2);
            x[i][0] = bf16x2_to_f32x2(u.x);
            x[i][1] = bf16x2_to_f32x2(u.y);
          }
#pragma unroll
          for (int kw = 0; kw < 3; ++kw) {
            const int t = (kd * 3 + kh) * 3 + kw;
#pragma unroll
            for (int ow = 0; ow < WT; ++ow) {
              ffma2(acc[ow][0], x[ow * S + kw][0], wreg[t][0]);
              ffma2(acc[ow][1], x[ow * S + kw][1], wreg[t][1]);
            }
          }
        }
      }
      __nv_bfloat16* orow = p.y + ((((long long)n * p.Do + od) * p.Ho + oh) * p.Wo) * p.C + c0;
#pragma unroll
      for (int ow = 0; ow < WT; ++ow) {
        const int wo = owb + ow;
        if (wo >= p.Wo) break;
        float a0, a1, a2, a3;
        unpack_f32x2(acc[ow][0], a0, a1);
        unpack_f32x2(acc[ow][1], a2, a3);
        a0 = clamp_floor(__fadd_rn(__fmul_rn(a0, sc.x), sh.x), p.floor);
        a1 = clamp_floor(__fadd_rn(__fmul_rn(a1, sc.y), sh.y), p.floor);
        a2 = clamp_floor(__fadd_rn(__fmul_rn(a2, sc.z), sh.z), p.floor);
        a3 = clamp_floor(__fadd_rn(__fmul_rn(a3, sc.w), sh.w), p.floor);
        *reinterpret_cast<uint2*>(orow + (long long)wo * p.C) = make_uint2(pack_bf16x2(a0, a1), pack_bf16x2(a2, a3));
      }
    }
    __syncthreads();   // tile[buf] is free again
  }
}

// ------------------------------------------------------------------------------------------------
// Stride 2, de-interleaved halo.  With stride 2 every input position one instruction touches has the same parity
// along each axis for all outputs, so with 64-byte voxels the four 8-lane groups of a warp hit the same 16 of the
// 32 banks: ncu showed 4 shared-memory wavefronts per 8-byte load instead of 2, and the kernel is bound by exactly
// that pipe.  Here the halo arrives as TWO boxes with a TMA traversal stride of 2 along W (E = halo columns
// 0, 2, .., 16; O = columns 1, 3, .., 17), the lane groups of a warp take four CONSECUTIVE output columns (so
// consecutive E / O entries: alternating bank halves) and a thread owns 4 channels x 2 outputs along H: 5 input
// rows x {E[w], O[w], E[w+1]} per kd = 45 loads per 2 outputs as before, every one conflict free.  Each output
// still accumulates its 27 taps in (kd, kh, kw) order: bit-identical to the direct kernel.
// ------------------------------------------------------------------------------------------------
struct DwS2 {
  static constexpr int TD = 4, TH = 4, TW = 8;
  static constexpr int TDI = 9, THI = 9, TWI = 9;                   // per parity box
  static constexpr int BOX_BYTES = TDI * THI * TWI * DW_CB * 2;     // 46656
  static constexpr int BOX_PITCH = (BOX_BYTES + 127) & ~127;
  static constexpr int PITCH = 2 * BOX_PITCH;
  static constexpr int ITEMS = TD * (TH / 2) * TW * 8;              // 512
  static constexpr size_t SMEM = 128 + 2 * (size_t)PITCH + 16;
};

__global__ void __launch_bounds__(256, 1) dw_tma_s2_kernel(const __grid_constant__ CUtensorMap tm, const DwTmaParams p) {
  using T = DwS2;
  extern __shared__ uint8_t dw_raw[];
  const uint32_t raw = smem_u32(dw_raw);
  uint8_t* smem = dw_raw + ((128u - (raw & 127u)) & 127u);
  uint8_t* tiles = smem;
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + 2 * T::PITCH);
  const int tid = threadIdx.x;
  if (tid == 0) {
    tma_prefetch_desc(&tm);
    mbar_init(&full[0], 1);
    mbar_init(&full[1], 1);
    fence_barrier_init();
  }
  __syncthreads();
  pdl_wait();
  pdl_launch_dependents();
  const int chunk = blockIdx.x % p.chunks;
  const int cbase = chunk * DW_CB;
  const int first = blockIdx.x / p.chunks;
  const int step = gridDim.x / p.chunks;
  auto decode = [&](int tile, int& ow0, int& oh0, int& od0, int& n) {
    int t = tile;
    ow0 = (t % p.tiles_w) * T::TW; t /= p.tiles_w;
    oh0 = (t % p.tiles_h) * T::TH; t /= p.tiles_h;
    od0 = (t % p.tiles_d) * T::TD;
    n = t / p.tiles_d;
  };
  auto issue = [&](int tile, int buf) {
    int ow0, oh0, od0, n;
    decode(tile, ow0, oh0, od0, n);
    uint8_t* dst = tiles + (size_t)buf * T::PITCH;
    mbar_arrive_expect_tx(&full[buf], (uint32_t)(2 * T::BOX_BYTES));
    tma_load_5d(dst, &tm, &full[buf], cbase, ow0 * 2 - 1, oh0 * 2 - 1, od0 * 2 - 1, n);
    tma_load_5d(dst + T::BOX_PITCH, &tm, &full[buf], cbase, ow0 * 2, oh0 * 2 - 1, od0 * 2 - 1, n);
  };
  if (tid == 0 && first < p.spatial_tiles) issue(first, 0);

  const int cv = tid & 7;
  const int c0 = cbase + cv * 4;
  f32x2 wreg[27][2];
#pragma unroll
  for (int t = 0; t < 27; ++t) {
    const uint2 u = __ldg(reinterpret_cast<const uint2*>(p.w + (size_t)t * p.C + c0));
    wreg[t][0] = bf16x2_to_f32x2(u.x);
    wreg[t][1] = bf16x2_to_f32x2(u.y);
  }
  const float4 sc = __ldg(reinterpret_cast<const float4*>(p.scale + c0));
  const float4 sh = __ldg(reinterpret_cast<const float4*>(p.shift + c0));

  int it = 0;
  for (int tile = first; tile < p.spatial_tiles; tile += step, ++it) {
    const int buf = it & 1;
    const int next = tile + step;
    if (tid == 0 && next < p.spatial_tiles) issue(next, buf ^ 1);   // released by the trailing barrier of it-1
    int ow0, oh0, od0, n;
    decode(tile, ow0, oh0, od0, n);
    mbar_wait(&full[buf], (uint32_t)((it >> 1) & 1));
    const uint8_t* in = tiles + (size_t)buf * T::PITCH;
#pragma unroll 1
    for (int item = tid; item < T::ITEMS; item += 256) {
      const int w = (item >> 3) & 7, hp = (item >> 6) & 1, d = item >> 7;
      const int od = od0 + d, oh = oh0 + 2 * hp, wo = ow0 + w;
      if (od >= p.Do || oh >= p.Ho || wo >= p.Wo) continue;
      f32x2 acc0[2] = {0ull, 0ull}, acc1[2] = {0ull, 0ull};
      const uint8_t* base = in + ((size_t)(((2 * d) * T::THI + 4 * hp) * T::TWI + w) * DW_CB + cv * 4) * 2;
#pragma unroll
      for (int kd = 0; kd < 3; ++kd) {
#pragma unroll
        for (int r = 0; r < 5; ++r) {
          const uint8_t* row = base + (size_t)((kd * T::THI + r) * T::TWI) * DW_CB * 2;
          const uint2 u0 = *reinterpret_cast<const uint2*>(row);                    // E[w]   : kw = 0
          const uint2 u1 = *reinterpret_cast<const uint2*>(row + T::BOX_PITCH);     // O[w]   : kw = 1
          const uint2 u2 = *reinterpret_cast<const uint2*>(row + DW_CB * 2);        // E[w+1] : kw = 2
          const f32x2 x0[2] = {bf16x2_to_f32x2(u0.x), bf16x2_to_f32x2(u0.y)};
          const f32x2 x1[2] = {bf16x2_to_f32x2(u1.x), bf16x2_to_f32x2(u1.y)};
          const f32x2 x2[2] = {bf16x2_to_f32x2(u2.x), bf16x2_to_f32x2(u2.y)};
          if (r <= 2) {          // output row 2hp: kh = r
            const int t = (kd * 3 + r) * 3;
            ffma2(acc0[0], x0[0], wreg[t][0]);     ffma2(acc0[1], x0[1], wreg[t][1]);
            ffma2(acc0[0], x1[0], wreg[t + 1][0]); ffma2(acc0[1], x1[1], wreg[t + 1][1]);
            ffma2(acc0[0], x2[0], wreg[t + 2][0]); ffma2(acc0[1], x2[1], wreg[t + 2][1]);
          }
          if (r >= 2) {          // output row 2hp + 1: kh = r - 2
            const int t = (kd * 3 + (r - 2)) * 3;
            ffma2(acc1[0], x0[0], wreg[t][0]);     ffma2(acc1[1], x0[1], wreg[t][1]);
            ffma2(acc1[0], x1[0], wreg[t + 1][0]); ffma2(acc1[1], x1[1], wreg[t + 1][1]);
            ffma2(acc1[0], x2[0], wreg[t + 2][0]); ffma2(acc1[1], x2[1], wreg[t + 2][1]);
          }
        }
      }
      __nv_bfloat16* o = p.y + ((((long long)n * p.Do + od) * p.Ho + oh) * p.Wo + wo) * p.C + c0;
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        if (e == 1 && oh + 1 >= p.Ho) break;
        float a0, a1, a2, a3;
        unpack_f32x2(e ? acc1[0] : acc0[0], a0, a1);
        unpack_f32x2(e ? acc1[1] : acc0[1], a2, a3);
        a0 = clamp_floor(__fadd_rn(__fmul_rn(a0, sc.x), sh.x), p.floor);
        a1 = clamp_floor(__fadd_rn(__fmul_rn(a1, sc.y), sh.y), p.floor);
        a2 = clamp_floor(__fadd_rn(__fmul_rn(a2, sc.z), sh.z), p.floor);
        a3 = clamp_floor(__fadd_rn(__fmul_rn(a3, sc.w), sh.w), p.floor);
        *reinterpret_cast<uint2*>(o + (long long)e * p.Wo * p.C) = make_uint2(pack_bf16x2(a0, a1), pack_bf16x2(a2, a3));
      }
    }
    __syncthreads();   // tile[buf] is free again
  }
}

static int launch_dw_tma_s2(const void* x, DwTmaParams& p, cudaStream_t st) {
  using T = DwS2;
  p.tiles_w = (p.Wo + T::TW - 1) / T::TW;
  p.tiles_h = (p.Ho + T::TH - 1) / T::TH;
  p.tiles_d = (p.Do + T::TD - 1) / T::TD;
  p.chunks = p.C / DW_CB;
  const long long spatial = (long long)p.tiles_w * p.tiles_h * p.tiles_d * p.N;
  if (spatial * p.chunks > 0x3fffffffll) return SSD3D_ERR_UNSUPPORTED;
  p.spatial_tiles = (int)spatial;
  CUtensorMap tm;
  const uint64_t dims[5] = {(uint64_t)p.C, (uint64_t)p.W, (uint64_t)p.H, (uint64_t)p.D, (uint64_t)p.N};
  const uint64_t strides[4] = {(uint64_t)p.C * 2, (uint64_t)p.W * p.C * 2, (uint64_t)p.H * p.W * p.C * 2,
                               (uint64_t)p.D * p.H * p.W * p.C * 2};
  // the box spans 17 columns of which every second one is loaded (9 per parity box)
  const uint32_t box[5] = {(uint32_t)DW_CB, 17u, (uint32_t)T::THI, (uint32_t)T::TDI, 1u};
  const uint32_t estr[5] = {1u, 2u, 1u, 1u, 1u};
  if (make_tma_bf16(&tm, x, 5, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_NONE, estr)) return SSD3D_ERR_TMA;
  cudaError_t e = cudaFuncSetAttribute(dw_tma_s2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)T::SMEM);
  if (e != cudaSuccess) return (int)e;
  const int n_sm = persistent_sms();
  long long grid = n_sm;
  if (grid > spatial * p.chunks) grid = spatial * p.chunks;
  grid = grid / p.chunks * p.chunks;
  if (grid < p.chunks) grid = p.chunks;
  SSD3D_LAUNCH_PDL(dw_tma_s2_kernel, dim3((unsigned)grid), dim3(256), T::SMEM, st, tm, p);
  return SSD3D_OK;
}

// ------------------------------------------------------------------------------------------------
// Depthwise WEIGHT gradient with the same tiling: dw[c][tap] = sum_o dz[o][c] * x[S*o + tap - 1][c].
// Roles swapped w.r.t. the forward kernel: the 27 x 4 accumulators live in registers for the whole kernel, the
// 4-channel dz vector of each output is the multiplier.  At the end the threads of a CTA that own the same
// channels are reduced (warp shuffles, then shared memory, fixed order) into one (32 channels x 27) block of the
// CTA's partial slab; ssd3d_dwconv3d_wgrad sums the slabs.
// ------------------------------------------------------------------------------------------------
template <int S, int WT, int TD, int TH, int TW>
__global__ void __launch_bounds__(256, 1) dw_wgrad_tma_kernel(const __grid_constant__ CUtensorMap tm,
                                                              const DwTmaParams p, const __nv_bfloat16* __restrict__ dz,
                                                              float* __restrict__ partial) {
  using T = DwTile<S, WT, TD, TH, TW>;
  constexpr int NI = (WT - 1) * S + 3;
  extern __shared__ uint8_t dw_raw[];
  const uint32_t raw = smem_u32(dw_raw);
  uint8_t* smem = dw_raw + ((128u - (raw & 127u)) & 127u);
  uint8_t* tiles = smem;
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + 2 * T::PITCH);
  const int tid = threadIdx.x;
  if (tid == 0) {
    tma_prefetch_desc(&tm);
    mbar_init(&full[0], 1);
    mbar_init(&full[1], 1);
    fence_barrier_init();
  }
  __syncthreads();
  pdl_wait();
  pdl_launch_dependents();
  const int chunk = blockIdx.x % p.chunks;
  const int cbase = chunk * DW_CB;
  const int first = blockIdx.x / p.chunks;
  const int step = gridDim.x / p.chunks;
  auto decode = [&](int tile, int& ow0, int& oh0, int& od0, int& n) {
    int t = tile;
    ow0 = (t % p.tiles_w) * TW; t /= p.tiles_w;
    oh0 = (t % p.tiles_h) * TH; t /= p.tiles_h;
    od0 = (t % p.tiles_d) * TD;
    n = t / p.tiles_d;
  };
  auto issue = [&](int tile, int buf) {
    int ow0, oh0, od0, n;
    decode(tile, ow0, oh0, od0, n);
    mbar_arrive_expect_tx(&full[buf], (uint32_t)T::BYTES);
    tma_load_5d(tiles + (size_t)buf * T::PITCH, &tm, &full[buf], cbase, ow0 * S - 1, oh0 * S - 1, od0 * S - 1, n);
  };
  if (tid == 0 && first < p.spatial_tiles) issue(first, 0);
  const int cv = tid & 7;
  const int c0 = cbase + cv * 4;
  f32x2 acc[27][2];
#pragma unroll
  for (int t = 0; t < 27; ++t) { acc[t][0] = 0ull; acc[t][1] = 0ull; }

  int it = 0;
  for (int tile = first; tile < p.spatial_tiles; tile += step, ++it) {
    const int buf = it & 1;
    const int next = tile + step;
    if (tid == 0 && next < p.spatial_tiles) issue(next, buf ^ 1);
    int ow0, oh0, od0, n;
    decode(tile, ow0, oh0, od0, n);
    mbar_wait(&full[buf], (uint32_t)((it >> 1) & 1));
    const uint8_t* in = tiles + (size_t)buf * T::PITCH;
#pragma unroll 1
    for (int item = tid; item < T::ITEMS; item += 256) {
      int r = item >> 3;
      const int h = r % TH; r /= TH;
      const int wq = r % T::WQ;
      const int d = r / T::WQ;
      const int od = od0 + d, oh = oh0 + h, owb = ow0 + wq * WT;
      if (od >= p.Do || oh >= p.Ho || owb >= p.Wo) continue;
      const __nv_bfloat16* grow = dz + ((((long long)n * p.Do + od) * p.Ho + oh) * p.Wo) * p.C + c0;
      f32x2 g[WT][2];
#pragma unroll
      for (int ow = 0; ow < WT; ++ow) {
        uint2 u = make_uint2(0u, 0u);
        if (owb + ow < p.Wo) u = __ldg(reinterpret_cast<const uint2*>(grow + (long long)(owb + ow) * p.C));
        g[ow][0] = bf16x2_to_f32x2(u.x);
        g[ow][1] = bf16x2_to_f32x2(u.y);
      }
      const uint8_t* base = in + ((size_t)(((d * S) * T::THI + h * S) * T::TWI + wq * WT * S) * DW_CB + cv * 4) * 2;
#pragma unroll
      for (int kd = 0; kd < 3; ++kd) {
#pragma unroll
        for (int kh = 0; kh < 3; ++kh) {
          const uint8_t* row = base + (size_t)((kd * T::THI + kh) * T::TWI) * DW_CB * 2;
          f32x2 x[NI][2];
#pragma unroll
          for (int i = 0; i < NI; ++i) {
            const uint2 u = *reinterpret_cast<const uint2*>(row + i * DW_CB * 2);
            x[i][0] = bf16x2_to_f32x2(u.x);
            x[i][1] = bf16x2_to_f32x2(u.y);
          }
#pragma unroll
          for (int kw = 0; kw < 3; ++kw) {
            const int t = (kd * 3 + kh) * 3 + kw;
#pragma unroll
            for (int ow = 0; ow < WT; ++ow) {
              ffma2(acc[t][0], x[ow * S + kw][0], g[ow][0]);
              ffma2(acc[t][1], x[ow * S + kw][1], g[ow][1]);
            }
          }
        }
      }
    }
    __syncthreads();
  }
  // ---- reduce over the threads that own the same 4 channels: lanes l, l^8, l^16, l^24 of a warp, then the 8 warps ----
  float* red = reinterpret_cast<float*>(tiles);      // [8 warps][8 cv][108]: 27.6 KB of the (now idle) tile buffers
  const int warp = tid >> 5, lane = tid & 31;
#pragma unroll
  for (int t = 0; t < 27; ++t) {
#pragma unroll
    for (int hsel = 0; hsel < 2; ++hsel) {
      float a, b;
      unpack_f32x2(acc[t][hsel], a, b);
      a += __shfl_xor_sync(0xffffffffu, a, 8);
      b += __shfl_xor_sync(0xffffffffu, b, 8);
      a += __shfl_xor_sync(0xffffffffu, a, 16);
      b += __shfl_xor_sync(0xffffffffu, b, 16);
      if (lane < 8) {
        red[(warp * 8 + cv) * 108 + t * 4 + hsel * 2] = a;
        red[(warp * 8 + cv) * 108 + t * 4 + hsel * 2 + 1] = b;
      }
    }
  }
  __syncthreads();
  // partial slab [C][27] of this CTA's spatial index; this CTA fills rows cbase .. cbase+31
  float* dst = partial + (size_t)(blockIdx.x / p.chunks) * p.C * 27;
  for (int i = tid; i < 32 * 27; i += 256) {
    const int ch = i / 27, t = i % 27;         // ch = cv*4 + j
    const int cvv = ch >> 2, j = ch & 3;
    float s = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) s += red[(w * 8 + cvv) * 108 + t * 4 + j];
    dst[(size_t)(cbase + ch) * 27 + t] = s;
  }
}

template <int S, int WT, int TD, int TH, int TW>
static int launch_dw_wgrad_tma(const void* x, DwTmaParams& p, const __nv_bfloat16* dz, float* partial, int max_slabs,
                               int* slabs_out, cudaStream_t st) {
  using T = DwTile<S, WT, TD, TH, TW>;
  p.tiles_w = (p.Wo + TW - 1) / TW;
  p.tiles_h = (p.Ho + TH - 1) / TH;
  p.tiles_d = (p.Do + TD - 1) / TD;
  p.chunks = p.C / DW_CB;
  const long long spatial = (long long)p.tiles_w * p.tiles_h * p.tiles_d * p.N;
  if (spatial * p.chunks > 0x3fffffffll) return SSD3D_ERR_UNSUPPORTED;
  p.spatial_tiles = (int)spatial;
  CUtensorMap tm;
  const uint64_t dims[5] = {(uint64_t)p.C, (uint64_t)p.W, (uint64_t)p.H, (uint64_t)p.D, (uint64_t)p.N};
  const uint64_t strides[4] = {(uint64_t)p.C * 2, (uint64_t)p.W * p.C * 2, (uint64_t)p.H * p.W * p.C * 2,
                               (uint64_t)p.D * p.H * p.W * p.C * 2};
  const uint32_t box[5] = {(uint32_t)DW_CB, (uint32_t)T::TWI, (uint32_t)T::THI, (uint32_t)T::TDI, 1u};
  if (make_tma_bf16(&tm, x, 5, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_NONE)) return SSD3D_ERR_TMA;
  size_t smem = T::SMEM;
  if (smem < 128 + 8 * 8 * 108 * 4 + 64) smem = 128 + 8 * 8 * 108 * 4 + 64;
  cudaError_t e = cudaFuncSetAttribute(dw_wgrad_tma_kernel<S, WT, TD, TH, TW>,
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return (int)e;
  const int n_sm = persistent_sms();
  long long grid = n_sm;
  if (grid > spatial * p.chunks) grid = spatial * p.chunks;
  grid = grid / p.chunks * p.chunks;
  if (grid < p.chunks) grid = p.chunks;
  if (grid / p.chunks > max_slabs) return SSD3D_ERR_UNSUPPORTED;
  *slabs_out = (int)(grid / p.chunks);
  SSD3D_LAUNCH_PDL((dw_wgrad_tma_kernel<S, WT, TD, TH, TW>), dim3((unsigned)grid), dim3(256), smem, st, tm, p, dz, partial);
  return SSD3D_OK;
}

template <int S, int WT, int TD, int TH, int TW>
static int launch_dw_tma(const void* x, DwTmaParams& p, cudaStream_t st) {
  using T = DwTile<S, WT, TD, TH, TW>;
  p.tiles_w = (p.Wo + TW - 1) / TW;
  p.tiles_h = (p.Ho + TH - 1) / TH;
  p.tiles_d = (p.Do + TD - 1) / TD;
  p.chunks = p.C / DW_CB;
  const long long spatial = (long long)p.tiles_w * p.tiles_h * p.tiles_d * p.N;
  if (spatial * p.chunks > 0x3fffffffll) return SSD3D_ERR_UNSUPPORTED;
  p.spatial_tiles = (int)spatial;
  CUtensorMap tm;
  const uint64_t dims[5] = {(uint64_t)p.C, (uint64_t)p.W, (uint64_t)p.H, (uint64_t)p.D, (uint64_t)p.N};
  const uint64_t strides[4] = {(uint64_t)p.C * 2, (uint64_t)p.W * p.C * 2, (uint64_t)p.H * p.W * p.C * 2,
                               (uint64_t)p.D * p.H * p.W * p.C * 2};
  const uint32_t box[5] = {(uint32_t)DW_CB, (uint32_t)T::TWI, (uint32_t)T::THI, (uint32_t)T::TDI, 1u};
  if (make_tma_bf16(&tm, x, 5, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_NONE)) return SSD3D_ERR_TMA;
  cudaError_t e = cudaFuncSetAttribute(dw_tma_kernel<S, WT, TD, TH, TW>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)T::SMEM);
  if (e != cudaSuccess) return (int)e;
  const int n_sm = persistent_sms();
  // persistent grid: one CTA per SM (the register-resident weights need 1 x 256 threads x ~200 registers),
  // rounded down to a multiple of the channel chunks so that every CTA keeps one chunk
  long long grid = n_sm;
  if (grid > spatial * p.chunks) grid = spatial * p.chunks;
  grid = grid / p.chunks * p.chunks;
  if (grid < p.chunks) grid = p.chunks;
  SSD3D_LAUNCH_PDL((dw_tma_kernel<S, WT, TD, TH, TW>), dim3((unsigned)grid), dim3(256), T::SMEM, st, tm, p);
  return SSD3D_OK;
}

}  // namespace ssd3d

using namespace ssd3d;

// Returns SSD3D_ERR_UNSUPPORTED when the layer is better served by the direct kernel (small maps, C % 32 != 0).
int ssd3d_dwconv3d_tma(const void* x, const void* w, const float* scale, const float* shift, void* y, int N, int C,
                       int D, int H, int W, int stride, float floor, cudaStream_t st) {
  const int Do = (D - 1) / stride + 1, Ho = (H - 1) / stride + 1, Wo = (W - 1) / stride + 1;
  if (C % DW_CB || Wo < 8 || Ho < 4 || Do < 4) return SSD3D_ERR_UNSUPPORTED;
  if ((reinterpret_cast<uintptr_t>(x) & 15) != 0) return SSD3D_ERR_UNSUPPORTED;
  DwTmaParams p{};
  p.N = N; p.C = C; p.D = D; p.H = H; p.W = W; p.Do = Do; p.Ho = Ho; p.Wo = Wo;
  p.w = static_cast<const __nv_bfloat16*>(w);
  p.scale = scale; p.shift = shift; p.y = static_cast<__nv_bfloat16*>(y); p.floor = floor;
  if (stride == 2) return launch_dw_tma_s2(x, p, st);
  return launch_dw_tma<1, 4, 4, 8, 8>(x, p, st);
}

// Weight gradient through the same tiles; fills `slabs` partial slabs of (C, 27) floats in `partial`
// (capacity max_slabs) that the caller sums.  SSD3D_ERR_UNSUPPORTED -> use the direct kernel.
int ssd3d_dwconv3d_wgrad_tma(const void* dz, const void* x, int N, int C, int D, int H, int W, int stride,
                             float* partial, int max_slabs, int* slabs, cudaStream_t st) {
  const int Do = (D - 1) / stride + 1, Ho = (H - 1) / stride + 1, Wo = (W - 1) / stride + 1;
  if (C % DW_CB || Wo < 8 || Ho < 4 || Do < 4) return SSD3D_ERR_UNSUPPORTED;
  if ((reinterpret_cast<uintptr_t>(x) & 15) != 0) return SSD3D_ERR_UNSUPPORTED;
  DwTmaParams p{};
  p.N = N; p.C = C; p.D = D; p.H = H; p.W = W; p.Do = Do; p.Ho = Ho; p.Wo = Wo;
  const __nv_bfloat16* g = static_cast<const __nv_bfloat16*>(dz);
  if (stride == 2) return launch_dw_wgrad_tma<2, 2, 4, 4, 8>(x, p, g, partial, max_slabs, slabs, st);
  return launch_dw_wgrad_tma<1, 4, 4, 8, 8>(x, p, g, partial, max_slabs, slabs, st);
}
