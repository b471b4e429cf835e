// Stem convolution (dense 3x3x3, Cin in {1..4} -> 32, stride (sd,2,2), + BN + ReLU) as a tcgen05 implicit
// GEMM (mobilenet.py:26-31 as instantiated at ssd3d.py:60-61).
//
// On CUDA cores this layer is compute-bound (1728 FMA per output voxel at Cin=2: ~300 us for the 2ch 128^3
// batch-8 workload against a 31 us HBM floor), so the contraction goes to the tensor cores:
//   * one CTA = 128 output voxels (TW x TH x TD box) x 32 channels = one UMMA M=128, N=32 accumulator;
//   * the input halo box of the NCDHW tensor is fetched by ONE 4-D TMA load; voxels outside the volume are
//     zero-filled by the TMA unit, which is the conv's zero padding;
//   * each thread gathers its voxel's 27*Cin taps from the shared-memory halo into one K-major row of the
//     A operand, written in the 128B-swizzle layout the UMMA descriptor expects (K padded to 64/128);
//   * 4 (or 8) UMMAs accumulate into 32 TMEM columns; the epilogue applies scale/shift/ReLU and writes
//     64 contiguous bytes per voxel (channels-last bf16).
// Several CTAs are resident per SM (about 30 KB of shared memory each), so TMA, gather, MMA and store of
// neighbouring tiles overlap without an intra-CTA pipeline.
#include "common.cuh"
#include "tma_host.h"

namespace ssd3d {

struct StemParams {
  int N, D, H, W, Do, Ho, Wo, sd;
  int TW, TH, TD;            // output tile (product 128)
  int TWI, THI, TDI;         // input halo tile (TWI padded so that a row is a multiple of 16 bytes)
  int tiles_w, tiles_h, tiles_d;
  const __nv_bfloat16* wt;   // (32, KPAD) bf16, k = ((ci*3+kd)*3+kh)*3+kw, zero padded
  const float* scale;
  const float* shift;
  __nv_bfloat16* y;          // (N, Do, Ho, Wo, 32)
  float floor;               // activation floor: 0 = ReLU, -inf = identity
};

__device__ __forceinline__ void tma_load_4d(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1,
                                            int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2),
      "r"(c3)
      : "memory");
}

__device__ __forceinline__ uint32_t bf16_bits(float f) {
  return (uint32_t)__bfloat16_as_ushort(__float2bfloat16_rn(f));
}

// byte offset of 16-byte chunk `chunk` (0..7) of row `row` inside a 128B-swizzled K-major tile
__device__ __forceinline__ uint32_t sw128_offset(int row, int chunk) {
  return (uint32_t)(row * 128 + ((chunk ^ (row & 7)) << 4));
}

// NaN-propagating ReLU in one instruction (max.NaN returns NaN if either input is NaN: torch.relu semantics)
__device__ __forceinline__ float relu_nan1(float v, float floor) {
  float r;
  asm("max.NaN.f32 %0, %1, %2;" : "=f"(r) : "f"(v), "f"(floor));
  return r;
}

// registers -> TMEM: 32 consecutive 32-bit columns of this thread's lane (thread i of a warp <-> lane base + i)
__device__ __forceinline__ void tmem_st_32x32b_x32(uint32_t taddr, const uint32_t* r) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
      "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]), "r"(r[18]),
      "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]),
      "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// D[tmem] (+)= A[tmem] * B[smem]^T: the A operand (128 rows x 16 bf16 = 8 columns of packed pairs) comes from
// tensor memory, where the gather wrote it with tcgen05.st -- it never touches shared memory.
__device__ __forceinline__ void umma_bf16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t desc_b, uint32_t idesc,
                                             uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}" ::"r"(tmem_d),
      "r"(tmem_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}

// Persistent CTA: loops over tiles t = blockIdx.x, blockIdx.x + gridDim.x, ...  Per tile
//   TMA halo box (double buffered, prefetched two tiles ahead)  ->  gather of the 27*CIN taps into registers  ->
//   tcgen05.st into the A operand in TENSOR MEMORY (double buffered; the A tile never exists in shared memory,
//   whose bandwidth was the kernel's limit: 16 KB written + 16 KB read back per tile)  ->  4*KB UMMAs (A from
//   TMEM, B from smem) into one of two 32-column TMEM accumulators (asynchronous)  ->  epilogue of the PREVIOUS
//   tile (TMEM -> scale/shift/ReLU -> swizzled staging tile -> TMA store) while this tile's UMMAs run.
// Weights (B operand), scale and shift are loaded once per CTA; 3 CTAs are resident per SM.
template <typename TIn, int CIN>
__global__ void __launch_bounds__(128, 4) stem_tc_kernel(const __grid_constant__ CUtensorMap tmX,
                                                         const __grid_constant__ CUtensorMap tmY, const StemParams p) {
  constexpr int KREAL = 27 * CIN;
  constexpr int KPAD = (KREAL <= 64) ? 64 : 128;
  constexpr int KB = KPAD / 64;
  constexpr int NREG = KPAD / 2;          // packed bf16 pairs per A row
  constexpr int PADL = 16 / (int)sizeof(TIn);   // left halo rounded up to 16 bytes (1 column is needed)
  constexpr int NG = 9 * CIN;             // (ci, kd, kh) groups of 3 consecutive taps

  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw = smem_u32(smem_raw);
  uint8_t* smem = smem_raw + ((1024u - (raw & 1023u)) & 1023u);
  uint8_t* sB = smem;                                   // KB x (32 rows x 128 B)
  constexpr uint32_t TMEM_COLS = (64 + 2 * NREG <= 128) ? 128u : 256u;   // 2 accumulators + 2 A buffers
  uint8_t* ctl = sB + KB * 4096;                        // mbarriers + TMEM slot (128 B), then scale/shift (256 B)
  const int tile_elems = CIN * p.TDI * p.THI * p.TWI;
  const uint32_t tile_bytes = (uint32_t)(tile_elems * sizeof(TIn));
  const uint32_t tile_pitch = (tile_bytes + 127u) & ~127u;
  float* s_sc = reinterpret_cast<float*>(ctl + 128);    // BN scale[32], shift[32]: shared, not 64 registers per
  float* s_sh = s_sc + 32;                              // thread, so that a 4th CTA fits on the SM
  uint8_t* sOut = ctl + 384 + 640;                      // 128 rows x 64 B output staging tile (1024-aligned), 64B-swizzled
  uint8_t* sX = sOut + 8192;                            // 2 x input halo tile [CIN][TDI][THI][TWI] of TIn
  uint64_t* bar_in = reinterpret_cast<uint64_t*>(ctl);  // [2]
  uint64_t* bar_mma = bar_in + 2;                       // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bar_in + 4);

  const int tid = threadIdx.x;
  const int warp = tid >> 5;
  const int total_tiles = p.tiles_w * p.tiles_h * p.tiles_d * p.N;

  // barrier init and TMA issue live in warp 1, so that warp 0 reaches the .sync.aligned TMEM
  // allocation fully converged (a lane still inside a divergent branch makes it an illegal instruction)
  if (tid == 32) {
    tma_prefetch_desc(&tmX);
    tma_prefetch_desc(&tmY);
    mbar_init(&bar_in[0], 1); mbar_init(&bar_in[1], 1);
    mbar_init(&bar_mma[0], 1); mbar_init(&bar_mma[1], 1);
    fence_barrier_init();
  }
  if (warp == 0) {
    __syncwarp();
    tmem_alloc(tmem_slot, TMEM_COLS);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  auto issue_tma = [&](int tile, int buf) {   // called by tid 32 only
    int t = tile;
    const int w0 = (t % p.tiles_w) * p.TW; t /= p.tiles_w;
    const int h0 = (t % p.tiles_h) * p.TH; t /= p.tiles_h;
    const int d0 = (t % p.tiles_d) * p.TD; t /= p.tiles_d;
    mbar_arrive_expect_tx(&bar_in[buf], tile_bytes);
    // TMA needs the box start to be 16-byte aligned along the innermost dimension (a start at column
    // 2*w0 - 1 is an illegal instruction): fetch from 2*w0 - PADL, PADL = 16 bytes of elements
    tma_load_4d(sX + (size_t)buf * tile_pitch, &tmX, &bar_in[buf], 2 * w0 - PADL, 2 * h0 - 1, p.sd * d0 - 1, t * CIN);
  };

  const int first = blockIdx.x;
  pdl_wait();                 // the input (and the output buffer's previous readers) belong to earlier work
  pdl_launch_dependents();
  if (tid == 32) {
    if (first < total_tiles) issue_tma(first, 0);
    if (first + (int)gridDim.x < total_tiles) issue_tma(first + gridDim.x, 1);
  }

  // weights -> swizzled B operand while the TMA is in flight: 32 rows x (KPAD/8) 16-byte chunks
  for (int c = tid; c < 32 * (KPAD / 8); c += 128) {
    const int row = c / (KPAD / 8), ch = c % (KPAD / 8);
    const uint4 v = __ldg(reinterpret_cast<const uint4*>(p.wt + row * KPAD + ch * 8));
    *reinterpret_cast<uint4*>(sB + (ch >> 3) * 4096 + sw128_offset(row, ch & 7)) = v;
  }
  if (tid < 32) { s_sc[tid] = __ldg(p.scale + tid); s_sh[tid] = __ldg(p.shift + tid); }
  __syncthreads();

  // this thread's output voxel inside a tile (w fastest) and its offset inside the halo tile
  const int wl = tid % p.TW;
  const int hl = (tid / p.TW) % p.TH;
  const int dl = tid / (p.TW * p.TH);
  const int vox_off = ((p.sd * dl) * p.THI + 2 * hl) * p.TWI + 2 * wl + PADL;
  const int plane = p.TDI * p.THI * p.TWI;
  const uint32_t taddr = tmem_base + ((uint32_t)(warp * 32) << 16);

  auto epilogue = [&](int tile, int buf) {
    uint32_t v0[16], v1[16];
    __syncwarp();
    tmem_ld_32x32b_x16(taddr + (uint32_t)(buf * 32), v0);
    tmem_ld_32x32b_x16(taddr + (uint32_t)(buf * 32 + 16), v1);
    tmem_ld_wait();
    // BN + activation, then the tile leaves through ONE TMA store: a thread owns a 64-byte row, so direct 16-byte
    // stores would touch 32 different rows per warp instruction (half-used sectors, 4 instructions per row)
    uint4 o4[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      uint32_t o[4];
      float sc[8], sh[8];
      *reinterpret_cast<float4*>(&sc[0]) = *reinterpret_cast<const float4*>(s_sc + q * 8);
      *reinterpret_cast<float4*>(&sc[4]) = *reinterpret_cast<const float4*>(s_sc + q * 8 + 4);
      *reinterpret_cast<float4*>(&sh[0]) = *reinterpret_cast<const float4*>(s_sh + q * 8);
      *reinterpret_cast<float4*>(&sh[4]) = *reinterpret_cast<const float4*>(s_sh + q * 8 + 4);
#pragma unroll
      for (int h = 0; h < 4; ++h) {
        const int c = q * 8 + h * 2;
        const float a0 = __uint_as_float(c < 16 ? v0[c & 15] : v1[c & 15]);
        const float a1 = __uint_as_float(c + 1 < 16 ? v0[(c + 1) & 15] : v1[(c + 1) & 15]);
        o[h] = pack_bf16x2(relu_nan1(__fadd_rn(__fmul_rn(a0, sc[h * 2]), sh[h * 2]), p.floor),
                           relu_nan1(__fadd_rn(__fmul_rn(a1, sc[h * 2 + 1]), sh[h * 2 + 1]), p.floor));
      }
      o4[q] = make_uint4(o[0], o[1], o[2], o[3]);
    }
    // (sOut is free: tid 32 waited for the previous store's read before this iteration's gather barrier)
#pragma unroll
    for (int q = 0; q < 4; ++q)      // 64-byte swizzle: 16-byte chunk ^= (row >> 1) & 3
      *reinterpret_cast<uint4*>(sOut + tid * 64 + ((q ^ ((tid >> 1) & 3)) << 4)) = o4[q];
    fence_proxy_async_smem();
    __syncthreads();
    if (tid == 32) {
      int t = tile;
      const int w0 = (t % p.tiles_w) * p.TW; t /= p.tiles_w;
      const int h0 = (t % p.tiles_h) * p.TH; t /= p.tiles_h;
      const int d0 = (t % p.tiles_d) * p.TD; t /= p.tiles_d;
      asm volatile(
          "cp.async.bulk.tensor.5d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5, %6}], [%1];" ::"l"(
              reinterpret_cast<uint64_t>(&tmY)),
          "r"(smem_u32(sOut)), "r"(0), "r"(w0), "r"(h0), "r"(d0), "r"(t)
          : "memory");
      asm volatile("cp.async.bulk.commit_group;" ::: "memory");
    }
  };

  int it = 0;
  int prev_tile = -1;
  for (int tile = first; tile < total_tiles; tile += gridDim.x, ++it) {
    const int buf = it & 1;
    const uint32_t par = (uint32_t)((it >> 1) & 1);
    mbar_wait(&bar_in[buf], par);

    // ---- gather the 27*CIN taps of this voxel into one K-major row (bf16 pairs in registers) ----
    uint32_t regs[NREG];
#pragma unroll
    for (int i = 0; i < NREG; ++i) regs[i] = 0u;
    const TIn* xt = reinterpret_cast<const TIn*>(sX + (size_t)buf * tile_pitch) + vox_off;
    if constexpr (sizeof(TIn) == 2) {
      // taps kw = 0..2 of group g sit at columns -1, 0, +1: words a = (col -2, col -1), b = (col 0, col +1).
      // Two groups give three packed registers with two byte permutes.
      uint32_t wa[NG], wb[NG];
#pragma unroll
      for (int g = 0; g < NG; ++g) {
        const int ci = g / 9, kd = (g / 3) % 3, kh = g % 3;
        const TIn* src = xt + ci * plane + (kd * p.THI + kh) * p.TWI;
        wa[g] = *reinterpret_cast<const uint32_t*>(src - 2);
        wb[g] = *reinterpret_cast<const uint32_t*>(src);
      }
#pragma unroll
      for (int g = 0; g + 1 < NG; g += 2) {
        const int r = (3 * g) >> 1;                           // 3g is even
        regs[r] = __byte_perm(wa[g], wb[g], 0x5432);          // (e0, e1) of group g
        regs[r + 1] = __byte_perm(wb[g], wa[g + 1], 0x7632);  // (e2 of g, e0 of g+1)
        regs[r + 2] = wb[g + 1];                              // (e1, e2) of group g+1
      }
      if constexpr (NG & 1) {
        const int g = NG - 1, r = (3 * g) >> 1;
        regs[r] = __byte_perm(wa[g], wb[g], 0x5432);
        regs[r + 1] = wb[g] >> 16;
      }
    } else {
#pragma unroll
      for (int g = 0; g < NG; ++g) {
        const int ci = g / 9, kd = (g / 3) % 3, kh = g % 3;
        const float* src = reinterpret_cast<const float*>(xt) + ci * plane + (kd * p.THI + kh) * p.TWI;
        const float a = src[-1];
        const float2 b = *reinterpret_cast<const float2*>(src);
        const uint32_t e0 = bf16_bits(a), e1 = bf16_bits(b.x), e2 = bf16_bits(b.y);
        const int k0 = g * 3;
        regs[(k0 + 0) >> 1] |= e0 << (16 * ((k0 + 0) & 1));
        regs[(k0 + 1) >> 1] |= e1 << (16 * ((k0 + 1) & 1));
        regs[(k0 + 2) >> 1] |= e2 << (16 * ((k0 + 2) & 1));
      }
    }
    // the A buffer of this parity was last read by the UMMAs of tile it-2: their completion was observed
    // in the epilogue of tile it-2 (bar_mma wait), which every thread has passed
    const uint32_t a_tmem = tmem_base + 64u + (uint32_t)(buf * NREG);
    __syncwarp();
#pragma unroll
    for (int j = 0; j < NREG; j += 32) tmem_st_32x32b_x32(a_tmem + ((uint32_t)(warp * 32) << 16) + (uint32_t)j, &regs[j]);
    tmem_st_wait();
    tc_fence_before();
    // the TMA store issued in the previous iteration has had the whole gather to read the staging tile: waiting
    // here (not in the epilogue) lets the barrier below also publish "sOut is free"
    if (tid == 32) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
    __syncthreads();              // all rows are in TMEM; everyone is also done reading sX[buf]; sOut is free

    if (tid == 32) {
      // the halo buffer is free: prefetch the tile two iterations ahead
      const int nxt = tile + 2 * (int)gridDim.x;
      if (nxt < total_tiles) issue_tma(nxt, buf);
      tc_fence_after();
      const uint32_t idesc = umma_idesc_bf16(128, 32);
#pragma unroll
      for (int kb = 0; kb < KB; ++kb) {
        const uint64_t db = umma_desc_k_sw128(smem_u32(sB + kb * 4096));
#pragma unroll
        for (int k = 0; k < 4; ++k)      // 16 bf16 of K = 8 TMEM columns of A
          umma_bf16_ts(tmem_base + (uint32_t)(buf * 32), a_tmem + (uint32_t)((kb * 4 + k) * 8), db + (uint64_t)(2 * k),
                       idesc, (kb | k) != 0 ? 1u : 0u);
      }
      umma_commit(&bar_mma[buf]);
    }
    __syncwarp();

    // ---- epilogue of the previous tile overlaps this tile's UMMAs ----
    if (prev_tile >= 0) {
      const int pb = (it - 1) & 1;
      mbar_wait(&bar_mma[pb], (uint32_t)(((it - 1) >> 1) & 1));
      tc_fence_after();
      epilogue(prev_tile, pb);
      tc_fence_before();
    }
    prev_tile = tile;
  }
  if (prev_tile >= 0) {
    const int pb = (it - 1) & 1;
    if (tid == 32) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");   // sOut free for the last tile
    __syncthreads();
    mbar_wait(&bar_mma[pb], (uint32_t)(((it - 1) >> 1) & 1));
    tc_fence_after();
    epilogue(prev_tile, pb);
  }

  if (tid == 32) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");   // every output tile has landed
  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    __syncwarp();
    tc_fence_after();
    tmem_dealloc(tmem_base, TMEM_COLS);
  }
}

// ------------------------------------------------------------------------------------------------
// Stem WEIGHT gradient on the same tiles: dW[co][k] = sum_voxels dz[v][co] * im2col(x)[v][k], k = ci*27 + tap.
// The forward kernel's machinery produces im2col rows from a TMA halo box in shared memory (36 four-byte LDS per
// voxel instead of 27 scalar global loads with index arithmetic); here the row goes to a padded smem tile and
// mma.sync (bf16, fp32 accumulate) contracts it with the voxel's 32 gradient channels.  Accumulators live in
// registers across all tiles of the persistent CTA; one (32, KPAD) partial slab per CTA, summed by the caller.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void sw_ldsm_x4_t(uint32_t addr, uint32_t (&r)[4]) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0, %1, %2, %3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}
__device__ __forceinline__ void sw_mma_bf16(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, "
      "{%0, %1, %2, %3};"
      : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

// FUSE: the BatchNorm + ReLU backward of the stem unit is applied to the gradient rows as they are loaded -- `dz`
// then is the gradient w.r.t. the ReLU OUTPUT and `f.z` the saved raw conv output; the rows
// dz = sc*dy + ka + z*kb (dy = g * [z*sc+sh > 0], the expression of the BatchNorm kernels, rounded to bf16 like the
// tensor they would have written) exist only in shared memory: the 113 MB gradient of the C3 stem is neither written
// nor read back.
struct StemBnFuse {
  const __nv_bfloat16* z;     // (M, 32) raw conv output
  const float* scale;
  const float* shift;
  const float* mean;
  const float* invstd;
  const float* dgamma;
  const float* dbeta;
  float inv_m;
};

template <typename TIn, int CIN, bool FUSE>
__global__ void __launch_bounds__(128, 4) stem_wgrad_tile_kernel(const __grid_constant__ CUtensorMap tmX,
                                                                 const StemParams p,
                                                                 const __nv_bfloat16* __restrict__ dz,
                                                                 float* __restrict__ partial, const StemBnFuse f) {
  __shared__ float s_bn[FUSE ? 4 : 1][32];      // scale, shift, ka, kb
  constexpr int KREAL = 27 * CIN;
  constexpr int KPAD = (KREAL <= 64) ? 64 : 128;
  constexpr int NREG = KPAD / 2;
  constexpr int PADL = 16 / (int)sizeof(TIn);
  constexpr int NG = 9 * CIN;
  constexpr int XP = KPAD + 8;            // padded pitches (elements): conflict-free ldmatrix
  constexpr int ZP = 40;
  constexpr int NB = KPAD / 64;           // 16-column groups per warp (each warp owns KPAD/4 columns)

  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw = smem_u32(smem_raw);
  uint8_t* smem = smem_raw + ((128u - (raw & 127u)) & 127u);
  __nv_bfloat16* sXc = reinterpret_cast<__nv_bfloat16*>(smem);                 // [128][XP]
  __nv_bfloat16* sZ = sXc + 128 * XP;                                          // [128][ZP]
  uint64_t* bar_in = reinterpret_cast<uint64_t*>(sZ + 128 * ZP);               // [2]
  const int tile_elems = CIN * p.TDI * p.THI * p.TWI;
  const uint32_t tile_bytes = (uint32_t)(tile_elems * sizeof(TIn));
  const uint32_t tile_pitch = (tile_bytes + 127u) & ~127u;
  uint8_t* sX = reinterpret_cast<uint8_t*>(bar_in) + 128;                      // 2 x halo tile

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int total_tiles = p.tiles_w * p.tiles_h * p.tiles_d * p.N;
  if (tid == 32) {
    tma_prefetch_desc(&tmX);
    mbar_init(&bar_in[0], 1);
    mbar_init(&bar_in[1], 1);
    fence_barrier_init();
  }
  __syncthreads();
  auto issue_tma = [&](int tile, int buf) {
    int t = tile;
    const int w0 = (t % p.tiles_w) * p.TW; t /= p.tiles_w;
    const int h0 = (t % p.tiles_h) * p.TH; t /= p.tiles_h;
    const int d0 = (t % p.tiles_d) * p.TD; t /= p.tiles_d;
    mbar_arrive_expect_tx(&bar_in[buf], tile_bytes);
    tma_load_4d(sX + (size_t)buf * tile_pitch, &tmX, &bar_in[buf], 2 * w0 - PADL, 2 * h0 - 1, p.sd * d0 - 1, t * CIN);
  };
  const int first = blockIdx.x;
  pdl_wait();
  pdl_launch_dependents();
  if (tid == 32) {
    if (first < total_tiles) issue_tma(first, 0);
    if (first + (int)gridDim.x < total_tiles) issue_tma(first + gridDim.x, 1);
  }
  if constexpr (FUSE) {
    if (tid < 32) {
      const float scj = f.scale[tid], isj = f.invstd[tid], muj = f.mean[tid];
      const float t = scj * isj * f.dgamma[tid] * f.inv_m;
      s_bn[0][tid] = scj;
      s_bn[1][tid] = f.shift[tid];
      s_bn[2][tid] = fmaf(muj, t, -(scj * f.dbeta[tid] * f.inv_m));
      s_bn[3][tid] = -t;
    }
    __syncthreads();
  }
  const int wl = tid % p.TW;
  const int hl = (tid / p.TW) % p.TH;
  const int dl = tid / (p.TW * p.TH);
  const int vox_off = ((p.sd * dl) * p.THI + 2 * hl) * p.TWI + 2 * wl + PADL;
  const int plane = p.TDI * p.THI * p.TWI;

  float acc[2][2 * NB][4];
#pragma unroll
  for (int a = 0; a < 2; ++a)
#pragma unroll
    for (int b = 0; b < 2 * NB; ++b)
#pragma unroll
      for (int c = 0; c < 4; ++c) acc[a][b][c] = 0.f;
  const uint32_t sXc_u = smem_u32(sXc), sZ_u = smem_u32(sZ);
  const int lq = lane >> 3, lr = lane & 7;

  int it = 0;
  for (int tile = first; tile < total_tiles; tile += gridDim.x, ++it) {
    const int buf = it & 1;
    mbar_wait(&bar_in[buf], (uint32_t)((it >> 1) & 1));
    // ---- im2col row of this thread's voxel (same gather as the forward kernel) ----
    uint32_t regs[NREG];
#pragma unroll
    for (int i = 0; i < NREG; ++i) regs[i] = 0u;
    const TIn* xt = reinterpret_cast<const TIn*>(sX + (size_t)buf * tile_pitch) + vox_off;
    if constexpr (sizeof(TIn) == 2) {
      uint32_t wa[NG], wb[NG];
#pragma unroll
      for (int g = 0; g < NG; ++g) {
        const int ci = g / 9, kd = (g / 3) % 3, kh = g % 3;
        const TIn* src = xt + ci * plane + (kd * p.THI + kh) * p.TWI;
        wa[g] = *reinterpret_cast<const uint32_t*>(src - 2);
        wb[g] = *reinterpret_cast<const uint32_t*>(src);
      }
#pragma unroll
      for (int g = 0; g + 1 < NG; g += 2) {
        const int r = (3 * g) >> 1;
        regs[r] = __byte_perm(wa[g], wb[g], 0x5432);
        regs[r + 1] = __byte_perm(wb[g], wa[g + 1], 0x7632);
        regs[r + 2] = wb[g + 1];
      }
      if constexpr (NG & 1) {
        const int g = NG - 1, r = (3 * g) >> 1;
        regs[r] = __byte_perm(wa[g], wb[g], 0x5432);
        regs[r + 1] = wb[g] >> 16;
      }
    } else {
#pragma unroll
      for (int g = 0; g < NG; ++g) {
        const int ci = g / 9, kd = (g / 3) % 3, kh = g % 3;
        const float* src = reinterpret_cast<const float*>(xt) + ci * plane + (kd * p.THI + kh) * p.TWI;
        const float a = src[-1];
        const float2 b = *reinterpret_cast<const float2*>(src);
        const uint32_t e0 = bf16_bits(a), e1 = bf16_bits(b.x), e2 = bf16_bits(b.y);
        const int k0 = g * 3;
        regs[(k0 + 0) >> 1] |= e0 << (16 * ((k0 + 0) & 1));
        regs[(k0 + 1) >> 1] |= e1 << (16 * ((k0 + 1) & 1));
        regs[(k0 + 2) >> 1] |= e2 << (16 * ((k0 + 2) & 1));
      }
    }
    // ---- this voxel's 32 gradient channels (zero outside the volume) ----
    int t = tile;
    const int wo = (t % p.tiles_w) * p.TW + wl; t /= p.tiles_w;
    const int ho = (t % p.tiles_h) * p.TH + hl; t /= p.tiles_h;
    const int dzo = (t % p.tiles_d) * p.TD + dl; t /= p.tiles_d;
    uint4 g4[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) g4[q] = make_uint4(0u, 0u, 0u, 0u);
    if (wo < p.Wo && ho < p.Ho && dzo < p.Do) {
      const long long row = (((long long)t * p.Do + dzo) * p.Ho + ho) * p.Wo + wo;
      const uint4* src = reinterpret_cast<const uint4*>(dz + row * 32);
#pragma unroll
      for (int q = 0; q < 4; ++q) g4[q] = __ldg(src + q);
      if constexpr (FUSE) {
        const uint4* zsrc = reinterpret_cast<const uint4*>(f.z + row * 32);
        uint4 z4[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) z4[q] = __ldg(zsrc + q);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const uint32_t zu[4] = {z4[q].x, z4[q].y, z4[q].z, z4[q].w};
          const uint32_t gu[4] = {g4[q].x, g4[q].y, g4[q].z, g4[q].w};
          uint32_t ou[4];
#pragma unroll
          for (int h = 0; h < 4; ++h) {
            float o2[2];
#pragma unroll
            for (int e = 0; e < 2; ++e) {
              const int c = q * 8 + h * 2 + e;
              const float zf = e ? bf16_hi(zu[h]) : bf16_lo(zu[h]);
              const float gf = e ? bf16_hi(gu[h]) : bf16_lo(gu[h]);
              const float scc = s_bn[0][c];
              const float pre = __fadd_rn(__fmul_rn(zf, scc), s_bn[1][c]);
              const float dy = (pre > 0.f) ? gf : 0.f;
              o2[e] = fmaf(zf, s_bn[3][c], fmaf(scc, dy, s_bn[2][c]));
            }
            ou[h] = pack_bf16x2(o2[0], o2[1]);
          }
          g4[q] = make_uint4(ou[0], ou[1], ou[2], ou[3]);
        }
      }
    }
    __syncthreads();            // the previous tile's fragments have been read; everyone is done with sX[buf]
    if (tid == 32) {
      const int nxt = tile + 2 * (int)gridDim.x;
      if (nxt < total_tiles) issue_tma(nxt, buf);
    }
#pragma unroll
    for (int j = 0; j < KPAD / 8; ++j)
      *reinterpret_cast<uint4*>(sXc + tid * XP + j * 8) = make_uint4(regs[4 * j], regs[4 * j + 1], regs[4 * j + 2], regs[4 * j + 3]);
#pragma unroll
    for (int q = 0; q < 4; ++q) *reinterpret_cast<uint4*>(sZ + tid * ZP + q * 8) = g4[q];
    __syncthreads();
#pragma unroll
    for (int ks = 0; ks < 8; ++ks) {
      const int kk = ks * 16;
      uint32_t afr[2][4];
#pragma unroll
      for (int a = 0; a < 2; ++a)      // A = dz^T (16 co x 16 voxels), transposed on load
        sw_ldsm_x4_t(sZ_u + (uint32_t)(((kk + (lq >> 1) * 8 + lr) * ZP + a * 16 + (lq & 1) * 8) * 2), afr[a]);
#pragma unroll
      for (int b = 0; b < NB; ++b) {
        uint32_t bfr[4];               // B = im2col rows (16 voxels x 16 k), two n8 tiles
        sw_ldsm_x4_t(sXc_u + (uint32_t)(((kk + (lq & 1) * 8 + lr) * XP + warp * (KPAD / 4) + b * 16 + (lq >> 1) * 8) * 2), bfr);
#pragma unroll
        for (int a = 0; a < 2; ++a) {
          sw_mma_bf16(acc[a][2 * b], afr[a], bfr[0], bfr[1]);
          sw_mma_bf16(acc[a][2 * b + 1], afr[a], bfr[2], bfr[3]);
        }
      }
    }
  }
  float* out = partial + (size_t)blockIdx.x * 32 * KPAD + warp * (KPAD / 4);
#pragma unroll
  for (int a = 0; a < 2; ++a)
#pragma unroll
    for (int b = 0; b < 2 * NB; ++b) {
      const int co = a * 16 + (lane >> 2), k = b * 8 + (lane & 3) * 2;
      *reinterpret_cast<float2*>(out + (size_t)co * KPAD + k) = make_float2(acc[a][b][0], acc[a][b][1]);
      *reinterpret_cast<float2*>(out + (size_t)(co + 8) * KPAD + k) = make_float2(acc[a][b][2], acc[a][b][3]);
    }
}

static inline int p2ceil(int v) {
  int r = 1;
  while (r < v) r <<= 1;
  return r;
}

template <typename TIn, int CIN>
static int launch_stem_tc(const void* x, const StemParams& p0, CUtensorMapDataType dt, cudaStream_t st) {
  StemParams p = p0;
  constexpr int KPAD = (27 * CIN <= 64) ? 64 : 128;
  constexpr int KB = KPAD / 64;
  CUtensorMap tm;
  {
    PFN_encodeTiled enc = get_encode_tiled();
    if (!enc) return SSD3D_ERR_TMA;
    const cuuint64_t es = sizeof(TIn);
    cuuint64_t gdim[4] = {(cuuint64_t)p.W, (cuuint64_t)p.H, (cuuint64_t)p.D, (cuuint64_t)p.N * CIN};
    cuuint64_t gstr[3] = {(cuuint64_t)p.W * es, (cuuint64_t)p.W * p.H * es, (cuuint64_t)p.W * p.H * p.D * es};
    cuuint32_t box[4] = {(cuuint32_t)p.TWI, (cuuint32_t)p.THI, (cuuint32_t)p.TDI, (cuuint32_t)CIN};
    cuuint32_t estr[4] = {1, 1, 1, 1};
    CUresult r = enc(&tm, dt, 4, const_cast<void*>(x), gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return SSD3D_ERR_TMA;
  }
  const size_t tile_pitch = ((size_t)CIN * p.TDI * p.THI * p.TWI * sizeof(TIn) + 127) & ~(size_t)127;
  const size_t smem = 1024 + (size_t)KB * 4096 + 1024 + 8192 + 2 * tile_pitch + 128;
  CUtensorMap tmY;
  {
    const uint64_t dims[5] = {32ull, (uint64_t)p.Wo, (uint64_t)p.Ho, (uint64_t)p.Do, (uint64_t)p.N};
    const uint64_t strides[4] = {64ull, (uint64_t)p.Wo * 64, (uint64_t)p.Ho * p.Wo * 64, (uint64_t)p.Do * p.Ho * p.Wo * 64};
    const uint32_t box[5] = {32u, (uint32_t)p.TW, (uint32_t)p.TH, (uint32_t)p.TD, 1u};
    if (make_tma_bf16(&tmY, p.y, 5, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_64B)) return SSD3D_ERR_TMA;
  }
  cudaError_t e = cudaFuncSetAttribute(stem_tc_kernel<TIn, CIN>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return (int)e;
  // persistent grid: CTAs per SM bounded by shared memory (~31 KB each), tensor memory (128 or 256 of 512
  // columns each) and registers (launch bounds 3); never more CTAs than tiles
  const int n_sm = persistent_sms();
  const long long tiles = (long long)p.tiles_w * p.tiles_h * p.tiles_d * p.N;
  long long per_sm = (smem + 1024) * 4 <= 227 * 1024 ? 4 : ((smem + 1024) * 3 <= 227 * 1024 ? 3 : (smem * 2 <= 220 * 1024 ? 2 : 1));
  if (KPAD > 64 && per_sm > 2) per_sm = 2;      // 256 TMEM columns per CTA
  const unsigned grid = (unsigned)(tiles < per_sm * n_sm ? tiles : per_sm * n_sm);
  SSD3D_LAUNCH_PDL((stem_tc_kernel<TIn, CIN>), dim3(grid), dim3(128), smem, st, tm, tmY, p);
  return SSD3D_OK;
}

template <typename TIn, int CIN>
static int launch_stem_wgrad(const void* x, const StemParams& p, CUtensorMapDataType dt, const __nv_bfloat16* dz,
                             float* partial, int max_slabs, int* slabs, cudaStream_t st, const StemBnFuse* fuse) {
  constexpr int KPAD = (27 * CIN <= 64) ? 64 : 128;
  CUtensorMap tm;
  {
    PFN_encodeTiled enc = get_encode_tiled();
    if (!enc) return SSD3D_ERR_TMA;
    const cuuint64_t es = sizeof(TIn);
    cuuint64_t gdim[4] = {(cuuint64_t)p.W, (cuuint64_t)p.H, (cuuint64_t)p.D, (cuuint64_t)p.N * CIN};
    cuuint64_t gstr[3] = {(cuuint64_t)p.W * es, (cuuint64_t)p.W * p.H * es, (cuuint64_t)p.W * p.H * p.D * es};
    cuuint32_t box[4] = {(cuuint32_t)p.TWI, (cuuint32_t)p.THI, (cuuint32_t)p.TDI, (cuuint32_t)CIN};
    cuuint32_t estr[4] = {1, 1, 1, 1};
    CUresult r = enc(&tm, dt, 4, const_cast<void*>(x), gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return SSD3D_ERR_TMA;
  }
  const size_t tile_pitch = ((size_t)CIN * p.TDI * p.THI * p.TWI * sizeof(TIn) + 127) & ~(size_t)127;
  const size_t smem = 128 + (size_t)128 * (KPAD + 8) * 2 + 128 * 40 * 2 + 128 + 2 * tile_pitch;
  cudaError_t e = fuse ? cudaFuncSetAttribute(stem_wgrad_tile_kernel<TIn, CIN, true>,
                                             cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)
                       : cudaFuncSetAttribute(stem_wgrad_tile_kernel<TIn, CIN, false>,
                                              cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return (int)e;
  const long long tiles = (long long)p.tiles_w * p.tiles_h * p.tiles_d * p.N;
  long long per_sm = (smem + 1024) * 4 <= 227 * 1024 ? 4 : ((smem + 1024) * 3 <= 227 * 1024 ? 3 : (smem * 2 <= 220 * 1024 ? 2 : 1));
  long long grid = per_sm * persistent_sms();
  if (grid > tiles) grid = tiles;
  if (grid > max_slabs) grid = max_slabs;
  if (grid < 1) return SSD3D_ERR_ARG;
  if (fuse) {
    SSD3D_LAUNCH_PDL((stem_wgrad_tile_kernel<TIn, CIN, true>), dim3((unsigned)grid), dim3(128), smem, st, tm, p, dz,
                     partial, *fuse);
  } else {
    SSD3D_LAUNCH_PDL((stem_wgrad_tile_kernel<TIn, CIN, false>), dim3((unsigned)grid), dim3(128), smem, st, tm, p, dz,
                     partial, StemBnFuse{});
  }
  *slabs = (int)grid;
  return SSD3D_OK;
}

}  // namespace ssd3d

using namespace ssd3d;

// 1 when the tensor-core stem can take this input (TMA needs 16-byte row strides), else 0
extern "C" int ssd3d_stem_tc_supported(int x_is_bf16, int Cin, int W) {
  if (Cin < 1 || Cin > 4) return 0;
  return ((W * (x_is_bf16 ? 2 : 4)) % 16 == 0) ? 1 : 0;
}

// output tile + halo box of one 128-voxel tile (shared by the forward and the weight-gradient kernels)
static int stem_tiling(StemParams& p, int x_is_bf16, int N, int D, int H, int W, int stride_d) {
  p.N = N; p.D = D; p.H = H; p.W = W; p.sd = stride_d;
  p.Do = (D - 1) / stride_d + 1; p.Ho = (H - 1) / 2 + 1; p.Wo = (W - 1) / 2 + 1;
  // output tile: widest W extent (<= 64) that wastes < 15 % of its columns, then H, then D
  int tw = 8;
  for (int c : {64, 32, 16, 8}) {
    if (c > p2ceil(p.Wo)) continue;
    const int padded = ((p.Wo + c - 1) / c) * c;
    if (padded * 100 <= p.Wo * 115 || c == 8) { tw = c; break; }
  }
  if (p2ceil(p.Wo) < tw) tw = p2ceil(p.Wo);
  p.TW = tw;
  int rest = 128 / p.TW;
  p.TH = p2ceil(p.Ho) < rest ? p2ceil(p.Ho) : rest;
  rest /= p.TH;
  p.TD = rest;                                 // whatever remains goes to D (rows past Do are masked)
  const int padl = x_is_bf16 ? 8 : 4;          // 16 bytes of elements on the left (see the kernel)
  p.TWI = 2 * p.TW + padl;                      // columns 2*w0 - padl .. 2*w0 + 2*TW - 1: a multiple of 16 bytes
  // every tile's first column 2*k*TW - padl must stay 16-byte aligned
  if (p.Wo > p.TW && ((2 * p.TW * (x_is_bf16 ? 2 : 4)) % 16) != 0) return SSD3D_ERR_UNSUPPORTED;
  p.THI = 2 * p.TH + 1;
  p.TDI = stride_d * (p.TD - 1) + 3;
  if (p.TWI > 256 || p.THI > 256 || p.TDI > 256) return SSD3D_ERR_UNSUPPORTED;
  p.tiles_w = (p.Wo + p.TW - 1) / p.TW;
  p.tiles_h = (p.Ho + p.TH - 1) / p.TH;
  p.tiles_d = (p.Do + p.TD - 1) / p.TD;
  return SSD3D_OK;
}

static int stem_tc(const void* x, int x_is_bf16, const void* w_tc, const float* scale, const float* shift, void* y,
                   int N, int Cin, int D, int H, int W, int stride_d, int relu, cudaStream_t st) {
  StemParams p{};
  p.floor = SSD3D_FLOOR(relu);
  if (const int rc = stem_tiling(p, x_is_bf16, N, D, H, W, stride_d)) return rc;
  p.wt = static_cast<const __nv_bfloat16*>(w_tc);
  p.scale = scale;
  p.shift = shift;
  p.y = static_cast<__nv_bfloat16*>(y);
#define STEM_CASE(T, DT, C) return launch_stem_tc<T, C>(x, p, DT, st)
  if (x_is_bf16) {
    switch (Cin) {
      case 1: STEM_CASE(__nv_bfloat16, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 1);
      case 2: STEM_CASE(__nv_bfloat16, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2);
      case 3: STEM_CASE(__nv_bfloat16, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3);
      default: STEM_CASE(__nv_bfloat16, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4);
    }
  } else {
    switch (Cin) {
      case 1: STEM_CASE(float, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 1);
      case 2: STEM_CASE(float, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2);
      case 3: STEM_CASE(float, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3);
      default: STEM_CASE(float, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4);
    }
  }
#undef STEM_CASE
}

extern "C" int ssd3d_stem_conv_affine_simt(const void* x, int x_is_bf16, const void* w, const float* scale,
                                           const float* shift, void* y, int N, int Cin, int D, int H, int W,
                                           int stride_d, int relu, void* stream);

extern "C" int ssd3d_stem_conv_affine_tz(const void* x, int x_is_bf16, const void* w, const float* scale,
                                         const float* shift, void* y, int N, int Cin, int D, int H, int W, int stride_d,
                                         int relu, void* stream);
extern "C" int ssd3d_stem_tz_supported(int x_is_bf16, int Cin, int W);

// Which tcgen05 stem kernel ssd3d_stem_conv_affine picks: the banded-B kernel (conv_stem_tz.cu) when its 32-voxel row
// slots are all full (W a multiple of 64: 43-44 us against 45.5 us for the gather kernel at the benchmark shape; both
// sit on the mixed read/write HBM floor), the gather kernel otherwise (Wo = 48 wastes a third of the second slot:
// 37-41 vs 37.3 us).
static bool stem_tz_wanted(int x_is_bf16, int Cin, int W) {
  return ssd3d_stem_tz_supported(x_is_bf16, Cin, W) && W % 64 == 0;
}

extern "C" int ssd3d_stem_conv_affine_tc(const void* x, int x_is_bf16, const void* w, const float* scale,
                                         const float* shift, void* y, int N, int Cin, int D, int H, int W, int stride_d,
                                         int relu, void* stream) {
  if (!x || !w || !scale || !shift || !y || N <= 0 || D <= 0 || H <= 0 || W <= 0) return SSD3D_ERR_ARG;
  if (stride_d != 1 && stride_d != 2) return SSD3D_ERR_ARG;
  if (!ssd3d_stem_tc_supported(x_is_bf16, Cin, W)) return SSD3D_ERR_UNSUPPORTED;
  return stem_tc(x, x_is_bf16, w, scale, shift, y, N, Cin, D, H, W, stride_d, relu, static_cast<cudaStream_t>(stream));
}

extern "C" int ssd3d_stem_conv_affine(const void* x, int x_is_bf16, const void* w, const float* scale,
                                      const float* shift, void* y, int N, int Cin, int D, int H, int W, int stride_d,
                                      int relu, void* stream) {
  if (!x || !w || !scale || !shift || !y || N <= 0 || D <= 0 || H <= 0 || W <= 0) return SSD3D_ERR_ARG;
  if (stride_d != 1 && stride_d != 2) return SSD3D_ERR_ARG;
  if (Cin < 1 || Cin > 4) return SSD3D_ERR_UNSUPPORTED;
  if (stem_tz_wanted(x_is_bf16, Cin, W)) {
    const int rc = ssd3d_stem_conv_affine_tz(x, x_is_bf16, w, scale, shift, y, N, Cin, D, H, W, stride_d, relu, stream);
    if (rc != SSD3D_ERR_UNSUPPORTED) return rc;
  }
  if (ssd3d_stem_tc_supported(x_is_bf16, Cin, W)) {
    const int rc = stem_tc(x, x_is_bf16, w, scale, shift, y, N, Cin, D, H, W, stride_d, relu,
                           static_cast<cudaStream_t>(stream));
    if (rc != SSD3D_ERR_UNSUPPORTED) return rc;
  }
  // rows that TMA cannot address (W * elemsize not a multiple of 16 bytes): CUDA-core kernel
  return ssd3d_stem_conv_affine_simt(x, x_is_bf16, w, scale, shift, y, N, Cin, D, H, W, stride_d, relu, stream);
}

extern "C" int ssd3d_stem_conv_bn_relu(const void* x, int x_is_bf16, const void* w, const float* scale,
                                       const float* shift, void* y, int N, int Cin, int D, int H, int W, int stride_d,
                                       void* stream) {
  return ssd3d_stem_conv_affine(x, x_is_bf16, w, scale, shift, y, N, Cin, D, H, W, stride_d, 1, stream);
}

// Tile-based stem weight gradient (used by ssd3d_stem_wgrad in train.cu): writes `*slabs` partial slabs of
// (32, *kpad) fp32 to `partial`; SSD3D_ERR_UNSUPPORTED when TMA cannot address the input rows.
namespace ssd3d {
// bn (optional, 8 pointers: z, scale, shift, mean, invstd, dgamma, dbeta, &inv_m): fuse the stem unit's BatchNorm + ReLU
// backward into the gradient load (`dz` is then the gradient w.r.t. the unit's output)
int stem_wgrad_tiles(const void* dz, const void* x, int x_is_bf16, int N, int Cin, int D, int H, int W, int stride_d,
                     float* partial, int max_slabs, int* slabs, int* kpad, cudaStream_t st, const void* const* bn) {
  if (!ssd3d_stem_tc_supported(x_is_bf16, Cin, W)) return SSD3D_ERR_UNSUPPORTED;
  StemParams p{};
  if (const int rc = stem_tiling(p, x_is_bf16, N, D, H, W, stride_d)) return rc;
  *kpad = (27 * Cin <= 64) ? 64 : 128;
  const __nv_bfloat16* g = static_cast<const __nv_bfloat16*>(dz);
  StemBnFuse fz{};
  const StemBnFuse* fuse = nullptr;
  if (bn) {
    fz.z = static_cast<const __nv_bfloat16*>(bn[0]);
    fz.scale = static_cast<const float*>(bn[1]); fz.shift = static_cast<const float*>(bn[2]);
    fz.mean = static_cast<const float*>(bn[3]);  fz.invstd = static_cast<const float*>(bn[4]);
    fz.dgamma = static_cast<const float*>(bn[5]); fz.dbeta = static_cast<const float*>(bn[6]);
    fz.inv_m = *static_cast<const float*>(bn[7]);
    fuse = &fz;
  }
#define STEM_WG(T, DT, C) return launch_stem_wgrad<T, C>(x, p, DT, g, partial, max_slabs, slabs, st, fuse)
  if (x_is_bf16) {
    switch (Cin) {
      case 1: STEM_WG(__nv_bfloat16, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 1);
      case 2: STEM_WG(__nv_bfloat16, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2);
      case 3: STEM_WG(__nv_bfloat16, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3);
      default: STEM_WG(__nv_bfloat16, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4);
    }
  } else {
    switch (Cin) {
      case 1: STEM_WG(float, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 1);
      case 2: STEM_WG(float, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2);
      case 3: STEM_WG(float, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3);
      default: STEM_WG(float, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4);
    }
  }
#undef STEM_WG
}
}  // namespace ssd3d
