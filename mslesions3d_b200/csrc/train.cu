// Training-step kernels of the SSD3D network (LSSD3D.training_step, ssd3d.py:467-531; the reference gets
// them from torch autograd over nn.Conv3d / nn.BatchNorm3d / nn.ReLU, mobilenet.py:26-49, ssd3d.py:131-167):
//   * train-mode BatchNorm: per-channel batch statistics of a raw conv output (two-stage, deterministic),
//     running-stat update, normalise + ReLU; and its backward (ReLU mask recomputed from the saved raw
//     output, dgamma / dbeta reductions, dz)
//   * weight gradients of the pointwise and stem (3x3x3, NCDHW input) convolutions as ONE split-M implicit GEMM
//     dW[n][k] = sum_m dz[m][n] * im2col(x)[m][k]   on mma.sync bf16 tensor cores (operands are channels-last,
//     i.e. M-major: fragments come from ldmatrix.trans), fixed-order reduction; the head (3x3x3) weight gradient
//     in an activation-stationary form of the same contraction
//   * data gradient of the head convs (transposed 3x3x3 conv, 16 -> C channels) as an mma.sync implicit GEMM
//   * depthwise 3x3x3 data and weight gradients (HBM-bound CUDA-core kernels, 16-byte channel vectors)
//   * packing of d(loss)/d(locs, scores) into the head's (voxel, 16) bf16 gradient rows
//   * fused Adam over the flat parameter / gradient buffers (ssd3d.py:704-722)
// Activations and activation gradients are channels-last bf16; every reduction accumulates in fp32 (fp64
// for the final cross-block sums) and is bit-reproducible run to run.
#include <algorithm>
#include "common.cuh"
#include "../../include/ssd3d_b200.h"

namespace ssd3d {

typedef __nv_bfloat16 bf16;

__device__ __forceinline__ uint4 ld_nc16(const void* p) {
  uint4 r;
  asm volatile("ld.global.nc.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
  return r;
}
__device__ __forceinline__ void unpack8f(const uint4& v, float (&f)[8]) {
  f[0] = bf16_lo(v.x); f[1] = bf16_hi(v.x);
  f[2] = bf16_lo(v.y); f[3] = bf16_hi(v.y);
  f[4] = bf16_lo(v.z); f[5] = bf16_hi(v.z);
  f[6] = bf16_lo(v.w); f[7] = bf16_hi(v.w);
}
__device__ __forceinline__ uint4 pack8f(const float (&v)[8]) {
  uint4 o;
  o.x = pack_bf16x2(v[0], v[1]);
  o.y = pack_bf16x2(v[2], v[3]);
  o.z = pack_bf16x2(v[4], v[5]);
  o.w = pack_bf16x2(v[6], v[7]);
  return o;
}
__device__ __forceinline__ void load8(const float* p, float (&f)[8]) {
  *reinterpret_cast<float4*>(&f[0]) = __ldg(reinterpret_cast<const float4*>(p));
  *reinterpret_cast<float4*>(&f[4]) = __ldg(reinterpret_cast<const float4*>(p + 4));
}

// ------------------------------------------------------------------------------------------------
// Column reductions over a channels-last (M, C) bf16 matrix; thread = 8 channels x a strided set of rows.
//   MODE 0 (BN forward) : s0 = sum z,  s1 = sum z^2
//   MODE 1 (BN backward): dy = g * [z*scale+shift > 0], xhat = (z-mean)*invstd;  s0 = sum dy, s1 = sum dy*xhat
// partial[(block*2 + {0,1}) * C + c]
// ------------------------------------------------------------------------------------------------
template <int MODE>
__global__ void __launch_bounds__(256) colreduce_kernel(const bf16* __restrict__ z, const bf16* __restrict__ g,
                                                        const float* __restrict__ scale,
                                                        const float* __restrict__ shift,
                                                        const float* __restrict__ mean,
                                                        const float* __restrict__ invstd, long long M, int C,
                                                        long long rows_per_block, float* __restrict__ partial) {
  __shared__ float red[256 * 16];
  pdl_wait();
  pdl_launch_dependents();
  const int CV = C >> 3;
  const int RP = blockDim.x / CV;
  const int cv = threadIdx.x % CV, r = threadIdx.x / CV;
  const int c0 = cv << 3;
  float s0[8], s1[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) { s0[j] = 0.f; s1[j] = 0.f; }
  float sc[8], sh[8], mu[8], is[8];
  if (MODE == 1) {
    load8(scale + c0, sc); load8(shift + c0, sh); load8(mean + c0, mu); load8(invstd + c0, is);
  }
  const long long m_begin = (long long)blockIdx.x * rows_per_block;
  const long long m_end = (m_begin + rows_per_block < M) ? m_begin + rows_per_block : M;
  // four rows in flight per thread (all loads first): the pass is latency-bound with one
  auto add_row = [&](const uint4& zu, const uint4& gu) {
    float zf[8];
    unpack8f(zu, zf);
    if (MODE == 0) {
#pragma unroll
      for (int j = 0; j < 8; ++j) { s0[j] += zf[j]; s1[j] = fmaf(zf[j], zf[j], s1[j]); }
    } else {
      float gf[8];
      unpack8f(gu, gf);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float pre = __fadd_rn(__fmul_rn(zf[j], sc[j]), sh[j]);
        const float dy = (pre > 0.f) ? gf[j] : 0.f;
        const float xh = (zf[j] - mu[j]) * is[j];
        s0[j] += dy;
        s1[j] = fmaf(dy, xh, s1[j]);
      }
    }
  };
  long long m = m_begin + r;
  for (; m + 3ll * RP < m_end; m += 4ll * RP) {
    uint4 zu[4], gu[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) zu[i] = ld_nc16(z + (m + (long long)i * RP) * C + c0);
    if (MODE == 1) {
#pragma unroll
      for (int i = 0; i < 4; ++i) gu[i] = ld_nc16(g + (m + (long long)i * RP) * C + c0);
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) add_row(zu[i], MODE == 1 ? gu[i] : zu[i]);
  }
  for (; m < m_end; m += RP) {
    const uint4 zu = ld_nc16(z + m * C + c0);
    add_row(zu, MODE == 1 ? ld_nc16(g + m * C + c0) : zu);
  }
#pragma unroll
  for (int j = 0; j < 8; ++j) { red[threadIdx.x * 16 + j] = s0[j]; red[threadIdx.x * 16 + 8 + j] = s1[j]; }
  __syncthreads();
  if (r == 0) {
    for (int rr = 1; rr < RP; ++rr) {
      const float* src = red + (rr * CV + cv) * 16;
#pragma unroll
      for (int j = 0; j < 8; ++j) { s0[j] += src[j]; s1[j] += src[8 + j]; }
    }
    float* dst = partial + (size_t)blockIdx.x * 2 * C;
#pragma unroll
    for (int j = 0; j < 8; ++j) { dst[c0 + j] = s0[j]; dst[C + c0 + j] = s1[j]; }
  }
}

// Cross-block sums of the column partials: 32 channels x 32 block lanes per CTA (1024 threads), fp64, combined in
// a fixed order.  The loads of a lane are independent (unrolled): the loop is L2-latency bound otherwise.
constexpr int FIN_LANES = 32;
__device__ __forceinline__ void colpartials_sum(const float* __restrict__ partial, int B, int C, int c, int lane,
                                                double (&red)[FIN_LANES][32][2], double& s, double& q) {
  double ls = 0.0, lq = 0.0;
  if (c < C) {
#pragma unroll 4
    for (int b = lane; b < B; b += FIN_LANES) {
      const float a0 = partial[(size_t)b * 2 * C + c];
      const float a1 = partial[(size_t)b * 2 * C + C + c];
      ls += (double)a0;
      lq += (double)a1;
    }
  }
  red[lane][threadIdx.x & 31][0] = ls;
  red[lane][threadIdx.x & 31][1] = lq;
  __syncthreads();
  s = 0.0; q = 0.0;
  if (lane == 0) {
#pragma unroll
    for (int l = 0; l < FIN_LANES; ++l) { s += red[l][threadIdx.x & 31][0]; q += red[l][threadIdx.x & 31][1]; }
  }
}

// BN forward finalize: batch mean / biased variance -> scale = gamma*invstd, shift = beta - mean*scale,
// running statistics (momentum update with the unbiased variance, as nn.BatchNorm3d in train mode).
__global__ void __launch_bounds__(1024) bn_finalize_fwd_kernel(const float* __restrict__ partial, int B, int C,
                                                              long long M, const float* __restrict__ gamma,
                                                              const float* __restrict__ beta, float eps,
                                                              float momentum, float* __restrict__ running_mean,
                                                              float* __restrict__ running_var,
                                                              float* __restrict__ scale, float* __restrict__ shift,
                                                              float* __restrict__ mean, float* __restrict__ invstd,
                                                              long long* __restrict__ num_batches_tracked) {
  __shared__ double red[FIN_LANES][32][2];
  pdl_wait();
  pdl_launch_dependents();
  if (num_batches_tracked && blockIdx.x == 0 && threadIdx.x == 0) *num_batches_tracked += 1;
  const int c = blockIdx.x * 32 + (threadIdx.x & 31), lane = threadIdx.x >> 5;
  double s, q;
  colpartials_sum(partial, B, C, c, lane, red, s, q);
  if (lane != 0 || c >= C) return;
  const double mu = s / (double)M;
  double var = q / (double)M - mu * mu;
  if (var < 0.0) var = 0.0;
  const float istd = (float)(1.0 / sqrt(var + (double)eps));
  const float ga = gamma ? gamma[c] : 1.f, be = beta ? beta[c] : 0.f;
  const float sc = ga * istd;
  scale[c] = sc;
  shift[c] = be - (float)mu * sc;
  mean[c] = (float)mu;
  invstd[c] = istd;
  if (running_mean && running_var) {
    const double unbiased = (M > 1) ? var * (double)M / (double)(M - 1) : var;
    running_mean[c] = (float)((1.0 - (double)momentum) * (double)running_mean[c] + (double)momentum * mu);
    running_var[c] = (float)((1.0 - (double)momentum) * (double)running_var[c] + (double)momentum * unbiased);
  }
}

// BN backward finalize: dbeta = sum dy, dgamma = sum dy*xhat (written into the parameter gradients).
__global__ void __launch_bounds__(1024) bn_finalize_bwd_kernel(const float* __restrict__ partial, int B, int C,
                                                              float* __restrict__ dgamma, float* __restrict__ dbeta) {
  __shared__ double red[FIN_LANES][32][2];
  pdl_wait();
  pdl_launch_dependents();
  const int c = blockIdx.x * 32 + (threadIdx.x & 31), lane = threadIdx.x >> 5;
  double s, q;
  colpartials_sum(partial, B, C, c, lane, red, s, q);
  if (lane != 0 || c >= C) return;
  dbeta[c] = (float)s;
  dgamma[c] = (float)q;
}

// a = relu(z*scale + shift)   (train-mode BN + ReLU on the raw conv output, mobilenet.py:29-30,44-45)
__global__ void __launch_bounds__(256) bn_apply_relu_kernel(const bf16* __restrict__ z,
                                                            const float* __restrict__ scale,
                                                            const float* __restrict__ shift, bf16* __restrict__ a,
                                                            long long total_vec, int CV, int* nan_flag) {
  pdl_wait();
  pdl_launch_dependents();
  bool bad = false;
  // the grid stride is a multiple of CV for power-of-two channel counts: scale/shift are loaded once per thread
  const long long stride = (long long)gridDim.x * blockDim.x;
  const bool fixed = (stride % CV) == 0;
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  float sc[8], sh[8];
  auto load_consts = [&](long long idx) {
    const int c0 = (int)(idx % CV) << 3;
    load8(scale + c0, sc);
    load8(shift + c0, sh);
  };
  auto apply = [&](long long idx, const uint4& zu) {
    float zf[8], o[8];
    unpack8f(zu, zf);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      o[j] = relu_nan(__fadd_rn(__fmul_rn(zf[j], sc[j]), sh[j]));
      bad |= (o[j] != o[j]);
    }
    *reinterpret_cast<uint4*>(a + idx * 8) = pack8f(o);
  };
  if (i < total_vec) load_consts(i);
  if (fixed) {
    for (; i + 3 * stride < total_vec; i += 4 * stride) {
      uint4 zu[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) zu[k] = ld_nc16(z + (i + k * stride) * 8);
#pragma unroll
      for (int k = 0; k < 4; ++k) apply(i + k * stride, zu[k]);
    }
  }
  for (; i < total_vec; i += stride) {
    if (!fixed) load_consts(i);
    apply(i, ld_nc16(z + i * 8));
  }
  if (bad && nan_flag) atomicOr(nan_flag, SSD3D_NAN_BACKBONE);
}

// dz = scale * (dy - dbeta/M - xhat * dgamma/M),  dy = g * [z*scale+shift > 0]      (dz may alias g)
__global__ void __launch_bounds__(256) bn_relu_bwd_apply_kernel(const bf16* __restrict__ z, const bf16* g,
                                                                const float* __restrict__ scale,
                                                                const float* __restrict__ shift,
                                                                const float* __restrict__ mean,
                                                                const float* __restrict__ invstd,
                                                                const float* __restrict__ dgamma,
                                                                const float* __restrict__ dbeta, float inv_m,
                                                                bf16* dz, long long total_vec, int CV) {
  pdl_wait();
  pdl_launch_dependents();
  // the grid stride is a multiple of CV for every channel count of the network (powers of two): a thread keeps its
  // channels, so the per-channel constants are loaded once; two vectors in flight per iteration
  const long long stride = (long long)gridDim.x * blockDim.x;
  const bool fixed = (stride % CV) == 0;
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  // dz = sc*(dy - dbeta/M - xhat*dgamma/M) with xhat = (z - mu)*invstd, regrouped as sc*dy + A + z*B
  float sc[8], sh[8], ka[8], kb[8];
  auto load_consts = [&](long long idx) {
    const int c0 = (int)(idx % CV) << 3;
    float mu[8], is[8], dg[8], db[8];
    load8(scale + c0, sc); load8(shift + c0, sh); load8(mean + c0, mu); load8(invstd + c0, is);
    load8(dgamma + c0, dg); load8(dbeta + c0, db);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float t = sc[j] * is[j] * dg[j] * inv_m;
      kb[j] = -t;
      ka[j] = fmaf(mu[j], t, -(sc[j] * db[j] * inv_m));
    }
  };
  auto apply = [&](long long idx, const uint4& zu, const uint4& gu) {
    float zf[8], gf[8], o[8];
    unpack8f(zu, zf);
    unpack8f(gu, gf);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float pre = __fadd_rn(__fmul_rn(zf[j], sc[j]), sh[j]);
      const float dy = (pre > 0.f) ? gf[j] : 0.f;
      o[j] = fmaf(zf[j], kb[j], fmaf(sc[j], dy, ka[j]));
    }
    *reinterpret_cast<uint4*>(dz + idx * 8) = pack8f(o);
  };
  if (i < total_vec) load_consts(i);
  if (fixed) {
    for (; i + stride < total_vec; i += 2 * stride) {
      const uint4 z0 = ld_nc16(z + i * 8), z1 = ld_nc16(z + (i + stride) * 8);
      const uint4 g0 = *reinterpret_cast<const uint4*>(g + i * 8), g1 = *reinterpret_cast<const uint4*>(g + (i + stride) * 8);
      apply(i, z0, g0);
      apply(i + stride, z1, g1);
    }
  }
  for (; i < total_vec; i += stride) {
    if (!fixed) load_consts(i);
    apply(i, ld_nc16(z + i * 8), *reinterpret_cast<const uint4*>(g + i * 8));
  }
}

// ------------------------------------------------------------------------------------------------
// mma.sync helpers (bf16 x bf16 -> fp32, m16n8k16)
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void ldsm_x4(uint32_t addr, uint32_t (&r)[4]) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0, %1, %2, %3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}
__device__ __forceinline__ void ldsm_x4_t(uint32_t addr, uint32_t (&r)[4]) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0, %1, %2, %3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}
__device__ __forceinline__ void mma_bf16(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, "
      "{%0, %1, %2, %3};"
      : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

// ------------------------------------------------------------------------------------------------
// Weight gradient as a split-M implicit GEMM:  dW[n][k] = sum_m dz[m][n] * X[m][k]
//   MODE 0 pointwise : X[m][k] = x[m*C + k], zero for k >= C                        (K = Cin rounded up to 64)
//   MODE 2 stem 3^3  : k = ci*27 + tap, X = bf16(x_ncdhw[n][ci][sd*do+kd-1][2*ho+kh-1][2*wo+kw-1])
// CTA: 128 threads, output tile NT (n) x 64 (k), rows [split*rows_per_split, ...) in chunks of 64.
// Both operands sit in smem as [m][n] / [m][k] (M-major); A (= dz^T) and B fragments are ldmatrix.trans.
// ------------------------------------------------------------------------------------------------
struct WgradParams {
  const bf16* dz;
  int ldz;
  long long M;
  int K;                      // padded to a multiple of 64
  const void* x;
  int x_is_bf16;              // stem only
  int C;                      // pointwise: Cin (row pitch)
  int N, D, H, W;             // stem: input volume
  int Do, Ho, Wo, sd, Cin;    // stem
  long long rows_per_split;
  int n_pad;                  // rows of one partial slab (multiple of NT)
  float* partial;             // [splits][n_pad][K]
};

template <int NT, int MODE, int KT>
__global__ void __launch_bounds__(128) wgrad_kernel(const WgradParams p) {
  constexpr int ZP = NT + 8;          // padded row pitch (elements): conflict-free ldmatrix
  constexpr int XP = KT + 8;
  constexpr int ZCH = NT / 8;         // 16-byte chunks per dz row
  constexpr int ZPT = (64 * ZCH + 127) / 128;
  constexpr int XCH = KT / 8;         // 16-byte chunks per X row (8 or 4)
  constexpr int XPT = 64 * XCH / 128; // chunks per thread (4 or 2)
  constexpr int XRS = 128 / XCH;      // row step between a thread's chunks (16 or 32)
  constexpr int NB = KT / 32;         // n8 tiles per warp along k (2 or 1)
  __shared__ __align__(16) bf16 sZ[64 * ZP];
  __shared__ __align__(16) bf16 sX[64 * XP];
  pdl_wait();
  pdl_launch_dependents();
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int k0 = blockIdx.x * KT;
  const int n0 = blockIdx.y * NT;
  const long long m_begin = (long long)blockIdx.z * p.rows_per_split;
  const long long m_end = (m_begin + p.rows_per_split < p.M) ? m_begin + p.rows_per_split : p.M;

  // ---- per-thread constants of the X gather ----
  const int xcc = tid % XCH;          // 16-byte chunk (8 k values) inside the KT-wide k tile
  const int xrow0 = tid / XCH;        // rows xrow0 + XRS*i, i < XPT
  int e_off[8];                                          // MODE 2: per element (ci, tap) -> offset, or -1
  int e_kd[8], e_kh[8], e_kw[8];
  if (MODE == 2) {
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const int k = k0 + xcc * 8 + e;
      const int ci = k / 27, tap = k - ci * 27;
      e_off[e] = (ci < p.Cin) ? ci : -1;
      e_kd[e] = tap / 9 - 1; e_kh[e] = (tap / 3) % 3 - 1; e_kw[e] = tap % 3 - 1;
    }
  }

  uint4 zr[ZPT], xr[XPT];
  auto load_tiles = [&](long long m0) {
#pragma unroll
    for (int i = 0; i < ZPT; ++i) {
      const int q = tid + i * 128;
      const int row = q / ZCH, cc = q % ZCH;
      const long long m = m0 + row;
      zr[i] = make_uint4(0u, 0u, 0u, 0u);
      if (q < 64 * ZCH && m < m_end) zr[i] = ld_nc16(p.dz + m * p.ldz + n0 + cc * 8);
    }
#pragma unroll
    for (int i = 0; i < XPT; ++i) {
      const long long m = m0 + xrow0 + XRS * i;
      xr[i] = make_uint4(0u, 0u, 0u, 0u);
      if (m >= m_end) continue;
      if (MODE == 0) {
        if (k0 + xcc * 8 < p.C) xr[i] = ld_nc16(static_cast<const bf16*>(p.x) + m * p.C + k0 + xcc * 8);
      } else {
        long long t = m;
        const int wo = (int)(t % p.Wo); t /= p.Wo;
        const int ho = (int)(t % p.Ho); t /= p.Ho;
        const int dz_ = (int)(t % p.Do); t /= p.Do;
        const long long plane = (long long)p.D * p.H * p.W;
        float v[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          v[e] = 0.f;
          const int d = dz_ * p.sd + e_kd[e], h = ho * 2 + e_kh[e], w = wo * 2 + e_kw[e];
          if (e_off[e] >= 0 && (unsigned)d < (unsigned)p.D && (unsigned)h < (unsigned)p.H && (unsigned)w < (unsigned)p.W) {
            const long long idx = ((long long)t * p.Cin + e_off[e]) * plane + ((long long)d * p.H + h) * p.W + w;
            v[e] = p.x_is_bf16 ? __bfloat162float(static_cast<const bf16*>(p.x)[idx])
                               : __ldg(static_cast<const float*>(p.x) + idx);
          }
        }
        xr[i] = pack8f(v);
      }
    }
  };

  float acc[NT / 16][NB][4];
#pragma unroll
  for (int a = 0; a < NT / 16; ++a)
#pragma unroll
    for (int b = 0; b < NB; ++b)
#pragma unroll
      for (int c = 0; c < 4; ++c) acc[a][b][c] = 0.f;

  const uint32_t sZ_u = smem_u32(sZ), sX_u = smem_u32(sX);
  const int lq = lane >> 3, lr = lane & 7;
  if (m_begin < m_end) load_tiles(m_begin);
  for (long long m0 = m_begin; m0 < m_end; m0 += 64) {
    __syncthreads();                       // the previous chunk's fragments have been read
#pragma unroll
    for (int i = 0; i < ZPT; ++i) {
      const int q = tid + i * 128;
      if (q < 64 * ZCH) *reinterpret_cast<uint4*>(&sZ[(q / ZCH) * ZP + (q % ZCH) * 8]) = zr[i];
    }
#pragma unroll
    for (int i = 0; i < XPT; ++i) *reinterpret_cast<uint4*>(&sX[(xrow0 + XRS * i) * XP + xcc * 8]) = xr[i];
    __syncthreads();
    if (m0 + 64 < m_end) load_tiles(m0 + 64);   // global loads of the next chunk fly during the MMAs
#pragma unroll
    for (int ks = 0; ks < 4; ++ks) {
      const int kk = ks * 16;
      uint32_t bfr[4];
      // B (k16 x NB n8 tiles): matrices {rows kk..+7 | kk+8..+15} x {cols w*8*NB (| +8)}; with NB = 1 the
      // upper two matrices re-read the first tile (their registers are unused)
      ldsm_x4_t(sX_u + (uint32_t)(((kk + (lq & 1) * 8 + lr) * XP + warp * 8 * NB + (NB == 2 ? (lq >> 1) * 8 : 0)) * 2),
                bfr);
#pragma unroll
      for (int a = 0; a < NT / 16; ++a) {
        uint32_t afr[4];
        // A = dz^T (16 n x k16): matrices {n 0-7 | 8-15} x {rows kk..+7 | kk+8..+15}, transposed on load
        ldsm_x4_t(sZ_u + (uint32_t)(((kk + (lq >> 1) * 8 + lr) * ZP + a * 16 + (lq & 1) * 8) * 2), afr);
        mma_bf16(acc[a][0], afr, bfr[0], bfr[1]);
        if (NB == 2) mma_bf16(acc[a][NB - 1], afr, bfr[2], bfr[3]);
      }
    }
  }
  float* out = p.partial + ((size_t)blockIdx.z * p.n_pad + n0) * p.K + k0 + warp * 8 * NB;
#pragma unroll
  for (int a = 0; a < NT / 16; ++a)
#pragma unroll
    for (int b = 0; b < NB; ++b) {
      const int n = a * 16 + (lane >> 2), k = b * 8 + (lane & 3) * 2;
      *reinterpret_cast<float2*>(out + (size_t)n * p.K + k) = make_float2(acc[a][b][0], acc[a][b][1]);
      *reinterpret_cast<float2*>(out + (size_t)(n + 8) * p.K + k) = make_float2(acc[a][b][2], acc[a][b][3]);
    }
}

// ------------------------------------------------------------------------------------------------
// Head weight gradient, activation-stationary form.  dW[n][c][tap] = sum_v dO[v][n] * x[v + off(tap)][c] is the
// same sum over u = v + off(tap):  sum_u x[u][c] * dO[u - off(tap)][n].  So a 64-voxel chunk of x (64 channels)
// is loaded ONCE and contracted against G[u][j*16 + n] = dO[u - off(kd, j)][n], the 9 (kh, kw) shifts of the
// 16-column gradient rows (32 bytes each, zero outside the map, L1/L2 resident), instead of gathering the 27
// shifted activation tiles.  CTA = (64-channel tile, kd, voxel split); cp.async double buffering; warp w owns
// channels 16w..16w+15 x 144 columns (72 accumulator registers).  Slab layout [split][16][C][27], the layout of
// the conv weight rows, so that the final sum is a plain contiguous reduction.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src, bool valid) {
  const int sz = valid ? 16 : 0;
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(sz) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

struct HeadWgradParams {
  const bf16* dO;             // (M, 16)
  const bf16* x;              // (M, C) channels-last
  int N, D, H, W, C;
  long long M;
  int chunks_per_split;
  float* partial;             // [splits][16][C][27]
};

constexpr int HW_XP = 72;     // sX pitch (elements)
constexpr int HW_GP = 152;    // sG pitch

__global__ void __launch_bounds__(128, 3) head_wgrad_g_kernel(const HeadWgradParams p) {
  extern __shared__ __align__(16) uint8_t hw_smem[];
  bf16* sX = reinterpret_cast<bf16*>(hw_smem);                   // [2][64][HW_XP]
  bf16* sG = sX + 2 * 64 * HW_XP;                                // [2][64][HW_GP]
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int c0 = blockIdx.x * 64, kd = blockIdx.y;
  const long long chunk0 = (long long)blockIdx.z * p.chunks_per_split;
  const long long n_chunks_all = (p.M + 63) / 64;
  long long rem = n_chunks_all - chunk0;
  const int n_chunks = (int)(rem < p.chunks_per_split ? rem : p.chunks_per_split);
  const uint32_t sX_u = smem_u32(sX), sG_u = smem_u32(sG);
  const int row = tid >> 1, half = tid & 1;

  pdl_wait();
  pdl_launch_dependents();
  auto load_chunk = [&](int ci, int buf) {
    const long long u0 = (chunk0 + ci) * 64;
    // activations: 64 rows x 8 chunks of 16 bytes
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int q = tid + i * 128, r = q >> 3, cc = q & 7;
      const long long u = u0 + r;
      const bool ok = u < p.M;
      cp_async16(sX_u + (uint32_t)(((buf * 64 + r) * HW_XP + cc * 8) * 2), p.x + (ok ? u : 0) * p.C + c0 + cc * 8, ok);
    }
    // shifted gradient rows: this thread's voxel, taps half, half+2, ...
    const long long u = u0 + row;
    const bool in = u < p.M;
    long long t = in ? u : 0;
    const int w = (int)(t % p.W); t /= p.W;
    const int h = (int)(t % p.H); t /= p.H;
    const int d = (int)(t % p.D);
    const int dd = d - (kd - 1);
    const bool okd = in && dd >= 0 && dd < p.D;
#pragma unroll
    for (int jj = 0; jj < 5; ++jj) {
      const int j = half + 2 * jj;
      if (j < 9) {
        const int kh = j / 3, kw = j % 3;
        const int hh = h - (kh - 1), ww = w - (kw - 1);
        const bool ok = okd && hh >= 0 && hh < p.H && ww >= 0 && ww < p.W;
        const long long v = ok ? u - ((long long)((kd - 1) * p.H + (kh - 1)) * p.W + (kw - 1)) : 0;
        const uint32_t dst = sG_u + (uint32_t)(((buf * 64 + row) * HW_GP + j * 16) * 2);
        cp_async16(dst, p.dO + v * 16, ok);
        cp_async16(dst + 16, p.dO + v * 16 + 8, ok);
      }
    }
  };

  float acc[18][4];
#pragma unroll
  for (int b = 0; b < 18; ++b)
#pragma unroll
    for (int c = 0; c < 4; ++c) acc[b][c] = 0.f;
  const int lq = lane >> 3, lr = lane & 7;

  if (n_chunks > 0) load_chunk(0, 0);
  cp_async_commit();
  for (int ci = 0; ci < n_chunks; ++ci) {
    const int buf = ci & 1;
    if (ci + 1 < n_chunks) load_chunk(ci + 1, buf ^ 1);
    cp_async_commit();
    cp_async_wait<1>();
    __syncthreads();
#pragma unroll
    for (int ks = 0; ks < 4; ++ks) {
      const int kk = ks * 16;
      uint32_t afr[4];        // A = x^T (16 channels x 16 voxels), transposed on load
      ldsm_x4_t(sX_u + (uint32_t)(((buf * 64 + kk + (lq >> 1) * 8 + lr) * HW_XP + warp * 16 + (lq & 1) * 8) * 2), afr);
#pragma unroll
      for (int j = 0; j < 9; ++j) {
        uint32_t bfr[4];      // B = G (16 voxels x 16 columns of tap j)
        ldsm_x4_t(sG_u + (uint32_t)(((buf * 64 + kk + (lq & 1) * 8 + lr) * HW_GP + j * 16 + (lq >> 1) * 8) * 2), bfr);
        mma_bf16(acc[2 * j], afr, bfr[0], bfr[1]);
        mma_bf16(acc[2 * j + 1], afr, bfr[2], bfr[3]);
      }
    }
    __syncthreads();
  }
  // acc[2j + hi][..]: row = channel c0 + 16*warp + lane/4 (+8), column n = hi*8 + (lane&3)*2 (+1) of tap kd*9 + j
  float* out = p.partial + (size_t)blockIdx.z * 16 * p.C * 27;
#pragma unroll
  for (int j = 0; j < 9; ++j)
#pragma unroll
    for (int hi = 0; hi < 2; ++hi) {
      const int c = c0 + warp * 16 + (lane >> 2), n = hi * 8 + (lane & 3) * 2, tap = kd * 9 + j;
      out[((size_t)n * p.C + c) * 27 + tap] = acc[2 * j + hi][0];
      out[((size_t)(n + 1) * p.C + c) * 27 + tap] = acc[2 * j + hi][1];
      out[((size_t)n * p.C + c + 8) * 27 + tap] = acc[2 * j + hi][2];
      out[((size_t)(n + 1) * p.C + c + 8) * 27 + tap] = acc[2 * j + hi][3];
    }
}

static int head_wgrad_splits(long long M, int C) {
  const long long chunks = (M + 63) / 64;
  const int tiles = (C / 64) * 3;
  long long s = (444 + tiles - 1) / tiles;
  if (s > chunks) s = chunks;
  if (s < 1) s = 1;
  return (int)s;
}

// out[r*dst_ld + c] = sum over splits of partial[s][r*src_ld + c],  c < cols.  1024/LANES outputs x LANES split
// lanes per CTA; lane l adds splits l, l+LANES, ... in order and the lane sums are combined in order: fixed for a
// given S.  LANES follows S (few slabs: one thread per output; many: 32 lanes) so that the pass stays a plain
// coalesced read of the slabs instead of a latency-bound serial loop or a mostly idle CTA.
template <int LANES>
__global__ void __launch_bounds__(1024) sum_partials_kernel(const float* __restrict__ partial, int S,
                                                           long long slab, int rows, int cols, int src_ld,
                                                           int dst_ld, int dst_cs, float* __restrict__ out) {
  constexpr int OUTS = 1024 / LANES;
  __shared__ float red[LANES > 1 ? LANES : 1][LANES > 1 ? OUTS : 1];
  pdl_wait();
  pdl_launch_dependents();
  const int ox = threadIdx.x % OUTS, lane = threadIdx.x / OUTS;
  const long long i = (long long)blockIdx.x * OUTS + ox;
  const bool valid = i < (long long)rows * cols;
  const int r = valid ? (int)(i / cols) : 0, c = valid ? (int)(i % cols) : 0;
  float s = 0.f;
  if (valid) {
#pragma unroll 4
    for (int k = lane; k < S; k += LANES) s += partial[(size_t)k * slab + (size_t)r * src_ld + c];
  }
  if constexpr (LANES == 1) {
    if (valid) out[(size_t)r * dst_ld + (size_t)c * dst_cs] = s;
  } else {
    red[lane][ox] = s;
    __syncthreads();
    if (lane == 0 && valid) {
      float t = red[0][ox];
#pragma unroll
      for (int l = 1; l < LANES; ++l) t += red[l][ox];
      out[(size_t)r * dst_ld + (size_t)c * dst_cs] = t;
    }
  }
}

// dst_cs: stride between the columns of the OUTPUT (1 = plain rows; the depthwise slabs are tap-major [27][C] and land
// as out[c*27 + tap]: rows = taps with dst_ld = 1, columns = channels with dst_cs = 27)
static int launch_sum_partials(const float* partial, int S, long long slab, int rows, int cols, int src_ld, int dst_ld,
                               float* out, cudaStream_t st, int dst_cs = 1) {
  const long long total = (long long)rows * cols;
  if (S <= 3) {
    SSD3D_LAUNCH_PDL(sum_partials_kernel<1>, dim3((unsigned)((total + 1023) / 1024)), dim3(1024), 0, st, partial, S, slab,
                     rows, cols, src_ld, dst_ld, dst_cs, out);
  } else if (S <= 24) {
    SSD3D_LAUNCH_PDL(sum_partials_kernel<4>, dim3((unsigned)((total + 255) / 256)), dim3(1024), 0, st, partial, S, slab,
                     rows, cols, src_ld, dst_ld, dst_cs, out);
  } else {
    SSD3D_LAUNCH_PDL(sum_partials_kernel<32>, dim3((unsigned)((total + 31) / 32)), dim3(1024), 0, st, partial, S, slab,
                     rows, cols, src_ld, dst_ld, dst_cs, out);
  }
  return SSD3D_OK;
}

// ------------------------------------------------------------------------------------------------
// Head gradient rows: dO[m][b*6+j] = dlocs[n][off + v*bpl + b][j], dO[m][bpl*6 + b*ncls + k] = dscores[...][k]
// (the column order of the fused head GEMM, gemm_tc.cu), zero padded to 16 columns; bias gradients are
// the column sums (second stage: sum_partials).
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) head_grad_pack_kernel(const float* __restrict__ dlocs,
                                                             const float* __restrict__ dscores, long long P,
                                                             long long prior_off, long long V, int N, int bpl,
                                                             int n_classes, int groups, bf16* __restrict__ dO,
                                                             float* __restrict__ bias_partial) {
  __shared__ float red[256][16];
  pdl_wait();
  pdl_launch_dependents();
  const long long M = (long long)N * V;
  const long long m = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int nl = bpl * 6, nc = bpl * n_classes;
  const float* lp = nullptr;
  const float* sp = nullptr;
  if (m < M) {
    const long long n = m / V, vox = m - n * V;
    lp = dlocs + (n * P + prior_off + vox * bpl) * 6;
    sp = dscores + (n * P + prior_off + vox * bpl) * n_classes;
  }
  // column group g holds columns 16g .. 16g+15 of [loc (bpl*6) | class (bpl*n_classes) | zero pad]; dO is
  // (groups, M, 16): every group is a contiguous 16-column matrix for the 16-column contraction kernels
  for (int g = 0; g < groups; ++g) {
    float v[16];
#pragma unroll
    for (int j = 0; j < 16; ++j) {
      const int col = g * 16 + j;
      v[j] = 0.f;
      if (m < M) {
        if (col < nl) v[j] = lp[col];
        else if (col < nl + nc) v[j] = sp[col - nl];
      }
    }
    if (m < M) {
      float lo[8], hi[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) { lo[j] = v[j]; hi[j] = v[8 + j]; }
      uint4* dst = reinterpret_cast<uint4*>(dO + ((long long)g * M + m) * 16);
      dst[0] = pack8f(lo);
      dst[1] = pack8f(hi);
    }
    // block-level column sums of the fp32 values (bias gradient), fixed order
    if (g) __syncthreads();
#pragma unroll
    for (int j = 0; j < 16; ++j) red[threadIdx.x][j] = v[j];
    __syncthreads();
    if (threadIdx.x < 16) {
      float s = 0.f;
      for (int t = 0; t < 256; ++t) s += red[t][threadIdx.x];
      bias_partial[(size_t)blockIdx.x * (groups * 16) + g * 16 + threadIdx.x] = s;
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Head data gradient: dx[m][c] = sum_tap sum_n dO[voxel(m) - (tap offsets - 1)][n] * w[n][tap*C + c]  (+ addend)
// implicit GEMM, M x C output, K = 27 taps x 16; CTA = 64 rows x 64 channels, 4 warps (16 rows each).
// ------------------------------------------------------------------------------------------------
struct HeadDgradParams {
  const bf16* dO;        // (groups, M, 16)
  const bf16* w;         // (16*groups, 27*C)
  const bf16* addend;    // (M, C) or null
  bf16* dx;              // (M, C)
  int N, D, H, W, C;
  long long M;
  int groups;            // 16 gradient columns each, accumulated in fp32 inside the kernel
};

__global__ void __launch_bounds__(128) head_dgrad_kernel(const HeadDgradParams p) {
  constexpr int BP = 72, AP = 24;
  extern __shared__ __align__(16) uint8_t hd_smem[];
  bf16* sB = reinterpret_cast<bf16*>(hd_smem);                 // [27*16][BP]
  bf16* sA = sB + 27 * 16 * BP;                                // [2][64][AP]
  pdl_wait();
  pdl_launch_dependents();
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const long long m0 = (long long)blockIdx.x * 64;
  const int c0 = blockIdx.y * 64;
  // gather role: row = tid/2, half = tid%2
  const int arow = tid >> 1, ahalf = tid & 1;
  const long long am = m0 + arow;
  int aw = 0, ah = 0, ad = 0;
  long long an = 0;
  if (am < p.M) {
    long long t = am;
    aw = (int)(t % p.W); t /= p.W;
    ah = (int)(t % p.H); t /= p.H;
    ad = (int)(t % p.D); t /= p.D;
    an = t;
  }
  float acc[8][4];
#pragma unroll
  for (int a = 0; a < 8; ++a)
#pragma unroll
    for (int c = 0; c < 4; ++c) acc[a][c] = 0.f;
  const uint32_t sA_u = smem_u32(sA), sB_u = smem_u32(sB);
  const int lq = lane >> 3, lr = lane & 7;
  for (int g = 0; g < p.groups; ++g) {
    const bf16* wg = p.w + (size_t)g * 16 * 27 * p.C;
    const bf16* dOg = p.dO + (size_t)g * p.M * 16;
    if (g) __syncthreads();                        // every warp is done with the previous group's weights / rows
    for (int q = tid; q < 27 * 16 * 8; q += 128) {
      const int row = q >> 3, cc = q & 7;          // row = tap*16 + n
      const int tap = row >> 4, n = row & 15;
      *reinterpret_cast<uint4*>(&sB[row * BP + cc * 8]) =
          ld_nc16(wg + (size_t)n * 27 * p.C + (size_t)tap * p.C + c0 + cc * 8);
    }
    for (int tap = 0; tap < 27; ++tap) {
      const int buf = tap & 1;
      uint4 v = make_uint4(0u, 0u, 0u, 0u);
      {
        const int d = ad - (tap / 9 - 1), h = ah - ((tap / 3) % 3 - 1), w = aw - (tap % 3 - 1);
        if (am < p.M && (unsigned)d < (unsigned)p.D && (unsigned)h < (unsigned)p.H && (unsigned)w < (unsigned)p.W)
          v = ld_nc16(dOg + ((((long long)an * p.D + d) * p.H + h) * p.W + w) * 16 + ahalf * 8);
      }
      *reinterpret_cast<uint4*>(&sA[(buf * 64 + arow) * AP + ahalf * 8]) = v;
      __syncthreads();
      uint32_t afr[4];
      // A (16 rows x k16): matrices {rows 0-7 | 8-15} x {cols 0-7 | 8-15}
      ldsm_x4(sA_u + (uint32_t)(((buf * 64 + warp * 16 + (lq & 1) * 8 + lr) * AP + (lq >> 1) * 8) * 2), afr);
#pragma unroll
      for (int jj = 0; jj < 4; ++jj) {
        uint32_t bfr[4];
        ldsm_x4_t(sB_u + (uint32_t)(((tap * 16 + (lq & 1) * 8 + lr) * BP + jj * 16 + (lq >> 1) * 8) * 2), bfr);
        mma_bf16(acc[jj * 2], afr, bfr[0], bfr[1]);
        mma_bf16(acc[jj * 2 + 1], afr, bfr[2], bfr[3]);
      }
    }
  }
#pragma unroll
  for (int half = 0; half < 2; ++half) {
    const long long m = m0 + warp * 16 + (lane >> 2) + half * 8;
    if (m >= p.M) continue;
#pragma unroll
    for (int a = 0; a < 8; ++a) {
      const int c = c0 + a * 8 + (lane & 3) * 2;
      float v0 = acc[a][half * 2], v1 = acc[a][half * 2 + 1];
      if (p.addend) {
        const uint32_t u = *reinterpret_cast<const uint32_t*>(p.addend + m * p.C + c);
        v0 += bf16_lo(u);
        v1 += bf16_hi(u);
      }
      *reinterpret_cast<uint32_t*>(p.dx + m * p.C + c) = pack_bf16x2(v0, v1);
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Depthwise 3x3x3 backward.  forward: y[o][c] = sum_k x[S*o + k - 1][c] * w[k][c]
// ------------------------------------------------------------------------------------------------
// data: dx[i][c] = sum_{k : (i + 1 - k) % S == 0} dz[(i + 1 - k)/S][c] * w[k][c];  thread = 8 channels x 1 voxel
template <int S>
__global__ void __launch_bounds__(256) dw_dgrad_kernel(const bf16* __restrict__ dz, const bf16* __restrict__ w,
                                                       bf16* __restrict__ dx, int N, int C, int D, int H, int W,
                                                       int Do, int Ho, int Wo, long long total) {
  pdl_wait();
  pdl_launch_dependents();
  const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (gid >= total) return;
  const int CV = C >> 3;
  const int cv = (int)(gid % CV);
  long long r = gid / CV;
  const int wi = (int)(r % W); r /= W;
  const int hi = (int)(r % H); r /= H;
  const int di = (int)(r % D);
  const int n = (int)(r / D);
  const int c0 = cv << 3;
  float acc[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) acc[j] = 0.f;
  // only taps with (i + 1 - k) divisible by S reach an output: for S = 2 that is k = parity, parity + 2
  // (1 or 2 taps per axis, 3.4 of 27 on average) -- walk exactly those
  if constexpr (S == 1) {
    // stride 1: every tap contributes.  One (kd) plane at a time: its nine gradient rows and nine weight vectors are
    // requested together (zero outside the map) -- with the loads inside the bounds branches the kernel paid one
    // L2 round trip per tap, 27 in a row (28 us for the 7 MB map of the C3 step's third block)
#pragma unroll 1
    for (int kd = 0; kd < 3; ++kd) {
      const int od = di + 1 - kd;
      if ((unsigned)od >= (unsigned)Do) continue;
      const bf16* zrow = dz + ((long long)n * Do + od) * Ho * (long long)Wo * C + c0;
      uint4 gu[9], wu[9];
#pragma unroll
      for (int t = 0; t < 9; ++t) {
        const int oh = hi + 1 - t / 3, ow = wi + 1 - t % 3;
        gu[t] = make_uint4(0u, 0u, 0u, 0u);
        if ((unsigned)oh < (unsigned)Ho && (unsigned)ow < (unsigned)Wo) gu[t] = ld_nc16(zrow + ((long long)oh * Wo + ow) * C);
        wu[t] = ld_nc16(w + (kd * 9 + t) * C + c0);
      }
#pragma unroll
      for (int t = 0; t < 9; ++t) {
        float gf[8], wf[8];
        unpack8f(gu[t], gf);
        unpack8f(wu[t], wf);
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[j] = fmaf(gf[j], wf[j], acc[j]);
      }
    }
    *reinterpret_cast<uint4*>(dx + gid * 8) = pack8f(acc);
    return;
  }
  const int pd = (S == 2) ? ((di + 1) & 1) : 0, ph = (S == 2) ? ((hi + 1) & 1) : 0, pw = (S == 2) ? ((wi + 1) & 1) : 0;
  for (int kd = pd; kd < 3; kd += S) {
    const int td = di + 1 - kd;
    if (td < 0) continue;
    const int od = td / S;
    if (od >= Do) continue;
    for (int kh = ph; kh < 3; kh += S) {
      const int th = hi + 1 - kh;
      if (th < 0) continue;
      const int oh = th / S;
      if (oh >= Ho) continue;
      for (int kw = pw; kw < 3; kw += S) {
        const int tw = wi + 1 - kw;
        if (tw < 0) continue;
        const int ow = tw / S;
        if (ow >= Wo) continue;
        float gf[8], wf[8];
        unpack8f(ld_nc16(dz + ((((long long)n * Do + od) * Ho + oh) * Wo + ow) * C + c0), gf);
        unpack8f(ld_nc16(w + ((kd * 3 + kh) * 3 + kw) * C + c0), wf);
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[j] = fmaf(gf[j], wf[j], acc[j]);
      }
    }
  }
  *reinterpret_cast<uint4*>(dx + gid * 8) = pack8f(acc);
}

// Stride-2 data gradient by PARITY CLASS.  An input voxel i receives tap k only when (i + 1 - k) is even: an even
// i gets k = 1 (from output i/2), an odd i = 2a+1 gets k = 0 (from a+1) and k = 2 (from a).  Voxels of one
// (d,h,w)-parity class therefore share a fixed tap set of 1..8 taps: blockIdx.y selects the class, the tap loops
// unroll at compile time, the class's weights sit in registers as fp32 pairs, and a thread produces 4 channels of
// four class-neighbours along W with packed FFMA2 -- 16 instead of 37 instructions per gradient element.
typedef unsigned long long f32x2_t;
__device__ __forceinline__ f32x2_t tr_bf16x2_to_f32x2(uint32_t u) {
  f32x2_t r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "r"(u << 16), "r"(u & 0xffff0000u));
  return r;
}
__device__ __forceinline__ void tr_ffma2(f32x2_t& acc, f32x2_t a, f32x2_t b) {
  asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(acc) : "l"(a), "l"(b));
}
__device__ __forceinline__ uint32_t tr_pack_bf16x2(f32x2_t v) {
  uint32_t a, b;
  asm("mov.b64 {%0, %1}, %2;" : "=r"(a), "=r"(b) : "l"(v));
  return pack_bf16x2(__uint_as_float(a), __uint_as_float(b));
}

template <int PD, int PH, int PW>
__device__ __forceinline__ void dw_dgrad_s2_class(const bf16* __restrict__ dz, const bf16* __restrict__ w,
                                                  bf16* __restrict__ dx, int N, int C, int D, int H, int W, int Do,
                                                  int Ho, int Wo) {
  constexpr int WT = 4;
  constexpr int ND = PD ? 1 : 2, NH = PH ? 1 : 2, NW = PW ? 1 : 2;     // taps per axis
  // class extents: parity 1 <-> even coordinate 2a, parity 0 <-> odd coordinate 2a + 1
  const int Ad = PD ? (D + 1) / 2 : D / 2, Ah = PH ? (H + 1) / 2 : H / 2, Aw = PW ? (W + 1) / 2 : W / 2;
  const int CV = C >> 2;
  const int WG = (Aw + WT - 1) / WT;
  const long long total = (long long)N * Ad * Ah * WG * CV;
  const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (gid >= total) return;
  const int cv = (int)(gid % CV);
  long long r = gid / CV;
  const int wg = (int)(r % WG); r /= WG;
  const int ah = (int)(r % Ah); r /= Ah;
  const int ad = (int)(r % Ad);
  const int n = (int)(r / Ad);
  const int c0 = cv << 2;
  // weights of this class: tap index along an axis is (parity ? 1 : 2*j), j < taps
  f32x2_t wr[ND * NH * NW][2];
#pragma unroll
  for (int a = 0; a < ND; ++a)
#pragma unroll
    for (int b = 0; b < NH; ++b)
#pragma unroll
      for (int c = 0; c < NW; ++c) {
        const int kd = PD ? 1 : 2 * a, kh = PH ? 1 : 2 * b, kw = PW ? 1 : 2 * c;
        const uint2 u = __ldg(reinterpret_cast<const uint2*>(w + ((kd * 3 + kh) * 3 + kw) * C + c0));
        wr[(a * NH + b) * NW + c][0] = tr_bf16x2_to_f32x2(u.x);
        wr[(a * NH + b) * NW + c][1] = tr_bf16x2_to_f32x2(u.y);
      }
  f32x2_t acc[WT][2];
#pragma unroll
  for (int i = 0; i < WT; ++i) { acc[i][0] = 0ull; acc[i][1] = 0ull; }
#pragma unroll
  for (int a = 0; a < ND; ++a) {
    const int od = PD ? ad : (a == 0 ? ad + 1 : ad);        // k = 0 -> output a+1, k = 2 (or 1) -> output a
    if (od >= Do) continue;
#pragma unroll
    for (int b = 0; b < NH; ++b) {
      const int oh = PH ? ah : (b == 0 ? ah + 1 : ah);
      if (oh >= Ho) continue;
      const bf16* grow = dz + ((((long long)n * Do + od) * Ho + oh) * Wo) * C + c0;
#pragma unroll
      for (int c = 0; c < NW; ++c) {
#pragma unroll
        for (int i = 0; i < WT; ++i) {
          const int aw = wg * WT + i;
          const int ow = PW ? aw : (c == 0 ? aw + 1 : aw);
          if (aw >= Aw || ow >= Wo) continue;
          const uint2 u = __ldg(reinterpret_cast<const uint2*>(grow + (long long)ow * C));
          tr_ffma2(acc[i][0], tr_bf16x2_to_f32x2(u.x), wr[(a * NH + b) * NW + c][0]);
          tr_ffma2(acc[i][1], tr_bf16x2_to_f32x2(u.y), wr[(a * NH + b) * NW + c][1]);
        }
      }
    }
  }
  const int di = PD ? 2 * ad : 2 * ad + 1, hi = PH ? 2 * ah : 2 * ah + 1;
  bf16* xrow = dx + ((((long long)n * D + di) * H + hi) * W) * C + c0;
#pragma unroll
  for (int i = 0; i < WT; ++i) {
    const int aw = wg * WT + i;
    if (aw >= Aw) break;
    const int wi = PW ? 2 * aw : 2 * aw + 1;
    *reinterpret_cast<uint2*>(xrow + (long long)wi * C) = make_uint2(tr_pack_bf16x2(acc[i][0]), tr_pack_bf16x2(acc[i][1]));
  }
}

__global__ void __launch_bounds__(256) dw_dgrad_s2_kernel(const bf16* __restrict__ dz, const bf16* __restrict__ w,
                                                          bf16* __restrict__ dx, int N, int C, int D, int H, int W,
                                                          int Do, int Ho, int Wo) {
  pdl_wait();
  pdl_launch_dependents();
  switch (blockIdx.y) {
    case 0: dw_dgrad_s2_class<0, 0, 0>(dz, w, dx, N, C, D, H, W, Do, Ho, Wo); break;
    case 1: dw_dgrad_s2_class<0, 0, 1>(dz, w, dx, N, C, D, H, W, Do, Ho, Wo); break;
    case 2: dw_dgrad_s2_class<0, 1, 0>(dz, w, dx, N, C, D, H, W, Do, Ho, Wo); break;
    case 3: dw_dgrad_s2_class<0, 1, 1>(dz, w, dx, N, C, D, H, W, Do, Ho, Wo); break;
    case 4: dw_dgrad_s2_class<1, 0, 0>(dz, w, dx, N, C, D, H, W, Do, Ho, Wo); break;
    case 5: dw_dgrad_s2_class<1, 0, 1>(dz, w, dx, N, C, D, H, W, Do, Ho, Wo); break;
    case 6: dw_dgrad_s2_class<1, 1, 0>(dz, w, dx, N, C, D, H, W, Do, Ho, Wo); break;
    default: dw_dgrad_s2_class<1, 1, 1>(dz, w, dx, N, C, D, H, W, Do, Ho, Wo); break;
  }
}

// Stride-2 data gradient by OUTPUT BLOCK (maps with C <= 256).  A thread produces 8 channels of the 2x2x2 block of
// dx voxels (2m + p), p in {0,1}^3, from the 2x2x2 block of gradient voxels (m + a): per axis p = 0 takes tap 1
// from a = 0, p = 1 takes tap 2 from a = 0 and tap 0 from a = 1 -- all 27 taps once, 8 gradient loads of 16 bytes
// and 8 stores of 16 bytes per 64 gradient elements, and a warp writes whole 128-byte lines (both W parities back
// to back) where the per-class kernel wrote every line in two far-apart halves.  Weights sit in shared memory as
// fp32 (two LDS.128 per tap), the products are packed FFMA2.
__global__ void __launch_bounds__(256, 2) dw_dgrad_s2_block_kernel(const bf16* __restrict__ dz, const bf16* __restrict__ w,
                                                                bf16* __restrict__ dx, int N, int C, int D, int H, int W,
                                                                int Do, int Ho, int Wo, int Md, int Mh, int Mw,
                                                                long long total) {
  extern __shared__ __align__(16) float dg_sw[];       // [27][C]
  pdl_wait();
  pdl_launch_dependents();
  for (int i = threadIdx.x; i < 27 * C; i += 256) dg_sw[i] = __bfloat162float(w[i]);
  __syncthreads();
  const long long gid = (long long)blockIdx.x * 256 + threadIdx.x;
  if (gid >= total) return;
  const int CV = C >> 3;
  const int cv = (int)(gid % CV);
  long long r = gid / CV;
  const int mw = (int)(r % Mw); r /= Mw;
  const int mh = (int)(r % Mh); r /= Mh;
  const int md = (int)(r % Md);
  const int n = (int)(r / Md);
  const int c0 = cv << 3;
  f32x2_t acc[8][4];
#pragma unroll
  for (int p = 0; p < 8; ++p)
#pragma unroll
    for (int q = 0; q < 4; ++q) acc[p][q] = 0ull;
  // all eight gradient vectors of the 2x2x2 block are requested before the first use (zero outside the map: a zero
  // gradient adds nothing) -- inside the bounds branches they were eight L2 round trips in a row
  uint4 gu8[8];
#pragma unroll
  for (int t = 0; t < 8; ++t) {
    const int od = md + (t >> 2), oh = mh + ((t >> 1) & 1), ow = mw + (t & 1);
    gu8[t] = make_uint4(0u, 0u, 0u, 0u);
    if (od < Do && oh < Ho && ow < Wo) gu8[t] = ld_nc16(dz + ((((long long)n * Do + od) * Ho + oh) * Wo + ow) * C + c0);
  }
#pragma unroll
  for (int a = 0; a < 2; ++a) {
#pragma unroll
    for (int b = 0; b < 2; ++b) {
#pragma unroll
      for (int c = 0; c < 2; ++c) {
        const uint4 u = gu8[(a * 2 + b) * 2 + c];
        const f32x2_t g[4] = {tr_bf16x2_to_f32x2(u.x), tr_bf16x2_to_f32x2(u.y), tr_bf16x2_to_f32x2(u.z),
                              tr_bf16x2_to_f32x2(u.w)};
#pragma unroll
        for (int pd = a; pd < 2; ++pd) {               // a = 1 only feeds odd coordinates
          const int kd = pd == 0 ? 1 : (a == 0 ? 2 : 0);
#pragma unroll
          for (int ph = b; ph < 2; ++ph) {
            const int kh = ph == 0 ? 1 : (b == 0 ? 2 : 0);
#pragma unroll
            for (int pw = c; pw < 2; ++pw) {
              const int kw = pw == 0 ? 1 : (c == 0 ? 2 : 0);
              const ulonglong2* wp = reinterpret_cast<const ulonglong2*>(dg_sw + ((kd * 3 + kh) * 3 + kw) * C + c0);
              const ulonglong2 w01 = wp[0], w23 = wp[1];
              f32x2_t(&o)[4] = acc[(pd * 2 + ph) * 2 + pw];
              tr_ffma2(o[0], g[0], w01.x);
              tr_ffma2(o[1], g[1], w01.y);
              tr_ffma2(o[2], g[2], w23.x);
              tr_ffma2(o[3], g[3], w23.y);
            }
          }
        }
      }
    }
  }
#pragma unroll
  for (int pd = 0; pd < 2; ++pd) {
    const int di = 2 * md + pd;
    if (di >= D) continue;
#pragma unroll
    for (int ph = 0; ph < 2; ++ph) {
      const int hi = 2 * mh + ph;
      if (hi >= H) continue;
#pragma unroll
      for (int pw = 0; pw < 2; ++pw) {
        const int wi = 2 * mw + pw;
        if (wi >= W) continue;
        const f32x2_t(&o)[4] = acc[(pd * 2 + ph) * 2 + pw];
        *reinterpret_cast<uint4*>(dx + ((((long long)n * D + di) * H + hi) * W + wi) * C + c0) =
            make_uint4(tr_pack_bf16x2(o[0]), tr_pack_bf16x2(o[1]), tr_pack_bf16x2(o[2]), tr_pack_bf16x2(o[3]));
      }
    }
  }
}

// weight: dw[c][k] = sum_o dz[o][c] * x[S*o + k - 1][c].  thread = (8 channels, kd, voxel lane g): 9 taps x 8
// channels of accumulators; block partial [27][C] (tap-major) after a fixed-order reduction over the voxel lanes.
template <int S>
__global__ void __launch_bounds__(256) dw_wgrad_kernel(const bf16* __restrict__ dz, const bf16* __restrict__ x,
                                                       int N, int C, int D, int H, int W, int Do, int Ho, int Wo,
                                                       long long Mo, long long vox_per_block, int G,
                                                       float* __restrict__ partial) {
  __shared__ float red[256 * 8];
  pdl_wait();
  pdl_launch_dependents();
  const int CV = C >> 3;
  const int cv = threadIdx.x % CV;
  const int kd = (threadIdx.x / CV) % 3;
  const int g = threadIdx.x / (CV * 3);
  const int c0 = cv << 3;
  float acc[9][8];
#pragma unroll
  for (int t = 0; t < 9; ++t)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[t][j] = 0.f;
  const long long o_begin = (long long)blockIdx.x * vox_per_block;
  const long long o_end = (o_begin + vox_per_block < Mo) ? o_begin + vox_per_block : Mo;
  // the ten loads of a voxel (gradient row + nine taps, zero outside the map) are issued together: with the loads
  // inside the bounds branches the loop ran one L2 latency per tap (22-35 us on the 3^3 / 6^3 maps of the C3 step)
  for (long long o = o_begin + g; o < o_end; o += G) {
    unsigned t = (unsigned)o;                 // Mo < 2^31 (checked by the launcher)
    const int ow = (int)(t % (unsigned)Wo); t /= (unsigned)Wo;
    const int oh = (int)(t % (unsigned)Ho); t /= (unsigned)Ho;
    const int od = (int)(t % (unsigned)Do); t /= (unsigned)Do;
    const int di = od * S + kd - 1;
    if ((unsigned)di >= (unsigned)D) continue;
    const uint4 gu = ld_nc16(dz + o * C + c0);
    const bf16* xrow = x + ((long long)t * D + di) * H * (long long)W * C + c0;
    uint4 xu[9];
#pragma unroll
    for (int kh = 0; kh < 3; ++kh) {
      const int hi = oh * S + kh - 1;
#pragma unroll
      for (int kw = 0; kw < 3; ++kw) {
        const int wi = ow * S + kw - 1;
        xu[kh * 3 + kw] = make_uint4(0u, 0u, 0u, 0u);
        if ((unsigned)hi < (unsigned)H && (unsigned)wi < (unsigned)W)
          xu[kh * 3 + kw] = ld_nc16(xrow + ((long long)hi * W + wi) * C);
      }
    }
    float gf[8];
    unpack8f(gu, gf);
#pragma unroll
    for (int k = 0; k < 9; ++k) {
      float xf[8];
      unpack8f(xu[k], xf);
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[k][j] = fmaf(gf[j], xf[j], acc[k][j]);
    }
  }
  float* dst = partial + (size_t)blockIdx.x * C * 27;
#pragma unroll
  for (int t = 0; t < 9; ++t) {
    if (G > 1) {
      __syncthreads();
#pragma unroll
      for (int j = 0; j < 8; ++j) red[threadIdx.x * 8 + j] = acc[t][j];
      __syncthreads();
      if (g == 0) {
        for (int gg = 1; gg < G; ++gg) {
          const float* src = red + (size_t)(gg * CV * 3 + kd * CV + cv) * 8;
#pragma unroll
          for (int j = 0; j < 8; ++j) acc[t][j] += src[j];
        }
      }
    }
    if (g == 0) {
      // tap-major slab [27][C]: the thread's 8 channels are one 32-byte run (the [C][27] layout scattered 72 single
      // floats per thread, 27 floats apart -- the slab writes, not the loads, were most of this kernel's time)
      float* d8 = dst + (size_t)(kd * 9 + t) * C + c0;
      *reinterpret_cast<float4*>(d8) = make_float4(acc[t][0], acc[t][1], acc[t][2], acc[t][3]);
      *reinterpret_cast<float4*>(d8 + 4) = make_float4(acc[t][4], acc[t][5], acc[t][6], acc[t][7]);
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Adam (torch.optim.Adam semantics: L2 weight decay folded into the gradient, bias-corrected moments)
// over flat buffers; elements >= bias_start use lr_bias (the reference's "biases at twice the lr" group).
// ------------------------------------------------------------------------------------------------
// status[0] |= 1 when any gradient element is NaN / Inf (a batch without a single positive prior makes the
// MultiBox loss 0/0, ssd3d.py:938-940: the reference raises; a fused step cannot raise without a host sync, so it
// must at least not poison the parameters)
__global__ void __launch_bounds__(256) grad_nonfinite_kernel(const float* __restrict__ g, long long n,
                                                             int* __restrict__ status) {
  pdl_wait();
  pdl_launch_dependents();
  bool bad = false;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const float x = g[i];
    bad |= !(fabsf(x) <= 3.0e38f);
  }
  if (__syncthreads_or(bad) && threadIdx.x == 0) atomicOr(status, 1);
}

__global__ void __launch_bounds__(256) adam_kernel(float* __restrict__ p, const float* __restrict__ g,
                                                   float* __restrict__ m, float* __restrict__ v, long long n,
                                                   long long bias_start, float lr, float lr_bias, float beta1,
                                                   float beta2, float eps, float weight_decay, float bc1,
                                                   float bc2_sqrt, float grad_scale, int* __restrict__ status) {
  pdl_wait();
  pdl_launch_dependents();
  if (status && (status[0] & 1)) {       // non-finite gradient: leave parameters and moments untouched
    if (blockIdx.x == 0 && threadIdx.x == 0) atomicAdd(status + 1, 1);
    return;
  }
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const float pi = p[i];
    const float gi = g[i] * grad_scale + weight_decay * pi;
    const float mi = m[i] + (gi - m[i]) * (1.f - beta1);
    const float vi = beta2 * v[i] + (1.f - beta2) * gi * gi;
    m[i] = mi;
    v[i] = vi;
    const float denom = sqrtf(vi) / bc2_sqrt + eps;
    const float step = (i >= bias_start ? lr_bias : lr) / bc1;
    p[i] = pi - step * (mi / denom);
  }
}

// ---- the same step with ALL of its state on the device (capturable in a CUDA graph, no host scalars) ----------
// state[0] non-finite flag of this step, state[1] skipped steps, state[2] applied steps, state[3] unused.
// One thread turns the step counter into the scalars of the step: the optimizer step counter and the position of
// CosineAnnealingLR(T_max) advance ONLY when the update is applied (a skipped step leaves both where they were --
// torch.optim / the reference apply no step when "Loss is NaN" is raised, ssd3d.py:938-940).
//   lr_k = eta_min + (base - eta_min) * (1 + cos(pi * k / T_max)) / 2,  k = applied step (1-based): the reference
//   steps the scheduler inside training_step, before the optimizer step of the same batch (ssd3d.py:525-527).
__global__ void adam_prepare_kernel(int* __restrict__ state, float* __restrict__ scal, float base_lr,
                                    float bias_lr_mult, int t_max, float beta1, float beta2) {
  pdl_wait();
  pdl_launch_dependents();
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  if (state[0] & 1) {
    state[1] += 1;
    scal[4] = 0.f;          // skip
    return;
  }
  const int k = ++state[2];
  double lr = (double)base_lr;
  if (t_max > 0) lr = lr * (1.0 + cos(3.14159265358979323846 * (double)k / (double)t_max)) * 0.5;
  scal[0] = (float)lr;
  scal[1] = (float)(lr * (double)bias_lr_mult);
  scal[2] = (float)(1.0 - pow((double)beta1, (double)k));
  scal[3] = (float)sqrt(1.0 - pow((double)beta2, (double)k));
  scal[4] = 1.f;
}

__global__ void __launch_bounds__(256) adam_dev_kernel(float* __restrict__ p, const float* __restrict__ g,
                                                       float* __restrict__ m, float* __restrict__ v, long long n,
                                                       long long bias_start, const float* __restrict__ scal,
                                                       float beta1, float beta2, float eps, float weight_decay,
                                                       float grad_scale) {
  pdl_wait();
  pdl_launch_dependents();
  if (scal[4] == 0.f) return;            // non-finite gradient: parameters and moments untouched
  const float lr = scal[0], lr_bias = scal[1], bc1 = scal[2], bc2_sqrt = scal[3];
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const float pi = p[i];
    const float gi = g[i] * grad_scale + weight_decay * pi;
    const float mi = m[i] + (gi - m[i]) * (1.f - beta1);
    const float vi = beta2 * v[i] + (1.f - beta2) * gi * gi;
    m[i] = mi;
    v[i] = vi;
    const float denom = sqrtf(vi) / bc2_sqrt + eps;
    const float step = (i >= bias_start ? lr_bias : lr) / bc1;
    p[i] = pi - step * (mi / denom);
  }
}

// ------------------------------------------------------------------------------------------------
// Weight packing for the next step as ONE launch: dst[i] = bf16(src[index[i]]) (index < 0 -> 0).  The index map
// (built once on the host) encodes every layout the kernels want -- stem (32, KPAD) zero padded, depthwise
// (27, C), pointwise (Cout, Cin) and its transpose, head (16, 27*C) with loc | class rows -- over the flat fp32
// parameter buffer the optimizer updates.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) gather_cast_bf16_kernel(const float* __restrict__ src,
                                                               const int* __restrict__ index, long long n,
                                                               bf16* __restrict__ dst) {
  pdl_wait();
  pdl_launch_dependents();
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const int k = index[i];
    dst[i] = __float2bfloat16_rn(k >= 0 ? src[k] : 0.f);
  }
}
__global__ void __launch_bounds__(256) gather_f32_kernel(const float* __restrict__ src, const int* __restrict__ index,
                                                         long long n, float* __restrict__ dst) {
  pdl_wait();
  pdl_launch_dependents();
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const int k = index[i];
    dst[i] = k >= 0 ? src[k] : 0.f;
  }
}

static inline int grid_for(long long total, int block, int cap) {
  long long b = (total + block - 1) / block;
  if (b > cap) b = cap;
  if (b < 1) b = 1;
  return (int)b;
}

}  // namespace ssd3d

using namespace ssd3d;

// ================================================================================================
// C ABI
// ================================================================================================
static const int COLRED_MAX_BLOCKS = 592;   // 4 x 148 SMs

static int colreduce_plan(long long M, int C, int* threads, long long* rows_per_block,
                          int max_blocks = COLRED_MAX_BLOCKS) {
  const int CV = C / 8;
  if (C <= 0 || (C & 7) || CV > 256) return -1;
  const int RP = 256 / CV;
  *threads = CV * RP;
  long long B = (M + RP * 4 - 1) / (RP * 4);
  if (B > max_blocks) B = max_blocks;
  if (B < 1) B = 1;
  long long rpb = (M + B - 1) / B;
  *rows_per_block = rpb;
  return (int)((M + rpb - 1) / rpb);
}

extern "C" int64_t ssd3d_bn_workspace_bytes(int C) { return (int64_t)COLRED_MAX_BLOCKS * 2 * C * 4; }

extern "C" int ssd3d_bn_train_fwd(const void* z, int64_t M, int C, const float* gamma, const float* beta, float eps,
                                  float momentum, float* running_mean, float* running_var,
                                  int64_t* num_batches_tracked, float* scale, float* shift, float* mean, float* invstd,
                                  void* a, int* nan_flag, void* workspace, int64_t workspace_bytes, void* stream) {
  if (!z || !scale || !shift || !mean || !invstd || !workspace || M <= 0) return SSD3D_ERR_ARG;
  int threads;
  long long rpb;
  const int B = colreduce_plan(M, C, &threads, &rpb);
  if (B < 0 || workspace_bytes < (int64_t)B * 2 * C * 4) return SSD3D_ERR_ARG;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  float* partial = static_cast<float*>(workspace);
  const bf16* zp = static_cast<const bf16*>(z);
  SSD3D_LAUNCH_PDL(colreduce_kernel<0>, dim3(B), dim3(threads), 0, st, zp, (const bf16*)nullptr, (const float*)nullptr,
                   (const float*)nullptr, (const float*)nullptr, (const float*)nullptr, (long long)M, C, rpb, partial);
  SSD3D_LAUNCH_PDL(bn_finalize_fwd_kernel, dim3((C + 31) / 32), dim3(1024), 0, st, (const float*)partial, B, C,
                   (long long)M, gamma, beta, eps, momentum, running_mean, running_var, scale, shift, mean, invstd,
                   reinterpret_cast<long long*>(num_batches_tracked));
  if (a) {
    const long long total_vec = (long long)M * (C / 8);
    SSD3D_LAUNCH_PDL(bn_apply_relu_kernel, dim3(grid_for(total_vec, 256, 148 * 8)), dim3(256), 0, st, zp,
                     (const float*)scale, (const float*)shift, static_cast<bf16*>(a), total_vec, C / 8, nan_flag);
  }
  return SSD3D_OK;
}

extern "C" int ssd3d_bn_relu_bwd(const void* z, const void* grad_a, int64_t M, int C, const float* scale,
                                 const float* shift, const float* mean, const float* invstd, float* dgamma,
                                 float* dbeta, void* dz, void* workspace, int64_t workspace_bytes, void* stream) {
  if (!z || !grad_a || !scale || !shift || !mean || !invstd || !dgamma || !dbeta || !dz || !workspace || M <= 0)
    return SSD3D_ERR_ARG;
  int threads;
  long long rpb;
  // the backward reduction holds 84 registers: three CTAs per SM are resident, so at most 3 x 148 blocks (a fourth
  // quarter of the grid would run as a second, mostly empty wave)
  const int B = colreduce_plan(M, C, &threads, &rpb, 444);
  if (B < 0 || workspace_bytes < (int64_t)B * 2 * C * 4) return SSD3D_ERR_ARG;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  float* partial = static_cast<float*>(workspace);
  const bf16* zp = static_cast<const bf16*>(z);
  const bf16* gp = static_cast<const bf16*>(grad_a);
  SSD3D_LAUNCH_PDL(colreduce_kernel<1>, dim3(B), dim3(threads), 0, st, zp, gp, scale, shift, mean, invstd, (long long)M,
                   C, rpb, partial);
  SSD3D_LAUNCH_PDL(bn_finalize_bwd_kernel, dim3((C + 31) / 32), dim3(1024), 0, st, (const float*)partial, B, C, dgamma,
                   dbeta);
  const long long total_vec = (long long)M * (C / 8);
  SSD3D_LAUNCH_PDL(bn_relu_bwd_apply_kernel, dim3(grid_for(total_vec, 256, 148 * 8)), dim3(256), 0, st, zp, gp, scale,
                   shift, mean, invstd, (const float*)dgamma, (const float*)dbeta, (float)(1.0 / (double)M),
                   static_cast<bf16*>(dz), total_vec, C / 8);
  return SSD3D_OK;
}

// ---- weight gradients ------------------------------------------------------------------------------
static int wgrad_splits(long long M, int tiles) {
  long long s = (592 + tiles - 1) / tiles;
  const long long chunks = (M + 63) / 64;
  if (s > chunks) s = chunks;
  if (s < 1) s = 1;
  return (int)s;
}

extern "C" int64_t ssd3d_wgrad_workspace_bytes(int64_t M, int n_out, int K) {
  const int kp = (K + 63) / 64 * 64;
  const int np = n_out <= 16 ? 16 : (n_out <= 32 ? 32 : (n_out + 63) / 64 * 64);
  const int nt = np <= 16 ? 16 : (np <= 32 ? 32 : 64);
  const int S = wgrad_splits(M, (kp / 64) * (np / nt));
  int64_t need = (int64_t)S * np * kp * 4;
  if (np == 16 && K % (27 * 64) == 0) {     // SSD head: slabs of the activation-stationary kernel
    const int C = K / 27;
    need = std::max<int64_t>(need, (int64_t)head_wgrad_splits(M, C) * 16 * 27 * C * 4);
  }
  return need;
}

template <int NT, int MODE, int KT>
static int run_wgrad(WgradParams& p, int n_out, cudaStream_t st, int* splits_out) {
  const int tiles = (p.K / KT) * (p.n_pad / NT);
  const int S = wgrad_splits(p.M, tiles);
  long long rps = (p.M + S - 1) / S;
  rps = (rps + 63) / 64 * 64;
  p.rows_per_split = rps;
  const int S2 = (int)((p.M + rps - 1) / rps);
  dim3 grid((unsigned)(p.K / KT), (unsigned)(p.n_pad / NT), (unsigned)S2);
  SSD3D_LAUNCH_PDL((wgrad_kernel<NT, MODE, KT>), grid, dim3(128), 0, st, p);
  *splits_out = S2;
  return SSD3D_OK;
}

// wgrad_tc.cu: the same contraction on tcgen05 (MN-major UMMA operands straight from TMA)
namespace ssd3d {
int64_t wgrad_tc_workspace_bytes(long long M, int Cin, int Cout);
int wgrad_tc_launch(const void* dz, const void* x, long long M, int Cin, int Cout, float* dw, float* partial,
                    cudaStream_t st);
int head_wgrad_tc_launch(const void* dO16, const void* x, int N, int C, int D, int H, int W, int g, int n_loc, int n_cls,
                         float* dw_loc, float* dw_cls, float* workspace, int64_t workspace_bytes, cudaStream_t st);
int head_dgrad_tc_launch(const void* dO, const void* w, const void* addend, void* dx, int N, int C, int D, int H, int W,
                         int groups, cudaStream_t st);
}

extern "C" int ssd3d_pwconv_wgrad(const void* dz, const void* x, int64_t M, int Cin, int Cout, float* dw,
                                  void* workspace, int64_t workspace_bytes, void* stream) {
  if (!dz || !x || !dw || !workspace || M <= 0) return SSD3D_ERR_ARG;
  if (Cin <= 0 || (Cin % 32) || Cout <= 0 || (Cout % 64)) return SSD3D_ERR_ARG;
  if (workspace_bytes < ssd3d_wgrad_workspace_bytes(M, Cout, Cin)) return SSD3D_ERR_ARG;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (workspace_bytes >= wgrad_tc_workspace_bytes(M, Cin, Cout)) {
    const int S = wgrad_tc_launch(dz, x, M, Cin, Cout, dw, static_cast<float*>(workspace), st);
    if (S == 1) return SSD3D_OK;
    if (S > 1)
      return launch_sum_partials((const float*)workspace, S, (long long)Cout * Cin, Cout, Cin, Cin, Cin, dw, st);
    if (S < -1) return SSD3D_ERR_ARG;       // -1: shape not taken by the tcgen05 tiling -> mma.sync kernel below
  }
  WgradParams p{};
  p.dz = static_cast<const bf16*>(dz); p.ldz = Cout; p.M = M;
  p.K = (Cin + 63) / 64 * 64;
  p.x = x; p.C = Cin; p.n_pad = Cout;
  p.partial = static_cast<float*>(workspace);
  int S = 0;
  const int rc = run_wgrad<64, 0, 64>(p, Cout, st, &S);
  if (rc) return rc;
  if (const int rc_s = launch_sum_partials((const float*)p.partial, S, (long long)p.n_pad * p.K, Cout, Cin, p.K, Cin, dw, st)) return rc_s;
  return SSD3D_OK;
}

// Rows 16g .. 16g+15 of the packed head weight [loc rows | class rows | pad] -> the two conv weight gradients:
// the slabs of column group g are [S][16][C][27]; its rows land in dw_loc / dw_cls as (at most) one contiguous run each.
static int head_wgrad_scatter(const float* partial, int S, int C, int g, int n_loc, int n_cls, float* dw_loc,
                              float* dw_cls, cudaStream_t st) {
  const long long slab = 16ll * 27 * C, row = 27ll * C;
  const int r0 = 16 * g, r1 = r0 + 16;
  const int l0 = r0 < n_loc ? r0 : n_loc, l1 = r1 < n_loc ? r1 : n_loc;                        // loc rows [l0, l1)
  if (l1 > l0)
    if (const int rc = launch_sum_partials(partial + (size_t)(l0 - r0) * row, S, slab, 1, (int)((l1 - l0) * row),
                                           (int)((l1 - l0) * row), (int)((l1 - l0) * row), dw_loc + (size_t)l0 * row, st))
      return rc;
  const int c0 = (r0 > n_loc ? r0 : n_loc), c1 = (r1 < n_loc + n_cls ? r1 : n_loc + n_cls);      // class rows [c0, c1)
  if (c1 > c0)
    if (const int rc = launch_sum_partials(partial + (size_t)(c0 - r0) * row, S, slab, 1, (int)((c1 - c0) * row),
                                           (int)((c1 - c0) * row), (int)((c1 - c0) * row),
                                           dw_cls + (size_t)(c0 - n_loc) * row, st))
      return rc;
  return SSD3D_OK;
}

extern "C" int ssd3d_head_wgrad(const void* dO, const void* x, int N, int C, int D, int H, int W, int n_loc, int n_cls,
                                float* dw_loc, float* dw_cls, void* workspace, int64_t workspace_bytes,
                                void* stream) {
  if (!dO || !x || !dw_loc || !dw_cls || !workspace || N <= 0 || D <= 0 || H <= 0 || W <= 0) return SSD3D_ERR_ARG;
  if (C <= 0 || (C % 64) || n_loc <= 0 || n_cls <= 0 || n_loc + n_cls > 256) return SSD3D_ERR_UNSUPPORTED;
  const long long M = (long long)N * D * H * W;
  if (workspace_bytes < ssd3d_wgrad_workspace_bytes(M, 16, 27 * C)) return SSD3D_ERR_ARG;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int groups = (n_loc + n_cls + 15) / 16;      // 16 output columns per pass (dO is (groups, M, 16))
  for (int g = 0; g < groups; ++g) {
    const bf16* dOg = static_cast<const bf16*>(dO) + (size_t)g * M * 16;
    const int rc = head_wgrad_tc_launch(dOg, x, N, C, D, H, W, g, n_loc, n_cls, dw_loc, dw_cls,
                                        static_cast<float*>(workspace), workspace_bytes, st);
    if (rc == 0) continue;
    if (rc < -1) return SSD3D_ERR_ARG;    // -1: no 64-voxel box fits this map -> mma.sync kernel below
    HeadWgradParams q{};
    q.dO = dOg; q.x = static_cast<const bf16*>(x);
    q.N = N; q.D = D; q.H = H; q.W = W; q.C = C; q.M = M;
    const long long chunks = (M + 63) / 64;
    const int S0 = head_wgrad_splits(M, C);
    q.chunks_per_split = (int)((chunks + S0 - 1) / S0);
    const int S = (int)((chunks + q.chunks_per_split - 1) / q.chunks_per_split);
    q.partial = static_cast<float*>(workspace);
    const size_t smem = (size_t)2 * 64 * (HW_XP + HW_GP) * 2;
    cudaError_t e = cudaFuncSetAttribute(head_wgrad_g_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    SSD3D_LAUNCH_PDL(head_wgrad_g_kernel, dim3((unsigned)(C / 64), 3u, (unsigned)S), dim3(128), smem, st, q);
    if (const int rc_s = head_wgrad_scatter(q.partial, S, C, g, n_loc, n_cls, dw_loc, dw_cls, st)) return rc_s;
  }
  return SSD3D_OK;
}

namespace ssd3d {
int stem_wgrad_tiles(const void* dz, const void* x, int x_is_bf16, int N, int Cin, int D, int H, int W, int stride_d,
                     float* partial, int max_slabs, int* slabs, int* kpad, cudaStream_t st,
                     const void* const* bn);   // conv_stem_tc.cu
}

// The stem unit's backward in two launches instead of three: `ssd3d_bn_unit_bwd` with dz = NULL leaves only the
// statistics (dgamma, dbeta); this entry point then applies the BatchNorm + ReLU backward to the gradient rows while
// it loads them for the weight gradient (conv_stem_tc.cu): dz of the first layer is never materialised (nothing
// upstream needs it).  SSD3D_ERR_UNSUPPORTED where the TMA tile kernel does not take the shape.
extern "C" int ssd3d_stem_wgrad_bn(const void* z, const void* grad_a, const void* x, int x_is_bf16, int N, int Cin, int D,
                                   int H, int W, int stride_d, const float* scale, const float* shift,
                                   const float* mean, const float* invstd, const float* dgamma, const float* dbeta,
                                   float* dw, void* workspace, int64_t workspace_bytes, void* stream) {
  if (!z || !grad_a || !x || !scale || !shift || !mean || !invstd || !dgamma || !dbeta || !dw || !workspace)
    return SSD3D_ERR_ARG;
  if (N <= 0 || D <= 0 || H <= 0 || W <= 0 || Cin < 1 || Cin > 4 || (stride_d != 1 && stride_d != 2)) return SSD3D_ERR_UNSUPPORTED;
  const int Do = (D - 1) / stride_d + 1, Ho = (H - 1) / 2 + 1, Wo = (W - 1) / 2 + 1;
  const long long M = (long long)N * Do * Ho * Wo;
  if (M < 128 * 148) return SSD3D_ERR_UNSUPPORTED;
  if (workspace_bytes < ssd3d_wgrad_workspace_bytes(M, 32, 27 * Cin)) return SSD3D_ERR_ARG;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const float inv_m = (float)(1.0 / (double)M);
  const void* bn[8] = {z, scale, shift, mean, invstd, dgamma, dbeta, &inv_m};
  const int kp = (27 * Cin <= 64) ? 64 : 128;
  const int max_slabs = (int)std::min<long long>(workspace_bytes / (32ll * kp * 4), 4096);
  int S = 0, kpad = 0;
  const int rc = stem_wgrad_tiles(grad_a, x, x_is_bf16, N, Cin, D, H, W, stride_d, static_cast<float*>(workspace),
                                  max_slabs, &S, &kpad, st, bn);
  if (rc != SSD3D_OK) return rc;
  return launch_sum_partials((const float*)workspace, S, 32ll * kpad, 32, 27 * Cin, kpad, 27 * Cin, dw, st);
}

extern "C" int ssd3d_stem_wgrad(const void* dz, const void* x, int x_is_bf16, int N, int Cin, int D, int H, int W,
                                int stride_d, float* dw, void* workspace, int64_t workspace_bytes, void* stream) {
  if (!dz || !x || !dw || !workspace || N <= 0 || D <= 0 || H <= 0 || W <= 0) return SSD3D_ERR_ARG;
  if (Cin < 1 || Cin > 4 || (stride_d != 1 && stride_d != 2)) return SSD3D_ERR_UNSUPPORTED;
  const int Do = (D - 1) / stride_d + 1, Ho = (H - 1) / 2 + 1, Wo = (W - 1) / 2 + 1;
  const long long M = (long long)N * Do * Ho * Wo;
  const int K = (27 * Cin <= 32) ? 32 : (27 * Cin + 63) / 64 * 64;     // one 32-wide k tile for Cin = 1
  if (workspace_bytes < ssd3d_wgrad_workspace_bytes(M, 32, 27 * Cin)) return SSD3D_ERR_ARG;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (M >= 128 * 148) {
    // halo tiles through TMA + im2col in shared memory (the forward stem's gather), one slab per persistent CTA
    const int kp = (27 * Cin <= 64) ? 64 : 128;
    const int max_slabs = (int)std::min<long long>(workspace_bytes / (32ll * kp * 4), 4096);
    int S = 0, kpad = 0;
    const int rc = stem_wgrad_tiles(dz, x, x_is_bf16, N, Cin, D, H, W, stride_d, static_cast<float*>(workspace),
                                    max_slabs, &S, &kpad, st, nullptr);
    if (rc == SSD3D_OK) {
      if (const int rc_s = launch_sum_partials((const float*)workspace, S, 32ll * kpad, 32, 27 * Cin, kpad, 27 * Cin, dw, st)) return rc_s;
      return SSD3D_OK;
    }
    if (rc != SSD3D_ERR_UNSUPPORTED) return rc;
  }
  WgradParams p{};
  p.dz = static_cast<const bf16*>(dz); p.ldz = 32; p.M = M;
  p.K = K;
  p.x = x; p.x_is_bf16 = x_is_bf16; p.N = N; p.D = D; p.H = H; p.W = W;
  p.Do = Do; p.Ho = Ho; p.Wo = Wo; p.sd = stride_d; p.Cin = Cin; p.n_pad = 32;
  p.partial = static_cast<float*>(workspace);
  int S = 0;
  const int rc = (K == 32) ? run_wgrad<32, 2, 32>(p, 32, st, &S) : run_wgrad<32, 2, 64>(p, 32, st, &S);
  if (rc) return rc;
  if (const int rc_s = launch_sum_partials((const float*)p.partial, S, (long long)p.n_pad * p.K, 32, 27 * Cin, p.K, 27 * Cin, dw, st)) return rc_s;
  return SSD3D_OK;
}

// ---- head gradient rows + bias gradient, head data gradient ---------------------------------------------
extern "C" int64_t ssd3d_head_grad_workspace_bytes(int N, int D, int H, int W, int n_cols) {
  const long long M = (long long)N * D * H * W;
  const int groups = (n_cols + 15) / 16;
  return (int64_t)((M + 255) / 256) * groups * 16 * 4;
}

extern "C" int ssd3d_head_grad_pack(const float* dlocs, const float* dscores, int N, int D, int H, int W, int bpl,
                                    int n_classes, int64_t P, int64_t prior_offset, void* dO, float* dbias_loc,
                                    float* dbias_cls, void* workspace, int64_t workspace_bytes, void* stream) {
  if (!dlocs || !dscores || !dO || !dbias_loc || !dbias_cls || !workspace || N <= 0) return SSD3D_ERR_ARG;
  const int n_cols = bpl * (6 + n_classes);
  if (bpl <= 0 || n_classes <= 0 || n_cols > 256) return SSD3D_ERR_UNSUPPORTED;
  const int groups = (n_cols + 15) / 16, ld = groups * 16;
  const long long V = (long long)D * H * W, M = (long long)N * V;
  const int blocks = (int)((M + 255) / 256);
  if (workspace_bytes < (int64_t)blocks * ld * 4) return SSD3D_ERR_ARG;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  float* partial = static_cast<float*>(workspace);
  SSD3D_LAUNCH_PDL(head_grad_pack_kernel, dim3(blocks), dim3(256), 0, st, dlocs, dscores, (long long)P,
                   (long long)prior_offset, V, N, bpl, n_classes, groups, static_cast<bf16*>(dO), partial);
  // column sums: partial is [blocks][ld] -> rows = 1, slab = ld
  if (const int rc_s = launch_sum_partials((const float*)partial, blocks, (long long)ld, 1, bpl * 6, ld,
                   bpl * 6, dbias_loc, st)) return rc_s;
  if (const int rc_s = launch_sum_partials((const float*)(partial + bpl * 6), blocks, (long long)ld, 1,
                   bpl * n_classes, ld, bpl * n_classes, dbias_cls, st)) return rc_s;
  return SSD3D_OK;
}

extern "C" int ssd3d_head_dgrad(const void* dO, const void* w, const void* addend, void* dx, int N, int C, int D,
                                int H, int W, int n_cols, void* stream) {
  if (!dO || !w || !dx || N <= 0 || D <= 0 || H <= 0 || W <= 0) return SSD3D_ERR_ARG;
  if (C <= 0 || (C % 64) || n_cols <= 0 || n_cols > 256) return SSD3D_ERR_UNSUPPORTED;
  const long long M = (long long)N * D * H * W;
  const int groups = (n_cols + 15) / 16;
  const int rc = head_dgrad_tc_launch(dO, w, addend, dx, N, C, D, H, W, groups, static_cast<cudaStream_t>(stream));
  if (rc == 0) return SSD3D_OK;
  if (rc < -1) return SSD3D_ERR_ARG;      // -1: no 128-voxel box fits this map -> mma.sync kernel below
  const size_t smem = (size_t)(27 * 16 * 72 + 2 * 64 * 24) * 2;
  cudaError_t e = cudaFuncSetAttribute(head_dgrad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return (int)e;
  dim3 grid((unsigned)((M + 63) / 64), (unsigned)(C / 64));
  // 16 gradient columns per group, all groups accumulated in fp32 registers inside ONE launch
  HeadDgradParams p{};
  p.dO = static_cast<const bf16*>(dO);
  p.w = static_cast<const bf16*>(w);
  p.addend = static_cast<const bf16*>(addend);
  p.dx = static_cast<bf16*>(dx);
  p.N = N; p.D = D; p.H = H; p.W = W; p.C = C; p.M = M; p.groups = groups;
  SSD3D_LAUNCH_PDL(head_dgrad_kernel, grid, dim3(128), smem, static_cast<cudaStream_t>(stream), p);
  return SSD3D_OK;
}

// ---- depthwise backward -------------------------------------------------------------------------------
extern "C" int ssd3d_dwconv3d_dgrad(const void* dz, const void* w, void* dx, int N, int C, int D, int H, int W,
                                    int stride, void* stream) {
  if (!dz || !w || !dx || N <= 0 || D <= 0 || H <= 0 || W <= 0) return SSD3D_ERR_ARG;
  if (C <= 0 || (C & 7) || (stride != 1 && stride != 2)) return SSD3D_ERR_ARG;
  const int Do = (D - 1) / stride + 1, Ho = (H - 1) / stride + 1, Wo = (W - 1) / stride + 1;
  const long long total = (long long)N * D * H * W * (C / 8);
  const unsigned blocks = (unsigned)((total + 255) / 256);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const bf16* gp = static_cast<const bf16*>(dz);
  const bf16* wp = static_cast<const bf16*>(w);
  if (stride == 1) {
    SSD3D_LAUNCH_PDL(dw_dgrad_kernel<1>, dim3(blocks), dim3(256), 0, st, gp, wp, static_cast<bf16*>(dx), N, C, D, H, W,
                     Do, Ho, Wo, total);
  } else if (C <= 256) {
    const int Md = (D + 1) / 2, Mh = (H + 1) / 2, Mw = (W + 1) / 2;
    const long long tot = (long long)N * Md * Mh * Mw * (C / 8);
    SSD3D_LAUNCH_PDL(dw_dgrad_s2_block_kernel, dim3((unsigned)((tot + 255) / 256)), dim3(256), (size_t)27 * C * 4, st, gp,
                     wp, static_cast<bf16*>(dx), N, C, D, H, W, Do, Ho, Wo, Md, Mh, Mw, tot);
  } else {
    // one block row per parity class; the largest class (all coordinates even) sizes the grid
    const long long biggest = (long long)N * ((D + 1) / 2) * ((H + 1) / 2) * (((W + 1) / 2 + 3) / 4) * (C / 4);
    dim3 grid((unsigned)((biggest + 255) / 256), 8);
    SSD3D_LAUNCH_PDL(dw_dgrad_s2_kernel, grid, dim3(256), 0, st, gp, wp, static_cast<bf16*>(dx), N, C, D, H, W, Do, Ho,
                     Wo);
  }
  return SSD3D_OK;
}

static int dw_wgrad_plan(long long Mo, int C, int* threads, int* G, long long* vpb) {
  const int CV = C / 8;
  if (C <= 0 || (C & 7) || CV * 3 > 256) return -1;
  *G = 256 / (CV * 3);
  *threads = CV * 3 * (*G);
  // voxels per voxel lane: the loop over them is serial (one L2 round trip + ~350 instructions each, 1-2 warps per
  // scheduler), so small maps get as few as 2 -- ~1.5 CTAs per SM -- and pay with more slabs; large ones 8
  long long vpl = Mo / ((long long)(*G) * 222);
  vpl = vpl < 2 ? 2 : (vpl > 8 ? 8 : vpl);
  long long B = (Mo + (*G) * vpl - 1) / ((*G) * vpl);       // >= vpl voxels per voxel lane
  if (B > 592) B = 592;
  if (B < 1) B = 1;
  *vpb = (Mo + B - 1) / B;
  return (int)((Mo + *vpb - 1) / *vpb);
}

extern "C" int64_t ssd3d_dw_wgrad_workspace_bytes(int C) { return (int64_t)592 * C * 27 * 4; }

// conv_dw_tma.cu
int ssd3d_dwconv3d_wgrad_tma(const void* dz, const void* x, int N, int C, int D, int H, int W, int stride,
                             float* partial, int max_slabs, int* slabs, cudaStream_t st);

extern "C" int ssd3d_dwconv3d_wgrad(const void* dz, const void* x, int N, int C, int D, int H, int W, int stride,
                                    float* dw, void* workspace, int64_t workspace_bytes, void* stream) {
  if (!dz || !x || !dw || !workspace || N <= 0 || D <= 0 || H <= 0 || W <= 0) return SSD3D_ERR_ARG;
  if (stride != 1 && stride != 2) return SSD3D_ERR_ARG;
  const int Do = (D - 1) / stride + 1, Ho = (H - 1) / stride + 1, Wo = (W - 1) / stride + 1;
  const long long Mo = (long long)N * Do * Ho * Wo;
  if (C > 0 && workspace_bytes >= ssd3d_dw_wgrad_workspace_bytes(C)) {
    // large maps: TMA halo tiles, register-resident accumulators (conv_dw_tma.cu)
    int slabs = 0;
    const int rc = ssd3d_dwconv3d_wgrad_tma(dz, x, N, C, D, H, W, stride, static_cast<float*>(workspace), 592, &slabs,
                                            static_cast<cudaStream_t>(stream));
    if (rc == SSD3D_OK) {
      return launch_sum_partials((const float*)workspace, slabs, (long long)C * 27, C, 27, 27, 27, dw,
                                 static_cast<cudaStream_t>(stream));
    }
    if (rc != SSD3D_ERR_UNSUPPORTED) return rc;
  }
  int threads, G;
  long long vpb;
  const int B = dw_wgrad_plan(Mo, C, &threads, &G, &vpb);
  if (B < 0 || Mo >= (1ll << 31)) return SSD3D_ERR_UNSUPPORTED;
  if (workspace_bytes < (int64_t)B * C * 27 * 4) return SSD3D_ERR_ARG;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  float* partial = static_cast<float*>(workspace);
  const bf16* gp = static_cast<const bf16*>(dz);
  const bf16* xp = static_cast<const bf16*>(x);
  if (stride == 1)
    SSD3D_LAUNCH_PDL(dw_wgrad_kernel<1>, dim3(B), dim3(threads), 0, st, gp, xp, N, C, D, H, W, Do, Ho, Wo, Mo, vpb, G,
                     partial);
  else
    SSD3D_LAUNCH_PDL(dw_wgrad_kernel<2>, dim3(B), dim3(threads), 0, st, gp, xp, N, C, D, H, W, Do, Ho, Wo, Mo, vpb, G,
                     partial);
  if (const int rc_s = launch_sum_partials((const float*)partial,
                   B, (long long)C * 27, 27, C, C, 1, dw, st, 27)) return rc_s;
  return SSD3D_OK;
}

// ---- optimizer ------------------------------------------------------------------------------------------
extern "C" int ssd3d_adam_step(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n,
                               int64_t bias_start, float lr, float lr_bias, float beta1, float beta2, float eps,
                               float weight_decay, int step, float grad_scale, int32_t* status, void* stream) {
  if (!param || !grad || !exp_avg || !exp_avg_sq || n <= 0 || step < 1) return SSD3D_ERR_ARG;
  const double bc1 = 1.0 - pow((double)beta1, (double)step);
  const double bc2 = 1.0 - pow((double)beta2, (double)step);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (status) {
    cudaError_t e = cudaMemsetAsync(status, 0, 4, st);
    if (e != cudaSuccess) return (int)e;
    SSD3D_LAUNCH_PDL(grad_nonfinite_kernel, dim3(grid_for(n, 256, 148 * 4)), dim3(256), 0, st, grad, (long long)n, status);
  }
  SSD3D_LAUNCH_PDL(adam_kernel, dim3(grid_for(n, 256, 148 * 8)), dim3(256), 0, st, param, grad, exp_avg, exp_avg_sq,
                   (long long)n, (long long)bias_start, lr, lr_bias, beta1, beta2, eps, weight_decay, (float)bc1,
                   (float)sqrt(bc2), grad_scale, status);
  return SSD3D_OK;
}

extern "C" int ssd3d_adam_step_dev(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n,
                                   int64_t bias_start, float base_lr, float bias_lr_mult, int t_max, float beta1,
                                   float beta2, float eps, float weight_decay, float grad_scale, int32_t* state,
                                   float* scalars, void* stream) {
  if (!param || !grad || !exp_avg || !exp_avg_sq || !state || !scalars || n <= 0 || t_max < 0) return SSD3D_ERR_ARG;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  cudaError_t e = cudaMemsetAsync(state, 0, 4, st);
  if (e != cudaSuccess) return (int)e;
  SSD3D_LAUNCH_PDL(grad_nonfinite_kernel, dim3(grid_for(n, 256, 148 * 4)), dim3(256), 0, st, grad, (long long)n, state);
  SSD3D_LAUNCH_PDL(adam_prepare_kernel, dim3(1), dim3(32), 0, st, state, scalars, base_lr, bias_lr_mult, t_max, beta1,
                   beta2);
  SSD3D_LAUNCH_PDL(adam_dev_kernel, dim3(grid_for(n, 256, 148 * 8)), dim3(256), 0, st, param, grad, exp_avg, exp_avg_sq,
                   (long long)n, (long long)bias_start, (const float*)scalars, beta1, beta2, eps, weight_decay,
                   grad_scale);
  return SSD3D_OK;
}

// ---- weight packing -------------------------------------------------------------------------------------
extern "C" int ssd3d_gather_cast(const float* src, const int32_t* index, int64_t n, void* dst, int dst_is_bf16,
                                 void* stream) {
  if (!src || !index || !dst || n <= 0) return SSD3D_ERR_ARG;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (dst_is_bf16)
    SSD3D_LAUNCH_PDL(gather_cast_bf16_kernel, dim3(grid_for(n, 256, 148 * 8)), dim3(256), 0, st, src, index, (long long)n,
                     static_cast<bf16*>(dst));
  else
    SSD3D_LAUNCH_PDL(gather_f32_kernel, dim3(grid_for(n, 256, 148 * 8)), dim3(256), 0, st, src, index, (long long)n,
                     static_cast<float*>(dst));
  return SSD3D_OK;
}
