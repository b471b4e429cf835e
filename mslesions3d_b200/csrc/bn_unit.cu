// Train-mode BatchNorm3d + ReLU as ONE launch per direction (mobilenet.py:29-30,44-45 under autograd) instead of the
// three dependent passes of train.cu (column partial sums, cross-block finalize, elementwise apply).  Three kernels,
// picked per shape by ssd3d_bn_unit_fwd / _bwd:
//   bn_cluster_kernel  maps up to 8192 rows: channel split over thread-block clusters, sums through distributed
//                      shared memory, no grid-wide barrier at all (below)
//   bn_tile_kernel     larger maps, channels a multiple of 32: (row chunk x 64-channel group) tiles, ONE barrier per
//                      channel group, every CTA finalizes its group redundantly (below)
//   bn_unit_kernel     the general fallback and the first version, described here: all CTAs resident (at most one
//                      per SM, cooperative launch), three phases separated by two grid-wide barriers
//
//   phase 1  CTA b owns rows [b*rows_per_cta, ...): thread = 8 channels x a strided set of rows, fp32 sums,
//            in-CTA tree (shuffles + shared memory), slab[b][2][C] to the workspace
//   barrier
//   phase 2  warp w finalizes channel w (, w + warps, ...): the slabs are added in fp64 in a fixed order
//            forward : mean / biased variance -> scale, shift, mean, invstd, running statistics
//            backward: dbeta = sum dy, dgamma = sum dy*xhat
//   barrier
//   phase 3  the CTA walks its own rows again (L2 hits for every map of the network but the first) and writes
//            a = relu(z*scale+shift)   /   dz = scale*(dy - dbeta/M - xhat*dgamma/M)
//
// The barrier words (zero before the first launch; 512 u32: bn_unit uses three, bn_tile two per channel group)
// belong to the caller's stream slot; the last CTA to leave a barrier zeroes its words again, so every launch (and
// every CUDA-graph replay) finds them clean.  Every reduction order is fixed by (M, C, grid): results are
// bit-reproducible run to run.
#include "common.cuh"
#include "../../include/ssd3d_b200.h"

namespace ssd3d {

typedef __nv_bfloat16 bf16;

namespace {

constexpr int BU_THREADS = 512;
constexpr int BU_WARPS = BU_THREADS / 32;

__device__ __forceinline__ uint4 bu_ld_nc16(const void* p) {
  uint4 r;
  asm volatile("ld.global.nc.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
  return r;
}
__device__ __forceinline__ void bu_unpack8(const uint4& v, float (&f)[8]) {
  f[0] = bf16_lo(v.x); f[1] = bf16_hi(v.x);
  f[2] = bf16_lo(v.y); f[3] = bf16_hi(v.y);
  f[4] = bf16_lo(v.z); f[5] = bf16_hi(v.z);
  f[6] = bf16_lo(v.w); f[7] = bf16_hi(v.w);
}
__device__ __forceinline__ uint4 bu_pack8(const float (&v)[8]) {
  uint4 o;
  o.x = pack_bf16x2(v[0], v[1]);
  o.y = pack_bf16x2(v[2], v[3]);
  o.z = pack_bf16x2(v[4], v[5]);
  o.w = pack_bf16x2(v[6], v[7]);
  return o;
}
// values another CTA of THIS grid wrote before a barrier: read them through L2 (never a stale L1 line)
__device__ __forceinline__ void bu_load8_cg(const float* p, float (&f)[8]) {
  const float4 a = __ldcg(reinterpret_cast<const float4*>(p));
  const float4 b = __ldcg(reinterpret_cast<const float4*>(p + 4));
  f[0] = a.x; f[1] = a.y; f[2] = a.z; f[3] = a.w; f[4] = b.x; f[5] = b.y; f[6] = b.z; f[7] = b.w;
}

__device__ __forceinline__ unsigned bu_ld_acquire(const unsigned* p) {
  unsigned v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
// All G CTAs are resident (G <= SM count, one CTA per SM fits by construction, cooperative launch), so spinning
// cannot starve a CTA that has not started yet.  bar.sync orders the CTA's earlier writes before thread 0's fence + arrive.
__device__ __forceinline__ void bu_grid_barrier(unsigned* word, unsigned G) {
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    atomicAdd(word, 1u);
    while (bu_ld_acquire(word) < G) {}
    __threadfence();
  }
  __syncthreads();
}

struct BnUnitParams {
  const bf16* z;
  const bf16* g;              // backward: gradient w.r.t. the ReLU output (dz may alias it)
  bf16* out;                  // forward: a (may be null: statistics only); backward: dz
  long long M;
  int C;
  long long rows_per_cta;
  float* slab;                // [G][2][C]
  unsigned* sync;             // 3 words
  // forward
  const float* gamma;
  const float* beta;
  float eps, momentum;
  float* running_mean;
  float* running_var;
  long long* num_batches_tracked;
  int* nan_flag;
  // forward: written in phase 2; backward: inputs
  float* scale;
  float* shift;
  float* mean;
  float* invstd;
  // backward
  float* dgamma;
  float* dbeta;
  float inv_m;
};

// MODE 0 forward, MODE 1 backward.  KEEP: at most 8 rows per thread (the 12^3-sized maps): they are loaded once and
// stay in registers across both barriers -- phase 3 starts without another trip to L2.
template <int MODE, bool KEEP>
__global__ void __launch_bounds__(BU_THREADS, 1) bn_unit_kernel(const BnUnitParams p) {
  __shared__ float red[BU_WARPS][2][8 * 32];      // cross-warp stage of phase 1 (32 KB)
  __shared__ double fin[BU_WARPS][32][2];         // phase 2 lane sums (8 KB)
  pdl_wait();
  pdl_launch_dependents();
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const unsigned G = gridDim.x;
  const int C = p.C, CV = C >> 3;                 // CV: power of two, 4 <= CV <= 512
  const int RP = BU_THREADS / CV;                 // row lanes of the CTA
  const int cv = tid % CV, r = tid / CV;
  const int c0 = cv << 3;
  const long long m_begin = (long long)blockIdx.x * p.rows_per_cta;
  const long long m_end = (m_begin + p.rows_per_cta < p.M) ? m_begin + p.rows_per_cta : p.M;

  float sc[8], sh[8], mu[8], is[8];
  if (MODE == 1) {
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      sc[j] = __ldg(p.scale + c0 + j); sh[j] = __ldg(p.shift + c0 + j);
      mu[j] = __ldg(p.mean + c0 + j);  is[j] = __ldg(p.invstd + c0 + j);
    }
  }

  uint4 zk[KEEP ? 8 : 1];
  // ---------------- phase 1: column partial sums over this CTA's rows ----------------
  {
    float s0[8], s1[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) { s0[j] = 0.f; s1[j] = 0.f; }
    auto add_row = [&](const uint4& zu, const uint4& gu) {
      float zf[8];
      bu_unpack8(zu, zf);
      if (MODE == 0) {
#pragma unroll
        for (int j = 0; j < 8; ++j) { s0[j] += zf[j]; s1[j] = fmaf(zf[j], zf[j], s1[j]); }
      } else {
        float gf[8];
        bu_unpack8(gu, gf);
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
    if constexpr (KEEP) {
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const long long mi = m_begin + r + (long long)i * RP;
        zk[i] = make_uint4(0u, 0u, 0u, 0u);
        if (mi < m_end) zk[i] = bu_ld_nc16(p.z + mi * C + c0);
      }
      if constexpr (MODE == 1) {
        // the gradient rows pass through in two batches of four (registers); phase 3 reads them again from L1/L2
#pragma unroll
        for (int i0 = 0; i0 < 8; i0 += 4) {
          uint4 gt[4];
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const long long mi = m_begin + r + (long long)(i0 + i) * RP;
            gt[i] = make_uint4(0u, 0u, 0u, 0u);
            if (mi < m_end) gt[i] = bu_ld_nc16(p.g + mi * C + c0);
          }
#pragma unroll
          for (int i = 0; i < 4; ++i) add_row(zk[i0 + i], gt[i]);
        }
      } else {
#pragma unroll
        for (int i = 0; i < 8; ++i) add_row(zk[i], zk[i]);
      }
    }
    constexpr int U = (MODE == 0) ? 8 : 4;        // 16-byte loads in flight per thread and operand
    // whole batches of U rows with every load issued before the first use; rows past the end are predicated off
    // and contribute zeros (z = 0 adds nothing to either sum; g = 0 gives dy = 0)
    for (long long m = m_begin + r; !KEEP && m < m_end; m += (long long)U * RP) {
      uint4 zu[U], gu[MODE == 1 ? U : 1];
#pragma unroll
      for (int i = 0; i < U; ++i) {
        const long long mi = m + (long long)i * RP;
        zu[i] = make_uint4(0u, 0u, 0u, 0u);
        if (mi < m_end) zu[i] = bu_ld_nc16(p.z + mi * C + c0);
      }
      if constexpr (MODE == 1) {
#pragma unroll
        for (int i = 0; i < U; ++i) {
          const long long mi = m + (long long)i * RP;
          gu[i] = make_uint4(0u, 0u, 0u, 0u);
          if (mi < m_end) gu[i] = bu_ld_nc16(p.g + mi * C + c0);
        }
      }
#pragma unroll
      for (int i = 0; i < U; ++i) {
        if constexpr (MODE == 1) add_row(zu[i], gu[i]);
        else add_row(zu[i], zu[i]);
      }
    }
    // in-warp: lanes with the same cv sit CV apart (CV < 32); then across the warps that share a cv
    if (CV < 32) {
      for (int off = CV; off < 32; off <<= 1) {
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          s0[j] += __shfl_xor_sync(0xffffffffu, s0[j], off);
          s1[j] += __shfl_xor_sync(0xffffffffu, s1[j], off);
        }
      }
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) { red[warp][0][j * 32 + lane] = s0[j]; red[warp][1][j * 32 + lane] = s1[j]; }
    __syncthreads();
    // writer threads: one per (cv, j-pair source); thread t < CV collects the warps that hold its cv
    if (tid < CV) {
      // warps holding cv = tid: CV <= 32 -> every warp (lane = tid);  CV > 32 -> warps w with (w*32)/... below
      const int wstep = (CV <= 32) ? 1 : CV / 32;          // warps per row lane
      const int w0 = (CV <= 32) ? 0 : tid / 32;            // first warp holding this cv
      const int ln = (CV <= 32) ? tid : (tid & 31);
      float t0[8], t1[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) { t0[j] = 0.f; t1[j] = 0.f; }
      for (int w = w0; w < BU_WARPS; w += wstep) {
#pragma unroll
        for (int j = 0; j < 8; ++j) { t0[j] += red[w][0][j * 32 + ln]; t1[j] += red[w][1][j * 32 + ln]; }
      }
      float* dst = p.slab + (size_t)blockIdx.x * 2 * C;
#pragma unroll
      for (int j = 0; j < 8; ++j) { dst[(tid << 3) + j] = t0[j]; dst[C + (tid << 3) + j] = t1[j]; }
    }
  }
  bu_grid_barrier(p.sync + 0, G);

  // ---------------- phase 2: cross-CTA sums, one warp per channel ----------------
  if (MODE == 0 && blockIdx.x == 0 && tid == 0 && p.num_batches_tracked) *p.num_batches_tracked += 1;
  for (int c = blockIdx.x * BU_WARPS + warp; c < C; c += (int)G * BU_WARPS) {
    // every slab value of this lane is requested before the first add (G <= 256: at most 8 per lane and sum); the
    // adds keep the order b = lane, lane + 32, ...
    float v0[8], v1[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const unsigned b = lane + 32u * i;
      v0[i] = 0.f; v1[i] = 0.f;
      if (b < G) {
        v0[i] = __ldcg(p.slab + (size_t)b * 2 * C + c);
        v1[i] = __ldcg(p.slab + (size_t)b * 2 * C + C + c);
      }
    }
    double ls = 0.0, lq = 0.0;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      if (lane + 32u * i < G) { ls += (double)v0[i]; lq += (double)v1[i]; }
    }
    fin[warp][lane][0] = ls;
    fin[warp][lane][1] = lq;
    __syncwarp();
    if (lane == 0) {
      double s = 0.0, q = 0.0;
      const int nl = G < 32u ? (int)G : 32;
      for (int l = 0; l < nl; ++l) { s += fin[warp][l][0]; q += fin[warp][l][1]; }
      if (MODE == 0) {
        const double mean = s / (double)p.M;
        double var = q / (double)p.M - mean * mean;
        if (var < 0.0) var = 0.0;
        const float istd = (float)(1.0 / sqrt(var + (double)p.eps));
        const float ga = p.gamma ? p.gamma[c] : 1.f, be = p.beta ? p.beta[c] : 0.f;
        const float scl = ga * istd;
        p.scale[c] = scl;
        p.shift[c] = be - (float)mean * scl;
        p.mean[c] = (float)mean;
        p.invstd[c] = istd;
        if (p.running_mean && p.running_var) {
          const double unbiased = (p.M > 1) ? var * (double)p.M / (double)(p.M - 1) : var;
          p.running_mean[c] = (float)((1.0 - (double)p.momentum) * (double)p.running_mean[c] + (double)p.momentum * mean);
          p.running_var[c] = (float)((1.0 - (double)p.momentum) * (double)p.running_var[c] + (double)p.momentum * unbiased);
        }
      } else {
        p.dbeta[c] = (float)s;
        p.dgamma[c] = (float)q;
      }
    }
    __syncwarp();
  }
  bu_grid_barrier(p.sync + 1, G);
  if (tid == 0) {
    // everybody has left barrier 0 long ago; the last CTA to leave barrier 1 clears all three words
    if (atomicAdd(p.sync + 2, 1u) == G - 1) {
      p.sync[0] = 0u; p.sync[1] = 0u; p.sync[2] = 0u;
      __threadfence();
    }
  }
  if (p.out == nullptr) return;

  // ---------------- phase 3: apply over the same rows ----------------
  if (MODE == 0) {
    bu_load8_cg(p.scale + c0, sc);
    bu_load8_cg(p.shift + c0, sh);
    bool bad = false;
    auto apply = [&](long long m, const uint4& zu) {
      float zf[8], o[8];
      bu_unpack8(zu, zf);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        o[j] = relu_nan(__fadd_rn(__fmul_rn(zf[j], sc[j]), sh[j]));
        bad |= (o[j] != o[j]);
      }
      *reinterpret_cast<uint4*>(p.out + m * C + c0) = bu_pack8(o);
    };
    if constexpr (KEEP) {
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const long long mi = m_begin + r + (long long)i * RP;
        if (mi < m_end) apply(mi, zk[i]);
      }
    }
    for (long long m = m_begin + r; !KEEP && m < m_end; m += 4ll * RP) {
      uint4 zu[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const long long mi = m + (long long)i * RP;
        if (mi < m_end) zu[i] = bu_ld_nc16(p.z + mi * C + c0);
      }
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const long long mi = m + (long long)i * RP;
        if (mi < m_end) apply(mi, zu[i]);
      }
    }
    if (bad && p.nan_flag) atomicOr(p.nan_flag, SSD3D_NAN_BACKBONE);
  } else {
    // dz = sc*(dy - dbeta/M - xhat*dgamma/M) with xhat = (z - mu)*invstd, regrouped as sc*dy + A + z*B
    // (the same expression, operation for operation, as bn_relu_bwd_apply_kernel)
    float dg[8], db[8], ka[8], kb[8];
    bu_load8_cg(p.dgamma + c0, dg);
    bu_load8_cg(p.dbeta + c0, db);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float t = sc[j] * is[j] * dg[j] * p.inv_m;
      kb[j] = -t;
      ka[j] = fmaf(mu[j], t, -(sc[j] * db[j] * p.inv_m));
    }
    auto apply = [&](long long m, const uint4& zu, const uint4& gu) {
      float zf[8], gf[8], o[8];
      bu_unpack8(zu, zf);
      bu_unpack8(gu, gf);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float pre = __fadd_rn(__fmul_rn(zf[j], sc[j]), sh[j]);
        const float dy = (pre > 0.f) ? gf[j] : 0.f;
        o[j] = fmaf(zf[j], kb[j], fmaf(sc[j], dy, ka[j]));
      }
      *reinterpret_cast<uint4*>(p.out + m * C + c0) = bu_pack8(o);
    };
    // g may be overwritten in place (out == g): every element is read and written by the same thread
    if constexpr (KEEP) {
#pragma unroll
      for (int i0 = 0; i0 < 8; i0 += 4) {
        uint4 gt[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const long long mi = m_begin + r + (long long)(i0 + i) * RP;
          if (mi < m_end) gt[i] = *reinterpret_cast<const uint4*>(p.g + mi * C + c0);
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const long long mi = m_begin + r + (long long)(i0 + i) * RP;
          if (mi < m_end) apply(mi, zk[i0 + i], gt[i]);
        }
      }
    }
    for (long long m = m_begin + r; !KEEP && m < m_end; m += 4ll * RP) {
      uint4 zu[4], gu[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const long long mi = m + (long long)i * RP;
        if (mi < m_end) {
          zu[i] = bu_ld_nc16(p.z + mi * C + c0);
          gu[i] = *reinterpret_cast<const uint4*>(p.g + mi * C + c0);
        }
      }
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const long long mi = m + (long long)i * RP;
        if (mi < m_end) apply(mi, zu[i], gu[i]);
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Small maps (M <= 8 x 1024 rows): channel-split, NO grid-wide barrier.  A thread-block cluster of K
// CTAs owns 8 channels (one 16-byte vector per row); CTA k takes rows [k*rows_per_cta, ...), thread t its rows
// t, t+256, ... -- at most R <= 4 per thread, loaded ONCE, all loads in flight together, and kept in registers for the
// apply.  Sums: thread -> warp shuffles ->
// shared memory -> the K CTAs' 16 partials through distributed shared memory (fp64, fixed order, every CTA
// redundantly, so that nothing has to be sent back) -> 8 threads finalize -> broadcast through shared memory.
// Two hardware cluster barriers replace the two trips through L2 atomics of the kernel above, and no CTA ever
// waits for a CTA outside its cluster.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void cluster_arrive() { asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory"); }
__device__ __forceinline__ void cluster_wait() { asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory"); }
__device__ __forceinline__ float ld_dsmem_f32(const float* local, unsigned rank) {
  const uint32_t a = (uint32_t)__cvta_generic_to_shared(local);
  uint32_t ra;
  float v;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(ra) : "r"(a), "r"(rank));
  asm volatile("ld.shared::cluster.f32 %0, [%1];" : "=f"(v) : "r"(ra) : "memory");
  return v;
}

constexpr int BC_THREADS = 256;     // lean CTAs (<= 32 K registers): they fit next to the side stream's kernels
constexpr int BC_WARPS = BC_THREADS / 32;

template <int MODE, int R>
__global__ void __launch_bounds__(BC_THREADS, 2) bn_cluster_kernel(const BnUnitParams p) {
  constexpr bool KEEP_G = (MODE == 1);
  __shared__ float wred[BC_WARPS][16];
  __shared__ float part[16];          // this CTA's sums: [0..7] s0, [8..15] s1 -- read by the whole cluster
  __shared__ double tot[16];
  __shared__ float cst[4][8];         // forward: scale, shift;  backward: ka, kb (see below)
  pdl_wait();
  pdl_launch_dependents();
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const unsigned K = gridDim.x, rank = blockIdx.x;
  const int C = p.C, c0 = blockIdx.y << 3;
  const long long m_begin = (long long)rank * p.rows_per_cta;
  const long long m_end = (m_begin + p.rows_per_cta < p.M) ? m_begin + p.rows_per_cta : p.M;

  float sc[8], sh[8], mu[8], is[8];
  if (MODE == 1) {
    bu_load8_cg(p.scale + c0, sc); bu_load8_cg(p.shift + c0, sh);
    bu_load8_cg(p.mean + c0, mu);  bu_load8_cg(p.invstd + c0, is);
  }
  // ---- load: every row of this thread at once ----
  uint4 zu[R], gu[KEEP_G ? R : 1];
#pragma unroll
  for (int i = 0; i < R; ++i) {
    const long long m = m_begin + tid + (long long)i * BC_THREADS;
    zu[i] = make_uint4(0u, 0u, 0u, 0u);
    if (m < m_end) zu[i] = bu_ld_nc16(p.z + m * C + c0);
  }
  float s0[8], s1[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) { s0[j] = 0.f; s1[j] = 0.f; }
  if constexpr (MODE == 0) {
#pragma unroll
    for (int i = 0; i < R; ++i) {
      float zf[8];
      bu_unpack8(zu[i], zf);
#pragma unroll
      for (int j = 0; j < 8; ++j) { s0[j] += zf[j]; s1[j] = fmaf(zf[j], zf[j], s1[j]); }
    }
  } else {
    constexpr int GB = R < 4 ? R : 4;      // gradient rows in flight
#pragma unroll
    for (int i0 = 0; i0 < R; i0 += GB) {
      uint4 gt[GB];
#pragma unroll
      for (int i = 0; i < GB; ++i) {
        const long long m = m_begin + tid + (long long)(i0 + i) * BC_THREADS;
        gt[i] = make_uint4(0u, 0u, 0u, 0u);
        if (m < m_end) gt[i] = bu_ld_nc16(p.g + m * C + c0);
      }
#pragma unroll
      for (int i = 0; i < GB; ++i) {
        if constexpr (KEEP_G) gu[i0 + i] = gt[i];
        float zf[8], gf[8];
        bu_unpack8(zu[i0 + i], zf);
        bu_unpack8(gt[i], gf);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float pre = __fadd_rn(__fmul_rn(zf[j], sc[j]), sh[j]);
          const float dy = (pre > 0.f) ? gf[j] : 0.f;
          const float xh = (zf[j] - mu[j]) * is[j];
          s0[j] += dy;
          s1[j] = fmaf(dy, xh, s1[j]);
        }
      }
    }
  }
  // ---- CTA sums: shuffle tree, then the 16 warps in order ----
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) {
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      s0[j] += __shfl_xor_sync(0xffffffffu, s0[j], off);
      s1[j] += __shfl_xor_sync(0xffffffffu, s1[j], off);
    }
  }
  if (lane == 0) {
#pragma unroll
    for (int j = 0; j < 8; ++j) { wred[warp][j] = s0[j]; wred[warp][8 + j] = s1[j]; }
  }
  __syncthreads();
  if (tid < 16) {
    float t = 0.f;
#pragma unroll
    for (int w = 0; w < BC_WARPS; ++w) t += wred[w][tid];
    part[tid] = t;
  }
  // ---- cluster sums through distributed shared memory ----
  cluster_arrive();
  cluster_wait();
  if (tid < 16) {
    double t = 0.0;
    for (unsigned k = 0; k < K; ++k) t += (double)ld_dsmem_f32(&part[tid], k);
    tot[tid] = t;
  }
  cluster_arrive();                     // this CTA has read its peers: they may exit (waited for at the very end)
  __syncthreads();
  if (tid < 8) {
    const int c = c0 + tid;
    const double s = tot[tid], q = tot[8 + tid];
    if (MODE == 0) {
      const double mean = s / (double)p.M;
      double var = q / (double)p.M - mean * mean;
      if (var < 0.0) var = 0.0;
      const float istd = (float)(1.0 / sqrt(var + (double)p.eps));
      const float ga = p.gamma ? p.gamma[c] : 1.f, be = p.beta ? p.beta[c] : 0.f;
      const float scl = ga * istd;
      const float sft = be - (float)mean * scl;
      cst[0][tid] = scl;
      cst[1][tid] = sft;
      if (rank == 0) {
        p.scale[c] = scl;
        p.shift[c] = sft;
        p.mean[c] = (float)mean;
        p.invstd[c] = istd;
        if (p.running_mean && p.running_var) {
          const double unbiased = (p.M > 1) ? var * (double)p.M / (double)(p.M - 1) : var;
          p.running_mean[c] = (float)((1.0 - (double)p.momentum) * (double)p.running_mean[c] + (double)p.momentum * mean);
          p.running_var[c] = (float)((1.0 - (double)p.momentum) * (double)p.running_var[c] + (double)p.momentum * unbiased);
        }
        if (tid == 0 && blockIdx.y == 0 && p.num_batches_tracked) *p.num_batches_tracked += 1;
      }
    } else {
      const float db = (float)s, dg = (float)q;
      if (rank == 0) { p.dbeta[c] = db; p.dgamma[c] = dg; }
      // dz = sc*(dy - dbeta/M - xhat*dgamma/M) regrouped as sc*dy + ka + z*kb (as bn_relu_bwd_apply_kernel)
      const float scj = __ldcg(p.scale + c), isj = __ldcg(p.invstd + c), muj = __ldcg(p.mean + c);
      const float t = scj * isj * dg * p.inv_m;
      cst[3][tid] = -t;
      cst[2][tid] = fmaf(muj, t, -(scj * db * p.inv_m));
    }
  }
  __syncthreads();
  if (p.out != nullptr) {
    if constexpr (MODE == 0) {
      float a_sc[8], a_sh[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) { a_sc[j] = cst[0][j]; a_sh[j] = cst[1][j]; }
      bool bad = false;
#pragma unroll
      for (int i = 0; i < R; ++i) {
        const long long m = m_begin + tid + (long long)i * BC_THREADS;
        if (m < m_end) {
          float zf[8], o[8];
          bu_unpack8(zu[i], zf);
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            o[j] = relu_nan(__fadd_rn(__fmul_rn(zf[j], a_sc[j]), a_sh[j]));
            bad |= (o[j] != o[j]);
          }
          *reinterpret_cast<uint4*>(p.out + m * C + c0) = bu_pack8(o);
        }
      }
      if (bad && p.nan_flag) atomicOr(p.nan_flag, SSD3D_NAN_BACKBONE);
    } else {
      float ka[8], kb[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) { ka[j] = cst[2][j]; kb[j] = cst[3][j]; }
      if constexpr (!KEEP_G) {
        // every element of g is read and (over)written by the same thread: in place is safe
#pragma unroll
        for (int i0 = 0; i0 < R; i0 += 4) {
          uint4 gt[4];
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const long long m = m_begin + tid + (long long)(i0 + i) * BC_THREADS;
            if (i0 + i < R && m < m_end) gt[i] = *reinterpret_cast<const uint4*>(p.g + m * C + c0);
          }
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const long long m = m_begin + tid + (long long)(i0 + i) * BC_THREADS;
            if (i0 + i < R && m < m_end) {
              float zf[8], gf[8], o[8];
              bu_unpack8(zu[i0 + i], zf);
              bu_unpack8(gt[i], gf);
#pragma unroll
              for (int j = 0; j < 8; ++j) {
                const float pre = __fadd_rn(__fmul_rn(zf[j], sc[j]), sh[j]);
                const float dy = (pre > 0.f) ? gf[j] : 0.f;
                o[j] = fmaf(zf[j], kb[j], fmaf(sc[j], dy, ka[j]));
              }
              *reinterpret_cast<uint4*>(p.out + m * C + c0) = bu_pack8(o);
            }
          }
        }
      } else {
#pragma unroll
        for (int i = 0; i < R; ++i) {
          const long long m = m_begin + tid + (long long)i * BC_THREADS;
          if (m < m_end) {
            float zf[8], gf[8], o[8];
            bu_unpack8(zu[i], zf);
            bu_unpack8(gu[i], gf);
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              const float pre = __fadd_rn(__fmul_rn(zf[j], sc[j]), sh[j]);
              const float dy = (pre > 0.f) ? gf[j] : 0.f;
              o[j] = fmaf(zf[j], kb[j], fmaf(sc[j], dy, ka[j]));
            }
            *reinterpret_cast<uint4*>(p.out + m * C + c0) = bu_pack8(o);
          }
        }
      }
    }
  }
  cluster_wait();                       // nobody leaves while a peer may still read its shared memory
}

// cluster plan: K CTAs per 8-channel group, at most 8 rows per thread; widen the cluster while the grid still fits
// one wave and a thread has more than one row
constexpr int BC_MAX_K = 8, BC_MAX_R = 4;
int bn_cluster_plan(long long M, int C, long long* rows_per_cta, int* R) {
  if (C <= 0 || (C & 7) || M <= 0 || M > (long long)BC_MAX_K * BC_MAX_R * BC_THREADS) return -1;
  int K = 1;
  while ((M + K - 1) / K > (long long)BC_MAX_R * BC_THREADS) K <<= 1;
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  while (K < BC_MAX_K && (C / 8) * (K * 2) <= sms && (M + K - 1) / K > BC_THREADS) K <<= 1;
  const long long rpc = (M + K - 1) / K;
  const long long r = (rpc + BC_THREADS - 1) / BC_THREADS;
  *rows_per_cta = rpc;
  *R = r <= 1 ? 1 : r <= 2 ? 2 : 4;
  return K;
}

// The grid-barrier kernel is launched COOPERATIVELY: the driver then guarantees that all CTAs are co-resident
// (and refuses grids that cannot be), also when kernels of other streams hold SMs, and two such grids of different
// streams cannot each end up half resident waiting for the other.  (No programmatic dependent launch on this one.)
template <int MODE>
cudaError_t launch_bn_unit(const BnUnitParams& p, int G, cudaStream_t st) {
  // forward only: with z AND the per-channel constants of the backward live, keeping rows spills (392 B measured)
  const bool keep = MODE == 0 && p.rows_per_cta <= 8ll * (BU_THREADS / (p.C / 8));
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((unsigned)G);
  cfg.blockDim = dim3(BU_THREADS);
  cfg.dynamicSmemBytes = 0;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeCooperative;
  attr[0].val.cooperative = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return keep ? cudaLaunchKernelEx(&cfg, bn_unit_kernel<MODE, true>, p)
              : cudaLaunchKernelEx(&cfg, bn_unit_kernel<MODE, false>, p);
}

template <int MODE, int R>
cudaError_t launch_bn_cluster(const BnUnitParams& p, int K, cudaStream_t st) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((unsigned)K, (unsigned)(p.C / 8), 1);
  cfg.blockDim = dim3(BC_THREADS);
  cfg.dynamicSmemBytes = 0;
  cfg.stream = st;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  attr[1].id = cudaLaunchAttributeClusterDimension;
  attr[1].val.clusterDim.x = (unsigned)K;
  attr[1].val.clusterDim.y = 1;
  attr[1].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 2;
  return cudaLaunchKernelEx(&cfg, bn_cluster_kernel<MODE, R>, p);
}

template <int MODE>
cudaError_t launch_bn_cluster_r(const BnUnitParams& p, int K, int R, cudaStream_t st) {
  switch (R) {
    case 1: return launch_bn_cluster<MODE, 1>(p, K, st);
    case 2: return launch_bn_cluster<MODE, 2>(p, K, st);
    default: return launch_bn_cluster<MODE, 4>(p, K, st);
  }
}

// ------------------------------------------------------------------------------------------------
// Larger maps, ONE barrier: 2-D split.  CTA (chunk i, group j) owns a contiguous row chunk x CG = 64 (or 32)
// channels -- a warp reads whole 128-byte (64-byte) row segments -- and writes its 2*CG column partials to slab
// [j][i].  The only synchronisation is between the RC CTAs of one channel group (one counter per group): after it
// EVERY CTA of the group adds the group's RC slabs itself (fp64, fixed order, all loads in flight: RC * 2*CG floats
// <= 38 KB from L2) and finalizes its CG channels redundantly, so nothing has to be published and waited for a second
// time; chunk 0 of each group writes the statistics / parameter gradients.  Against bn_unit_kernel this removes one
// grid barrier and two dependent L2 round trips per launch.  Cooperative launch as above (<= one CTA per SM).
// ------------------------------------------------------------------------------------------------
struct BnTileParams {
  BnUnitParams u;
  int CG;                 // channels per group: 64 or 32
  int RC;                 // row chunks (CTAs per group)
};

template <int MODE, bool KEEP>
__global__ void __launch_bounds__(BU_THREADS, 1) bn_tile_kernel(const BnTileParams q) {
  const BnUnitParams& p = q.u;
  __shared__ float red[BU_WARPS][8][16];          // [warp][cv of the group][s0 x8 | s1 x8]
  __shared__ double part[4][128];                 // phase 2: four slab lanes per column
  __shared__ float cst[4][64];                    // forward: scale, shift; backward: ka, kb
  pdl_wait();
  pdl_launch_dependents();
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int C = p.C, CG = q.CG, RC = q.RC;
  const int CVB = CG >> 3;                        // 16-byte vectors per row of the tile: 8 or 4
  const int RL = BU_THREADS / CVB;                // row lanes: 64 or 128
  const int grp = blockIdx.x / RC, chunk = blockIdx.x - grp * RC;
  const int cv = tid % CVB, r = tid / CVB;
  const int c0 = grp * CG + (cv << 3);
  const long long m_begin = (long long)chunk * p.rows_per_cta;
  const long long m_end = (m_begin + p.rows_per_cta < p.M) ? m_begin + p.rows_per_cta : p.M;

  float sc[8], sh[8], mu[8], is[8];
  if (MODE == 1) {
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      sc[j] = __ldg(p.scale + c0 + j); sh[j] = __ldg(p.shift + c0 + j);
      mu[j] = __ldg(p.mean + c0 + j);  is[j] = __ldg(p.invstd + c0 + j);
    }
  }
  uint4 zk[KEEP ? 8 : 1];
  // ---------------- phase 1 ----------------
  {
    float s0[8], s1[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) { s0[j] = 0.f; s1[j] = 0.f; }
    auto add_row = [&](const uint4& zu, const uint4& gu) {
      float zf[8];
      bu_unpack8(zu, zf);
      if (MODE == 0) {
#pragma unroll
        for (int j = 0; j < 8; ++j) { s0[j] += zf[j]; s1[j] = fmaf(zf[j], zf[j], s1[j]); }
      } else {
        float gf[8];
        bu_unpack8(gu, gf);
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
    if constexpr (KEEP) {
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const long long mi = m_begin + r + (long long)i * RL;
        zk[i] = make_uint4(0u, 0u, 0u, 0u);
        if (mi < m_end) zk[i] = bu_ld_nc16(p.z + mi * C + c0);
      }
#pragma unroll
      for (int i = 0; i < 8; ++i) add_row(zk[i], zk[i]);
    }
    constexpr int U = (MODE == 0) ? 8 : 4;
    for (long long m = m_begin + r; !KEEP && m < m_end; m += (long long)U * RL) {
      uint4 zu[U], gu[MODE == 1 ? U : 1];
#pragma unroll
      for (int i = 0; i < U; ++i) {
        const long long mi = m + (long long)i * RL;
        zu[i] = make_uint4(0u, 0u, 0u, 0u);
        if (mi < m_end) zu[i] = bu_ld_nc16(p.z + mi * C + c0);
      }
      if constexpr (MODE == 1) {
#pragma unroll
        for (int i = 0; i < U; ++i) {
          const long long mi = m + (long long)i * RL;
          gu[i] = make_uint4(0u, 0u, 0u, 0u);
          if (mi < m_end) gu[i] = bu_ld_nc16(p.g + mi * C + c0);
        }
      }
#pragma unroll
      for (int i = 0; i < U; ++i) {
        if constexpr (MODE == 1) add_row(zu[i], gu[i]);
        else add_row(zu[i], zu[i]);
      }
    }
    // lanes with the same cv sit CVB apart
    for (int off = CVB; off < 32; off <<= 1) {
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        s0[j] += __shfl_xor_sync(0xffffffffu, s0[j], off);
        s1[j] += __shfl_xor_sync(0xffffffffu, s1[j], off);
      }
    }
    if (lane < CVB) {
#pragma unroll
      for (int j = 0; j < 8; ++j) { red[warp][lane][j] = s0[j]; red[warp][lane][8 + j] = s1[j]; }
    }
    __syncthreads();
    if (tid < 2 * CG) {
      // column t of the slab row: [s0 of the CG channels | s1 of the CG channels]
      const int which = tid / CG, ch = tid - which * CG;
      float t = 0.f;
#pragma unroll
      for (int w = 0; w < BU_WARPS; ++w) t += red[w][ch >> 3][which * 8 + (ch & 7)];
      p.slab[((size_t)grp * RC + chunk) * 128 + tid] = t;
    }
  }
  // ---------------- the group's barrier ----------------
  bu_grid_barrier(p.sync + grp, (unsigned)RC);
  if (tid == 0) {
    // last CTA of the group to get here clears the group's two words (all have left the spin: they only leave it
    // after the counter reached RC, and each adds to the exit word afterwards)
    if (atomicAdd(p.sync + 256 + grp, 1u) == (unsigned)RC - 1) {
      p.sync[grp] = 0u;
      p.sync[256 + grp] = 0u;
      __threadfence();
    }
  }
  // ---------------- phase 2: the group's totals, in every CTA ----------------
  {
    const int col = tid & 127, ln = tid >> 7;                 // 128 columns x 4 slab lanes
    double acc = 0.0;
    if (col < 2 * CG) {
      const float* src = p.slab + (size_t)grp * RC * 128 + col;
      for (int b0 = ln; b0 < RC; b0 += 32) {                   // 8 slabs of this lane per batch, loads first
        float v[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const int b = b0 + 4 * i;
          v[i] = (b < RC) ? __ldcg(src + (size_t)b * 128) : 0.f;
        }
#pragma unroll
        for (int i = 0; i < 8; ++i) acc += (double)v[i];
      }
    }
    part[ln][col] = acc;
    __syncthreads();
    if (tid < CG) {
      const double s = part[0][tid] + part[1][tid] + part[2][tid] + part[3][tid];
      const double qq = part[0][CG + tid] + part[1][CG + tid] + part[2][CG + tid] + part[3][CG + tid];
      const int c = grp * CG + tid;
      if (MODE == 0) {
        const double mean = s / (double)p.M;
        double var = qq / (double)p.M - mean * mean;
        if (var < 0.0) var = 0.0;
        const float istd = (float)(1.0 / sqrt(var + (double)p.eps));
        const float ga = p.gamma ? p.gamma[c] : 1.f, be = p.beta ? p.beta[c] : 0.f;
        const float scl = ga * istd;
        const float sft = be - (float)mean * scl;
        cst[0][tid] = scl;
        cst[1][tid] = sft;
        if (chunk == 0) {
          p.scale[c] = scl;
          p.shift[c] = sft;
          p.mean[c] = (float)mean;
          p.invstd[c] = istd;
          if (p.running_mean && p.running_var) {
            const double unbiased = (p.M > 1) ? var * (double)p.M / (double)(p.M - 1) : var;
            p.running_mean[c] = (float)((1.0 - (double)p.momentum) * (double)p.running_mean[c] + (double)p.momentum * mean);
            p.running_var[c] = (float)((1.0 - (double)p.momentum) * (double)p.running_var[c] + (double)p.momentum * unbiased);
          }
          if (c == 0 && p.num_batches_tracked) *p.num_batches_tracked += 1;
        }
      } else {
        const float db = (float)s, dg = (float)qq;
        if (chunk == 0) { p.dbeta[c] = db; p.dgamma[c] = dg; }
        const float scj = __ldg(p.scale + c), isj = __ldg(p.invstd + c), muj = __ldg(p.mean + c);
        const float t = scj * isj * dg * p.inv_m;
        cst[3][tid] = -t;
        cst[2][tid] = fmaf(muj, t, -(scj * db * p.inv_m));
      }
    }
    __syncthreads();
  }
  if (p.out == nullptr) return;
  // ---------------- phase 3 ----------------
  const int cl = cv << 3;                                      // channel within the group
  if constexpr (MODE == 0) {
    float a_sc[8], a_sh[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) { a_sc[j] = cst[0][cl + j]; a_sh[j] = cst[1][cl + j]; }
    bool bad = false;
    auto apply = [&](long long m, const uint4& zu) {
      float zf[8], o[8];
      bu_unpack8(zu, zf);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        o[j] = relu_nan(__fadd_rn(__fmul_rn(zf[j], a_sc[j]), a_sh[j]));
        bad |= (o[j] != o[j]);
      }
      *reinterpret_cast<uint4*>(p.out + m * C + c0) = bu_pack8(o);
    };
    if constexpr (KEEP) {
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const long long mi = m_begin + r + (long long)i * RL;
        if (mi < m_end) apply(mi, zk[i]);
      }
    }
    for (long long m = m_begin + r; !KEEP && m < m_end; m += 4ll * RL) {
      uint4 zu[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const long long mi = m + (long long)i * RL;
        if (mi < m_end) zu[i] = bu_ld_nc16(p.z + mi * C + c0);
      }
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const long long mi = m + (long long)i * RL;
        if (mi < m_end) apply(mi, zu[i]);
      }
    }
    if (bad && p.nan_flag) atomicOr(p.nan_flag, SSD3D_NAN_BACKBONE);
  } else {
    float ka[8], kb[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) { ka[j] = cst[2][cl + j]; kb[j] = cst[3][cl + j]; }
    auto apply = [&](long long m, const uint4& zu, const uint4& gu) {
      float zf[8], gf[8], o[8];
      bu_unpack8(zu, zf);
      bu_unpack8(gu, gf);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float pre = __fadd_rn(__fmul_rn(zf[j], sc[j]), sh[j]);
        const float dy = (pre > 0.f) ? gf[j] : 0.f;
        o[j] = fmaf(zf[j], kb[j], fmaf(sc[j], dy, ka[j]));
      }
      *reinterpret_cast<uint4*>(p.out + m * C + c0) = bu_pack8(o);
    };
    for (long long m = m_begin + r; m < m_end; m += 4ll * RL) {
      uint4 zu[4], gu[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const long long mi = m + (long long)i * RL;
        if (mi < m_end) {
          zu[i] = bu_ld_nc16(p.z + mi * C + c0);
          gu[i] = *reinterpret_cast<const uint4*>(p.g + mi * C + c0);
        }
      }
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const long long mi = m + (long long)i * RL;
        if (mi < m_end) apply(mi, zu[i], gu[i]);
      }
    }
  }
}

// tile plan: CG = 64 (32 when C is an odd multiple of 32), RC chunks per group with NG * RC <= SMs
int bn_tile_plan(long long M, int C, BnTileParams* q) {
  if (C <= 0 || (C % 32) || M <= 0) return -1;
  const int CG = (C % 64 == 0) ? 64 : 32;
  const int NG = C / CG;
  int dev = 0, sms = 0;
  cudaGetDevice(&dev);
  if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms <= 0) return -1;
  if (NG > sms || NG > 256) return -1;
  const int RL = BU_THREADS / (CG / 8);
  long long rc = sms / NG;
  const long long by_rows = (M + RL * 4 - 1) / (RL * 4);      // at least four rows per row lane
  if (rc > by_rows) rc = by_rows;
  if (rc < 1) rc = 1;
  const long long rpc = (M + rc - 1) / rc;
  q->u.rows_per_cta = rpc;
  q->CG = CG;
  q->RC = (int)((M + rpc - 1) / rpc);
  return NG * q->RC;
}

template <int MODE>
cudaError_t launch_bn_tile(const BnTileParams& q, int G, cudaStream_t st) {
  const bool keep = MODE == 0 && q.u.rows_per_cta <= 8ll * (BU_THREADS / (q.CG / 8));
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((unsigned)G);
  cfg.blockDim = dim3(BU_THREADS);
  cfg.dynamicSmemBytes = 0;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeCooperative;
  attr[0].val.cooperative = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return keep ? cudaLaunchKernelEx(&cfg, bn_tile_kernel<MODE, true>, q)
              : cudaLaunchKernelEx(&cfg, bn_tile_kernel<MODE, false>, q);
}

// grid: every CTA gets at least four rows per row lane; never more CTAs than SMs (all must be resident)
int bn_unit_plan(long long M, int C, long long* rows_per_cta) {
  const int CV = C / 8;
  if (C <= 0 || (C & 7) || CV < 4 || CV > BU_THREADS || (CV & (CV - 1))) return -1;
  const int RP = BU_THREADS / CV;
  int dev = 0, sms = 0;
  cudaGetDevice(&dev);
  if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms <= 0) return -1;
  long long G = (M + RP * 4 - 1) / (RP * 4);
  if (G > sms) G = sms;
  if (G > 256) G = 256;            // phase 2 holds at most 8 slabs per lane
  if (G < 1) G = 1;
  const long long rpc = (M + G - 1) / G;
  *rows_per_cta = rpc;
  return (int)((M + rpc - 1) / rpc);
}

}  // namespace
}  // namespace ssd3d

using namespace ssd3d;

// A launch the driver REFUSES (cooperative grid larger than what can be co-resident on this context -- MPS / green
// contexts with fewer SMs --, cluster shape not schedulable, ...) has not run anything: clear the error and report
// "unsupported", so that the caller takes the three-launch passes of train.cu instead of failing.
static int bn_launch_result(cudaError_t e) {
  if (e == cudaSuccess) return SSD3D_OK;
  if (e == cudaErrorCooperativeLaunchTooLarge || e == cudaErrorLaunchOutOfResources || e == cudaErrorNotSupported ||
      e == cudaErrorInvalidClusterSize || e == cudaErrorInvalidConfiguration) {
    (void)cudaGetLastError();
    return SSD3D_ERR_UNSUPPORTED;
  }
  return (int)e;
}

extern "C" int ssd3d_bn_unit_supported(int64_t M, int C) {
  long long rpc;
  int R;
  if (M <= 0) return 0;
  if (bn_cluster_plan(M, C, &rpc, &R) > 0) return 1;
  return bn_unit_plan(M, C, &rpc) > 0 ? 1 : 0;
}

extern "C" int64_t ssd3d_bn_unit_workspace_bytes(int C) {
  const int64_t unit = (int64_t)256 * 2 * C * 4, tile = (int64_t)256 * 128 * 4;    // slabs of either kernel
  return unit > tile ? unit : tile;
}

extern "C" int ssd3d_bn_unit_fwd(const void* z, int64_t M, int C, const float* gamma, const float* beta, float eps,
                                 float momentum, float* running_mean, float* running_var,
                                 int64_t* num_batches_tracked, float* scale, float* shift, float* mean, float* invstd,
                                 void* a, int* nan_flag, void* workspace, int64_t workspace_bytes, uint32_t* sync_words,
                                 void* stream) {
  if (!z || !scale || !shift || !mean || !invstd || !workspace || !sync_words || M <= 0) return SSD3D_ERR_ARG;
  BnUnitParams p{};
  int R = 0;
  const int K = bn_cluster_plan(M, C, &p.rows_per_cta, &R);
  const int G = K > 0 ? 0 : bn_unit_plan(M, C, &p.rows_per_cta);
  if (G < 0 || workspace_bytes < (int64_t)G * 2 * C * 4) return SSD3D_ERR_ARG;
  p.z = static_cast<const bf16*>(z);
  p.out = static_cast<bf16*>(a);
  p.M = M; p.C = C;
  p.slab = static_cast<float*>(workspace);
  p.sync = sync_words;
  p.gamma = gamma; p.beta = beta; p.eps = eps; p.momentum = momentum;
  p.running_mean = running_mean; p.running_var = running_var;
  p.num_batches_tracked = reinterpret_cast<long long*>(num_batches_tracked);
  p.nan_flag = nan_flag;
  p.scale = scale; p.shift = shift; p.mean = mean; p.invstd = invstd;
  if (K > 0) {
    const cudaError_t e = launch_bn_cluster_r<0>(p, K, R, static_cast<cudaStream_t>(stream));
    return bn_launch_result(e);
  }
  BnTileParams q{};
  q.u = p;
  const int GT = bn_tile_plan(M, C, &q);
  if (GT > 0 && workspace_bytes >= (int64_t)GT * 128 * 4) {
    const cudaError_t e = launch_bn_tile<0>(q, GT, static_cast<cudaStream_t>(stream));
    return bn_launch_result(e);
  }
  const cudaError_t e = launch_bn_unit<0>(p, G, static_cast<cudaStream_t>(stream));
  return bn_launch_result(e);
}

extern "C" int ssd3d_bn_unit_bwd(const void* z, const void* grad_a, int64_t M, int C, const float* scale,
                                 const float* shift, const float* mean, const float* invstd, float* dgamma,
                                 float* dbeta, void* dz, void* workspace, int64_t workspace_bytes, uint32_t* sync_words,
                                 void* stream) {
  // dz == NULL: statistics only (dgamma, dbeta) -- the caller applies the backward elsewhere (ssd3d_stem_wgrad_bn)
  if (!z || !grad_a || !scale || !shift || !mean || !invstd || !dgamma || !dbeta || !workspace || !sync_words || M <= 0)
    return SSD3D_ERR_ARG;
  BnUnitParams p{};
  int R = 0;
  const int K = bn_cluster_plan(M, C, &p.rows_per_cta, &R);
  const int G = K > 0 ? 0 : bn_unit_plan(M, C, &p.rows_per_cta);
  if (G < 0 || workspace_bytes < (int64_t)G * 2 * C * 4) return SSD3D_ERR_ARG;
  p.z = static_cast<const bf16*>(z);
  p.g = static_cast<const bf16*>(grad_a);
  p.out = static_cast<bf16*>(dz);
  p.M = M; p.C = C;
  p.slab = static_cast<float*>(workspace);
  p.sync = sync_words;
  p.scale = const_cast<float*>(scale); p.shift = const_cast<float*>(shift);
  p.mean = const_cast<float*>(mean); p.invstd = const_cast<float*>(invstd);
  p.dgamma = dgamma; p.dbeta = dbeta;
  p.inv_m = (float)(1.0 / (double)M);
  if (K > 0) {
    const cudaError_t e = launch_bn_cluster_r<1>(p, K, R, static_cast<cudaStream_t>(stream));
    return bn_launch_result(e);
  }
  BnTileParams q{};
  q.u = p;
  const int GT = bn_tile_plan(M, C, &q);
  if (GT > 0 && workspace_bytes >= (int64_t)GT * 128 * 4) {
    const cudaError_t e = launch_bn_tile<1>(q, GT, static_cast<cudaStream_t>(stream));
    return bn_launch_result(e);
  }
  const cudaError_t e = launch_bn_unit<1>(p, G, static_cast<cudaStream_t>(stream));
  return bn_launch_result(e);
}
