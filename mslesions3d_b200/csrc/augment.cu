// Training batches from a device-resident data set (sampling + augmentation), and the packing of their ground truth
// into the static buffers of the captured training step.  Every step of an epoch runs in one CUDA-graph replay:
// nothing here reads a host scalar that changes between steps.
//
// ssd3d_augment_batch: slot b of the batch takes subject order[(step*N*world + rank*N + b) mod S]
// (DistributedSampler's split, the last batch wraps around) and draws, from Philox4x32-10 with
// key = seed and counter = (global slot rank*N + b, draw counter low, draw counter high, call):
//   call 0: {positive crop u, box pick, rot90 u, rot90 k}   call 1: {crop offset d, h, w, -}
//   call 2: {flip d, h, w, -}                               call 3: {scale u, shift u, -, -}
//   u01(u) = (u >> 8) * 2^-24, a Bernoulli(p) draw is u01 < p, randint(lo, hi) = lo + ((u * (hi - lo)) >> 32)
// then applies crop -> rot90 (np.rot90 semantics) -> flips (np.flip) -> y = x * (1 + f) + o (two fp32 roundings,
// then bf16 round to nearest) to the image and the crop -> rot90 -> flips to the mask.  The geometry is one signed
// axis permutation plus an offset, so the source address of an output voxel is linear in its index: the kernel
// walks output tiles of 32 (W) x 32 (the output axis that reads source W, or H) through shared memory -- reads run
// along the source's contiguous axis, writes are 16-byte stores along the output's.  The last block to finish
// advances the draw counter and the step, so consecutive replays draw fresh batches.
#include "common.cuh"
#include "philox.cuh"

namespace ssd3d {

constexpr int AUG_T = 32;        // output tile: AUG_T (the tile axis) x AUG_T (W)
constexpr int AUG_YB = 8;        // planes of the remaining axis per block

struct AugArgs {
  int S, C, Ds, Hs, Ws, N, d, h, w, ra0, ra1, X;      // X: the tile axis (0 or 1), the same for every draw
  float pos_ratio, flip_prob, rot90_prob, scale, shift;
};

__device__ __forceinline__ float u01(uint32_t u) { return (float)(u >> 8) * (1.f / 16777216.f); }

// the draws of slot b into rec[16] (layout in include/ssd3d_b200.h)
__device__ void aug_draw(const AugArgs& a, const long long* __restrict__ state, const int* __restrict__ order,
                         const int* __restrict__ boxes, const int* __restrict__ box_off, int b, int* rec) {
  const unsigned long long seed = (unsigned long long)state[0], ctr = (unsigned long long)state[1];
  const long long step = state[2], rank = state[3], world = state[4];
  const uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
  const long long g = rank * a.N + b;
  const int subj = order[(int)((step * a.N * world + g) % a.S)];
  Philox4 r[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) r[i] = philox4x32_10((uint32_t)g, (uint32_t)ctr, (uint32_t)(ctr >> 32), (uint32_t)i, k0, k1);
  const int b0 = box_off[subj], nb = box_off[subj + 1] - b0;
  const bool pos = nb > 0 && u01(r[0].v[0]) < a.pos_ratio;
  const int box = pos ? randint_ms(r[0].v[1], 0, nb) : -1;
  const int src[3] = {a.Ds, a.Hs, a.Ws}, out[3] = {a.d, a.h, a.w};
  rec[0] = subj;
#pragma unroll
  for (int ax = 0; ax < 3; ++ax) {
    int lo = 0, hi = src[ax] - out[ax];
    if (pos) {
      const int bl = boxes[(b0 + box) * 6 + ax], bh = boxes[(b0 + box) * 6 + 3 + ax];
      if (bh - bl + 1 <= out[ax]) {                    // every window that contains the whole box
        lo = max(0, bh - out[ax] + 1);
        hi = min(bl, src[ax] - out[ax]);
      } else {                                         // box larger than the window: windows holding its centre
        const int c = (bl + bh) / 2;
        lo = max(0, c - out[ax] + 1);
        hi = min(c, src[ax] - out[ax]);
      }
    }
    rec[1 + ax] = randint_ms(r[1].v[ax], lo, hi + 1);
    rec[5 + ax] = u01(r[2].v[ax]) < a.flip_prob ? 1 : 0;
  }
  rec[4] = u01(r[0].v[2]) < a.rot90_prob ? randint_ms(r[0].v[3], 1, 4) : 0;
  rec[8] = pos ? 1 : 0;
  rec[9] = box;
  const float f = __fmul_rn(a.scale, __fsub_rn(__fmul_rn(2.f, u01(r[3].v[0])), 1.f));
  const float o = __fmul_rn(a.shift, __fsub_rn(__fmul_rn(2.f, u01(r[3].v[1])), 1.f));
  rec[10] = __float_as_int(f);
  rec[11] = __float_as_int(o);
  rec[12] = (int)step;
  rec[13] = (int)(uint32_t)ctr;
  rec[14] = (int)g;
  rec[15] = nb;
}

// the geometry of record rec as a signed permutation: crop axis c takes output axis q[c], reversed or not -- rot90
// first (np.rot90 on the crop), then the flips of the output axes
__device__ __forceinline__ void aug_perm(const AugArgs& a, const int* rec, int* q, int* rev) {
  q[0] = 0; q[1] = 1; q[2] = 2;
  int r[3] = {0, 0, 0};
  const int k = rec[4], a0 = a.ra0, a1 = a.ra1;
  if (k == 1) { q[a0] = a1; q[a1] = a0; r[a1] = 1; }
  else if (k == 2) { r[a0] = 1; r[a1] = 1; }
  else if (k == 3) { q[a0] = a1; q[a1] = a0; r[a0] = 1; }
#pragma unroll
  for (int c = 0; c < 3; ++c) rev[c] = r[c] ^ rec[5 + q[c]];
}

// every block has read the state (before its own increment below): the last one advances it for the next batch
__device__ __forceinline__ void aug_advance_state(long long* state) {
  __threadfence();
  const unsigned long long total = (unsigned long long)gridDim.x * gridDim.y * gridDim.z;
  if (atomicAdd(reinterpret_cast<unsigned long long*>(state + 5), 1ull) == total - 1) {
    state[1] += 1;
    state[2] += 1;
    state[5] = 0;
    __threadfence();
  }
}

// grid: (tiles over (tile axis, W), AUG_YB-plane groups of the remaining axis, N); 256 threads
template <typename TIn>
__global__ void __launch_bounds__(256) augment_kernel(AugArgs a, const TIn* __restrict__ src,
                                                      const uint8_t* __restrict__ masks, const int* __restrict__ order,
                                                      long long* __restrict__ state, const int* __restrict__ boxes,
                                                      const int* __restrict__ box_off, __nv_bfloat16* __restrict__ out,
                                                      uint8_t* __restrict__ out_mask, int* __restrict__ record) {
  __shared__ int rec[16];
  __shared__ long long s_base, s_coef[3];
  __shared__ float tile[AUG_T][AUG_T + 1];
  __shared__ __align__(16) uint8_t mtile[AUG_T][AUG_T + 16];
  const int tid = threadIdx.x, b = blockIdx.z;
  const int ext[3] = {a.d, a.h, a.w};
  if (tid == 0) {
    aug_draw(a, state, order, boxes, box_off, b, rec);
    int q[3], rev[3];
    aug_perm(a, rec, q, rev);
    const long long ss[3] = {(long long)a.Hs * a.Ws, (long long)a.Ws, 1};
    long long base = 0;
    for (int c = 0; c < 3; ++c) {
      base += (long long)(rec[1 + c] + (rev[c] ? ext[q[c]] - 1 : 0)) * ss[c];
      s_coef[q[c]] = rev[c] ? -ss[c] : ss[c];
    }
    s_base = base;
    if (blockIdx.x == 0 && blockIdx.y == 0) for (int i = 0; i < 16; ++i) record[b * 16 + i] = rec[i];
  }
  __syncthreads();
  const int X = a.X, Y = 1 - a.X, ext_x = X ? a.h : a.d;
  const bool along_x = s_coef[X] == 1 || s_coef[X] == -1;    // source W is read along the tile axis
  const int tiles_w = (a.w + AUG_T - 1) / AUG_T;
  const int tx = blockIdx.x / tiles_w, tw = blockIdx.x % tiles_w, ext_y = Y ? a.h : a.d;
  const long long vox_s = (long long)a.Ds * a.Hs * a.Ws, vox_o = (long long)a.d * a.h * a.w;
  const long long cx = s_coef[X], cw = s_coef[2];
  const float scale1 = __fadd_rn(1.f, __int_as_float(rec[10])), shift = __int_as_float(rec[11]);
  // output index of the tile row x: y * stride(Y) + x * stride(X)
  const long long str_x = X ? a.w : (long long)a.h * a.w, str_y = Y ? a.w : (long long)a.h * a.w;
  // AUG_YB planes of the remaining axis per block: the draws and the setup above are paid once for all of them
  for (int y = blockIdx.y * AUG_YB; y < min(ext_y, (int)(blockIdx.y + 1) * AUG_YB); ++y) {
    const long long mbase = (long long)rec[0] * vox_s + s_base + (long long)y * s_coef[Y];
    const long long sbase = mbase + (long long)rec[0] * (a.C - 1) * vox_s;
    const long long obase = (long long)y * str_y + (long long)tx * AUG_T * str_x + (long long)tw * AUG_T;
    for (int c = 0; c < a.C; ++c) {
      const TIn* sc = src + sbase + (long long)c * vox_s;
#pragma unroll
      for (int it = 0; it < AUG_T * AUG_T / 256; ++it) {
        const int idx = it * 256 + tid;
        const int x = along_x ? (idx & (AUG_T - 1)) : idx / AUG_T, wl = along_x ? idx / AUG_T : (idx & (AUG_T - 1));
        const int ox = tx * AUG_T + x, ow = tw * AUG_T + wl;
        if (ox < ext_x && ow < a.w) {
          const long long s = (long long)ox * cx + (long long)ow * cw;
          tile[x][wl] = (float)sc[s];
          if (c == 0) mtile[x][wl] = masks[mbase + s];
        }
      }
      __syncthreads();
      if (tid < AUG_T * AUG_T / 8) {                           // 8 bf16 = one 16-byte store per thread
        const int x = tid / (AUG_T / 8), w0 = (tid % (AUG_T / 8)) * 8;
        if (tx * AUG_T + x < ext_x && tw * AUG_T + w0 < a.w) {
          uint32_t pk[4];
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const float v0 = __fadd_rn(__fmul_rn(tile[x][w0 + 2 * j], scale1), shift);
            const float v1 = __fadd_rn(__fmul_rn(tile[x][w0 + 2 * j + 1], scale1), shift);
            const __nv_bfloat162 p = __halves2bfloat162(__float2bfloat16_rn(v0), __float2bfloat16_rn(v1));
            pk[j] = *reinterpret_cast<const uint32_t*>(&p);
          }
          __nv_bfloat16* dst = out + ((long long)b * a.C + c) * vox_o + obase + (long long)x * str_x + w0;
          *reinterpret_cast<uint4*>(dst) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
        }
      } else if (c == 0 && tid < AUG_T * AUG_T / 8 + AUG_T * AUG_T / 16) {   // 16 mask bytes per thread
        const int t = tid - AUG_T * AUG_T / 8;
        const int x = t / (AUG_T / 16), w0 = (t % (AUG_T / 16)) * 16;
        if (tx * AUG_T + x < ext_x && tw * AUG_T + w0 < a.w)
          *reinterpret_cast<uint4*>(out_mask + (long long)b * vox_o + obase + (long long)x * str_x + w0) =
              *reinterpret_cast<const uint4*>(&mtile[x][w0]);
      }
      __syncthreads();
    }
  }
  if (tid == 0) aug_advance_state(state);
}

constexpr int AFF_TW = 64;       // output tile of one warp: AFF_TW (W) x 4 (H) of one D plane; 8 voxels per lane
constexpr int AFF_WARPS = 4;     // warps per block = D planes per tile
constexpr int AFF_DB = 4;        // tiles along D per block (the draws are paid once for all of them)

struct AffArgs {
  float prob, rot[3], zoom[3];
};

// words 16..31 of slot b's record: affine drawn, theta, z, M (layout in include/ssd3d_b200.h)
__device__ void affine_draw(const AugArgs& a, const AffArgs& f, const long long* __restrict__ state, int b,
                            int* rec) {
  const unsigned long long seed = (unsigned long long)state[0], ctr = (unsigned long long)state[1];
  const uint32_t g = (uint32_t)(state[3] * a.N + b), k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
  const Philox4 r4 = philox4x32_10(g, (uint32_t)ctr, (uint32_t)(ctr >> 32), 4u, k0, k1);
  const Philox4 r5 = philox4x32_10(g, (uint32_t)ctr, (uint32_t)(ctr >> 32), 5u, k0, k1);
  const bool on = u01(r4.v[0]) < f.prob;
  float th[3] = {0.f, 0.f, 0.f}, z[3] = {1.f, 1.f, 1.f}, M[3][3] = {{1.f, 0.f, 0.f}, {0.f, 1.f, 0.f}, {0.f, 0.f, 1.f}};
  if (on) {
    float s[3], c[3];
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      th[i] = __fmul_rn(f.rot[i], __fsub_rn(__fmul_rn(2.f, u01(r4.v[1 + i])), 1.f));
      z[i] = __fadd_rn(1.f, __fmul_rn(f.zoom[i], __fsub_rn(__fmul_rn(2.f, u01(r5.v[i])), 1.f)));
      sincosf(th[i], &s[i], &c[i]);
    }
    // R0 in the (h, w) plane, R1 in (d, w), R2 in (d, h): R[lo][lo] = R[hi][hi] = cos, R[lo][hi] = -sin, R[hi][lo] = sin
    const float R0[3][3] = {{1.f, 0.f, 0.f}, {0.f, c[0], -s[0]}, {0.f, s[0], c[0]}};
    const float R1[3][3] = {{c[1], 0.f, -s[1]}, {0.f, 1.f, 0.f}, {s[1], 0.f, c[1]}};
    const float R2[3][3] = {{c[2], -s[2], 0.f}, {s[2], c[2], 0.f}, {0.f, 0.f, 1.f}};
    float T[3][3];
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
      for (int j = 0; j < 3; ++j)
        T[i][j] = __fadd_rn(__fadd_rn(__fmul_rn(R0[i][0], R1[0][j]), __fmul_rn(R0[i][1], R1[1][j])),
                            __fmul_rn(R0[i][2], R1[2][j]));
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
      for (int j = 0; j < 3; ++j)
        M[i][j] = __fdiv_rn(__fadd_rn(__fadd_rn(__fmul_rn(T[i][0], R2[0][j]), __fmul_rn(T[i][1], R2[1][j])),
                                      __fmul_rn(T[i][2], R2[2][j])), z[j]);
  }
  rec[16] = on ? 1 : 0;
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    rec[17 + i] = __float_as_int(th[i]);
    rec[20 + i] = __float_as_int(z[i]);
  }
#pragma unroll
  for (int i = 0; i < 9; ++i) rec[23 + i] = __float_as_int(M[i / 3][i % 3]);
}

// fp32_rn(fp32_rn(v0 * (1 - t)) + fp32_rn(v1 * t)), omt = fp32_rn(1 - t)
__device__ __forceinline__ float aff_lerp(float v0, float v1, float t, float omt) {
  return __fadd_rn(__fmul_rn(v0, omt), __fmul_rn(v1, t));
}

constexpr int ELA_GMAX = 16;    // control points per crop axis, at most
constexpr int ELA_DROW = AFF_TW + 8;   // a row of the warp's field table (the pad keeps the 4 rows' lanes apart)

struct ElaArgs {
  float prob, m[3], r[3];        // r_c = fp32_rn((G_c - 3) / (n_c - 1)), 0 when n_c = 1
  int G[3], gmax;                // gmax = max G_c: the stride of the shared tables
};

// dynamic shared memory of the field, in floats: s_v (4 rows x K x L x 3), s_t (per warp 4 rows x L x 3), s_d (per
// warp 3 components x 4 rows x ELA_DROW), then the 4 rows' R weights and intervals
__host__ __device__ __forceinline__ int ela_smem_floats(int gmax) {
  return 4 * gmax * gmax * 3 + AFF_WARPS * 4 * gmax * 3 + AFF_WARPS * 3 * 4 * ELA_DROW + 4 * 4 + 4;
}

__device__ __forceinline__ int sel3(int c, int v0, int v1, int v2) { return c == 0 ? v0 : (c == 1 ? v1 : v2); }
__device__ __forceinline__ float sel3f(int c, float v0, float v1, float v2) { return c == 0 ? v0 : (c == 1 ? v1 : v2); }

// the cubic B-spline interval and weights of crop index p on an axis with inverse spacing r and G control points:
// t = fp32_rn(p * r), j = min(floor(t), G - 4), f = t - j (exact), w = {h(1 - f), c(f), c(1 - f), h(f)} with
// h(x) = x^3 / 6 and c(x) = x^3 / 2 - x^2 + 2 / 3, every operation rounded as written in include/ssd3d_b200.h
__device__ __forceinline__ float bspline_h(float x) {
  return __fmul_rn(__fmul_rn(__fmul_rn(x, x), x), 1.f / 6.f);
}
__device__ __forceinline__ float bspline_c(float x) {
  const float x2 = __fmul_rn(x, x);
  return __fadd_rn(__fsub_rn(__fmul_rn(0.5f, __fmul_rn(x2, x)), x2), 2.f / 3.f);
}
__device__ __forceinline__ int bspline_j(int p, float r, int G) {
  return min((int)floorf(__fmul_rn((float)p, r)), G - 4);
}
__device__ __forceinline__ int bspline_w(int p, float r, int G, float* w) {
  const float t = __fmul_rn((float)p, r);
  const int j = min((int)floorf(t), G - 4);
  const float f = __fsub_rn(t, (float)j), g = __fsub_rn(1.f, f);
  w[0] = bspline_h(g);
  w[1] = bspline_c(f);
  w[2] = bspline_c(g);
  w[3] = bspline_h(f);
  return j;
}

// word 32 of slot b's record: whether the slot draws the field (Philox call 6)
__device__ __forceinline__ int elastic_drawn(const AugArgs& a, const ElaArgs& e, const long long* __restrict__ state,
                                             int b) {
  const unsigned long long seed = (unsigned long long)state[0], ctr = (unsigned long long)state[1];
  const uint32_t g = (uint32_t)(state[3] * a.N + b);
  const Philox4 r6 = philox4x32_10(g, (uint32_t)ctr, (uint32_t)(ctr >> 32), 6u, (uint32_t)seed, (uint32_t)(seed >> 32));
  return u01(r6.v[0]) < e.prob ? 1 : 0;
}

// grid: (W tiles x H tiles of 4, groups of AFF_DB * AFF_WARPS D planes, N); 32 * AFF_WARPS threads.  Warp wz of
// the block computes output plane od = (blockIdx.y * AFF_DB + it) * AFF_WARPS + wz, rows oh = tile_h * 4 + lane / 8,
// voxels ow = tile_w * AFF_TW + j * 8 + lane % 8 (adjacent lanes read adjacent source voxels when M is near the
// identity); results go through shared memory so that each lane stores 8 consecutive W voxels (one 16-byte bf16
// store per channel, one 8-byte mask store).
//
// ELASTIC (ssd3d_augment_elastic_batch) adds the B-spline displacement to the crop coordinate before M.  The crop
// axes read from output D, H and W (K, R and L below) follow from the slot's rot90 permutation; a block's output box
// spans 16 D planes, 4 H rows and 64 W voxels, so it touches at most G control points per axis.  The block draws
// those once and contracts R (s_v: 4 rows x K x L x 3); each warp contracts its plane's K per iteration (s_t: 4 rows
// x L x 3) and then sums 4 L taps per component for its 4 x 64 voxels (s_d), which the voxel loop adds to u.  That
// nesting is the summation order the header states.  The tables are dynamic shared memory and e is the last
// parameter, so the ELASTIC = false instantiation compiles to the same code as before the field existed.
// (ELASTIC: at least 6 blocks per SM, which holds it to 77 registers without spills; 96 unbounded)
template <typename TIn, bool ELASTIC>
__global__ void __launch_bounds__(32 * AFF_WARPS, ELASTIC ? 6 : 0) augment_affine_kernel(
    AugArgs a, AffArgs f, const TIn* __restrict__ src, const uint8_t* __restrict__ masks,
    const int* __restrict__ order, long long* __restrict__ state, const int* __restrict__ boxes,
    const int* __restrict__ box_off, __nv_bfloat16* __restrict__ out, uint8_t* __restrict__ out_mask,
    int* __restrict__ record, ElaArgs e) {
  constexpr int RW = ELASTIC ? 33 : 32;                                   // record words
  extern __shared__ float s_ela[];                                        // ELASTIC: ela_smem_floats(e.gmax)
  const int gs = e.gmax;
  float* s_v = s_ela;
  float* s_t = s_v + 4 * gs * gs * 3;
  float* s_d = s_t + AFF_WARPS * 4 * gs * 3;
  float* s_wR = s_d + AFF_WARPS * 3 * 4 * ELA_DROW;
  int* s_jR = reinterpret_cast<int*>(s_wR + 16);
  __shared__ int rec[RW];
  __shared__ int s_q[3], s_rev[3];
  __shared__ __align__(16) __nv_bfloat16 s_img[AFF_WARPS][4][AFF_TW];
  __shared__ __align__(16) uint8_t s_msk[AFF_WARPS][4][AFF_TW];
  const int tid = threadIdx.x, b = blockIdx.z, lane = tid & 31, wz = tid >> 5, tx = lane & 7, ty = lane >> 3;
  if (tid == 0) {
    aug_draw(a, state, order, boxes, box_off, b, rec);
    affine_draw(a, f, state, b, rec);
    if constexpr (ELASTIC) rec[32] = elastic_drawn(a, e, state, b);
    int q[3], rev[3];
    aug_perm(a, rec, q, rev);
    for (int c = 0; c < 3; ++c) { s_q[c] = q[c]; s_rev[c] = rev[c]; }
    if (blockIdx.x == 0 && blockIdx.y == 0) for (int i = 0; i < RW; ++i) record[b * RW + i] = rec[i];
  }
  __syncthreads();
  const int ext[3] = {a.d, a.h, a.w}, srcx[3] = {a.Ds, a.Hs, a.Ws};
  float M[3][3], half[3], cen[3];
  int q[3], rev[3];
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    q[c] = s_q[c];
    rev[c] = s_rev[c];
    half[c] = __fmul_rn(0.5f, (float)(ext[c] - 1));                       // (n_c - 1) / 2, exact
    cen[c] = __fadd_rn((float)rec[1 + c], half[c]);                       // o_c + (n_c - 1) / 2, exact
#pragma unroll
    for (int j = 0; j < 3; ++j) M[c][j] = __int_as_float(rec[23 + c * 3 + j]);
  }
  const int subj = rec[0];
  const float scale1 = __fadd_rn(1.f, __int_as_float(rec[10])), shift = __int_as_float(rec[11]);
  const int plane = a.Hs * a.Ws;
  const long long vox_s = (long long)a.Ds * plane, vox_o = (long long)a.d * a.h * a.w;
  const uint8_t* msrc = masks + (long long)subj * vox_s;
  const TIn* isrc = src + (long long)subj * a.C * vox_s;
  const int tiles_w = (a.w + AFF_TW - 1) / AFF_TW;
  const int oh = (blockIdx.x / tiles_w) * 4 + ty, ow_t = (blockIdx.x % tiles_w) * AFF_TW;
  // the field's per-block set-up (ELASTIC, slot draws it): crop axes cK, cR, cL read from output D, H, W
  bool el_on = false;
  int revK = 0, revL = 0, GK = 4, GL = 4, kK0 = 0, kL0 = 0, nL = 4;
  float rK = 0.f, rL = 0.f;
  if constexpr (ELASTIC) {
    el_on = rec[32] != 0;
    if (el_on) {
      const int cK = q[0] == 0 ? 0 : (q[1] == 0 ? 1 : 2), cR = q[0] == 1 ? 0 : (q[1] == 1 ? 1 : 2), cL = 3 - cK - cR;
      const int revR = sel3(cR, rev[0], rev[1], rev[2]), GR = sel3(cR, e.G[0], e.G[1], e.G[2]);
      const float rR = sel3f(cR, e.r[0], e.r[1], e.r[2]);
      revK = sel3(cK, rev[0], rev[1], rev[2]);
      revL = sel3(cL, rev[0], rev[1], rev[2]);
      GK = sel3(cK, e.G[0], e.G[1], e.G[2]);
      GL = sel3(cL, e.G[0], e.G[1], e.G[2]);
      rK = sel3f(cK, e.r[0], e.r[1], e.r[2]);
      rL = sel3f(cL, e.r[0], e.r[1], e.r[2]);
      // the block's output box, clamped to the output; crop index p = rev ? n - 1 - o : o (n_c = ext of the output
      // axis it reads: rot90 only swaps axes of equal extent), so the touched control points are [j(lo), j(hi) + 3]
      const int od0 = blockIdx.y * AFF_DB * AFF_WARPS, od1 = min(od0 + AFF_DB * AFF_WARPS, a.d) - 1;
      const int oh0 = (blockIdx.x / tiles_w) * 4, oh1 = min(oh0 + 4, a.h) - 1, ow1 = min(ow_t + AFF_TW, a.w) - 1;
      kK0 = bspline_j(revK ? a.d - 1 - od1 : od0, rK, GK);
      const int nK = bspline_j(revK ? a.d - 1 - od0 : od1, rK, GK) + 4 - kK0;
      const int kR0 = bspline_j(revR ? a.h - 1 - oh1 : oh0, rR, GR);
      const int nR = bspline_j(revR ? a.h - 1 - oh0 : oh1, rR, GR) + 4 - kR0;
      kL0 = bspline_j(revL ? a.w - 1 - ow1 : ow_t, rL, GL);
      nL = bspline_j(revL ? a.w - 1 - ow_t : ow1, rL, GL) + 4 - kL0;
      if (tid < 4) {                                                      // the 4 rows' R weights
        const int o = min(oh0 + tid, oh1);
        s_jR[tid] = bspline_w(revR ? a.h - 1 - o : o, rR, GR, s_wR + tid * 4);
      }
      __syncthreads();
      const int G1 = e.G[1], G2 = e.G[2];
      const int sK = sel3(cK, G1 * G2, G2, 1), sR = sel3(cR, G1 * G2, G2, 1), sL = sel3(cL, G1 * G2, G2, 1);
      // the state is read here by every thread: it cannot advance before this block has finished (aug_advance_state)
      const unsigned long long seed = (unsigned long long)state[0], ctr = (unsigned long long)state[1];
      const uint32_t g = (uint32_t)(state[3] * a.N + b), k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
      for (int i = tid; i < nK * nL; i += 32 * AFF_WARPS) {
        const int kk = i / nL, kl = i % nL;
        float acc[4][3];
#pragma unroll
        for (int r = 0; r < 4; ++r)
#pragma unroll
          for (int c = 0; c < 3; ++c) acc[r][c] = 0.f;
        for (int kr = kR0; kr < kR0 + nR; ++kr) {
          // control point k of the slot: Philox call 7 + k, displacement {d, h, w} = m * (2 u01 - 1)
          const uint32_t k = (uint32_t)((kK0 + kk) * sK + kr * sR + (kL0 + kl) * sL);
          const Philox4 pr = philox4x32_10(g, (uint32_t)ctr, (uint32_t)(ctr >> 32), 7u + k, k0, k1);
          float dl[3];
#pragma unroll
          for (int c = 0; c < 3; ++c) dl[c] = __fmul_rn(e.m[c], __fsub_rn(__fmul_rn(2.f, u01(pr.v[c])), 1.f));
#pragma unroll
          for (int r = 0; r < 4; ++r) {
            const int bb = kr - s_jR[r];
            if (bb >= 0 && bb < 4) {
              const float wb = s_wR[r * 4 + bb];
#pragma unroll
              for (int c = 0; c < 3; ++c) acc[r][c] = __fadd_rn(acc[r][c], __fmul_rn(wb, dl[c]));
            }
          }
        }
#pragma unroll
        for (int r = 0; r < 4; ++r)
#pragma unroll
          for (int c = 0; c < 3; ++c) s_v[((r * gs + kk) * gs + kl) * 3 + c] = acc[r][c];
      }
      __syncthreads();                                                    // block-uniform: el_on is the slot's
    }
  }
  for (int it = 0; it < AFF_DB; ++it) {
    const int od = (blockIdx.y * AFF_DB + it) * AFF_WARPS + wz;
    if (od >= a.d) break;                                                 // warp-uniform
    if constexpr (ELASTIC) {
      if (el_on) {                                                        // this plane's K contraction
        float wK[4];
        const int jK = bspline_w(revK ? a.d - 1 - od : od, rK, GK, wK) - kK0;
        for (int i = lane; i < 4 * nL; i += 32) {
          const int r = i / nL, kl = i % nL;
#pragma unroll
          for (int c = 0; c < 3; ++c) {
            float s = 0.f;
#pragma unroll
            for (int ai = 0; ai < 4; ++ai)
              s = __fadd_rn(s, __fmul_rn(wK[ai], s_v[((r * gs + jK + ai) * gs + kl) * 3 + c]));
            s_t[((wz * 4 + r) * gs + kl) * 3 + c] = s;
          }
        }
        __syncwarp();
        // the field of the warp's 4 x 64 voxels: 4 L taps per component (voxels past the output take the last one's)
        for (int i = lane; i < 4 * AFF_TW; i += 32) {
          const int r = i / AFF_TW, ol = i % AFF_TW, ow = min(ow_t + ol, a.w - 1);
          float wL[4];
          const int jl = bspline_w(revL ? a.w - 1 - ow : ow, rL, GL, wL) - kL0;
          const float* tr = s_t + ((wz * 4 + r) * gs + jl) * 3;
#pragma unroll
          for (int c = 0; c < 3; ++c) {
            float s = 0.f;
#pragma unroll
            for (int ei = 0; ei < 4; ++ei) s = __fadd_rn(s, __fmul_rn(wL[ei], tr[ei * 3 + c]));
            s_d[((wz * 3 + c) * 4 + r) * ELA_DROW + ol] = s;
          }
        }
        __syncwarp();
      }
    }
    const bool row = oh < a.h;
    const bool store = row && ow_t + tx * 8 < a.w;
    const long long obase = (long long)od * a.h * a.w + (long long)oh * a.w + ow_t + tx * 8;
    // the coordinates are recomputed per channel: cheaper than holding 8 voxels' taps and weights in registers
    for (int ch = 0; ch < a.C; ++ch) {
      const TIn* sc = isrc + (long long)ch * vox_s;
#pragma unroll 4
      for (int j = 0; j < 8; ++j) {
        const int o[3] = {od, oh, ow_t + j * 8 + tx};
        const bool live = row && o[2] < a.w;
        float u[3];
#pragma unroll
        for (int c = 0; c < 3; ++c) {
          const int oq = o[q[c]];
          u[c] = __fsub_rn((float)(rev[c] ? ext[c] - 1 - oq : oq), half[c]);
        }
        if constexpr (ELASTIC) {
          if (el_on) {                                                    // u += the field
            const float* dr = s_d + (wz * 12 + ty) * ELA_DROW + j * 8 + tx;
#pragma unroll
            for (int c = 0; c < 3; ++c) u[c] = __fadd_rn(u[c], dr[c * 4 * ELA_DROW]);
          }
        }
        int i0[3], nn[3];
        bool lo[3], hi[3];
        float t[3];
#pragma unroll
        for (int c = 0; c < 3; ++c) {
          const float x = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(M[c][0], u[0]), __fmul_rn(M[c][1], u[1])),
                                              __fmul_rn(M[c][2], u[2])), cen[c]);
          const float fl = floorf(x);
          i0[c] = (int)fl;
          t[c] = __fsub_rn(x, fl);
          nn[c] = (int)floorf(__fadd_rn(x, 0.5f));
          lo[c] = i0[c] >= 0 && i0[c] < srcx[c];                           // tap i0 inside the source
          hi[c] = i0[c] >= -1 && i0[c] < srcx[c] - 1;                      // tap i0 + 1 inside the source
        }
        if (ch == 0) {
          const bool in = live && nn[0] >= 0 && nn[0] < a.Ds && nn[1] >= 0 && nn[1] < a.Hs && nn[2] >= 0 &&
                          nn[2] < a.Ws;
          s_msk[wz][ty][j * 8 + tx] = in ? __ldg(msrc + (nn[0] * a.Hs + nn[1]) * a.Ws + nn[2]) : (uint8_t)0;
        }
        const int base = (i0[0] * a.Hs + i0[1]) * a.Ws + i0[2];
        float v[8];                                                         // taps (dd, dh, dw), dw fastest
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          const int dd = k >> 2, dh = (k >> 1) & 1, dw = k & 1;
          const bool ok = live && (dd ? hi[0] : lo[0]) && (dh ? hi[1] : lo[1]) && (dw ? hi[2] : lo[2]);
          v[k] = ok ? (float)__ldg(sc + base + dd * plane + dh * a.Ws + dw) : 0.f;
        }
        const float mw = __fsub_rn(1.f, t[2]), mh = __fsub_rn(1.f, t[1]), md = __fsub_rn(1.f, t[0]);
        const float c00 = aff_lerp(v[0], v[1], t[2], mw), c01 = aff_lerp(v[2], v[3], t[2], mw);
        const float c10 = aff_lerp(v[4], v[5], t[2], mw), c11 = aff_lerp(v[6], v[7], t[2], mw);
        const float val = aff_lerp(aff_lerp(c00, c01, t[1], mh), aff_lerp(c10, c11, t[1], mh), t[0], md);
        s_img[wz][ty][j * 8 + tx] = __float2bfloat16_rn(__fadd_rn(__fmul_rn(val, scale1), shift));
      }
      __syncwarp();
      if (store) {
        *reinterpret_cast<uint4*>(out + ((long long)b * a.C + ch) * vox_o + obase) =
            *reinterpret_cast<const uint4*>(&s_img[wz][ty][tx * 8]);
        if (ch == 0)
          *reinterpret_cast<uint2*>(out_mask + b * vox_o + obase) =
              *reinterpret_cast<const uint2*>(&s_msk[wz][ty][tx * 8]);
      }
      __syncwarp();
    }
  }
  if (tid == 0) aug_advance_state(state);
}

// MR intensity augmentation (ssd3d_augment_intensity_batch): gamma, bias field and Gaussian noise, a point-wise pass
// in place over the bf16 batch the augment kernels above have written.  Two launches: intensity_slot_kernel draws
// every slot's values into the record and, when gamma_prob > 0, the per-(slot, chunk) min / max partials of the
// slots that draw gamma; intensity_voxel_kernel reduces those partials per block in a fixed order and streams 16-byte
// bf16 vectors.  Every draw is a pure function of (seed, draw counter, global slot, voxel index).
constexpr int INT_WORDS = 27;                   // record words per slot (layout in include/ssd3d_b200.h)
constexpr int INT_NCOEF = 20;                   // monomials u_d^i u_h^j u_w^k, i + j + k <= 3
constexpr uint32_t INT_CALL_SLOT = 1u << 16;    // per-slot draws: Philox calls 2^16 + j
constexpr uint32_t INT_CALL_NOISE = 1u << 24;   // noise: call 2^24 + q for the voxel quad q of the slot
constexpr int INT_CHUNK = 16384;                // bf16 values per min / max partial: 256 threads x 8 16-byte vectors
constexpr int INT_VPT = 4;                      // 8-voxel vectors per thread of the per-voxel pass

struct IntArgs {
  int N, C, d, h, w, chunks;                    // chunks: partials per slot, 0 when gamma_prob == 0
  float bias_prob, bias_coef, gamma_prob, gamma_log_range, noise_prob, noise_std;
  float su[2], ou[2];                           // u = fp32_rn(fp32_rn(p * su) - ou) on d and h (su = ou = 0: n = 1)
  float sw;                                     // the same on w (w >= 16)
};

// Philox4x32-10 of global slot g at the draw counter the preceding augment launch consumed (state[1] - 1)
__device__ __forceinline__ Philox4 int_philox(const long long* __restrict__ state, uint32_t g, uint32_t call) {
  const unsigned long long seed = (unsigned long long)state[0], ctr = (unsigned long long)state[1] - 1ull;
  return philox4x32_10(g, (uint32_t)ctr, (uint32_t)(ctr >> 32), call, (uint32_t)seed, (uint32_t)(seed >> 32));
}

__device__ __forceinline__ uint32_t int_slot(const IntArgs& a, const long long* __restrict__ state, int b) {
  return (uint32_t)(state[3] * a.N + b);
}

// the draws of slot b into rec[INT_WORDS]; lo and hi (words 4, 5) are left 0 for the per-voxel pass
__device__ void intensity_draw(const IntArgs& a, const long long* __restrict__ state, int b, int* rec) {
  const uint32_t g = int_slot(a, state, b);
  const Philox4 r0 = int_philox(state, g, INT_CALL_SLOT), r1 = int_philox(state, g, INT_CALL_SLOT + 1u);
  const bool gon = u01(r0.v[0]) < a.gamma_prob, bon = u01(r0.v[1]) < a.bias_prob, non = u01(r0.v[2]) < a.noise_prob;
  float gamma = 1.f, sigma = 0.f;
  if (gon) gamma = expf(__fmul_rn(a.gamma_log_range, __fsub_rn(__fmul_rn(2.f, u01(r0.v[3])), 1.f)));
  if (non) sigma = __fmul_rn(a.noise_std, u01(r1.v[0]));
  rec[0] = gon ? 1 : 0;
  rec[1] = bon ? 1 : 0;
  rec[2] = non ? 1 : 0;
  rec[3] = __float_as_int(gamma);
  rec[4] = 0;
  rec[5] = 0;
  rec[6] = __float_as_int(sigma);
  for (int q = 0; q < INT_NCOEF / 4; ++q) {
    const Philox4 rc = int_philox(state, g, INT_CALL_SLOT + 2u + (uint32_t)q);
#pragma unroll
    for (int e = 0; e < 4; ++e)
      rec[7 + q * 4 + e] =
          __float_as_int(bon ? __fmul_rn(a.bias_coef, __fsub_rn(__fmul_rn(2.f, u01(rc.v[e])), 1.f)) : 0.f);
  }
}

// grid: (max(chunks, 1), N); 256 threads.  Block (0, b) writes slot b's record; with chunks > 0 block (k, b) of a
// slot that draws gamma writes the min and max of the slot's bf16 values [k, k + 1) * INT_CHUNK (all channels)
__global__ void __launch_bounds__(256) intensity_slot_kernel(IntArgs a, const __nv_bfloat16* __restrict__ img,
                                                             const long long* __restrict__ state,
                                                             int* __restrict__ record, float2* __restrict__ partial) {
  __shared__ float s_lo[8], s_hi[8];
  const int b = blockIdx.y, tid = threadIdx.x;
  if (blockIdx.x == 0 && tid == 0) {
    int rec[INT_WORDS];
    intensity_draw(a, state, b, rec);
    for (int i = 0; i < INT_WORDS; ++i) record[b * INT_WORDS + i] = rec[i];
  }
  if (a.chunks == 0 || !(u01(int_philox(state, int_slot(a, state, b), INT_CALL_SLOT).v[0]) < a.gamma_prob)) return;
  const long long n = (long long)a.C * a.d * a.h * a.w;
  const uint4* src = reinterpret_cast<const uint4*>(img + (long long)b * n);
  const long long v1 = min((long long)(blockIdx.x + 1) * (INT_CHUNK / 8), n / 8);
  const __nv_bfloat162 inf2 = __floats2bfloat162_rn(INFINITY, INFINITY);
  __nv_bfloat162 lo2 = inf2, hi2 = __hneg2(inf2);
  for (long long v = (long long)blockIdx.x * (INT_CHUNK / 8) + tid; v < v1; v += 256) {
    const uint4 q = src[v];
    const uint32_t u[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const __nv_bfloat162 p = *reinterpret_cast<const __nv_bfloat162*>(&u[j]);
      lo2 = __hmin2(lo2, p);
      hi2 = __hmax2(hi2, p);
    }
  }
  float lo = fminf(__low2float(lo2), __high2float(lo2)), hi = fmaxf(__low2float(hi2), __high2float(hi2));
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    lo = fminf(lo, __shfl_xor_sync(0xffffffffu, lo, o));
    hi = fmaxf(hi, __shfl_xor_sync(0xffffffffu, hi, o));
  }
  if ((tid & 31) == 0) { s_lo[tid >> 5] = lo; s_hi[tid >> 5] = hi; }
  __syncthreads();
  if (tid == 0) {
    for (int i = 1; i < 8; ++i) { lo = fminf(lo, s_lo[i]); hi = fmaxf(hi, s_hi[i]); }
    partial[(long long)b * a.chunks + blockIdx.x] = make_float2(lo, hi);
  }
}

// the standard normals of the 8 voxels [i, i + 8) of a slot (i = c * d * h * w + 8 * vector, a multiple of 8): voxel
// quad q takes Philox call 2^24 + q, and Box-Muller on words (0, 1) and (2, 3) gives its voxels {r cos, r sin} each
__device__ __forceinline__ void int_normals(const long long* __restrict__ state, uint32_t g, uint32_t quad, float* n) {
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    const Philox4 r = int_philox(state, g, INT_CALL_NOISE + quad + (uint32_t)h);
#pragma unroll
    for (int p = 0; p < 2; ++p) {
      const float u1 = (float)((r.v[2 * p] >> 8) + 1u) * (1.f / 16777216.f);     // (0, 1]: the log is finite
      const float u2 = u01(r.v[2 * p + 1]);                                       // [0, 1)
      const float rad = sqrtf(__fmul_rn(-2.f, logf(u1)));
      float s, c;
      sincospif(__fmul_rn(2.f, u2), &s, &c);
      n[h * 4 + p * 2] = __fmul_rn(rad, c);
      n[h * 4 + p * 2 + 1] = __fmul_rn(rad, s);
    }
  }
}

// grid: (ceil(d * h * w / 8 / (256 * INT_VPT)), N); 256 threads, each INT_VPT vectors of 8 W voxels, every channel
__global__ void __launch_bounds__(256) intensity_voxel_kernel(IntArgs a, __nv_bfloat16* __restrict__ img,
                                                              const long long* __restrict__ state,
                                                              int* __restrict__ record,
                                                              const float2* __restrict__ partial) {
  __shared__ int s_rec[INT_WORDS];
  __shared__ float s_lohi[2];
  const int b = blockIdx.y, tid = threadIdx.x;
  if (tid < INT_WORDS) s_rec[tid] = record[b * INT_WORDS + tid];
  __syncthreads();
  const bool gon = s_rec[0] != 0, bon = s_rec[1] != 0, non = s_rec[2] != 0;
  if (!gon && !bon && !non) return;                                       // block-uniform: the slot draws nothing
  if (gon) {                                                              // lo, hi: min / max of the partials
    if (tid < 32) {
      float lo = INFINITY, hi = -INFINITY;
      for (int i = tid; i < a.chunks; i += 32) {
        const float2 p = partial[(long long)b * a.chunks + i];
        lo = fminf(lo, p.x);
        hi = fmaxf(hi, p.y);
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        lo = fminf(lo, __shfl_xor_sync(0xffffffffu, lo, o));
        hi = fmaxf(hi, __shfl_xor_sync(0xffffffffu, hi, o));
      }
      if (tid == 0) {
        s_lohi[0] = lo;
        s_lohi[1] = hi;
        if (blockIdx.x == 0) {
          record[b * INT_WORDS + 4] = __float_as_int(lo);
          record[b * INT_WORDS + 5] = __float_as_int(hi);
        }
      }
    }
    __syncthreads();
  }
  const float gamma = __int_as_float(s_rec[3]), sigma = __int_as_float(s_rec[6]);
  const float lo = gon ? s_lohi[0] : 0.f, hi = gon ? s_lohi[1] : 0.f;
  const bool g_act = gon && gamma != 1.f && hi != lo, n_act = non && sigma != 0.f;
  if (!g_act && !bon && !n_act) return;                                   // zero strengths: the identity
  const float r = __fsub_rn(hi, lo), rinv = g_act ? __frcp_rn(r) : 0.f;
  float cf[INT_NCOEF];
#pragma unroll
  for (int i = 0; i < INT_NCOEF; ++i) cf[i] = __int_as_float(s_rec[7 + i]);
  const uint32_t g = int_slot(a, state, b);
  const int wv = a.w / 8;
  const long long vox = (long long)a.d * a.h * a.w, nvec = vox / 8;
  __nv_bfloat16* base = img + (long long)b * a.C * vox;
  // 32-bit index arithmetic: d h w / 8 < 2^31 (the entry point bounds C d h w / 4 by 2^32)
  const unsigned nvec32 = (unsigned)nvec, hh = (unsigned)a.h;
#pragma unroll 1
  for (int k = 0; k < INT_VPT; ++k) {
    const unsigned v = (blockIdx.x * INT_VPT + k) * 256u + tid;
    if (v >= nvec32) break;
    const unsigned row = v / (unsigned)wv, zz = row / hh;
    const int x0 = (int)(v - row * wv) * 8, z = (int)zz, y = (int)(row - zz * hh);
    float field[8];
    if (bon) {
      // the row's cubic in u_w: a_k = sum over (i, j) in coefficient order of c_ijk * (u_d^i u_h^j)
      const float ud = __fsub_rn(__fmul_rn((float)z, a.su[0]), a.ou[0]);
      const float uh = __fsub_rn(__fmul_rn((float)y, a.su[1]), a.ou[1]);
      const float pd[4] = {1.f, ud, __fmul_rn(ud, ud), __fmul_rn(__fmul_rn(ud, ud), ud)};
      const float ph[4] = {1.f, uh, __fmul_rn(uh, uh), __fmul_rn(__fmul_rn(uh, uh), uh)};
      float ak[4] = {0.f, 0.f, 0.f, 0.f};
      int idx = 0;
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4 - i; ++j)
#pragma unroll
          for (int kk = 0; kk < 4 - i - j; ++kk)
            ak[kk] = __fadd_rn(ak[kk], __fmul_rn(cf[idx++], __fmul_rn(pd[i], ph[j])));
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const float uw = __fsub_rn(__fmul_rn((float)(x0 + e), a.sw), 1.f);
        const float p = __fadd_rn(__fmul_rn(__fadd_rn(__fmul_rn(__fadd_rn(__fmul_rn(ak[3], uw), ak[2]), uw), ak[1]),
                                            uw), ak[0]);
        field[e] = __expf(p);
      }
    }
#pragma unroll 1
    for (int c = 0; c < a.C; ++c) {
      uint4* ptr = reinterpret_cast<uint4*>(base + (long long)c * vox) + v;
      const uint4 q = *ptr;
      uint32_t u[4] = {q.x, q.y, q.z, q.w};
      float nz[8];
      if (n_act) int_normals(state, g, (uint32_t)(((long long)c * vox + (long long)v * 8) >> 2), nz);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float2 f = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u[j]));
        float x[2] = {f.x, f.y};
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          if (g_act) {
            const float t = fminf(__fmul_rn(__fsub_rn(x[e], lo), rinv), 1.f);
            x[e] = __fadd_rn(lo, __fmul_rn(r, exp2f(__fmul_rn(gamma, __log2f(t)))));
          }
          if (bon) x[e] = __fmul_rn(x[e], field[2 * j + e]);
          if (n_act) x[e] = __fadd_rn(x[e], __fmul_rn(sigma, nz[2 * j + e]));
        }
        const __nv_bfloat162 o = __floats2bfloat162_rn(x[0], x[1]);
        u[j] = *reinterpret_cast<const uint32_t*>(&o);
      }
      *ptr = make_uint4(u[0], u[1], u[2], u[3]);
    }
  }
}

// one block: per-volume overflow test, offsets (exclusive scan of the counts) and the row copy
__global__ void __launch_bounds__(256) gt_pack_kernel(const float* __restrict__ boxes, const long long* __restrict__ labels,
                                                      const int* __restrict__ counts, const int* __restrict__ n_comp,
                                                      int N, int max_boxes, int per_volume, float* __restrict__ gt_boxes,
                                                      long long* __restrict__ gt_labels, int* __restrict__ offsets,
                                                      int* __restrict__ status) {
  extern __shared__ int s_off[];
  __shared__ int s_bad;
  if (threadIdx.x == 0) s_bad = 0;
  __syncthreads();
  for (int i = threadIdx.x; i < N; i += blockDim.x)
    if (n_comp[i] > max_boxes || counts[i] > per_volume) atomicOr(&s_bad, 1);
  __syncthreads();
  const int bad = s_bad;
  if (threadIdx.x == 0) {
    int o = 0;
    for (int i = 0; i < N; ++i) { s_off[i] = o; o += bad ? 0 : counts[i]; }
    s_off[N] = o;
    status[0] = bad;
    if (bad) status[1] += 1;
  }
  __syncthreads();
  for (int i = threadIdx.x; i <= N; i += blockDim.x) offsets[i] = s_off[i];
  if (bad) return;
  for (int t = threadIdx.x; t < N * max_boxes; t += blockDim.x) {
    const int i = t / max_boxes, r = t % max_boxes;
    if (r >= counts[i]) continue;
    const long long dst = s_off[i] + r;
#pragma unroll
    for (int j = 0; j < 6; ++j) gt_boxes[dst * 6 + j] = boxes[(long long)t * 6 + j];
    gt_labels[dst] = labels[t];
  }
}

}  // namespace ssd3d

using namespace ssd3d;

// the argument checks shared by ssd3d_augment_batch and ssd3d_augment_affine_batch
static int aug_check(const void* src, const uint8_t* masks, const int32_t* order, const int64_t* state,
                     const int32_t* boxes, const int32_t* box_offsets, const void* out, const uint8_t* out_mask,
                     const int32_t* record, int S, int C, int Ds, int Hs, int Ws, int N, int d, int h, int w,
                     float pos_ratio, float flip_prob, float rot90_prob, int rot_axis0, int rot_axis1, float scale,
                     float shift) {
  if (!src || !masks || !order || !state || !boxes || !box_offsets || !out || !out_mask || !record) return SSD3D_ERR_ARG;
  if (S <= 0 || C <= 0 || N <= 0 || d <= 0 || h <= 0 || w <= 0 || d > Ds || h > Hs || w > Ws) return SSD3D_ERR_ARG;
  if (!(pos_ratio >= 0.f && pos_ratio <= 1.f) || !(flip_prob >= 0.f && flip_prob <= 1.f) ||
      !(rot90_prob >= 0.f && rot90_prob <= 1.f) || !(scale >= 0.f) || !(shift >= 0.f))
    return SSD3D_ERR_ARG;
  if (rot_axis0 < 0 || rot_axis0 > 2 || rot_axis1 < 0 || rot_axis1 > 2 || rot_axis0 == rot_axis1) return SSD3D_ERR_ARG;
  const int ext[3] = {d, h, w};
  if (rot90_prob > 0.f && ext[rot_axis0] != ext[rot_axis1]) return SSD3D_ERR_ARG;
  if (w % 16 != 0 || (long long)Ds * Hs * Ws >= (1ll << 31) || h > 65535 || d > 65535) return SSD3D_ERR_UNSUPPORTED;
  return SSD3D_OK;
}

// the affine arguments of ssd3d_augment_affine_batch and ssd3d_augment_elastic_batch
static int aff_check(float affine_prob, const float* rotate_range, const float* zoom_range, AffArgs* f) {
  if (!rotate_range || !zoom_range || !(affine_prob >= 0.f && affine_prob <= 1.f)) return SSD3D_ERR_ARG;
  *f = AffArgs{affine_prob, {0.f, 0.f, 0.f}, {0.f, 0.f, 0.f}};
  for (int i = 0; i < 3; ++i) {
    // the negated comparisons also refuse NaN; fp32(pi) = 3.14159274f (rounded up) is accepted
    if (!(rotate_range[i] >= 0.f && rotate_range[i] <= 3.14159274f) || !(zoom_range[i] >= 0.f && zoom_range[i] < 1.f))
      return SSD3D_ERR_ARG;
    f->rot[i] = rotate_range[i];
    f->zoom[i] = zoom_range[i];
  }
  return SSD3D_OK;
}

// the launch of augment_affine_kernel<TIn, ELASTIC> shared by ssd3d_augment_affine_batch and ssd3d_augment_elastic_batch
template <bool ELASTIC>
static int aff_launch(const AugArgs& a, const AffArgs& f, const ElaArgs& e, const void* src, int src_is_bf16,
                      const uint8_t* masks, const int32_t* order, int64_t* state, const int32_t* boxes,
                      const int32_t* box_offsets, void* out, uint8_t* out_mask, int32_t* record, void* stream) {
  const dim3 grid((unsigned)(((a.w + AFF_TW - 1) / AFF_TW) * ((a.h + 3) / 4)),
                  (unsigned)((a.d + AFF_DB * AFF_WARPS - 1) / (AFF_DB * AFF_WARPS)), (unsigned)a.N);
  const size_t smem = ELASTIC ? (size_t)ela_smem_floats(e.gmax) * sizeof(float) : 0;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (src_is_bf16)
    augment_affine_kernel<__nv_bfloat16, ELASTIC><<<grid, 32 * AFF_WARPS, smem, st>>>(
        a, f, static_cast<const __nv_bfloat16*>(src), masks, order, reinterpret_cast<long long*>(state), boxes,
        box_offsets, static_cast<__nv_bfloat16*>(out), out_mask, record, e);
  else
    augment_affine_kernel<float, ELASTIC><<<grid, 32 * AFF_WARPS, smem, st>>>(
        a, f, static_cast<const float*>(src), masks, order, reinterpret_cast<long long*>(state), boxes, box_offsets,
        static_cast<__nv_bfloat16*>(out), out_mask, record, e);
  SSD3D_CHECK_LAUNCH();
  return SSD3D_OK;
}

extern "C" int ssd3d_augment_affine_batch(const void* src, int src_is_bf16, const uint8_t* masks, int S, int C, int Ds,
                                          int Hs, int Ws, const int32_t* order, int64_t* state, const int32_t* boxes,
                                          const int32_t* box_offsets, int N, int d, int h, int w, float pos_ratio,
                                          float flip_prob, float rot90_prob, int rot_axis0, int rot_axis1, float scale,
                                          float shift, float affine_prob, const float* rotate_range,
                                          const float* zoom_range, void* out, uint8_t* out_mask, int32_t* record,
                                          void* stream) {
  const int rc = aug_check(src, masks, order, state, boxes, box_offsets, out, out_mask, record, S, C, Ds, Hs, Ws, N, d,
                           h, w, pos_ratio, flip_prob, rot90_prob, rot_axis0, rot_axis1, scale, shift);
  if (rc != SSD3D_OK) return rc;
  AffArgs f;
  if (aff_check(affine_prob, rotate_range, zoom_range, &f) != SSD3D_OK) return SSD3D_ERR_ARG;
  const AugArgs a{S, C, Ds, Hs, Ws, N, d, h, w, rot_axis0, rot_axis1, 1, pos_ratio, flip_prob, rot90_prob, scale, shift};
  return aff_launch<false>(a, f, ElaArgs{}, src, src_is_bf16, masks, order, state, boxes, box_offsets, out, out_mask, record,
                         stream);
}

extern "C" int ssd3d_augment_elastic_batch(const void* src, int src_is_bf16, const uint8_t* masks, int S, int C, int Ds,
                                           int Hs, int Ws, const int32_t* order, int64_t* state, const int32_t* boxes,
                                           const int32_t* box_offsets, int N, int d, int h, int w, float pos_ratio,
                                           float flip_prob, float rot90_prob, int rot_axis0, int rot_axis1,
                                           float scale, float shift, float affine_prob, const float* rotate_range,
                                           const float* zoom_range, float elastic_prob, const int32_t* elastic_points,
                                           const float* elastic_magnitude, void* out, uint8_t* out_mask,
                                           int32_t* record, void* stream) {
  int rc = aug_check(src, masks, order, state, boxes, box_offsets, out, out_mask, record, S, C, Ds, Hs, Ws, N, d, h, w,
                     pos_ratio, flip_prob, rot90_prob, rot_axis0, rot_axis1, scale, shift);
  if (rc != SSD3D_OK) return rc;
  AffArgs f;
  if ((rc = aff_check(affine_prob, rotate_range, zoom_range, &f)) != SSD3D_OK) return rc;
  if (!elastic_points || !elastic_magnitude || !(elastic_prob >= 0.f && elastic_prob <= 1.f)) return SSD3D_ERR_ARG;
  ElaArgs e{elastic_prob, {0.f, 0.f, 0.f}, {0.f, 0.f, 0.f}, {4, 4, 4}, 4};
  const int ext[3] = {d, h, w};
  for (int c = 0; c < 3; ++c) {
    const int G = elastic_points[c];
    const float m = elastic_magnitude[c];
    if (G < 4 || G > ELA_GMAX || !(m >= 0.f && m <= 3.40282347e38f)) return SSD3D_ERR_ARG;
    // |delta| <= m < 0.4 s keeps the cubic B-spline warp injective (Choi & Lee 2000: s / 2.48)
    if (m > 0.f && (double)m >= 0.4 * (double)(ext[c] - 1) / (double)(G - 3)) return SSD3D_ERR_ARG;
    e.G[c] = G;
    e.gmax = max(e.gmax, G);
    e.m[c] = m;
    e.r[c] = ext[c] > 1 ? (float)(G - 3) / (float)(ext[c] - 1) : 0.f;     // one correctly rounded fp32 division
  }
  const AugArgs a{S, C, Ds, Hs, Ws, N, d, h, w, rot_axis0, rot_axis1, 1, pos_ratio, flip_prob, rot90_prob, scale, shift};
  return aff_launch<true>(a, f, e, src, src_is_bf16, masks, order, state, boxes, box_offsets, out, out_mask, record,
                         stream);
}

extern "C" int ssd3d_augment_batch(const void* src, int src_is_bf16, const uint8_t* masks, int S, int C, int Ds, int Hs,
                                   int Ws, const int32_t* order, int64_t* state, const int32_t* boxes,
                                   const int32_t* box_offsets, int N, int d, int h, int w, float pos_ratio,
                                   float flip_prob, float rot90_prob, int rot_axis0, int rot_axis1, float scale,
                                   float shift, void* out, uint8_t* out_mask, int32_t* record, void* stream) {
  const int rc = aug_check(src, masks, order, state, boxes, box_offsets, out, out_mask, record, S, C, Ds, Hs, Ws, N, d,
                           h, w, pos_ratio, flip_prob, rot90_prob, rot_axis0, rot_axis1, scale, shift);
  if (rc != SSD3D_OK) return rc;
  const int ext[3] = {d, h, w};
  // Source W is read along output W, or -- after a rotation in a plane holding W -- along that plane's other
  // axis, which then is the tile axis for every draw (the planes' extents are equal, so the grid is the same)
  const int X = rot90_prob > 0.f && rot_axis0 == 2 ? rot_axis1 : (rot90_prob > 0.f && rot_axis1 == 2 ? rot_axis0 : 1);
  AugArgs a{S, C, Ds, Hs, Ws, N, d, h, w, rot_axis0, rot_axis1, X, pos_ratio, flip_prob, rot90_prob, scale, shift};
  const dim3 grid((unsigned)(((ext[X] + AUG_T - 1) / AUG_T) * ((w + AUG_T - 1) / AUG_T)),
                  (unsigned)((ext[1 - X] + AUG_YB - 1) / AUG_YB), (unsigned)N);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (src_is_bf16)
    augment_kernel<__nv_bfloat16><<<grid, 256, 0, st>>>(a, static_cast<const __nv_bfloat16*>(src), masks, order, reinterpret_cast<long long*>(state),
                                                        boxes, box_offsets, static_cast<__nv_bfloat16*>(out), out_mask,
                                                        record);
  else
    augment_kernel<float><<<grid, 256, 0, st>>>(a, static_cast<const float*>(src), masks, order, reinterpret_cast<long long*>(state), boxes,
                                                box_offsets, static_cast<__nv_bfloat16*>(out), out_mask, record);
  SSD3D_CHECK_LAUNCH();
  return SSD3D_OK;
}

static long long int_chunks(int C, int d, int h, int w) {
  return ((long long)C * d * h * w + INT_CHUNK - 1) / INT_CHUNK;
}

extern "C" int64_t ssd3d_augment_intensity_workspace_bytes(int N, int C, int d, int h, int w) {
  if (N <= 0 || C <= 0 || d <= 0 || h <= 0 || w <= 0) return 0;
  return (int64_t)N * int_chunks(C, d, h, w) * (int64_t)sizeof(float2);
}

extern "C" int ssd3d_augment_intensity_batch(void* image, int N, int C, int d, int h, int w, const int64_t* state,
                                             float bias_prob, float bias_coefficient, float gamma_prob,
                                             float gamma_log_range, float noise_prob, float noise_std,
                                             int32_t* record, void* workspace, int64_t workspace_bytes,
                                             void* stream) {
  if (!image || !state || !record) return SSD3D_ERR_ARG;
  if (N <= 0 || C <= 0 || d <= 0 || h <= 0 || w <= 0 || w % 16 != 0) return SSD3D_ERR_ARG;
  // the negated comparisons also refuse NaN
  if (!(bias_prob >= 0.f && bias_prob <= 1.f) || !(gamma_prob >= 0.f && gamma_prob <= 1.f) ||
      !(noise_prob >= 0.f && noise_prob <= 1.f) || !(bias_coefficient >= 0.f && bias_coefficient <= 1.f) ||
      !(gamma_log_range >= 0.f && gamma_log_range < 1.f) || !(noise_std >= 0.f && noise_std <= 3.40282347e38f))
    return SSD3D_ERR_ARG;
  const long long chunks = int_chunks(C, d, h, w);
  if (gamma_prob > 0.f && (!workspace || workspace_bytes < (int64_t)N * chunks * (int64_t)sizeof(float2)))
    return SSD3D_ERR_ARG;
  // noise call numbers 2^24 + quad stay below 2^32; N is the grid's y extent
  const long long vox = (long long)d * h * w;
  if (N > 65535 || (long long)C * vox / 4 > (1ll << 32) - (1ll << 24)) return SSD3D_ERR_UNSUPPORTED;
  IntArgs a{N, C, d, h, w, gamma_prob > 0.f ? (int)chunks : 0, bias_prob, bias_coefficient, gamma_prob,
            gamma_log_range, noise_prob, noise_std, {0.f, 0.f}, {0.f, 0.f}, 2.f / (float)(w - 1)};
  const int ext[2] = {d, h};
  for (int i = 0; i < 2; ++i)
    if (ext[i] > 1) { a.su[i] = 2.f / (float)(ext[i] - 1); a.ou[i] = 1.f; }    // one correctly rounded division
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  intensity_slot_kernel<<<dim3((unsigned)(a.chunks > 0 ? a.chunks : 1), (unsigned)N), 256, 0, st>>>(
      a, static_cast<const __nv_bfloat16*>(image), reinterpret_cast<const long long*>(state), record,
      static_cast<float2*>(workspace));
  SSD3D_CHECK_LAUNCH();
  const long long blocks = (vox / 8 + 256 * INT_VPT - 1) / (256 * INT_VPT);
  intensity_voxel_kernel<<<dim3((unsigned)blocks, (unsigned)N), 256, 0, st>>>(
      a, static_cast<__nv_bfloat16*>(image), reinterpret_cast<const long long*>(state), record,
      static_cast<const float2*>(workspace));
  SSD3D_CHECK_LAUNCH();
  return SSD3D_OK;
}

extern "C" int ssd3d_gt_pack(const float* boxes, const int64_t* labels, const int32_t* counts,
                             const int32_t* n_components, int N, int max_boxes, int per_volume, float* gt_boxes,
                             int64_t* gt_labels, int32_t* offsets, int32_t* status, void* stream) {
  if (!boxes || !labels || !counts || !n_components || !gt_boxes || !gt_labels || !offsets || !status) return SSD3D_ERR_ARG;
  if (N <= 0 || N > 8192 || max_boxes <= 0 || per_volume <= 0) return SSD3D_ERR_ARG;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  gt_pack_kernel<<<1, 256, (size_t)(N + 1) * 4, st>>>(boxes, reinterpret_cast<const long long*>(labels), counts,
                                                      n_components, N, max_boxes, per_volume, gt_boxes,
                                                      reinterpret_cast<long long*>(gt_labels), offsets, status);
  SSD3D_CHECK_LAUNCH();
  return SSD3D_OK;
}
