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
    // crop axis c takes output axis q[c], reversed or not: rot90 first (np.rot90 on the crop), then the flips of
    // the output axes
    int q[3] = {0, 1, 2}, rev[3] = {0, 0, 0};
    const int k = rec[4], a0 = a.ra0, a1 = a.ra1;
    if (k == 1) { q[a0] = a1; q[a1] = a0; rev[a1] = 1; }
    else if (k == 2) { rev[a0] = 1; rev[a1] = 1; }
    else if (k == 3) { q[a0] = a1; q[a1] = a0; rev[a0] = 1; }
    const long long ss[3] = {(long long)a.Hs * a.Ws, (long long)a.Ws, 1};
    long long base = 0;
    for (int c = 0; c < 3; ++c) {
      const int r = rev[c] ^ rec[5 + q[c]];
      base += (long long)(rec[1 + c] + (r ? ext[q[c]] - 1 : 0)) * ss[c];
      s_coef[q[c]] = r ? -ss[c] : ss[c];
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
  // every block has read the state (before its own increment below): the last one advances it for the next batch
  if (tid == 0) {
    __threadfence();
    const unsigned long long total = (unsigned long long)gridDim.x * gridDim.y * gridDim.z;
    if (atomicAdd(reinterpret_cast<unsigned long long*>(state + 5), 1ull) == total - 1) {
      state[1] += 1;
      state[2] += 1;
      state[5] = 0;
      __threadfence();
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

extern "C" int ssd3d_augment_batch(const void* src, int src_is_bf16, const uint8_t* masks, int S, int C, int Ds, int Hs,
                                   int Ws, const int32_t* order, int64_t* state, const int32_t* boxes,
                                   const int32_t* box_offsets, int N, int d, int h, int w, float pos_ratio,
                                   float flip_prob, float rot90_prob, int rot_axis0, int rot_axis1, float scale,
                                   float shift, void* out, uint8_t* out_mask, int32_t* record, void* stream) {
  if (!src || !masks || !order || !state || !boxes || !box_offsets || !out || !out_mask || !record) return SSD3D_ERR_ARG;
  if (S <= 0 || C <= 0 || N <= 0 || d <= 0 || h <= 0 || w <= 0 || d > Ds || h > Hs || w > Ws) return SSD3D_ERR_ARG;
  if (!(pos_ratio >= 0.f && pos_ratio <= 1.f) || !(flip_prob >= 0.f && flip_prob <= 1.f) ||
      !(rot90_prob >= 0.f && rot90_prob <= 1.f) || !(scale >= 0.f) || !(shift >= 0.f))
    return SSD3D_ERR_ARG;
  if (rot_axis0 < 0 || rot_axis0 > 2 || rot_axis1 < 0 || rot_axis1 > 2 || rot_axis0 == rot_axis1) return SSD3D_ERR_ARG;
  const int ext[3] = {d, h, w};
  if (rot90_prob > 0.f && ext[rot_axis0] != ext[rot_axis1]) return SSD3D_ERR_ARG;
  if (w % 16 != 0 || (long long)Ds * Hs * Ws >= (1ll << 31) || h > 65535 || d > 65535) return SSD3D_ERR_UNSUPPORTED;
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
