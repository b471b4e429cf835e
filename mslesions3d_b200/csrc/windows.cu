// Sliding-window inference over scans larger than the network input.
//
// ssd3d_window_gather copies the window grid of S scans (S, C, D, H, W) into the network's input batch
// (S*T, C, d, h, w) bf16.  Per spatial axis a the windows start at o_i = min(i * stride_a, S_a - w_a),
// i < n_a = ceil((S_a - w_a) / stride_a) + 1, so the last one ends flush with the scan; window
// t = (i_d * n_h + i_h) * n_w + i_w and the batch is scan-major.  A block copies a tile of rows of one
// (window, channel, z) plane: every warp reads whole source rows with consecutive lanes on consecutive
// elements (coalesced whatever the origin's alignment), converts them to bf16 (round to nearest even,
// torch.Tensor.to(torch.bfloat16) for every non-NaN value) into shared memory, and the block writes the tile,
// contiguous in the output, with 16-byte stores.
//
// ssd3d_merge_windows merges the per-window detections of ssd3d_detect_objects into per-scan ones.  Its stage-1
// kernel turns entry r < count[t] of window t into candidate j = t * K + r of its scan (label 0, the "nothing
// found" placeholder, and scores <= min_score are skipped), maps the box into the scan's fractional coordinates
// (coordinates k and k + 3 belong to spatial axis k: x' = x * (w_k / S_k) + o_k / S_k, both factors fp32 from the
// host, two rounded operations) and appends the key {~orderable(score), j} to the (scan, label) list.  Stages 2-4
// of detect_objects then run unchanged on those lists (detect_select).
#include <cuda_bf16.h>

#include "detect.cuh"

namespace ssd3d {

constexpr int GATHER_TILE = 8192;    // bf16 elements of one block's tile (16 KB)

struct WindowGrid {
  int S, C, D, H, W, d, h, w;
  int nd, nh, nw, sd, sh, sw;        // windows and stride per axis
  int rows_per_tile, tiles;          // tiles of whole output rows per (window, channel, z) plane
};

__device__ __forceinline__ unsigned short bf16_bits(float v) {
  return __bfloat16_as_ushort(__float2bfloat16_rn(v));
}

template <bool SRC_BF16>
__global__ void __launch_bounds__(256) window_gather_kernel(const void* __restrict__ src, const WindowGrid g,
                                                            unsigned short* __restrict__ dst) {
  __shared__ __align__(16) unsigned short tile[GATHER_TILE];
  const long long block = blockIdx.x;
  const int tix = (int)(block % g.tiles);
  long long q = block / g.tiles;                 // plane = ((scan * T + t) * C + c) * d + z
  const long long plane = q;
  const int z = (int)(q % g.d); q /= g.d;
  const int c = (int)(q % g.C); q /= g.C;
  const int T = g.nd * g.nh * g.nw;
  const int t = (int)(q % T);
  const int scan = (int)(q / T);
  const int iw = t % g.nw, ih = (t / g.nw) % g.nh, id = t / (g.nw * g.nh);
  const int od = min(id * g.sd, g.D - g.d), oh = min(ih * g.sh, g.H - g.h), ow = min(iw * g.sw, g.W - g.w);
  const int y0 = tix * g.rows_per_tile;
  const int rows = min(g.rows_per_tile, g.h - y0);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long src_plane = (((long long)scan * g.C + c) * g.D + od + z) * g.H + oh + y0;
  for (int r = warp; r < rows; r += 8) {
    const long long row = (src_plane + r) * g.W + ow;
    unsigned short* trow = tile + r * g.w;
    if constexpr (SRC_BF16) {
      const unsigned short* s = static_cast<const unsigned short*>(src) + row;
#pragma unroll 4
      for (int x = lane; x < g.w; x += 32) trow[x] = __ldg(s + x);
    } else {
      const float* s = static_cast<const float*>(src) + row;
#pragma unroll 4
      for (int x = lane; x < g.w; x += 32) trow[x] = bf16_bits(__ldg(s + x));
    }
  }
  __syncthreads();
  const int n16 = rows * g.w / 8;
  uint4* out = reinterpret_cast<uint4*>(dst + (plane * g.h + y0) * g.w);
  const uint4* in = reinterpret_cast<const uint4*>(tile);
  for (int i = threadIdx.x; i < n16; i += 256) out[i] = in[i];
}

// stage 1 of the merge: one thread per (scan, window entry)
__global__ void __launch_bounds__(256) window_candidates_kernel(
    const float* __restrict__ win_boxes, const float* __restrict__ win_scores, const long long* __restrict__ win_labels,
    const int* __restrict__ win_count, int T, int K, const float* __restrict__ win_offset, float scale_d,
    float scale_h, float scale_w, int C, float min_score, long long P, float* __restrict__ boxes,
    unsigned long long* __restrict__ cand, int* __restrict__ count) {
  pdl_wait();
  pdl_launch_dependents();
  const long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int scan = blockIdx.y;
  if (j >= P) return;
  const int t = (int)(j / K), r = (int)(j - (long long)t * K);
  const long long w = (long long)scan * T + t;
  if (r >= win_count[w]) return;
  const long long e = w * K + r;
  const long long label = win_labels[e];
  const float score = win_scores[e];
  if (label < 1 || label >= C || !(score > min_score)) return;
  const Box6 b = load_box(win_boxes + e * 6);
  const float sc[3] = {scale_d, scale_h, scale_w};
  const float* off = win_offset + (long long)t * 3;
  Box6 m;
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    m.v[k] = __fadd_rn(__fmul_rn(b.v[k], sc[k]), off[k]);
    m.v[k + 3] = __fadd_rn(__fmul_rn(b.v[k + 3], sc[k]), off[k]);
  }
  store_box(boxes + ((long long)scan * P + j) * 6, m);
  const int seg = scan * (C - 1) + (int)(label - 1);
  const int slot = atomicAdd(&count[seg], 1);
  cand[(long long)seg * P + slot] = ((unsigned long long)(~float_orderable(score)) << 32) | (unsigned long long)j;
}

static inline int window_count(int S, int w, int stride) { return (S - w + stride - 1) / stride + 1; }

}  // namespace ssd3d

using namespace ssd3d;

extern "C" int ssd3d_window_gather(const void* src, int src_is_bf16, int S, int C, int D, int H, int W, int d, int h,
                                   int w, int stride_d, int stride_h, int stride_w, void* out, void* stream) {
  if (!src || !out || S <= 0 || C <= 0 || d <= 0 || h <= 0 || w <= 0 || d > D || h > H || w > W || stride_d < 1 ||
      stride_h < 1 || stride_w < 1)
    return SSD3D_ERR_ARG;
  if (w % 8 != 0 || w > GATHER_TILE) return SSD3D_ERR_UNSUPPORTED;       // 16-byte stores of whole rows
  WindowGrid g;
  g.S = S; g.C = C; g.D = D; g.H = H; g.W = W; g.d = d; g.h = h; g.w = w;
  g.sd = stride_d; g.sh = stride_h; g.sw = stride_w;
  g.nd = window_count(D, d, stride_d);
  g.nh = window_count(H, h, stride_h);
  g.nw = window_count(W, w, stride_w);
  g.rows_per_tile = GATHER_TILE / w < h ? GATHER_TILE / w : h;
  g.tiles = (h + g.rows_per_tile - 1) / g.rows_per_tile;
  const long long blocks = (long long)S * g.nd * g.nh * g.nw * C * d * g.tiles;
  if (blocks > 0x7fffffffll) return SSD3D_ERR_UNSUPPORTED;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (src_is_bf16)
    window_gather_kernel<true><<<(unsigned)blocks, 256, 0, st>>>(src, g, static_cast<unsigned short*>(out));
  else
    window_gather_kernel<false><<<(unsigned)blocks, 256, 0, st>>>(src, g, static_cast<unsigned short*>(out));
  SSD3D_CHECK_LAUNCH();
  return SSD3D_OK;
}

extern "C" int64_t ssd3d_merge_windows_workspace_bytes(int n_scans, int n_windows, int K, int n_classes, int top_k) {
  const long long P = (long long)n_windows * K;
  if (n_scans <= 0 || n_windows <= 0 || K <= 0 || n_classes < 2 || top_k <= 0 || P > 0x7fffffffll) return 0;
  return detect_layout(n_scans, P, n_classes, top_k).total;
}

extern "C" int ssd3d_merge_windows(const float* win_boxes, const float* win_scores, const int64_t* win_labels,
                                   const int32_t* win_count, int n_scans, int n_windows, int K, const float* win_offset,
                                   float scale_d, float scale_h, float scale_w, int n_classes, float min_score,
                                   float max_overlap, int top_k, float* out_boxes, float* out_scores,
                                   int64_t* out_labels, int64_t* out_cand, int32_t* out_count, void* workspace,
                                   int64_t workspace_bytes, int32_t* status, void* stream) {
  if (!win_boxes || !win_scores || !win_labels || !win_count || !win_offset || !out_boxes || !out_scores ||
      !out_labels || !out_cand || !out_count || !workspace)
    return SSD3D_ERR_ARG;
  const long long P = (long long)n_windows * K;
  if (n_scans <= 0 || n_windows <= 0 || K <= 0 || n_classes < 2 || top_k <= 0 || P > 0x7fffffffll) return SSD3D_ERR_ARG;
  const DetectLayout L = detect_layout(n_scans, P, n_classes, top_k);
  if (workspace_bytes < L.total) return SSD3D_ERR_ARG;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  uint8_t* ws = static_cast<uint8_t*>(workspace);
  cudaError_t e = cudaMemsetAsync(ws + L.off_count, 0, (size_t)(L.off_boxes - L.off_count), st);
  if (e != cudaSuccess) return (int)e;
  if (status) {
    e = cudaMemsetAsync(status, 0, 4, st);
    if (e != cudaSuccess) return (int)e;
  }
  {
    dim3 grid((unsigned)((P + 255) / 256), (unsigned)n_scans);
    SSD3D_LAUNCH_PDL(window_candidates_kernel, grid, dim3(256), 0, st, win_boxes, win_scores,
                     reinterpret_cast<const long long*>(win_labels), win_count, n_windows, K, win_offset, scale_d,
                     scale_h, scale_w, n_classes, min_score, P, reinterpret_cast<float*>(ws + L.off_boxes),
                     reinterpret_cast<unsigned long long*>(ws + L.off_cand), reinterpret_cast<int*>(ws + L.off_count));
  }
  return detect_select(L, ws, n_scans, P, n_classes, max_overlap, top_k, out_boxes, out_scores, out_labels, out_cand,
                       out_count, status, st);
}
