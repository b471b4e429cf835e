// LSSD3D.detect_objects on the device (ssd3d.py:344-460), batched over images and classes, with no
// host synchronisation inside:
//   1. decode_filter : softmax over classes, decode offsets -> boundary boxes (utils.py:50-68), keep
//                      candidates with score > min_score (warp-ballot compaction into per-(image,class) lists)
//   2. sort_segments : per (image,class) bitonic sort of 64-bit keys {~orderable(score), prior index}
//                      = descending score, ascending prior index on ties; truncate to 10*top_k
//   3. nms_mask      : IoU > max_overlap bit matrix (64-bit words) over the sorted candidates
//   4. nms_select    : greedy scan of the bit matrix (ssd3d.py:414-426), per-image merge of the classes,
//                      final top-k cut (ssd3d.py:449-453), placeholder for empty images (ssd3d.py:437-440)
#include "detect.cuh"

namespace ssd3d {

// ------------------------------------------------------------------------------------------------
// stage 1: softmax + decode (+ filter)
// ------------------------------------------------------------------------------------------------
// softmax of one prior's class scores: exp(x - max) * (1 / sum), classes summed in index order
template <typename F>
__device__ __forceinline__ void softmax_small(const float* s, int C, F&& emit) {
  float m = s[0];
  for (int k = 1; k < C; ++k) m = fmaxf(m, s[k]);
  float sum = 0.f;
  for (int k = 0; k < C; ++k) sum = __fadd_rn(sum, expf(__fsub_rn(s[k], m)));
  const float inv = __fdiv_rn(1.0f, sum);
  for (int k = 0; k < C; ++k) emit(k, __fmul_rn(expf(__fsub_rn(s[k], m)), inv));
}

__global__ void __launch_bounds__(256) decode_softmax_kernel(const float* __restrict__ locs,
                                                             const float* __restrict__ scores,
                                                             const PriorSrc priors, long long P, int C,
                                                             float* __restrict__ probs, float* __restrict__ boxes) {
  const long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int img = blockIdx.y;
  if (p >= P) return;
  const long long ip = (long long)img * P + p;
  const Box6 xyz = cxcycz_to_xyz(gcxgcygcz_to_cxcycz(load_box(locs + ip * 6), load_prior(priors, p)));
  store_box(boxes + ip * 6, xyz);
  const float* s = scores + ip * C;
  float* o = probs + ip * C;
  softmax_small(s, C, [&](int k, float v) { o[k] = v; });
}

// cand layout: segment seg = img*(C-1) + (c-1) owns cand[seg*P .. seg*P + count[seg])
__global__ void __launch_bounds__(256) decode_filter_kernel(const float* __restrict__ locs,
                                                            const float* __restrict__ scores,
                                                            const PriorSrc priors, long long P, int C,
                                                            float min_score, float* __restrict__ boxes,
                                                            unsigned long long* __restrict__ cand,
                                                            int* __restrict__ count) {
  pdl_wait();
  pdl_launch_dependents();
  const long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int img = blockIdx.y;
  const bool live = p < P;
  const long long ip = (long long)img * P + (live ? p : 0);
  if (live) {
    const Box6 xyz = cxcycz_to_xyz(gcxgcygcz_to_cxcycz(load_box(locs + ip * 6), load_prior(priors, p)));
    store_box(boxes + ip * 6, xyz);
  }
  const float* s = scores + ip * C;
  const int lane = threadIdx.x & 31;
  // every lane walks the classes together so that the ballots are warp-uniform
  float m = s[0];
  for (int k = 1; k < C; ++k) m = fmaxf(m, s[k]);
  float sum = 0.f;
  for (int k = 0; k < C; ++k) sum = __fadd_rn(sum, expf(__fsub_rn(s[k], m)));
  const float inv = __fdiv_rn(1.0f, sum);
  for (int c = 1; c < C; ++c) {
    const float prob = __fmul_rn(expf(__fsub_rn(s[c], m)), inv);
    const bool pass = live && (prob > min_score);
    const unsigned ballot = __ballot_sync(0xffffffffu, pass);
    if (ballot == 0u) continue;
    const int seg = img * (C - 1) + (c - 1);
    int base = 0;
    if (lane == 0) base = atomicAdd(&count[seg], __popc(ballot));
    base = __shfl_sync(0xffffffffu, base, 0);
    if (pass) {
      const int slot = base + __popc(ballot & ((1u << lane) - 1u));
      const unsigned long long key =
          ((unsigned long long)(~float_orderable(prob)) << 32) | (unsigned long long)(uint32_t)p;
      cand[(long long)seg * P + slot] = key;
    }
  }
}

// ------------------------------------------------------------------------------------------------
// stage 2: per-segment sort (shared-memory bitonic network on 64-bit keys)
//
// A block sorts at most SSD3D_SORT_MAX keys.  Longer candidate lists (the >1M-prior whole-brain config) are
// reduced hierarchically: every 16384-key chunk is sorted by its own block which keeps the chunk's best
// `nmax` keys, the survivors form the next level's list, until one chunk is left.  Keys are unique
// ({~orderable(score), prior index}), so the result is exactly the first `nmax` entries of the full sort.
// Empty slots hold the sentinel ~0, which sorts last and is dropped at the end.
// ------------------------------------------------------------------------------------------------
// Stages whose compare-exchange distance j fits inside a warp's own contiguous chunk of np2 / nwarps keys
// (2j <= chunk) only need __syncwarp: for 8192 keys on 32 warps that is 76 of the 91 stages, and the block-wide
// barrier -- what the network's run time was made of -- remains for the 15 long-distance ones.
__device__ __forceinline__ int bitonic_sort_smem(unsigned long long* keys, const unsigned long long* src, int n) {
  int np2 = 1;
  while (np2 < n) np2 <<= 1;
  for (int i = threadIdx.x; i < np2; i += blockDim.x) keys[i] = (i < n) ? src[i] : ~0ull;
  __syncthreads();
  const int nwarps = blockDim.x >> 5, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  int chunk = np2 / nwarps;                     // power of two (blockDim.x is a power of two), maybe < 2
  if (chunk < 2) chunk = 0;
  auto cmpx = [&](int t, int j, int k) {
    const int lo = ((t & ~(j - 1)) << 1) | (t & (j - 1));
    const int hi = lo | j;
    const bool up = (lo & k) == 0;
    const unsigned long long a = keys[lo], b = keys[hi];
    if ((a > b) == up) { keys[lo] = b; keys[hi] = a; }
  };
  for (int k = 2; k <= np2; k <<= 1) {
    int j = k >> 1;
    for (; j > 0 && 2 * j > chunk; j >>= 1) {   // long distance: the whole block, one barrier per stage
      for (int t = threadIdx.x; t < (np2 >> 1); t += blockDim.x) cmpx(t, j, k);
      __syncthreads();
    }
    if (j > 0) {                                // the rest of this level stays inside each warp's chunk
      const int t0 = warp * (chunk >> 1);
      for (; j > 0; j >>= 1) {
        for (int t = lane; t < (chunk >> 1); t += 32) cmpx(t0 + t, j, k);
        __syncwarp();
      }
      __syncthreads();
    }
  }
  return np2;
}

// one level of the hierarchical reduction: block (chunk, seg) -> best `nmax` keys of its chunk (or sentinels)
__global__ void __launch_bounds__(1024) topk_reduce_kernel(const unsigned long long* __restrict__ src,
                                                           long long src_stride, const int* __restrict__ count,
                                                           int fixed_len, unsigned long long* __restrict__ dst,
                                                           long long dst_stride, int nmax, int chunk_len) {
  extern __shared__ unsigned long long keys[];
  pdl_wait();
  pdl_launch_dependents();
  const int chunk = blockIdx.x, seg = blockIdx.y;
  const long long len = count ? (long long)count[seg] : (long long)fixed_len;
  const long long begin = (long long)chunk * chunk_len;
  long long n = len - begin;
  if (n > chunk_len) n = chunk_len;
  unsigned long long* out = dst + (long long)seg * dst_stride + (long long)chunk * nmax;
  if (n <= 0) {
    for (int i = threadIdx.x; i < nmax; i += blockDim.x) out[i] = ~0ull;
    return;
  }
  bitonic_sort_smem(keys, src + (long long)seg * src_stride + begin, (int)n);
  for (int i = threadIdx.x; i < nmax; i += blockDim.x) out[i] = (i < n) ? keys[i] : ~0ull;
}

__global__ void __launch_bounds__(1024) sort_segments_kernel(const unsigned long long* __restrict__ cand,
                                                             long long cand_stride, const int* __restrict__ count,
                                                             int fixed_len, int* __restrict__ nkeep,
                                                             const float* __restrict__ boxes, long long P, int C,
                                                             int nmax, int sort_cap, float* __restrict__ sboxes,
                                                             float* __restrict__ sscores, int* __restrict__ sprior,
                                                             int* __restrict__ status) {
  extern __shared__ unsigned long long keys[];
  __shared__ int s_valid;
  pdl_wait();
  pdl_launch_dependents();
  const int seg = blockIdx.x;
  const int img = seg / (C - 1);
  int n = count ? count[seg] : fixed_len;
  if (n > sort_cap) {
    if (threadIdx.x == 0 && status) atomicOr(status, 1);
    n = sort_cap;
  }
  if (threadIdx.x == 0) s_valid = 0;
  const int np2 = bitonic_sort_smem(keys, cand + (long long)seg * cand_stride, n);
  // sentinels (empty slots of a reduced list) sort last: the valid prefix ends at the first one
  for (int i = threadIdx.x; i < n; i += blockDim.x)
    if (keys[i] != ~0ull && (i + 1 == np2 || keys[i + 1] == ~0ull)) s_valid = i + 1;
  __syncthreads();
  const int nv = s_valid;
  const int nk = nv < nmax ? nv : nmax;
  if (threadIdx.x == 0) nkeep[seg] = nk;
  for (int i = threadIdx.x; i < nk; i += blockDim.x) {
    const unsigned long long key = keys[i];
    const uint32_t p = (uint32_t)(key & 0xffffffffull);
    const long long o = (long long)seg * nmax + i;
    sprior[o] = (int)p;
    sscores[o] = float_from_orderable(~(uint32_t)(key >> 32));
    store_box(sboxes + o * 6, load_box(boxes + ((long long)img * P + p) * 6));
  }
}

// ------------------------------------------------------------------------------------------------
// stage 3: suppression bit matrix over the score-sorted candidates.
//   off-diagonal word (w > i/64): bit b  <=>  IoU(i, 64 w + b) > thr              (all of them later boxes)
//   diagonal word    (w = i/64): bit b  <=>  64 w + b != i and IoU(i, 64 w + b) > thr   (both directions:
//                                 IoU is exactly symmetric, so this word also lists the EARLIER neighbours)
// Words w < i/64 are never written nor read.
// ------------------------------------------------------------------------------------------------
// fl(inter / uni) > thr without the IEEE divide in the common case: a multiply pre-test with a 2^-18
// guard band (>> the 2^-23 rounding of the two products) decides all but near-threshold pairs; those,
// and every degenerate union, take the exactly rounded division the reference performs (utils.py:149).
__device__ __forceinline__ bool iou_exceeds(float inter, float uni, float thr) {
  if (thr > 0.0f && uni > 1e-30f && uni < 1e30f) {
    const float t = thr * uni;
    if (inter > t * 1.000004f) return true;
    if (inter < t * 0.999996f) return false;
  }
  return __fdiv_rn(inter, uni) > thr;
}

// exact fallback of iou_exceeds, kept out of the hot loop
__device__ __noinline__ bool iou_exceeds_exact(float inter, float uni, float thr) { return __fdiv_rn(inter, uni) > thr; }

template <bool TR>
__device__ __forceinline__ void nms_mask_body(const float* __restrict__ sboxes, const int* __restrict__ nkeep,
                                              int n_fixed, long long seg_stride_boxes, int words,
                                              long long seg_stride_mask, float thr,
                                              unsigned long long* __restrict__ mask,
                                              unsigned long long* __restrict__ block_flags, int flag_words) {
  pdl_wait();
  pdl_launch_dependents();
  const int cb = blockIdx.x, rb = blockIdx.y, seg = blockIdx.z;
  if (cb < rb) return;
  const int n = nkeep ? nkeep[seg] : n_fixed;
  if (rb * 64 >= n || cb * 64 >= n) return;
  // column boxes as two 16-byte records each: {x0, y0, z0, x1}, {y1, z1, volume, -}: two broadcast LDS.128 per pair
  __shared__ float4 cb0[64], cb1[64];
  const float* base = sboxes + (long long)seg * seg_stride_boxes;
  const int t = threadIdx.x;
  const int cj = cb * 64 + t;
  if (cj < n) {
    const Box6 b = load_box(base + (long long)cj * 6);
    cb0[t] = make_float4(b.v[0], b.v[1], b.v[2], b.v[3]);
    cb1[t] = make_float4(b.v[4], b.v[5], box_volume(b), 0.f);
  }
  __syncthreads();
  const int i = rb * 64 + t;
  unsigned long long bits = 0ull;
  if (i < n) {
    const Box6 a = load_box(base + (long long)i * 6);
    const float va = box_volume(a);
    const int jn = min(64, n - cb * 64);
    const bool thr_pos = thr > 0.0f;
    const float thr_hi = thr * 1.000004f, thr_lo = thr * 0.999996f;
    (void)thr_hi; (void)thr_lo;
    unsigned int half[2] = {0u, 0u};
#pragma unroll
    for (int hb = 0; hb < 2; ++hb) {
      unsigned int acc = 0u;
#pragma unroll 8
      for (int bb = 0; bb < 32; ++bb) {
        const int b = hb * 32 + bb;
        if (b >= jn) break;
        const float4 p = cb0[b], q = cb1[b];
        // utils.py:119-122, one rounded op at a time (clamp: NaN propagates like torch.clamp)
        const float d0 = clamp_min0(__fsub_rn(fminf(a.v[3], p.w), fmaxf(a.v[0], p.x)));
        const float d1 = clamp_min0(__fsub_rn(fminf(a.v[4], q.x), fmaxf(a.v[1], p.y)));
        const float d2 = clamp_min0(__fsub_rn(fminf(a.v[5], q.y), fmaxf(a.v[2], p.z)));
        const float inter = __fmul_rn(__fmul_rn(d0, d1), d2);
        const float uni = __fsub_rn(__fadd_rn(va, q.z), inter);
        // iou_exceeds: multiply pre-test with a guard band, exact IEEE division only near the threshold / for
        // degenerate unions
        const float tt = thr * uni;
        const bool yes = inter > tt * 1.000004f, no = inter < tt * 0.999996f;
        bool hit;
        if (thr_pos && uni > 1e-30f && uni < 1e30f && (yes || no)) hit = yes;
        else hit = iou_exceeds_exact(inter, uni, thr);
        acc |= hit ? (1u << bb) : 0u;
      }
      half[hb] = acc;
    }
    bits = ((unsigned long long)half[1] << 32) | half[0];
    if (cb == rb) bits &= ~(1ull << t);       // a box does not suppress itself (ssd3d.py:425-426)
    // TR: word-major layout [word][row] with `words` = rows per word-row (coalesced for the chunk scan)
    if (TR) mask[(long long)seg * seg_stride_mask + (long long)cb * words + i] = bits;
    else mask[(long long)seg * seg_stride_mask + (long long)i * words + cb] = bits;
  }
  if constexpr (TR) {
    // one flag per 64 x 64 block that holds any bit: most blocks of a sparse scene are empty and the scan
    // skips them (and whole steps) without touching the matrix
    if (__syncthreads_or(bits != 0ull) && t == 0)
      atomicOr(&block_flags[(long long)rb * flag_words + (cb >> 6)], 1ull << (cb & 63));
  }
}

__global__ void __launch_bounds__(64) nms_mask_kernel(const float* __restrict__ sboxes, const int* __restrict__ nkeep,
                                                      int n_fixed, long long seg_stride_boxes, int words,
                                                      long long seg_stride_mask, float thr,
                                                      unsigned long long* __restrict__ mask) {
  nms_mask_body<false>(sboxes, nkeep, n_fixed, seg_stride_boxes, words, seg_stride_mask, thr, mask, nullptr, 0);
}
// same bits, stored word-major: mask[word * row_stride + row], plus the per-block "any bit" flags
// block_flags[row_word * flag_words + col_word / 64] bit (col_word % 64)
__global__ void __launch_bounds__(64) nms_mask_tr_kernel(const float* __restrict__ sboxes, int n, int row_stride,
                                                         float thr, unsigned long long* __restrict__ mask,
                                                         unsigned long long* __restrict__ block_flags, int flag_words) {
  nms_mask_body<true>(sboxes, nullptr, n, 0, row_stride, 0, thr, mask, block_flags, flag_words);
}

// Greedy scan of one segment's bit matrix M (rows `stride` words apart; shared or global memory).
// `removed` is scratch of ceil(n/64) words, `keptw` receives the keep bits.  All threads call it.
//
// Chunk k (64 boxes) is resolved by warp 0 in rounds instead of a 64-step serial chain: lane l owns boxes
// l and l+32 with the masks of their EARLIER neighbours inside the chunk.  A box with a kept earlier
// neighbour is removed; a box none of whose earlier neighbours is kept or still undecided is kept.  The
// lowest undecided box is always decidable, so the loop ends, normally after a handful of rounds, with
// exactly the greedy result of ssd3d.py:414-426.  The rows of the kept boxes are then OR-ed into the later
// words, one warp per word, with redux.or across the 32 lanes.
__device__ __forceinline__ void nms_scan_core(const unsigned long long* M, int n, int stride,
                                              unsigned long long* removed, unsigned long long* keptw,
                                              const unsigned long long* removed_init = nullptr) {
  const int words = (n + 63) >> 6;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
  for (int w = threadIdx.x; w < words; w += blockDim.x) removed[w] = removed_init ? removed_init[w] : 0ull;
  __syncthreads();
  // OR of the rows of chunk k's kept boxes, word w, by one warp (redux.or across the lanes)
  auto or_word = [&](int k, unsigned long long kept, int w) {
    unsigned int lo = 0u, hi = 0u;
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int b = h * 32 + lane;
      unsigned long long v = 0ull;
      if ((kept >> b) & 1ull) v = M[(long long)(k * 64 + b) * stride + w];
      lo |= __reduce_or_sync(0xffffffffu, (unsigned int)v);
      hi |= __reduce_or_sync(0xffffffffu, (unsigned int)(v >> 32));
    }
    if (lane == 0) atomicOr(&removed[w], ((unsigned long long)hi << 32) | lo);
  };
  // ONE block barrier per chunk.  In iteration k warp 0 resolves chunk k and immediately ORs its kept rows into
  // word k+1 (all the next chunk needs from this one); meanwhile the other warps spread chunk k-1's kept rows
  // over the words >= k+1.  Word k is complete when warp 0 reads it: chunk k-1's part was added by warp 0 itself
  // one iteration ago, the parts of chunks <= k-2 by the helpers at least one barrier ago.
  for (int k = 0; k <= words; ++k) {
    if (warp == 0) {
      if (nwarps == 1 && k >= 1) {                        // no helpers in a one-warp block: do their part first
        const unsigned long long kp = keptw[k - 1];
        if (kp != 0ull)
          for (int w = k + 1; w < words; ++w) or_word(k - 1, kp, w);
        __syncwarp();
      }
      if (k < words) {
        const int rows = min(64, n - k * 64);
        const unsigned long long r0 = (lane < rows) ? M[(long long)(k * 64 + lane) * stride + k] : 0ull;
        const unsigned long long r1 = (lane + 32 < rows) ? M[(long long)(k * 64 + lane + 32) * stride + k] : 0ull;
        const unsigned long long e0 = r0 & ((1ull << lane) - 1ull);
        const unsigned long long e1 = r1 & ((1ull << (lane + 32)) - 1ull);
        unsigned long long rem = removed[k];
        if (rows < 64) rem |= (~0ull) << rows;            // rows past the end are never kept
        unsigned long long und = ~rem, kept = 0ull;
        while (und != 0ull) {
          const bool u0 = (und >> lane) & 1ull, u1 = (und >> (lane + 32)) & 1ull;
          const bool x0 = u0 && (e0 & kept) != 0ull, x1 = u1 && (e1 & kept) != 0ull;
          const bool k0 = u0 && !x0 && (e0 & und) == 0ull, k1 = u1 && !x1 && (e1 & und) == 0ull;
          const unsigned long long nk = (unsigned long long)__ballot_sync(0xffffffffu, k0) |
                                        ((unsigned long long)__ballot_sync(0xffffffffu, k1) << 32);
          const unsigned long long nx = (unsigned long long)__ballot_sync(0xffffffffu, x0) |
                                        ((unsigned long long)__ballot_sync(0xffffffffu, x1) << 32);
          kept |= nk;
          und &= ~(nk | nx);
        }
        if (lane == 0) keptw[k] = kept;
        if (kept != 0ull && k + 1 < words) or_word(k, kept, k + 1);
      }
    } else if (k >= 1) {                                    // (nwarps > 1 here)
      const unsigned long long kept = keptw[k - 1];       // published before the previous barrier
      if (kept != 0ull)
        for (int w = k + 1 + (warp - 1); w < words; w += nwarps - 1) or_word(k - 1, kept, w);
    }
    __syncthreads();
  }
}

// Stage the upper-triangular words of the bit matrix in shared memory when they fit (the default
// 10*top_k = 1000 candidates need 125 KB), so that the serial chain runs at shared-memory latency.
__device__ void nms_scan(const unsigned long long* __restrict__ mask, int n, int row_stride,
                         unsigned long long* removed, unsigned long long* keptw, unsigned long long* stage,
                         long long stage_words) {
  const int words = (n + 63) >> 6;
  if ((long long)n * words <= stage_words) {
    // only the words w >= i / 64 of row i exist; a half-warp copies one row (words <= 16 for the default 1000)
    const int hw = threadIdx.x >> 4, hl = threadIdx.x & 15, nhw = blockDim.x >> 4;
    for (int i = hw; i < n; i += nhw)
      for (int w = (i >> 6) + hl; w < words; w += 16) stage[i * words + w] = mask[(long long)i * row_stride + w];
    __syncthreads();
    nms_scan_core(stage, n, words, removed, keptw);
  } else {
    nms_scan_core(mask, n, row_stride, removed, keptw);
  }
}

// ------------------------------------------------------------------------------------------------
// stage 4: per image: scan every class, merge, top-k, write outputs
// ------------------------------------------------------------------------------------------------
// number of entries of the descending list s[0..n) that are > v (strict) or >= v
__device__ __forceinline__ int count_greater(const float* s, int n, float v, bool or_equal) {
  int lo = 0, hi = n;
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    const bool before = or_equal ? (s[mid] >= v) : (s[mid] > v);
    if (before) lo = mid + 1; else hi = mid;
  }
  return lo;
}

__global__ void __launch_bounds__(512) nms_select_kernel(const unsigned long long* __restrict__ mask,
                                                         const int* __restrict__ nkeep, int C, int nmax, int words_max,
                                                         long long stage_words, const float* __restrict__ sboxes,
                                                         const float* __restrict__ sscores,
                                                         const int* __restrict__ sprior, int* __restrict__ kept_pos,
                                                         float* __restrict__ kept_score, int* __restrict__ kept_cnt,
                                                         int top_k, float* __restrict__ out_boxes,
                                                         float* __restrict__ out_scores, long long* __restrict__ out_labels,
                                                         long long* __restrict__ out_prior, int* __restrict__ out_count) {
  extern __shared__ unsigned long long sm[];
  unsigned long long* removed = sm;
  unsigned long long* keptw = sm + words_max;
  unsigned long long* stage = sm + 2 * words_max;
  __shared__ int s_total;
  pdl_wait();
  pdl_launch_dependents();
  const int img = blockIdx.x;
  const int nseg = C - 1;

  // ---- greedy NMS per class; compact kept positions (in sorted order) ----
  for (int c = 0; c < nseg; ++c) {
    const int seg = img * nseg + c;
    const int n = nkeep[seg];
    const int words = (n + 63) >> 6;
    int* kp = kept_pos + (long long)seg * nmax;
    float* ks = kept_score + (long long)seg * nmax;
    if (n > 0) {
      nms_scan(mask + (long long)seg * nmax * words_max, n, words_max, removed, keptw, stage, stage_words);
      __syncthreads();
      // exclusive prefix of the kept counts per word (kept in `removed`, which the scan is done with)
      if (threadIdx.x == 0) {
        int run = 0;
        for (int w = 0; w < words; ++w) {
          removed[w] = (unsigned long long)run;
          run += __popcll(keptw[w]);
        }
        kept_cnt[seg] = run;
      }
      __syncthreads();
      for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const unsigned long long kw = keptw[i >> 6];
        if ((kw >> (i & 63)) & 1ull) {
          const int pos = (int)removed[i >> 6] + __popcll(kw & ((1ull << (i & 63)) - 1ull));
          kp[pos] = i;
          ks[pos] = sscores[(long long)seg * nmax + i];
        }
      }
    } else if (threadIdx.x == 0) {
      kept_cnt[seg] = 0;
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    int t = 0;
    for (int c = 0; c < nseg; ++c) t += kept_cnt[img * nseg + c];
    s_total = t;
  }
  __syncthreads();
  const int total = s_total;
  float* ob = out_boxes + (long long)img * top_k * 6;
  float* os = out_scores + (long long)img * top_k;
  long long* ol = out_labels + (long long)img * top_k;
  long long* op = out_prior + (long long)img * top_k;

  if (total == 0) {  // ssd3d.py:437-440
    if (threadIdx.x == 0) {
      ob[0] = 0.f; ob[1] = 0.f; ob[2] = 0.f; ob[3] = 1.f; ob[4] = 1.f; ob[5] = 1.f;
      os[0] = 0.f;
      ol[0] = 0;
      op[0] = -1;
      out_count[img] = 1;
    }
    return;
  }
  if (threadIdx.x == 0) out_count[img] = total < top_k ? total : top_k;

  // ---- merge classes.  total <= top_k: concatenation in class order (ssd3d.py:443-446).  Otherwise
  // the stable descending sort of the concatenation (ssd3d.py:449-453): an entry's rank is its own
  // position in its class list + entries of earlier classes with score >= its score + entries of later
  // classes with score > its score. ----
  int class_base = 0;
  for (int c = 0; c < nseg; ++c) {
    const int seg = img * nseg + c;
    const int cnt = kept_cnt[seg];
    const int* kp = kept_pos + (long long)seg * nmax;
    const float* ks = kept_score + (long long)seg * nmax;
    for (int r = threadIdx.x; r < cnt; r += blockDim.x) {
      int rank;
      if (total <= top_k) {
        rank = class_base + r;
      } else {
        const float v = ks[r];
        rank = r;
        for (int c2 = 0; c2 < nseg; ++c2) {
          if (c2 == c) continue;
          const int seg2 = img * nseg + c2;
          rank += count_greater(kept_score + (long long)seg2 * nmax, kept_cnt[seg2], v, c2 < c);
        }
      }
      if (rank < top_k) {
        const long long src = (long long)seg * nmax + kp[r];
        store_box(ob + (long long)rank * 6, load_box(sboxes + src * 6));
        os[rank] = sscores[src];
        ol[rank] = (long long)(c + 1);
        op[rank] = (long long)sprior[src];
      }
    }
    class_base += cnt;
  }
}

// standalone scan for ssd3d_nms3d_sorted
__global__ void __launch_bounds__(256) nms_scan_kernel(const unsigned long long* __restrict__ mask, int n, int words,
                                                       long long stage_words, uint8_t* __restrict__ keep) {
  extern __shared__ unsigned long long sm[];
  unsigned long long* removed = sm;
  unsigned long long* keptw = sm + words;
  unsigned long long* stage = sm + 2 * words;
  nms_scan(mask, n, words, removed, keptw, stage, stage_words);
  for (int i = threadIdx.x; i < n; i += blockDim.x) keep[i] = (uint8_t)((keptw[i >> 6] >> (i & 63)) & 1ull);
}


// ------------------------------------------------------------------------------------------------
// Greedy NMS over score-sorted lists of ANY length (the NMS-stress setting: min_score = 0 and a top_k
// that defeats the 10*top_k truncation, SURVEY.md 8d C4/C5).  The reference's n x n IoU matrix
// (ssd3d.py:407) is 25 TB at n = 2.5 M; the bit matrix above would still be 390 GB.  Here the list is
// walked in chunks of B boxes (score order):
//   cross : every box of the chunk against the boxes KEPT so far -> initial `removed` bits of the chunk.
//           With a threshold >= 0 through the spatial grid further down (nms_cross_grid_query); otherwise,
//           and for the "delta" of the grid path, the dense kernel below: one thread per chunk box, a range of
//           the compact kept list (32 B per box: corners + volume) streamed through shared memory in tiles
//           of 256, tiles strided over gridDim.y.
//   mask  : the bit matrix of the chunk alone (B x B/64 words, word-major, with per-block flags)
//   scan  : the greedy scan, started from the cross bits; kept boxes are appended to the list.
// A box is removed iff an earlier KEPT box overlaps it by more than the threshold, which is exactly the
// reference's loop (ssd3d.py:414-426); the decisions use the same iou_exceeds() as the bit matrix.
// Two launches per chunk (nms_scan_mask_kernel, which also carries the mask and grid cross test of the NEXT
// chunk, and the dense cross / delta pass); nothing is read back by the host.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) nms_cross_kernel(const float* __restrict__ boxes, int n,
                                                        const float4* __restrict__ kept_all,
                                                        const long long* __restrict__ lo_ptr,
                                                        const long long* __restrict__ hi_ptr, float thr,
                                                        unsigned int* __restrict__ rem32) {
  // kept-list entries [*lo_ptr, *hi_ptr): everything kept so far (dense mode) or the previous chunk's (delta)
  __shared__ float4 tile[256][2];
  const long long lo = *lo_ptr;
  const long long nk = *hi_ptr - lo;
  const float4* kept = kept_all + 2 * lo;
  const long long tiles = (nk + 255) >> 8;
  if ((long long)blockIdx.y >= tiles) return;
  const int i = blockIdx.x * 256 + threadIdx.x;
  const bool live = i < n;
  Box6 a;
#pragma unroll
  for (int k = 0; k < 6; ++k) a.v[k] = 0.f;
  if (live) a = load_box(boxes + (long long)i * 6);
  const float va = box_volume(a);
  bool rem = false;
  for (long long t = blockIdx.y; t < tiles; t += gridDim.y) {
    __syncthreads();
    const long long j = t * 256 + threadIdx.x;
    if (j < nk) {
      tile[threadIdx.x][0] = kept[2 * j];
      tile[threadIdx.x][1] = kept[2 * j + 1];
    }
    __syncthreads();
    const long long left = nk - t * 256;
    const int jn = left < 256 ? (int)left : 256;
    if (live && !rem) {
      for (int b = 0; b < jn; ++b) {
        const float4 p = tile[b][0], q = tile[b][1];
        Box6 o;
        o.v[0] = p.x; o.v[1] = p.y; o.v[2] = p.z; o.v[3] = p.w; o.v[4] = q.x; o.v[5] = q.y;
        const float inter = box_intersection(a, o);
        const float uni = __fsub_rn(__fadd_rn(va, q.z), inter);
        if (iou_exceeds(inter, uni, thr)) rem = true;
      }
    }
  }
  const unsigned ballot = __ballot_sync(0xffffffffu, live && rem);
  if ((threadIdx.x & 31) == 0 && ballot != 0u) atomicOr(&rem32[i >> 5], ballot);
}

// The greedy scan of nms_scan_core on the word-major matrix MT[word * stride + row], driven by the block flags:
//   * a step whose row of blocks is empty off the diagonal concerns nobody but warp 0, which resolves it
//     (kept = not removed, when the diagonal block is empty too) and moves on WITHOUT a barrier; the other
//     warps skip the step, so a sparse scene costs a few dozen instructions per 64 boxes;
//   * otherwise: resolve -> barrier -> the flagged words are dealt round-robin to the warps, whose 64 rows
//     are contiguous (one 512-byte request) -> OR-reduction -> barrier.
// Rows past n hold garbage that the kept bits mask out.  `sflags` is the shared-memory copy of the flags.
__device__ __forceinline__ void nms_scan_core_tr(const unsigned long long* __restrict__ MT, int n, int stride,
                                                 unsigned long long* removed, unsigned long long* keptw,
                                                 const unsigned long long* __restrict__ removed_init,
                                                 const unsigned long long* sflags, int fw) {
  const int words = (n + 63) >> 6;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
  for (int w = threadIdx.x; w < words; w += blockDim.x) removed[w] = removed_init ? removed_init[w] : 0ull;
  __syncthreads();
  for (int k = 0; k < words; ++k) {
    const int rows = min(64, n - k * 64);
    const unsigned long long* fr = sflags + k * fw;
    const int kq = k >> 6;
    const unsigned long long kbit = 1ull << (k & 63);
    bool od_any = false;
    for (int q = kq; q < fw; ++q) od_any |= ((q == kq) ? (fr[q] & ~kbit) : fr[q]) != 0ull;
    if (warp == 0) {
      unsigned long long rem = removed[k];
      if (rows < 64) rem |= (~0ull) << rows;            // rows past the end are never kept
      unsigned long long und = ~rem, kept = 0ull;
      if ((fr[kq] & kbit) == 0ull) {
        kept = und;                                     // no overlaps inside the word: everything left is kept
      } else if (und != 0ull) {
        const long long d = (long long)k * stride + k * 64;
        const unsigned long long r0 = (lane < rows) ? MT[d + lane] : 0ull;
        const unsigned long long r1 = (lane + 32 < rows) ? MT[d + lane + 32] : 0ull;
        const unsigned long long e0 = r0 & ((1ull << lane) - 1ull);
        const unsigned long long e1 = r1 & ((1ull << (lane + 32)) - 1ull);
        while (und != 0ull) {
          const bool u0 = (und >> lane) & 1ull, u1 = (und >> (lane + 32)) & 1ull;
          const bool x0 = u0 && (e0 & kept) != 0ull, x1 = u1 && (e1 & kept) != 0ull;
          const bool k0 = u0 && !x0 && (e0 & und) == 0ull, k1 = u1 && !x1 && (e1 & und) == 0ull;
          const unsigned long long nk = (unsigned long long)__ballot_sync(0xffffffffu, k0) |
                                        ((unsigned long long)__ballot_sync(0xffffffffu, k1) << 32);
          const unsigned long long nx = (unsigned long long)__ballot_sync(0xffffffffu, x0) |
                                        ((unsigned long long)__ballot_sync(0xffffffffu, x1) << 32);
          kept |= nk;
          und &= ~(nk | nx);
        }
      }
      if (lane == 0) keptw[k] = kept;
    }
    if (!od_any) continue;                              // block-uniform: nobody else needs this step
    __syncthreads();
    const unsigned long long kept = keptw[k];
    if (kept != 0ull) {
      const unsigned long long m0 = ((kept >> lane) & 1ull) ? ~0ull : 0ull;
      const unsigned long long m1 = ((kept >> (lane + 32)) & 1ull) ? ~0ull : 0ull;
      int idx = 0;
      for (int q = kq; q < fw; ++q) {
        unsigned long long f = (q == kq) ? (fr[q] & ~kbit) : fr[q];
        while (f != 0ull) {
          const int b = __ffsll((long long)f) - 1;
          f &= f - 1ull;
          if ((idx++ % nwarps) != warp) continue;
          const int w = q * 64 + b;
          const unsigned long long* row = MT + (long long)w * stride + k * 64;
          const unsigned long long v = (row[lane] & m0) | (row[lane + 32] & m1);
          const unsigned int lo = __reduce_or_sync(0xffffffffu, (unsigned int)v);
          const unsigned int hi = __reduce_or_sync(0xffffffffu, (unsigned int)(v >> 32));
          if (lane == 0) removed[w] |= ((unsigned long long)hi << 32) | lo;
        }
      }
    }
    __syncthreads();
  }
}

// ------------------------------------------------------------------------------------------------
// Spatial pruning of the cross test.  With a threshold >= 0 only boxes that really intersect can suppress
// each other, so the kept boxes a chunk box has to be tested against lie in a small neighbourhood.  Once
// per call ALL n boxes are counting-sorted into a uniform G^3 grid by their minimum corner (x fastest),
// as 32-byte records {corners, volume}, with one `state` BIT per slot that the scan kernel sets when the
// box is kept.  A kept box o can intersect a query box a only if, per axis,
//     o.min <= a.max   and   o.min >= a.min - wmax      (wmax = largest extent of any box, rounded up)
// and cell() is monotone, so the slots to visit are the cells [cell(a.min - wmax), cell(a.max)]: per
// (y, z) row one contiguous slot range.  One warp per query box: lanes stride over the range, look at the
// state bits and test only kept boxes.  Boxes of the same or later chunks still have state 0, which is
// exactly the "earlier kept boxes" the greedy loop asks for.  Decisions are unchanged (same iou_exceeds).
// ------------------------------------------------------------------------------------------------
// Size levels: a single very large box would widen every query's neighbourhood, so the grid is replicated
// NMS_LEVELS times and a box goes to the finest level l whose bound W / 2^l (W = largest extent of any box,
// any axis) still covers its largest extent; a query walks level l with that bound instead of W.  A level
// whose boxes are all too small to reach the threshold against the query box (volume <= bound^3 and
// IoU <= min volume / max volume) ends the walk.
#define NMS_LEVELS 4
struct GridMap {
  float lo[3], scale[3], wmax[3], W;
  int G;
};
// rng: [0..2] orderable min of the min corners, [3..5] orderable max, [6..8] bits of the largest extents
__device__ __forceinline__ GridMap load_grid(const unsigned int* __restrict__ rng, int G) {
  GridMap m;
  m.G = G;
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const float lo = float_from_orderable(rng[k]), hi = float_from_orderable(rng[3 + k]);
    const float d = hi - lo;
    m.lo[k] = lo;
    m.scale[k] = (d > 0.f && d < 3.0e38f) ? (float)G / d : 0.f;
    m.wmax[k] = __uint_as_float(rng[6 + k]);
  }
  m.W = fmaxf(m.wmax[0], fmaxf(m.wmax[1], m.wmax[2]));
  return m;
}
// finest level whose bound W / 2^l is >= every extent of the box (extents rounded up, as in wmax)
__device__ __forceinline__ int box_level(const GridMap& m, const Box6& b) {
  float e = 0.f;
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const float ext = __fsub_ru(b.v[3 + k], b.v[k]);
    if (ext > e) e = ext;
  }
  int l = 0;
  float w = m.W * 0.5f;
  while (l < NMS_LEVELS - 1 && e <= w) {
    ++l;
    w *= 0.5f;
  }
  return l;
}
// monotone non-decreasing in x (NaN -> 0)
__device__ __forceinline__ int cell_coord(const GridMap& m, int k, float x) {
  const float f = floorf((x - m.lo[k]) * m.scale[k]);
  return (f >= (float)m.G) ? m.G - 1 : ((f > 0.f) ? (int)f : 0);
}

__global__ void __launch_bounds__(256) nms_grid_range_kernel(const float* __restrict__ boxes, long long n,
                                                             unsigned int* __restrict__ rng) {
  unsigned int mn[3] = {0xffffffffu, 0xffffffffu, 0xffffffffu}, mx[3] = {0u, 0u, 0u}, wx[3] = {0u, 0u, 0u};
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const Box6 b = load_box(boxes + i * 6);
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      const unsigned int o = float_orderable(b.v[k]);
      mn[k] = min(mn[k], o);
      mx[k] = max(mx[k], o);
      float ext = __fsub_ru(b.v[3 + k], b.v[k]);
      if (!(ext > 0.f)) ext = 0.f;
      wx[k] = max(wx[k], __float_as_uint(ext));
    }
  }
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const unsigned int a = __reduce_min_sync(0xffffffffu, mn[k]);
    const unsigned int b = __reduce_max_sync(0xffffffffu, mx[k]);
    const unsigned int c = __reduce_max_sync(0xffffffffu, wx[k]);
    if ((threadIdx.x & 31) == 0) {
      atomicMin(&rng[k], a);
      atomicMax(&rng[3 + k], b);
      atomicMax(&rng[6 + k], c);
    }
  }
}

__global__ void __launch_bounds__(256) nms_grid_count_kernel(const float* __restrict__ boxes, long long n,
                                                             const unsigned int* __restrict__ rng, int G,
                                                             int* __restrict__ cell_count, int* __restrict__ cell_of) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const GridMap m = load_grid(rng, G);
  const Box6 b = load_box(boxes + i * 6);
  const int c = ((box_level(m, b) * G + cell_coord(m, 2, b.v[2])) * G + cell_coord(m, 1, b.v[1])) * G +
                cell_coord(m, 0, b.v[0]);
  cell_of[i] = c;
  atomicAdd(&cell_count[c], 1);
}

// exclusive scan of the cell counts (one block, 1024 cells per pass): cell_start[0..cells], counts reset to 0
// for the scatter
__global__ void __launch_bounds__(1024) nms_grid_scan_kernel(int* __restrict__ cell_count, int cells,
                                                             int* __restrict__ cell_start) {
  __shared__ int wsum[32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int carry = 0;
  for (int base = 0; base < cells; base += 1024) {
    const int c = base + threadIdx.x;
    const int v = (c < cells) ? cell_count[c] : 0;
    int x = v;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
      const int y = __shfl_up_sync(0xffffffffu, x, off);
      if (lane >= off) x += y;
    }
    if (lane == 31) wsum[warp] = x;
    __syncthreads();
    if (warp == 0) {
      int t = wsum[lane];
#pragma unroll
      for (int off = 1; off < 32; off <<= 1) {
        const int y = __shfl_up_sync(0xffffffffu, t, off);
        if (lane >= off) t += y;
      }
      wsum[lane] = t;
    }
    __syncthreads();
    const int before = (warp > 0 ? wsum[warp - 1] : 0) + x - v;
    const int total = wsum[31];
    if (c < cells) {
      cell_start[c] = carry + before;
      cell_count[c] = 0;
    }
    carry += total;
    __syncthreads();
  }
  if (threadIdx.x == 0) cell_start[cells] = carry;
}

__global__ void __launch_bounds__(256) nms_grid_scatter_kernel(const float* __restrict__ boxes, long long n,
                                                               const int* __restrict__ cell_start,
                                                               int* __restrict__ cursor, int* __restrict__ slot_of,
                                                               float4* __restrict__ sorted) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int c = slot_of[i];
  const int slot = cell_start[c] + atomicAdd(&cursor[c], 1);
  const Box6 b = load_box(boxes + i * 6);
  sorted[2ll * slot] = make_float4(b.v[0], b.v[1], b.v[2], b.v[3]);
  sorted[2ll * slot + 1] = make_float4(b.v[4], b.v[5], box_volume(b), 0.f);
  slot_of[i] = slot;
}

__device__ __forceinline__ void nms_cross_grid_query(int gw, const float* __restrict__ boxes, int n,
                                                     const unsigned int* __restrict__ rng, int G,
                                                     const int* __restrict__ cell_start,
                                                     const float4* __restrict__ sorted,
                                                     const unsigned int* __restrict__ state32, float thr,
                                                     unsigned int* __restrict__ rem32, int split) {
  // `split` warps share a query (they take alternate batches of 32 rows): a chunk has too few boxes to fill
  // the machine with one latency-bound warp each
  const int lane = threadIdx.x & 31;
  const int i = gw / split, part = gw - i * split;
  if (i >= n) return;                                   // whole warp
  const GridMap m = load_grid(rng, G);
  const Box6 a = load_box(boxes + (long long)i * 6);
  const float va = box_volume(a);
  // IoU > thr needs, on every axis, overlap_k > thr * extent_k(a) (inter / vol(a) <= overlap_k / extent_k), i.e.
  //   o.min_k < a.max_k - s_k   and   o.max_k > a.min_k + s_k,   s_k = thr' * extent_k(a)
  // with thr' = thr (1 - 1e-4): the margin dwarfs the few-ulp difference between the exact fp32 test and real
  // arithmetic; s_k is rounded down and the bounds outwards.  No shrink for volumes near the denormal range.
  float sh[3] = {0.f, 0.f, 0.f};
  if (thr > 0.f && va > 1e-20f) {
    const float thr1 = __fmul_rd(thr, 0.9999f);
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      const float ext = __fsub_rd(a.v[3 + k], a.v[k]);
      sh[k] = ext > 0.f ? __fmul_rd(thr1, ext) : 0.f;
    }
  }
  int chi[3];
#pragma unroll
  for (int k = 0; k < 3; ++k) chi[k] = cell_coord(m, k, __fsub_ru(a.v[3 + k], sh[k]));
  bool found = false;
  // Levels are walked starting from the query's own size class (where its suppressor most likely lives, so
  // a removed box leaves early).  A level is skipped when
  //   * its boxes are too small: volume <= w^3 < thr * vol(a)  (IoU <= min volume / max volume), or
  //   * its boxes are too large: IoU > thr also needs extent_k(o) < extent_k(a) / thr on every axis, and every
  //     box of level l < last has a largest extent > W / 2^(l+1).
  // Both with margins far above the few-ulp rounding of the exact test; false for NaN / non-positive volumes.
  const int own = box_level(m, a);
  float too_large = 3.0e38f;
  if (thr > 0.f && va > 1e-20f) {
    float e = 0.f;
#pragma unroll
    for (int k = 0; k < 3; ++k) e = fmaxf(e, __fsub_ru(a.v[3 + k], a.v[k]));
    too_large = __fmul_ru(__fdiv_ru(e, __fmul_rd(thr, 0.9999f)), 1.001f);
  }
  for (int li = 0; li < NMS_LEVELS && !found; ++li) {
    const int level = (own + li) % NMS_LEVELS;
    const float w = m.W * (1.0f / (float)(1 << level));          // exact power-of-two scaling
    if (__fmul_rn(__fmul_rn(__fmul_rn(w, w), w), 1.01f) < __fmul_rn(thr, va)) continue;
    if (level < NMS_LEVELS - 1 && w * 0.5f >= too_large) continue;
    int clo[3], hi[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      clo[k] = cell_coord(m, k, __fsub_rd(__fadd_rd(a.v[k], sh[k]), fminf(w, m.wmax[k])));
      hi[k] = chi[k] < clo[k] ? clo[k] : chi[k];         // malformed box (max < min): still a valid range
    }
    const int ny = hi[1] - clo[1] + 1;
    const int nrows = ny * (hi[2] - clo[2] + 1);
    for (int r0 = part * 32; r0 < nrows && !found; r0 += 32 * split) {
      // Every lane owns one (y, z) row = one contiguous slot range, and reads the kept BITS of that range one
      // 32-slot word per round (a row is 1-3 words).  The set bits of all 32 lanes are then dealt out evenly:
      // candidate j lives in the lane s with excl[s] <= j < incl[s] (binary search over the lanes' prefix sums),
      // at the (j - excl[s] + 1)-th set bit of that lane's word.  One memory round trip fetches the state of up
      // to 1024 slots, and every box load that follows is a really kept box.
      int begin = 0, end = 0;
      const int r = r0 + lane;
      if (r < nrows) {
        const int cz = clo[2] + r / ny, cy = clo[1] + r % ny;
        const int base = ((level * G + cz) * G + cy) * G;
        begin = cell_start[base + clo[0]];
        end = cell_start[base + hi[0] + 1];
      }
      bool more = end > begin;
      int wi = begin >> 5;
      const int wlast = (end - 1) >> 5;
      while (!found && __any_sync(0xffffffffu, more)) {
        unsigned int bits = 0u;
        if (more) {
          bits = state32[wi];
          const int lo_bit = begin - (wi << 5), hi_bit = end - (wi << 5);
          if (lo_bit > 0) bits &= 0xffffffffu << lo_bit;
          if (hi_bit < 32) bits &= (1u << hi_bit) - 1u;
        }
        const int base_slot = wi << 5;
        const int pc = __popc(bits);
        int incl = pc;
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
          const int y = __shfl_up_sync(0xffffffffu, incl, off);
          if (lane >= off) incl += y;
        }
        const int excl = incl - pc;
        const int total = __shfl_sync(0xffffffffu, incl, 31);
        for (int j0 = 0; j0 < total && !found; j0 += 32) {
          const int j = j0 + lane;
          int src = 0;                                  // largest lane with excl <= j
#pragma unroll
          for (int step = 16; step >= 1; step >>= 1) {
            const int cand = src + step;
            const int ex = __shfl_sync(0xffffffffu, excl, cand & 31);
            if (cand < 32 && ex <= j) src = cand;
          }
          const unsigned int word_s = __shfl_sync(0xffffffffu, bits, src);
          const int base_s = __shfl_sync(0xffffffffu, base_slot, src);
          const int excl_s = __shfl_sync(0xffffffffu, excl, src);
          bool hit = false;
          if (j < total) {
            const long long k = base_s + (int)__fns(word_s, 0u, j - excl_s + 1);
            const float4 p = sorted[2 * k], q = sorted[2 * k + 1];
            Box6 o;
            o.v[0] = p.x; o.v[1] = p.y; o.v[2] = p.z; o.v[3] = p.w; o.v[4] = q.x; o.v[5] = q.y;
            const float inter = box_intersection(a, o);
            const float uni = __fsub_rn(__fadd_rn(va, q.z), inter);
            hit = iou_exceeds(inter, uni, thr);
          }
          found = __any_sync(0xffffffffu, hit);
        }
        if (more) {
          if (wi >= wlast) more = false;
          else ++wi;
        }
      }
    }
  }
  if (lane == 0 && found) atomicOr(&rem32[i >> 5], 1u << (i & 31));
}

// One launch per chunk: CTA 0 resolves chunk c (greedy scan + append / flag the kept boxes, kept-list length
// recorded in nk_hist[c+1]); the other CTAs -- the scan leaves 147 SMs idle -- already work for chunk c+1:
//   * CTAs 1 .. mask_blocks: its word-major bit matrix and block flags into the other buffer (8 tiles of
//     64 x 64 per CTA);
//   * the rest: its grid-pruned cross test (16 warps per CTA).  They read `state` while CTA 0 may be setting
//     bits of chunk c: harmless, a set bit is always a really kept EARLIER box; what they can miss -- boxes
//     kept in chunk c -- is covered afterwards by a dense "delta" pass over kept-list entries
//     [nk_hist[c], nk_hist[c+1]) (at most one chunk of boxes, ~10 us).
// This takes both the matrix and the cross test off the serial path: per chunk it is scan + delta.
__global__ void __launch_bounds__(512) nms_scan_mask_kernel(
    const unsigned long long* __restrict__ mask, const float* __restrict__ boxes, int n, int words, int stride,
    const unsigned long long* __restrict__ removed_init, float4* __restrict__ kept, long long* __restrict__ nk_ptr,
    uint8_t* __restrict__ keep, const int* __restrict__ slot_of, unsigned int* __restrict__ state,
    unsigned long long* __restrict__ block_flags, int fw,
    const float* __restrict__ boxes_next, int n_next, float thr, unsigned long long* __restrict__ mask_next,
    unsigned long long* __restrict__ flags_next, long long* __restrict__ nk_hist_next, int mask_blocks,
    const unsigned int* __restrict__ rng, int G, const int* __restrict__ cell_start,
    const float4* __restrict__ sorted, unsigned int* __restrict__ rem32_next, int split) {
  extern __shared__ unsigned long long sm[];
  if ((int)blockIdx.x > mask_blocks) {
    const int gw = ((int)blockIdx.x - 1 - mask_blocks) * (blockDim.x >> 5) + (threadIdx.x >> 5);
    nms_cross_grid_query(gw, boxes_next, n_next, rng, G, cell_start, sorted, state, thr, rem32_next, split);
    return;
  }
  if (blockIdx.x != 0) {
    __shared__ float cbox[8][64][6];
    __shared__ float cvol[8][64];
    const int words_next = (n_next + 63) >> 6;
    const int sub = threadIdx.x >> 6, t = threadIdx.x & 63;
    const long long tile = (long long)(blockIdx.x - 1) * 8 + sub;
    const int rb = (int)(tile / words_next), cb = (int)(tile - (long long)rb * words_next);
    const bool active = rb < words_next && cb >= rb;
    if (active) {
      const int cj = cb * 64 + t;
      if (cj < n_next) {
        const Box6 bx = load_box(boxes_next + (long long)cj * 6);
#pragma unroll
        for (int k = 0; k < 6; ++k) cbox[sub][t][k] = bx.v[k];
        cvol[sub][t] = box_volume(bx);
      }
    }
    __syncthreads();
    if (!active) return;
    const int i = rb * 64 + t;
    unsigned long long bits = 0ull;
    if (i < n_next) {
      const Box6 a = load_box(boxes_next + (long long)i * 6);
      const float va = box_volume(a);
      const int jn = min(64, n_next - cb * 64);
      for (int b = 0; b < jn; ++b) {
        Box6 o;
#pragma unroll
        for (int k = 0; k < 6; ++k) o.v[k] = cbox[sub][b][k];
        const float inter = box_intersection(a, o);
        const float uni = __fsub_rn(__fadd_rn(va, cvol[sub][b]), inter);
        if (iou_exceeds(inter, uni, thr)) bits |= (1ull << b);
      }
      if (cb == rb) bits &= ~(1ull << t);       // a box does not suppress itself (ssd3d.py:425-426)
      mask_next[(long long)cb * stride + i] = bits;
    }
    const unsigned any = __ballot_sync(0xffffffffu, bits != 0ull);
    if (any != 0u && (threadIdx.x & 31) == 0) atomicOr(&flags_next[(long long)rb * fw + (cb >> 6)], 1ull << (cb & 63));
    return;
  }
  unsigned long long* removed = sm;
  unsigned long long* keptw = sm + words;
  unsigned long long* sflags = sm + 2 * words;
  int* prefix = reinterpret_cast<int*>(sm + 2 * words + words * fw);
  __shared__ long long s_base;
  for (int e = threadIdx.x; e < words * fw; e += blockDim.x) {
    sflags[e] = block_flags[e];
    block_flags[e] = 0ull;                               // ready for the mask of the chunk after next
  }
  nms_scan_core_tr(mask, n, stride, removed, keptw, removed_init, sflags, fw);
  __syncthreads();
  if (threadIdx.x == 0) {
    int run = 0;
    for (int w = 0; w < words; ++w) {
      prefix[w] = run;
      run += __popcll(keptw[w]);
    }
    const long long base = *nk_ptr;
    s_base = base;
    *nk_ptr = base + run;
    *nk_hist_next = base + run;
  }
  __syncthreads();
  const long long base = s_base;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const unsigned long long kw = keptw[i >> 6];
    const bool k = (kw >> (i & 63)) & 1ull;
    keep[i] = (uint8_t)k;
    if (k) {
      const long long pos = base + prefix[i >> 6] + __popcll(kw & ((1ull << (i & 63)) - 1ull));
      const Box6 b = load_box(boxes + (long long)i * 6);
      kept[2 * pos] = make_float4(b.v[0], b.v[1], b.v[2], b.v[3]);
      kept[2 * pos + 1] = make_float4(b.v[4], b.v[5], box_volume(b), 0.f);
      if (slot_of) {
        const int slot = slot_of[i];
        atomicOr(&state[slot >> 5], 1u << (slot & 31));
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------
// 64-bit key sort of any length (ascending, stable): 16384-key chunks by the shared-memory bitonic
// network, then log2(chunks) merge passes in which every key finds its output slot by a binary search in
// the sibling run (left run first on ties).  Used for candidate lists the single-block sort cannot hold.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(1024) sort_chunks_kernel(unsigned long long* __restrict__ data, long long n) {
  extern __shared__ unsigned long long keys[];
  const long long begin = (long long)blockIdx.x * SSD3D_SORT_MAX;
  long long len = n - begin;
  if (len > SSD3D_SORT_MAX) len = SSD3D_SORT_MAX;
  if (len <= 0) return;
  bitonic_sort_smem(keys, data + begin, (int)len);
  for (int i = threadIdx.x; i < (int)len; i += blockDim.x) data[begin + i] = keys[i];
}

__global__ void __launch_bounds__(256) merge_pass_kernel(const unsigned long long* __restrict__ src,
                                                         unsigned long long* __restrict__ dst, long long n,
                                                         long long run) {
  const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n) return;
  const long long r = e / run;
  const long long i = e - r * run;
  const unsigned long long key = src[e];
  const long long sib = (r ^ 1ll) * run;
  long long sib_len = n - sib;
  if (sib_len > run) sib_len = run;
  long long lo = 0;
  if (sib_len > 0) {
    const unsigned long long* s = src + sib;
    long long hi = sib_len;
    const bool right = (r & 1ll) != 0;       // right run: count sibling keys <= key; left run: < key
    while (lo < hi) {
      const long long mid = (lo + hi) >> 1;
      const unsigned long long v = s[mid];
      const bool before = right ? (v <= key) : (v < key);
      if (before) lo = mid + 1; else hi = mid;
    }
  }
  dst[(r & ~1ll) * run + i + lo] = key;
}

static inline long long align256(long long v) { return (v + 255) & ~255ll; }

// shared-memory words available for staging the bit matrix of up to n_max candidates (<= ~200 KB)
static inline long long nms_stage_words(int words, long long n_max) {
  const long long budget = (200ll * 1024) / 8 - 2ll * words;
  const long long want = n_max * (long long)words;
  return want < budget ? want : (budget > 0 ? budget : 0);
}

DetectLayout detect_layout(int N, long long P, int C, int top_k) {
  DetectLayout L;
  L.S = N * (C - 1);
  long long nm = 10ll * (long long)top_k;
  if (nm > P) nm = P;
  if (nm > SSD3D_SORT_MAX) nm = SSD3D_SORT_MAX;
  if (nm < 1) nm = 1;
  L.nmax = (int)nm;
  L.words = (L.nmax + 63) / 64;
  long long o = 0;
  L.off_count = o; o += align256(4ll * L.S);
  L.off_nkeep = o; o += align256(4ll * L.S);
  L.off_keptcnt = o; o += align256(4ll * L.S);
  L.off_boxes = o; o += align256(4ll * N * P * 6);
  L.off_cand = o; o += align256(8ll * L.S * P);
  // second key buffer for the hierarchical top-k (only when one block cannot hold all candidates)
  L.cand2_stride = (P > SSD3D_SORT_MAX) ? ((P + SSD3D_SORT_MAX - 1) / SSD3D_SORT_MAX) * L.nmax : 0;
  L.off_cand2 = o; o += align256(8ll * L.S * L.cand2_stride);
  L.off_sboxes = o; o += align256(4ll * L.S * L.nmax * 6);
  L.off_sscores = o; o += align256(4ll * L.S * L.nmax);
  L.off_sprior = o; o += align256(4ll * L.S * L.nmax);
  L.off_mask = o; o += align256(8ll * L.S * L.nmax * L.words);
  L.off_keptpos = o; o += align256(4ll * L.S * L.nmax);
  L.off_keptscore = o; o += align256(4ll * L.S * L.nmax);
  L.total = o;
  return L;
}

}  // namespace ssd3d

using namespace ssd3d;

extern "C" int64_t ssd3d_detect_workspace_bytes(int N, int64_t P, int n_classes, int top_k) {
  if (N <= 0 || P <= 0 || n_classes < 2 || top_k <= 0) return 0;
  return detect_layout(N, P, n_classes, top_k).total;
}

namespace ssd3d {
__global__ void __launch_bounds__(256) prior_boxes_kernel(const ssd3d_prior_table* __restrict__ tbl, long long P,
                                                          float* __restrict__ out) {
  const long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (p < P) store_box(out + p * 6, prior_from_table(tbl, p));
}
}  // namespace ssd3d

extern "C" int ssd3d_prior_boxes(const ssd3d_prior_table* table, int64_t P, float* out, void* stream) {
  if (!table || !out || P <= 0) return SSD3D_ERR_ARG;
  prior_boxes_kernel<<<(unsigned)((P + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(table, (long long)P, out);
  SSD3D_CHECK_LAUNCH();
  return SSD3D_OK;
}

static int decode_softmax_impl(const float* locs, const float* scores, PriorSrc priors, int N, int64_t P,
                               int n_classes, float* probs, float* boxes_xyz, void* stream) {
  if (!locs || !scores || (!priors.ptr && !priors.tbl) || !probs || !boxes_xyz || N <= 0 || P <= 0 || n_classes < 1)
    return SSD3D_ERR_ARG;
  dim3 grid((unsigned)((P + 255) / 256), (unsigned)N);
  decode_softmax_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(locs, scores, priors, P, n_classes, probs,
                                                                            boxes_xyz);
  SSD3D_CHECK_LAUNCH();
  return SSD3D_OK;
}
extern "C" int ssd3d_decode_softmax(const float* locs, const float* scores, const float* priors, int N, int64_t P,
                                    int n_classes, float* probs, float* boxes_xyz, void* stream) {
  return decode_softmax_impl(locs, scores, PriorSrc{priors, nullptr}, N, P, n_classes, probs, boxes_xyz, stream);
}
extern "C" int ssd3d_decode_softmax_analytic(const float* locs, const float* scores, const ssd3d_prior_table* table,
                                             int N, int64_t P, int n_classes, float* probs, float* boxes_xyz,
                                             void* stream) {
  return decode_softmax_impl(locs, scores, PriorSrc{nullptr, table}, N, P, n_classes, probs, boxes_xyz, stream);
}

extern "C" int ssd3d_nms3d_sorted(const float* boxes_xyz, int64_t n, float max_overlap, uint8_t* keep, void* mask_ws,
                                  void* stream) {
  if (!boxes_xyz || !keep || !mask_ws || n <= 0 || n > 131072) return SSD3D_ERR_ARG;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int words = (int)((n + 63) / 64);
  dim3 grid((unsigned)words, (unsigned)words, 1);
  nms_mask_kernel<<<grid, 64, 0, st>>>(boxes_xyz, nullptr, (int)n, 0, words, 0, max_overlap,
                                       static_cast<unsigned long long*>(mask_ws));
  SSD3D_CHECK_LAUNCH();
  const long long stage_words = nms_stage_words(words, n);
  const size_t smem = (size_t)(2 * words + stage_words) * 8;
  if (smem > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(nms_scan_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
  }
  nms_scan_kernel<<<1, 256, smem, st>>>(static_cast<const unsigned long long*>(mask_ws), (int)n, words, stage_words,
                                        keep);
  SSD3D_CHECK_LAUNCH();
  return SSD3D_OK;
}

// ---- chunked NMS / long sort / filter stage entry points ------------------------------------------
namespace ssd3d {
struct ChunkedNmsLayout {
  int chunk, G, cells;
  long long flags_bytes, mask_bytes;
  long long off_removed, off_nk, off_rng, off_hist, off_flags, off_kept, off_mask, off_cellstart, off_cursor, off_sorted, off_slot, off_state,
      total;
};
static ChunkedNmsLayout chunked_nms_layout(long long n, int chunk) {
  ChunkedNmsLayout L;
  if (chunk <= 0) chunk = 4096;                          // measured optimum from 64 k to 2.5 M candidates
  L.chunk = chunk;
  int G = (int)cbrt((double)n / 8.0);
  L.G = G < 1 ? 1 : (G > 64 ? 64 : G);
  L.cells = NMS_LEVELS * L.G * L.G * L.G;
  const long long cw = chunk / 64;
  const long long chunks = (n + chunk - 1) / chunk;
  long long o = 0;
  L.off_removed = o; o += align256(8ll * chunks * cw);
  L.off_nk = o; o += 256;
  L.off_rng = o; o += 256;
  L.off_hist = o; o += align256(8ll * (chunks + 1));
  L.flags_bytes = align256(8ll * cw * ((cw + 63) / 64));
  L.off_flags = o; o += 2 * L.flags_bytes;
  L.off_kept = o; o += align256(32ll * n);
  L.mask_bytes = align256(8ll * chunk * cw);
  L.off_mask = o; o += 2 * L.mask_bytes;
  L.off_cellstart = o; o += align256(4ll * (L.cells + 1));
  L.off_cursor = o; o += align256(4ll * L.cells);
  L.off_sorted = o; o += align256(32ll * n);
  L.off_slot = o; o += align256(4ll * n);
  L.off_state = o; o += align256(n);
  L.total = o;
  return L;
}
static inline bool chunk_ok(int chunk) { return chunk == 0 || (chunk >= 64 && chunk <= SSD3D_SORT_MAX && chunk % 64 == 0); }
}  // namespace ssd3d

extern "C" int64_t ssd3d_nms3d_chunked_workspace_bytes(int64_t n, int chunk) {
  if (n <= 0 || n > 0x7fffffffll || !chunk_ok(chunk)) return 0;
  return chunked_nms_layout(n, chunk).total;
}

extern "C" int ssd3d_nms3d_sorted_chunked(const float* boxes_xyz, int64_t n, float max_overlap, uint8_t* keep,
                                          int64_t* kept_count, void* workspace, int64_t workspace_bytes, int chunk,
                                          int flags, void* stream) {
  if (!boxes_xyz || !keep || !workspace || n <= 0 || n > 0x7fffffffll || !chunk_ok(chunk)) return SSD3D_ERR_ARG;
  const ChunkedNmsLayout L = chunked_nms_layout(n, chunk);
  if (workspace_bytes < L.total) return SSD3D_ERR_ARG;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  uint8_t* ws = static_cast<uint8_t*>(workspace);
  unsigned long long* removed = reinterpret_cast<unsigned long long*>(ws + L.off_removed);
  long long* nk = reinterpret_cast<long long*>(ws + L.off_nk);
  unsigned int* rng = reinterpret_cast<unsigned int*>(ws + L.off_rng);
  float4* kept = reinterpret_cast<float4*>(ws + L.off_kept);
  int* cell_start = reinterpret_cast<int*>(ws + L.off_cellstart);
  int* cursor = reinterpret_cast<int*>(ws + L.off_cursor);
  float4* sorted = reinterpret_cast<float4*>(ws + L.off_sorted);
  int* slot_of = reinterpret_cast<int*>(ws + L.off_slot);
  unsigned int* state = reinterpret_cast<unsigned int*>(ws + L.off_state);   // one kept bit per grid slot
  cudaError_t e = cudaMemsetAsync(ws, 0, (size_t)L.off_kept, st);      // removed bits, kept counter, grid range, flags
  if (e != cudaSuccess) return (int)e;
  const int B = L.chunk, cw = B / 64, fw = (cw + 63) / 64;
  const long long chunks = (n + B - 1) / B;
  // The grid only helps when disjoint boxes cannot suppress each other (threshold >= 0; NaN compares false).
  const bool use_grid = chunks > 1 && max_overlap >= 0.0f && !(flags & SSD3D_NMS_NO_GRID);
  if (use_grid) {
    e = cudaMemsetAsync(rng, 0xff, 12, st);                            // running minima start at the top
    if (e != cudaSuccess) return (int)e;
    e = cudaMemsetAsync(cursor, 0, (size_t)L.cells * 4, st);
    if (e != cudaSuccess) return (int)e;
    e = cudaMemsetAsync(state, 0, (size_t)((n + 31) / 32) * 4, st);
    if (e != cudaSuccess) return (int)e;
    const unsigned nb = (unsigned)((n + 255) / 256);
    nms_grid_range_kernel<<<nb < 1184u ? nb : 1184u, 256, 0, st>>>(boxes_xyz, (long long)n, rng);
    SSD3D_CHECK_LAUNCH();
    nms_grid_count_kernel<<<nb, 256, 0, st>>>(boxes_xyz, (long long)n, rng, L.G, cursor, slot_of);
    SSD3D_CHECK_LAUNCH();
    nms_grid_scan_kernel<<<1, 1024, 0, st>>>(cursor, L.cells, cell_start);
    SSD3D_CHECK_LAUNCH();
    nms_grid_scatter_kernel<<<nb, 256, 0, st>>>(boxes_xyz, (long long)n, cell_start, cursor, slot_of, sorted);
    SSD3D_CHECK_LAUNCH();
  }
  long long* hist = reinterpret_cast<long long*>(ws + L.off_hist);      // hist[c] = kept boxes before chunk c
  for (long long c = 0; c < chunks; ++c) {
    const long long first = c * B;
    const int rows = (int)((n - first) < B ? (n - first) : B);
    const int words = (rows + 63) / 64;
    const float* cb = boxes_xyz + first * 6;
    unsigned long long* crem = removed + c * cw;
    if (c > 0) {
      // grid mode: the grid-pruned cross test of this chunk ran inside the previous launch; what is left are
      // the boxes kept in chunk c-1.  Dense mode: the whole kept list.  x (B / 256) row blocks.
      dim3 grid((unsigned)((rows + 255) / 256), use_grid ? 16u : 74u);
      nms_cross_kernel<<<grid, 256, 0, st>>>(cb, rows, kept, use_grid ? hist + (c - 1) : hist, hist + c, max_overlap,
                                             reinterpret_cast<unsigned int*>(crem));
      SSD3D_CHECK_LAUNCH();
    }
    unsigned long long* mask_cur = reinterpret_cast<unsigned long long*>(ws + L.off_mask + (c & 1) * L.mask_bytes);
    unsigned long long* mask_nxt = reinterpret_cast<unsigned long long*>(ws + L.off_mask + ((c + 1) & 1) * L.mask_bytes);
    unsigned long long* flags_cur = reinterpret_cast<unsigned long long*>(ws + L.off_flags + (c & 1) * L.flags_bytes);
    unsigned long long* flags_nxt = reinterpret_cast<unsigned long long*>(ws + L.off_flags + ((c + 1) & 1) * L.flags_bytes);
    if (c == 0) {                                       // later chunks get their matrix from the previous launch
      dim3 mgrid((unsigned)words, (unsigned)words, 1);
      nms_mask_tr_kernel<<<mgrid, 64, 0, st>>>(cb, rows, B, max_overlap, mask_cur, flags_cur, fw);
      SSD3D_CHECK_LAUNCH();
    }
    const long long nfirst = first + B;
    const int nrows = (c + 1 < chunks) ? (int)((n - nfirst) < B ? (n - nfirst) : B) : 0;
    const long long nwords = (nrows + 63) / 64;
    const int mask_blocks = (int)((nwords * nwords + 7) / 8);
    const int split = nrows <= 4736 ? 2 : 1;            // 148 SMs x 64 warps = 9472 resident warps
    const int cross_blocks = use_grid ? (int)(((long long)nrows * split + 15) / 16) : 0;
    const size_t smem = (size_t)(2 * words + words * fw) * 8 + (size_t)(words + 2) * 4;
    nms_scan_mask_kernel<<<(unsigned)(1 + mask_blocks + cross_blocks), 512, smem, st>>>(
        mask_cur, cb, rows, words, B, crem, kept, nk, keep + first, use_grid ? slot_of + first : (const int*)nullptr,
        state, flags_cur, fw, boxes_xyz + nfirst * 6, nrows, max_overlap, mask_nxt, flags_nxt, hist + (c + 1),
        mask_blocks, rng, L.G, cell_start, sorted, reinterpret_cast<unsigned int*>(removed + (c + 1) * cw), split);
    SSD3D_CHECK_LAUNCH();
  }
  if (kept_count) {
    e = cudaMemcpyAsync(kept_count, nk, 8, cudaMemcpyDeviceToDevice, st);
    if (e != cudaSuccess) return (int)e;
  }
  return SSD3D_OK;
}

extern "C" int ssd3d_sort_keys_u64(uint64_t* keys, int64_t n, uint64_t* tmp, void* stream) {
  if (!keys || n < 0 || (n > SSD3D_SORT_MAX && !tmp)) return SSD3D_ERR_ARG;
  if (n <= 1) return SSD3D_OK;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  int cap = 1;
  while (cap < n && cap < SSD3D_SORT_MAX) cap <<= 1;
  const size_t smem = (size_t)cap * 8;
  if (smem > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(sort_chunks_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
  }
  const long long chunks = (n + SSD3D_SORT_MAX - 1) / SSD3D_SORT_MAX;
  sort_chunks_kernel<<<(unsigned)chunks, 1024, smem, st>>>(reinterpret_cast<unsigned long long*>(keys), (long long)n);
  SSD3D_CHECK_LAUNCH();
  unsigned long long* src = reinterpret_cast<unsigned long long*>(keys);
  unsigned long long* dst = reinterpret_cast<unsigned long long*>(tmp);
  for (long long run = SSD3D_SORT_MAX; run < n; run <<= 1) {
    merge_pass_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(src, dst, (long long)n, run);
    SSD3D_CHECK_LAUNCH();
    unsigned long long* t = src; src = dst; dst = t;
  }
  if (src != reinterpret_cast<unsigned long long*>(keys)) {
    cudaError_t e = cudaMemcpyAsync(keys, src, (size_t)n * 8, cudaMemcpyDeviceToDevice, st);
    if (e != cudaSuccess) return (int)e;
  }
  return SSD3D_OK;
}

static int decode_filter_impl(const float* locs, const float* scores, PriorSrc priors, int N, int64_t P,
                              int n_classes, float min_score, float* boxes_xyz, uint64_t* cand, int32_t* count,
                              void* stream) {
  if (!locs || !scores || (!priors.ptr && !priors.tbl) || !boxes_xyz || !cand || !count) return SSD3D_ERR_ARG;
  if (N <= 0 || P <= 0 || n_classes < 2 || P > 0x7fffffffll) return SSD3D_ERR_ARG;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  cudaError_t e = cudaMemsetAsync(count, 0, (size_t)N * (n_classes - 1) * 4, st);
  if (e != cudaSuccess) return (int)e;
  dim3 grid((unsigned)((P + 255) / 256), (unsigned)N);
  decode_filter_kernel<<<grid, 256, 0, st>>>(locs, scores, priors, (long long)P, n_classes, min_score, boxes_xyz,
                                             reinterpret_cast<unsigned long long*>(cand), count);
  SSD3D_CHECK_LAUNCH();
  return SSD3D_OK;
}

extern "C" int ssd3d_decode_filter(const float* locs, const float* scores, const float* priors, int N, int64_t P,
                                   int n_classes, float min_score, float* boxes_xyz, uint64_t* cand, int32_t* count,
                                   void* stream) {
  return decode_filter_impl(locs, scores, PriorSrc{priors, nullptr}, N, P, n_classes, min_score, boxes_xyz, cand, count,
                            stream);
}
extern "C" int ssd3d_decode_filter_analytic(const float* locs, const float* scores, const ssd3d_prior_table* table,
                                            int N, int64_t P, int n_classes, float min_score, float* boxes_xyz,
                                            uint64_t* cand, int32_t* count, void* stream) {
  return decode_filter_impl(locs, scores, PriorSrc{nullptr, table}, N, P, n_classes, min_score, boxes_xyz, cand, count,
                            stream);
}

namespace ssd3d {
// Stages 2-4 of detect_objects on the per-(image, class) candidate lists that a stage-1 kernel left in the workspace
// (count, cand and the boxes they index, laid out by detect_layout): sort -> 10*top_k truncation -> bit-matrix NMS ->
// per-image class merge, top-k and placeholder.  ssd3d_detect_objects and ssd3d_merge_windows share it.
int detect_select(const DetectLayout& L, uint8_t* ws, int N, long long P, int n_classes, float max_overlap, int top_k,
                  float* out_boxes, float* out_scores, int64_t* out_labels, int64_t* out_prior, int32_t* out_count,
                  int32_t* status, cudaStream_t st) {
  cudaError_t e = cudaSuccess;
  int* count = reinterpret_cast<int*>(ws + L.off_count);
  int* nkeep = reinterpret_cast<int*>(ws + L.off_nkeep);
  int* keptcnt = reinterpret_cast<int*>(ws + L.off_keptcnt);
  float* boxes = reinterpret_cast<float*>(ws + L.off_boxes);
  unsigned long long* cand = reinterpret_cast<unsigned long long*>(ws + L.off_cand);
  float* sboxes = reinterpret_cast<float*>(ws + L.off_sboxes);
  float* sscores = reinterpret_cast<float*>(ws + L.off_sscores);
  int* sprior = reinterpret_cast<int*>(ws + L.off_sprior);
  unsigned long long* mask = reinterpret_cast<unsigned long long*>(ws + L.off_mask);
  int* keptpos = reinterpret_cast<int*>(ws + L.off_keptpos);
  float* keptscore = reinterpret_cast<float*>(ws + L.off_keptscore);
  {
    int cap = 1;
    while (cap < P && cap < SSD3D_SORT_MAX) cap <<= 1;
    const size_t smem = (size_t)cap * 8;
    if (smem > 48 * 1024) {
      e = cudaFuncSetAttribute(sort_segments_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
      if (e != cudaSuccess) return (int)e;
      e = cudaFuncSetAttribute(topk_reduce_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
      if (e != cudaSuccess) return (int)e;
    }
    if (P <= SSD3D_SORT_MAX) {
      SSD3D_LAUNCH_PDL(sort_segments_kernel, dim3(L.S), dim3(1024), smem, st, cand, (long long)P, count, 0, nkeep, boxes,
                       (long long)P, n_classes, L.nmax, cap, sboxes, sscores, sprior, status);
    } else {
      // hierarchical top-nmax: every level shrinks the list by SORT_MAX / nmax (>= 2)
      if (L.nmax > SSD3D_SORT_MAX / 2) return SSD3D_ERR_UNSUPPORTED;
      unsigned long long* cand2 = reinterpret_cast<unsigned long long*>(ws + L.off_cand2);
      const unsigned long long* src = cand;
      long long src_stride = P;
      unsigned long long* dst = cand2;
      long long dst_stride = L.cand2_stride;
      const int* cnt = count;
      long long len = P;
      while (len > SSD3D_SORT_MAX) {
        const long long chunks = (len + SSD3D_SORT_MAX - 1) / SSD3D_SORT_MAX;
        dim3 grid((unsigned)chunks, (unsigned)L.S);
        SSD3D_LAUNCH_PDL(topk_reduce_kernel, grid, dim3(1024), smem, st, src, src_stride, cnt, (int)len, dst, dst_stride,
                         L.nmax, SSD3D_SORT_MAX);
        len = chunks * L.nmax;
        cnt = nullptr;
        // ping-pong: the buffer just read becomes the next destination
        unsigned long long* next_dst = (dst == cand2) ? cand : cand2;
        const long long next_stride = (dst == cand2) ? P : L.cand2_stride;
        src = dst; src_stride = dst_stride;
        dst = next_dst; dst_stride = next_stride;
      }
      SSD3D_LAUNCH_PDL(sort_segments_kernel, dim3(L.S), dim3(1024), smem, st, src, src_stride, (const int*)nullptr, (int)len,
                       nkeep, boxes, (long long)P, n_classes, L.nmax, cap, sboxes, sscores, sprior, status);
    }
  }
  {
    dim3 grid((unsigned)L.words, (unsigned)L.words, (unsigned)L.S);
    SSD3D_LAUNCH_PDL(nms_mask_kernel, grid, dim3(64), 0, st, sboxes, nkeep, 0, (long long)L.nmax * 6, L.words,
                     (long long)L.nmax * L.words, max_overlap, mask);
  }
  {
    const long long stage_words = nms_stage_words(L.words, L.nmax);
    const size_t smem = (size_t)(2 * L.words + stage_words) * 8;
    if (smem > 48 * 1024) {
      e = cudaFuncSetAttribute(nms_select_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
      if (e != cudaSuccess) return (int)e;
    }
    SSD3D_LAUNCH_PDL(nms_select_kernel, dim3(N), dim3(512), smem, st, mask, nkeep, n_classes, L.nmax, L.words, stage_words,
                     sboxes, sscores, sprior, keptpos, keptscore, keptcnt, top_k, out_boxes, out_scores,
                     reinterpret_cast<long long*>(out_labels), reinterpret_cast<long long*>(out_prior), out_count);
  }
  return SSD3D_OK;
}
}  // namespace ssd3d

static int detect_objects_impl(const float* locs, const float* scores, PriorSrc priors, int N, int64_t P,
                               int n_classes, float min_score, float max_overlap, int top_k, float* out_boxes,
                               float* out_scores, int64_t* out_labels, int64_t* out_prior, int32_t* out_count,
                               void* workspace, int64_t workspace_bytes, int32_t* status, void* stream) {
  if (!locs || !scores || (!priors.ptr && !priors.tbl) || !out_boxes || !out_scores || !out_labels || !out_prior || !out_count || !workspace)
    return SSD3D_ERR_ARG;
  if (N <= 0 || P <= 0 || n_classes < 2 || top_k <= 0 || P > 0x7fffffffll) return SSD3D_ERR_ARG;
  const DetectLayout L = detect_layout(N, P, n_classes, top_k);
  if (workspace_bytes < L.total) return SSD3D_ERR_ARG;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  uint8_t* ws = static_cast<uint8_t*>(workspace);
  int* count = reinterpret_cast<int*>(ws + L.off_count);
  float* boxes = reinterpret_cast<float*>(ws + L.off_boxes);
  unsigned long long* cand = reinterpret_cast<unsigned long long*>(ws + L.off_cand);

  cudaError_t e = cudaMemsetAsync(count, 0, (size_t)(L.off_boxes - L.off_count), st);
  if (e != cudaSuccess) return (int)e;
  if (status) {
    e = cudaMemsetAsync(status, 0, 4, st);
    if (e != cudaSuccess) return (int)e;
  }
  {
    dim3 grid((unsigned)((P + 255) / 256), (unsigned)N);
    SSD3D_LAUNCH_PDL(decode_filter_kernel, grid, dim3(256), 0, st, locs, scores, priors, (long long)P, n_classes, min_score, boxes,
                     cand, count);
  }
  return detect_select(L, ws, N, P, n_classes, max_overlap, top_k, out_boxes, out_scores, out_labels, out_prior,
                       out_count, status, st);
}

extern "C" int ssd3d_detect_objects(const float* locs, const float* scores, const float* priors, int N, int64_t P,
                                    int n_classes, float min_score, float max_overlap, int top_k, float* out_boxes,
                                    float* out_scores, int64_t* out_labels, int64_t* out_prior, int32_t* out_count,
                                    void* workspace, int64_t workspace_bytes, int32_t* status, void* stream) {
  return detect_objects_impl(locs, scores, PriorSrc{priors, nullptr}, N, P, n_classes, min_score, max_overlap, top_k,
                             out_boxes, out_scores, out_labels, out_prior, out_count, workspace, workspace_bytes, status,
                             stream);
}

extern "C" int ssd3d_detect_objects_analytic(const float* locs, const float* scores, const ssd3d_prior_table* table,
                                             int N, int64_t P, int n_classes, float min_score, float max_overlap,
                                             int top_k, float* out_boxes, float* out_scores, int64_t* out_labels,
                                             int64_t* out_prior, int32_t* out_count, void* workspace,
                                             int64_t workspace_bytes, int32_t* status, void* stream) {
  return detect_objects_impl(locs, scores, PriorSrc{nullptr, table}, N, P, n_classes, min_score, max_overlap, top_k,
                             out_boxes, out_scores, out_labels, out_prior, out_count, workspace, workspace_bytes, status,
                             stream);
}
