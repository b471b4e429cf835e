// tcgen05 / TMEM GEMMs of the SSD3D network, operands staged by TMA into 128B/64B-swizzled shared memory:
//   * pointwise 1x1x1 conv + BN + ReLU            y[M, Cout] = relu((x[M, Cin] . w[Cout, Cin]^T) * scale + shift)
//     (mobilenet.py:40,45; NaN check of mobilenet.py:46 folded into the epilogue)
//   * SSD head: loc conv and class conv (3x3x3, pad 1, bias) of one feature map as ONE implicit GEMM.
//     The im2col never exists: for tap (kd,kh,kw) the A tile is a 5-D TMA box of the channels-last
//     activation shifted by (kd-1,kh-1,kw-1); out-of-bounds voxels are zero-filled by the TMA unit, which
//     is exactly the conv's zero padding.  The epilogue adds the bias and writes directly into the
//     concatenated (N,P,6) / (N,P,n_classes) outputs at the layer's prior offset (ssd3d.py:131-167).
//
// Warp roles (192 threads): warps 0-3 epilogue (TMEM lane quarter = warp id), warp 4 TMA producer,
// warp 5 TMEM allocator + single-thread UMMA issuer.  smem ring of `stages` {A,B} slots with
// full/empty mbarriers; accumulator = 128 lanes x BN fp32 columns of TMEM.
#include "common.cuh"
#include "tma_host.h"

namespace ssd3d {

struct GemmParams {
  int num_kb;        // K iterations of BK elements
  int BN;            // tile width in N (UMMA N), multiple of 16, <= 256
  int stages;        // smem ring depth
  int tmem_cols;     // power of two >= max(32, BN)
  int* nan_flag;
  float floor;       // activation floor of the pointwise epilogue: 0 = ReLU, -inf = identity
  // ---- pointwise ----
  long long M;
  int Cout;
  __nv_bfloat16* y;
  const float* scale;
  const float* shift;
  // ---- head ----
  int C, D, H, W, N;
  int TW, TH, TD, TN;          // spatial/batch extent of one 128-row tile
  int tiles_w, tiles_h, tiles_d;
  int n_loc, n_cls;            // bpl*6, bpl*n_classes
  int bpl, n_classes;
  long long P, prior_off;
  float* locs;
  float* scores;
  const float* bias;
};

template <int BK>
struct SmemCfg {
  static constexpr int A_BYTES = 128 * BK * 2;
  static constexpr uint32_t SBO = 8 * BK * 2;           // bytes between 8-row groups
  static constexpr uint32_t LAYOUT = (BK == 64) ? 2u : 4u;  // SWIZZLE_128B : SWIZZLE_64B
};

template <int BK>
__device__ __forceinline__ uint64_t make_desc(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFFu) >> 4);
  d |= (uint64_t)1 << 16;                                  // LBO: unused for swizzled K-major
  d |= (uint64_t)(SmemCfg<BK>::SBO >> 4) << 32;
  d |= (uint64_t)1 << 46;                                  // descriptor version (Blackwell)
  d |= (uint64_t)SmemCfg<BK>::LAYOUT << 61;
  return d;
}

template <int BK, bool HEAD>
__global__ void __launch_bounds__(192, 1) gemm_tc_kernel(const __grid_constant__ CUtensorMap tmA,
                                                         const __grid_constant__ CUtensorMap tmB,
                                                         const GemmParams p) {
  extern __shared__ uint8_t smem_raw[];
  // 1024-byte alignment: required by the 128B swizzle atom (8 rows x 128 B)
  const uint32_t raw = smem_u32(smem_raw);
  uint8_t* smem = smem_raw + ((1024u - (raw & 1023u)) & 1023u);
  constexpr int A_BYTES = SmemCfg<BK>::A_BYTES;
  const int B_BYTES = p.BN * BK * 2;
  const int STAGE_BYTES = A_BYTES + B_BYTES;
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + (size_t)p.stages * STAGE_BYTES);
  uint64_t* empty = full + p.stages;
  uint64_t* tmem_full = empty + p.stages;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_full + 1);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  if (warp == 4 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    for (int s = 0; s < p.stages; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], 1);
    }
    mbar_init(tmem_full, 1);
    fence_barrier_init();
  }
  if (warp == 5) {
    tmem_alloc(tmem_slot, (uint32_t)p.tmem_cols);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_wait();                 // prologue above overlapped the previous kernel's tail
  pdl_launch_dependents();

  // ---- tile coordinates ----
  int m0 = 0, n0 = 0;                   // pointwise
  int tw0 = 0, th0 = 0, td0 = 0, tn0 = 0;  // head
  if constexpr (!HEAD) {
    m0 = blockIdx.x * 128;
    n0 = blockIdx.y * p.BN;
  } else {
    int t = blockIdx.x;
    tw0 = (t % p.tiles_w) * p.TW; t /= p.tiles_w;
    th0 = (t % p.tiles_h) * p.TH; t /= p.tiles_h;
    td0 = (t % p.tiles_d) * p.TD; t /= p.tiles_d;
    tn0 = t * p.TN;
  }

  if (warp == 4) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      const int KC = HEAD ? (p.C / BK) : 1;
      for (int kb = 0; kb < p.num_kb; ++kb) {
        const int s = kb % p.stages;
        const int use = kb / p.stages;
        if (use > 0) mbar_wait(&empty[s], (uint32_t)((use - 1) & 1));
        uint8_t* a_dst = smem + (size_t)s * STAGE_BYTES;
        uint8_t* b_dst = a_dst + A_BYTES;
        mbar_arrive_expect_tx(&full[s], (uint32_t)STAGE_BYTES);
        if constexpr (!HEAD) {
          tma_load_2d(a_dst, &tmA, &full[s], kb * BK, m0);
          tma_load_2d(b_dst, &tmB, &full[s], kb * BK, n0);
        } else {
          const int tap = kb / KC, kc = kb - tap * KC;
          const int kd = tap / 9, kh = (tap / 3) % 3, kw = tap % 3;
          tma_load_5d(a_dst, &tmA, &full[s], kc * BK, tw0 + kw - 1, th0 + kh - 1, td0 + kd - 1, tn0);
          tma_load_2d(b_dst, &tmB, &full[s], tap * p.C + kc * BK, 0);
        }
      }
    }
    __syncwarp();
  } else if (warp == 5) {
    // ===================== UMMA issuer =====================
    if (lane == 0) {
      const uint32_t idesc = umma_idesc_bf16(128, p.BN);
      for (int kb = 0; kb < p.num_kb; ++kb) {
        const int s = kb % p.stages;
        mbar_wait(&full[s], (uint32_t)((kb / p.stages) & 1));
        tc_fence_after();
        const uint32_t a_addr = smem_u32(smem + (size_t)s * STAGE_BYTES);
        const uint64_t da = make_desc<BK>(a_addr);
        const uint64_t db = make_desc<BK>(a_addr + A_BYTES);
#pragma unroll
        for (int k = 0; k < BK / 16; ++k) {
          // advance 16 bf16 = 32 bytes along K inside the swizzled row: +2 in the (addr >> 4) field
          umma_bf16_ss(tmem_base, da + (uint64_t)(2 * k), db + (uint64_t)(2 * k), idesc, (kb | k) != 0 ? 1u : 0u);
        }
        umma_commit(&empty[s]);   // smem slot reusable once these MMAs have read it
      }
      umma_commit(tmem_full);     // accumulator complete
    }
    __syncwarp();
  } else {
    // ===================== epilogue: TMEM -> registers -> global =====================
    mbar_wait(tmem_full, 0);
    __syncwarp();               // tcgen05.ld is .sync.aligned: reconverge after the per-thread poll loop
    tc_fence_after();
    const int row = warp * 32 + lane;                  // tile row == TMEM lane
    const uint32_t taddr = tmem_base + ((uint32_t)(warp * 32) << 16);
    bool bad = false;
    if constexpr (!HEAD) {
      const long long m = (long long)m0 + row;
      __nv_bfloat16* yrow = p.y + m * p.Cout + n0;
      for (int c = 0; c < p.BN; c += 16) {
        uint32_t v[16];
        tmem_ld_32x32b_x16(taddr + (uint32_t)c, v);
        tmem_ld_wait();
        if (m < p.M && (n0 + c) < p.Cout) {
          uint32_t o[8];
#pragma unroll
          for (int j = 0; j < 16; j += 4) {
            const float4 sc = __ldg(reinterpret_cast<const float4*>(p.scale + n0 + c + j));
            const float4 sh = __ldg(reinterpret_cast<const float4*>(p.shift + n0 + c + j));
            const float r0 = clamp_floor(__fadd_rn(__fmul_rn(__uint_as_float(v[j + 0]), sc.x), sh.x), p.floor);
            const float r1 = clamp_floor(__fadd_rn(__fmul_rn(__uint_as_float(v[j + 1]), sc.y), sh.y), p.floor);
            const float r2 = clamp_floor(__fadd_rn(__fmul_rn(__uint_as_float(v[j + 2]), sc.z), sh.z), p.floor);
            const float r3 = clamp_floor(__fadd_rn(__fmul_rn(__uint_as_float(v[j + 3]), sc.w), sh.w), p.floor);
            bad |= (r0 != r0) | (r1 != r1) | (r2 != r2) | (r3 != r3);
            o[j / 2] = pack_bf16x2(r0, r1);
            o[j / 2 + 1] = pack_bf16x2(r2, r3);
          }
          uint4* dst = reinterpret_cast<uint4*>(yrow + c);
          dst[0] = make_uint4(o[0], o[1], o[2], o[3]);
          dst[1] = make_uint4(o[4], o[5], o[6], o[7]);
        }
      }
      if (bad && p.nan_flag) atomicOr(p.nan_flag, SSD3D_NAN_BACKBONE);
    } else {
      // row -> (w, h, d, n) inside the tile, w fastest (the order the TMA box is laid out in smem)
      int r = row;
      const int w = tw0 + r % p.TW; r /= p.TW;
      const int h = th0 + r % p.TH; r /= p.TH;
      const int d = td0 + r % p.TD; r /= p.TD;
      const int n = tn0 + r;
      const bool valid = (w < p.W) && (h < p.H) && (d < p.D) && (n < p.N);
      const long long prior = p.prior_off + (((long long)d * p.H + h) * p.W + w) * p.bpl;
      float* lp = p.locs + ((long long)n * p.P + prior) * 6;
      float* sp = p.scores + ((long long)n * p.P + prior) * p.n_classes;
      bool bad_l = false, bad_s = false;
      for (int c = 0; c < p.BN; c += 16) {
        uint32_t v[16];
        tmem_ld_32x32b_x16(taddr + (uint32_t)c, v);
        tmem_ld_wait();
        if (valid) {
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            const int col = c + j;
            const float val = __fadd_rn(__uint_as_float(v[j]), __ldg(p.bias + col));
            if (col < p.n_loc) {
              lp[col] = val;
              bad_l |= (val != val);
            } else if (col < p.n_loc + p.n_cls) {
              sp[col - p.n_loc] = val;
              bad_s |= (val != val);
            }
          }
        }
      }
      if (p.nan_flag) {
        if (bad_l) atomicOr(p.nan_flag, SSD3D_NAN_LOCS);
        if (bad_s) atomicOr(p.nan_flag, SSD3D_NAN_SCORES);
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 5) {
    tc_fence_after();
    tmem_dealloc(tmem_base, (uint32_t)p.tmem_cols);
  }
}

static inline int pow2_ceil(int v) {
  int r = 1;
  while (r < v) r <<= 1;
  return r;
}

static inline size_t gemm_smem_bytes(int BK, int BN, int stages) {
  return (size_t)stages * (128 * BK * 2 + BN * BK * 2) + (2 * stages + 1) * 8 + 16 + 1024;
}

template <int BK, bool HEAD>
static int launch_gemm(const CUtensorMap& tmA, const CUtensorMap& tmB, const GemmParams& p, dim3 grid,
                       cudaStream_t st) {
  const size_t smem = gemm_smem_bytes(BK, p.BN, p.stages);
  cudaError_t e = cudaFuncSetAttribute(gemm_tc_kernel<BK, HEAD>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return (int)e;
  SSD3D_LAUNCH_PDL((gemm_tc_kernel<BK, HEAD>), grid, dim3(192), smem, st, tmA, tmB, p);
  return SSD3D_OK;
}

}  // namespace ssd3d

using namespace ssd3d;

// gemm_pw.cu: persistent, double-buffered-TMEM variant for problems with many tiles
int ssd3d_pwconv_persistent(const void* x, const void* w, const float* scale, const float* shift, void* y, int64_t M,
                            int Cin, int Cout, float floor, int* nan_flag, cudaStream_t st);

extern "C" int ssd3d_pwconv_affine(const void* x, const void* w, const float* scale, const float* shift, void* y,
                                   int64_t M, int Cin, int Cout, int relu, int* nan_flag, void* stream) {
  if (!x || !w || !scale || !shift || !y || M <= 0) return SSD3D_ERR_ARG;
  if (Cin <= 0 || (Cin % 32) || Cout <= 0 || (Cout % 16)) return SSD3D_ERR_ARG;
  {
    const int rc = ssd3d_pwconv_persistent(x, w, scale, shift, y, M, Cin, Cout, SSD3D_FLOOR(relu), nan_flag,
                                           static_cast<cudaStream_t>(stream));
    if (rc != SSD3D_ERR_UNSUPPORTED) return rc;
  }
  const int BK = (Cin % 64 == 0) ? 64 : 32;
  const long long m_tiles = (M + 127) / 128;
  // tile width: the widest of {256,128,64,32,16} dividing Cout, narrowed while the grid would leave
  // most of the 148 SMs idle (tail layers: M = 512 rows)
  int BN = 16;
  for (int c : {256, 128, 64, 32, 16})
    if (Cout % c == 0) { BN = c; break; }
  while (BN > 32 && m_tiles * (Cout / BN) < 148) BN >>= 1;
  GemmParams p{};
  p.num_kb = Cin / BK;
  p.BN = BN;
  p.stages = p.num_kb < 4 ? p.num_kb : 4;
  p.tmem_cols = pow2_ceil(BN < 32 ? 32 : BN);
  p.nan_flag = nan_flag;
  p.floor = SSD3D_FLOOR(relu);
  p.M = M;
  p.Cout = Cout;
  p.y = static_cast<__nv_bfloat16*>(y);
  p.scale = scale;
  p.shift = shift;

  CUtensorMap tmA, tmB;
  const CUtensorMapSwizzle sw = (BK == 64) ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B;
  {
    const uint64_t dims[2] = {(uint64_t)Cin, (uint64_t)M};
    const uint64_t strides[1] = {(uint64_t)Cin * 2};
    const uint32_t box[2] = {(uint32_t)BK, 128u};
    if (make_tma_bf16(&tmA, x, 2, dims, strides, box, sw)) return SSD3D_ERR_TMA;
  }
  {
    const uint64_t dims[2] = {(uint64_t)Cin, (uint64_t)Cout};
    const uint64_t strides[1] = {(uint64_t)Cin * 2};
    const uint32_t box[2] = {(uint32_t)BK, (uint32_t)BN};
    if (make_tma_bf16(&tmB, w, 2, dims, strides, box, sw)) return SSD3D_ERR_TMA;
  }
  dim3 grid((unsigned)m_tiles, (unsigned)(Cout / BN));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (BK == 64) return launch_gemm<64, false>(tmA, tmB, p, grid, st);
  return launch_gemm<32, false>(tmA, tmB, p, grid, st);
}

extern "C" int ssd3d_pwconv_bn_relu(const void* x, const void* w, const float* scale, const float* shift, void* y,
                                    int64_t M, int Cin, int Cout, int* nan_flag, void* stream) {
  return ssd3d_pwconv_affine(x, w, scale, shift, y, M, Cin, Cout, 1, nan_flag, stream);
}

// conv_head_tc.cu: halo-tile kernel (one activation load per 64-channel chunk)
int ssd3d_head_conv_halo(const void* x, const void* w, const float* bias, float* locs, float* scores, int N, int C,
                         int D, int H, int W, int bpl, int n_classes, int NPAD, int64_t P, int64_t prior_offset,
                         int* nan_flag, void* workspace, int64_t workspace_bytes, cudaStream_t st);

// conv_head_kw.cu: kw-GEMM + stencil for large maps
int ssd3d_head_conv_kw(const void* x, const void* w, int w_is_kw, const float* bias, float* locs, float* scores, int N,
                       int C, int D, int H, int W, int bpl, int n_classes, int NPAD, int64_t P, int64_t prior_offset,
                       int* nan_flag, void* workspace, int64_t workspace_bytes, cudaStream_t st);

extern "C" int ssd3d_head_conv(const void* x, const void* w, const float* bias, float* locs, float* scores, int N,
                               int C, int D, int H, int W, int bpl, int n_classes, int NPAD, int64_t P,
                               int64_t prior_offset, int* nan_flag, void* workspace, int64_t workspace_bytes,
                               int algo, void* stream) {
  if (!x || !w || !bias || !locs || !scores || N <= 0 || D <= 0 || H <= 0 || W <= 0) return SSD3D_ERR_ARG;
  if (C <= 0 || (C % 32) || bpl <= 0 || n_classes <= 0) return SSD3D_ERR_ARG;
  if (NPAD % 16 || NPAD > 256 || NPAD < bpl * (6 + n_classes)) return SSD3D_ERR_ARG;
  if (prior_offset < 0 || prior_offset + (int64_t)D * H * W * bpl > P) return SSD3D_ERR_ARG;
  // auto, in order of preference:
  //   kw-GEMM + (kd,kh) stencil (C % 64 == 0, NPAD == 16, >= 256 voxels): N = 144 columns per UMMA, 3 instead of
  //     27 activation reads -- 16-22 us on the benchmark's three heads;
  //   halo-tile kernel on small maps, where it can split K across CTAs (8^3: 23.6 vs 49 us, 4^3: 23.6 vs 88 us);
  //   per-tap kernel otherwise (e.g. the 32-channel layer-0 head): both older kernels are bound by the UMMA issue
  //     rate (~128 cycles per M=128 instruction whatever N) and the per-tap one issues fewer (30.7 vs 43.9 us)
  if (algo == 4)     // kw path, `w` already in the (144, 3*C) tiling of ssd3d_head_weight_kw
    return ssd3d_head_conv_kw(x, w, 1, bias, locs, scores, N, C, D, H, W, bpl, n_classes, NPAD, P, prior_offset, nan_flag,
                              workspace, workspace_bytes, static_cast<cudaStream_t>(stream));
  if (algo == 3 || algo == 0) {
    const int rc = ssd3d_head_conv_kw(x, w, 0, bias, locs, scores, N, C, D, H, W, bpl, n_classes, NPAD, P, prior_offset,
                                      nan_flag, workspace, workspace_bytes, static_cast<cudaStream_t>(stream));
    if (rc != SSD3D_ERR_UNSUPPORTED || algo == 3) return rc;
  }
  const bool small_map = (long long)N * D * H * W < 128ll * 128;
  if (algo == 2 || (algo == 0 && small_map)) {
    const int rc = ssd3d_head_conv_halo(x, w, bias, locs, scores, N, C, D, H, W, bpl, n_classes, NPAD, P, prior_offset,
                                        nan_flag, workspace, workspace_bytes, static_cast<cudaStream_t>(stream));
    if (rc != SSD3D_ERR_UNSUPPORTED || algo == 2) return rc;
  }
  const int BK = (C % 64 == 0) ? 64 : 32;
  GemmParams p{};
  p.num_kb = 27 * (C / BK);
  p.BN = NPAD;
  p.stages = 6;
  p.tmem_cols = pow2_ceil(NPAD < 32 ? 32 : NPAD);
  p.nan_flag = nan_flag;
  p.C = C; p.D = D; p.H = H; p.W = W; p.N = N;
  p.TW = pow2_ceil(W) < 8 ? pow2_ceil(W) : 8;
  p.TH = pow2_ceil(H) < 4 ? pow2_ceil(H) : 4;
  {
    const int rest = 128 / (p.TW * p.TH);
    p.TD = pow2_ceil(D) < rest ? pow2_ceil(D) : rest;
  }
  p.TN = 128 / (p.TW * p.TH * p.TD);
  p.tiles_w = (W + p.TW - 1) / p.TW;
  p.tiles_h = (H + p.TH - 1) / p.TH;
  p.tiles_d = (D + p.TD - 1) / p.TD;
  const int tiles_n = (N + p.TN - 1) / p.TN;
  p.bpl = bpl;
  p.n_classes = n_classes;
  p.n_loc = bpl * 6;
  p.n_cls = bpl * n_classes;
  p.P = P;
  p.prior_off = prior_offset;
  p.locs = locs;
  p.scores = scores;
  p.bias = bias;
  while (p.stages > 2 && gemm_smem_bytes(BK, NPAD, p.stages) > 220 * 1024) --p.stages;

  CUtensorMap tmA, tmB;
  const CUtensorMapSwizzle sw = (BK == 64) ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B;
  {
    const uint64_t dims[5] = {(uint64_t)C, (uint64_t)W, (uint64_t)H, (uint64_t)D, (uint64_t)N};
    const uint64_t strides[4] = {(uint64_t)C * 2, (uint64_t)W * C * 2, (uint64_t)H * W * C * 2,
                                 (uint64_t)D * H * W * C * 2};
    const uint32_t box[5] = {(uint32_t)BK, (uint32_t)p.TW, (uint32_t)p.TH, (uint32_t)p.TD, (uint32_t)p.TN};
    if (make_tma_bf16(&tmA, x, 5, dims, strides, box, sw)) return SSD3D_ERR_TMA;
  }
  {
    const uint64_t dims[2] = {(uint64_t)27 * C, (uint64_t)NPAD};
    const uint64_t strides[1] = {(uint64_t)27 * C * 2};
    const uint32_t box[2] = {(uint32_t)BK, (uint32_t)NPAD};
    if (make_tma_bf16(&tmB, w, 2, dims, strides, box, sw)) return SSD3D_ERR_TMA;
  }
  dim3 grid((unsigned)(p.tiles_w * p.tiles_h * p.tiles_d * tiles_n));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (BK == 64) return launch_gemm<64, true>(tmA, tmB, p, grid, st);
  return launch_gemm<32, true>(tmA, tmB, p, grid, st);
}
