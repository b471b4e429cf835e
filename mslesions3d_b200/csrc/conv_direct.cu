// Bandwidth-bound convolutions of the 3-D MobileNet backbone, channels-last-3d bf16, fp32 accumulate,
// BN(scale/shift) + ReLU fused into the store:
//   * stem   dense 3x3x3, Cin in {1..4} -> 32, stride (sd,2,2)      (mobilenet.py:26-31, ssd3d.py:60-61)
//   * dw     depthwise 3x3x3, stride 1|2                              (mobilenet.py:38,44)
// Both are HBM-roofline kernels (SURVEY.md section 8d): every global access is a 16-byte vector (dw) or a
// fully used sector (stem), halo re-reads are served by L1/L2, and each thread keeps a sliding window of
// the W axis in registers so that an input vector is fetched once per (kd,kh) row, not once per tap.
#include "common.cuh"
#include "../../include/ssd3d_b200.h"

namespace ssd3d {

// ------------------------------------------------------------------------------------------------
// depthwise 3x3x3
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint4 ldg_nc_v4(const void* p) {
  uint4 r;
  asm volatile("ld.global.nc.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
  return r;
}

__device__ __forceinline__ void unpack8(const uint4& v, float (&f)[8]) {
  f[0] = bf16_lo(v.x); f[1] = bf16_hi(v.x);
  f[2] = bf16_lo(v.y); f[3] = bf16_hi(v.y);
  f[4] = bf16_lo(v.z); f[5] = bf16_hi(v.z);
  f[6] = bf16_lo(v.w); f[7] = bf16_hi(v.w);
}

// One thread: 8 channels x WT consecutive outputs along W.  Lanes run over channel vectors first, so a
// warp reads whole contiguous (voxel, channel) spans.
template <int S, int WT>
__global__ void __launch_bounds__(256, 2) dwconv3d_kernel(const __nv_bfloat16* __restrict__ x,
                                                       const __nv_bfloat16* __restrict__ w,
                                                       const float* __restrict__ scale,
                                                       const float* __restrict__ shift,
                                                       __nv_bfloat16* __restrict__ y, int N, int C, int D, int H, int W,
                                                       int Do, int Ho, int Wo, long long total, float floor) {
  constexpr int NI = (WT - 1) * S + 3;  // input columns needed by WT outputs
  pdl_wait();
  pdl_launch_dependents();
  const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (gid >= total) return;
  const int CV = C >> 3;
  const int WR = (Wo + WT - 1) / WT;
  int cv = (int)(gid % CV);
  long long r = gid / CV;
  const int wr = (int)(r % WR); r /= WR;
  const int ho = (int)(r % Ho); r /= Ho;
  const int dz = (int)(r % Do);
  const int n = (int)(r / Do);
  const int c0 = cv << 3;
  const int wo0 = wr * WT;
  const int wi0 = wo0 * S - 1;  // first input column of the window

  float acc[WT][8];
#pragma unroll
  for (int i = 0; i < WT; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;

#pragma unroll
  for (int kd = 0; kd < 3; ++kd) {
    const int di = dz * S - 1 + kd;
    if ((unsigned)di >= (unsigned)D) continue;
#pragma unroll
    for (int kh = 0; kh < 3; ++kh) {
      const int hi = ho * S - 1 + kh;
      if ((unsigned)hi >= (unsigned)H) continue;
      const __nv_bfloat16* row = x + ((((long long)n * D + di) * H + hi) * W) * C + c0;
      uint4 in[NI];
#pragma unroll
      for (int i = 0; i < NI; ++i) {
        const int wi = wi0 + i;
        if ((unsigned)wi < (unsigned)W) in[i] = ldg_nc_v4(row + (long long)wi * C);
        else in[i] = make_uint4(0u, 0u, 0u, 0u);
      }
      const __nv_bfloat16* wrow = w + ((kd * 3 + kh) * 3) * C + c0;
#pragma unroll
      for (int kw = 0; kw < 3; ++kw) {
        float wf[8];
        unpack8(ldg_nc_v4(wrow + kw * C), wf);
#pragma unroll
        for (int ow = 0; ow < WT; ++ow) {
          float xf[8];
          unpack8(in[ow * S + kw], xf);
#pragma unroll
          for (int j = 0; j < 8; ++j) acc[ow][j] = fmaf(xf[j], wf[j], acc[ow][j]);
        }
      }
    }
  }

  float sc[8], sh[8];
  *reinterpret_cast<float4*>(&sc[0]) = __ldg(reinterpret_cast<const float4*>(scale + c0));
  *reinterpret_cast<float4*>(&sc[4]) = __ldg(reinterpret_cast<const float4*>(scale + c0 + 4));
  *reinterpret_cast<float4*>(&sh[0]) = __ldg(reinterpret_cast<const float4*>(shift + c0));
  *reinterpret_cast<float4*>(&sh[4]) = __ldg(reinterpret_cast<const float4*>(shift + c0 + 4));
  __nv_bfloat16* orow = y + ((((long long)n * Do + dz) * Ho + ho) * Wo) * C + c0;
#pragma unroll
  for (int ow = 0; ow < WT; ++ow) {
    const int wo = wo0 + ow;
    if (wo >= Wo) break;
    float v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = clamp_floor(__fadd_rn(__fmul_rn(acc[ow][j], sc[j]), sh[j]), floor);
    uint4 o;
    o.x = pack_bf16x2(v[0], v[1]);
    o.y = pack_bf16x2(v[2], v[3]);
    o.z = pack_bf16x2(v[4], v[5]);
    o.w = pack_bf16x2(v[6], v[7]);
    *reinterpret_cast<uint4*>(orow + (long long)wo * C) = o;
  }
}

// ------------------------------------------------------------------------------------------------
// stem: dense 3x3x3, tiny Cin, 32 output channels.  NCDHW input (fp32 or bf16), NDHWC bf16 output.
// One thread: two W-adjacent output voxels x 32 channels; weights broadcast from shared memory.
// ------------------------------------------------------------------------------------------------
template <typename T> __device__ __forceinline__ float load_in(const T* p);
template <> __device__ __forceinline__ float load_in<float>(const float* p) {
  // the product path stores activations in bf16: round the fp32 input the same way
  return __bfloat162float(__float2bfloat16_rn(__ldg(p)));
}
template <> __device__ __forceinline__ float load_in<__nv_bfloat16>(const __nv_bfloat16* p) {
  return __bfloat162float(*p);
}

template <typename T, int CIN>
__global__ void __launch_bounds__(128) stem_conv_kernel(const T* __restrict__ x, const __nv_bfloat16* __restrict__ w,
                                                        const float* __restrict__ scale,
                                                        const float* __restrict__ shift,
                                                        __nv_bfloat16* __restrict__ y, int N, int D, int H, int W,
                                                        int Do, int Ho, int Wo, int sd, long long total_pairs, float floor) {
  // w is (32, KPAD) bf16 with k = ci*27 + tap (PyTorch's flattened (Cin,3,3,3)); shared copy is
  // [tap*CIN + ci][32] fp32 so that one tap's 32 output-channel weights are contiguous
  constexpr int KPAD = (27 * CIN <= 64) ? 64 : 128;
  __shared__ __align__(16) float ws[27 * CIN * 32];
  for (int i = threadIdx.x; i < 27 * CIN * 32; i += blockDim.x) {
    const int c = i & 31, kk = i >> 5;
    const int tap = kk / CIN, ci = kk - tap * CIN;
    ws[i] = __bfloat162float(w[c * KPAD + ci * 27 + tap]);
  }
  __syncthreads();
  const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (gid >= total_pairs) return;
  const int WP = (Wo + 1) >> 1;
  const int wp = (int)(gid % WP);
  long long r = gid / WP;
  const int ho = (int)(r % Ho); r /= Ho;
  const int dz = (int)(r % Do);
  const int n = (int)(r / Do);
  const int wo0 = wp * 2;
  const int wi0 = wo0 * 2 - 1;

  float acc0[32], acc1[32];
#pragma unroll
  for (int j = 0; j < 32; ++j) { acc0[j] = 0.f; acc1[j] = 0.f; }

  const long long plane = (long long)D * H * W;
#pragma unroll 1
  for (int kd = 0; kd < 3; ++kd) {
    const int di = dz * sd - 1 + kd;
    if ((unsigned)di >= (unsigned)D) continue;
#pragma unroll 1
    for (int kh = 0; kh < 3; ++kh) {
      const int hi = ho * 2 - 1 + kh;
      if ((unsigned)hi >= (unsigned)H) continue;
#pragma unroll
      for (int ci = 0; ci < CIN; ++ci) {
        const T* row = x + ((long long)n * CIN + ci) * plane + ((long long)di * H + hi) * W;
        float v[5];
#pragma unroll
        for (int i = 0; i < 5; ++i) {
          const int wi = wi0 + i;
          v[i] = ((unsigned)wi < (unsigned)W) ? load_in<T>(row + wi) : 0.f;
        }
#pragma unroll
        for (int kw = 0; kw < 3; ++kw) {
          const float4* wr4 = reinterpret_cast<const float4*>(&ws[((((kd * 3 + kh) * 3 + kw) * CIN) + ci) * 32]);
          const float a0 = v[kw], a1 = v[kw + 2];
#pragma unroll
          for (int q = 0; q < 8; ++q) {
            const float4 wv = wr4[q];
            acc0[q * 4 + 0] = fmaf(a0, wv.x, acc0[q * 4 + 0]);
            acc0[q * 4 + 1] = fmaf(a0, wv.y, acc0[q * 4 + 1]);
            acc0[q * 4 + 2] = fmaf(a0, wv.z, acc0[q * 4 + 2]);
            acc0[q * 4 + 3] = fmaf(a0, wv.w, acc0[q * 4 + 3]);
            acc1[q * 4 + 0] = fmaf(a1, wv.x, acc1[q * 4 + 0]);
            acc1[q * 4 + 1] = fmaf(a1, wv.y, acc1[q * 4 + 1]);
            acc1[q * 4 + 2] = fmaf(a1, wv.z, acc1[q * 4 + 2]);
            acc1[q * 4 + 3] = fmaf(a1, wv.w, acc1[q * 4 + 3]);
          }
        }
      }
    }
  }

  __nv_bfloat16* o = y + ((((long long)n * Do + dz) * Ho + ho) * Wo + wo0) * 32;
  const bool second = (wo0 + 1) < Wo;
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    uint4 p0, p1;
    uint32_t* u0 = reinterpret_cast<uint32_t*>(&p0);
    uint32_t* u1 = reinterpret_cast<uint32_t*>(&p1);
#pragma unroll
    for (int h = 0; h < 4; ++h) {
      const int c = q * 8 + h * 2;
      const float s0 = __ldg(scale + c), s1 = __ldg(scale + c + 1);
      const float b0 = __ldg(shift + c), b1 = __ldg(shift + c + 1);
      u0[h] = pack_bf16x2(clamp_floor(__fadd_rn(__fmul_rn(acc0[c], s0), b0), floor),
                          clamp_floor(__fadd_rn(__fmul_rn(acc0[c + 1], s1), b1), floor));
      u1[h] = pack_bf16x2(clamp_floor(__fadd_rn(__fmul_rn(acc1[c], s0), b0), floor),
                          clamp_floor(__fadd_rn(__fmul_rn(acc1[c + 1], s1), b1), floor));
    }
    *reinterpret_cast<uint4*>(o + q * 8) = p0;
    if (second) *reinterpret_cast<uint4*>(o + 32 + q * 8) = p1;
  }
}

template <typename T>
static int launch_stem(const void* x, const __nv_bfloat16* w, const float* scale, const float* shift, void* y, int N,
                       int Cin, int D, int H, int W, int sd, float floor, cudaStream_t st) {
  const int Do = (D - 1) / sd + 1, Ho = (H - 1) / 2 + 1, Wo = (W - 1) / 2 + 1;
  const long long total = (long long)N * Do * Ho * ((Wo + 1) / 2);
  const unsigned blocks = (unsigned)((total + 127) / 128);
  const T* xp = static_cast<const T*>(x);
  __nv_bfloat16* yp = static_cast<__nv_bfloat16*>(y);
  switch (Cin) {
    case 1: stem_conv_kernel<T, 1><<<blocks, 128, 0, st>>>(xp, w, scale, shift, yp, N, D, H, W, Do, Ho, Wo, sd, total, floor); break;
    case 2: stem_conv_kernel<T, 2><<<blocks, 128, 0, st>>>(xp, w, scale, shift, yp, N, D, H, W, Do, Ho, Wo, sd, total, floor); break;
    case 3: stem_conv_kernel<T, 3><<<blocks, 128, 0, st>>>(xp, w, scale, shift, yp, N, D, H, W, Do, Ho, Wo, sd, total, floor); break;
    case 4: stem_conv_kernel<T, 4><<<blocks, 128, 0, st>>>(xp, w, scale, shift, yp, N, D, H, W, Do, Ho, Wo, sd, total, floor); break;
    default: return SSD3D_ERR_UNSUPPORTED;
  }
  SSD3D_CHECK_LAUNCH();
  return SSD3D_OK;
}

}  // namespace ssd3d

static int stem_simt(const void* x, int x_is_bf16, const void* w, const float* scale, const float* shift, void* y,
                     int N, int Cin, int D, int H, int W, int stride_d, int relu, void* stream) {
  if (!x || !w || !scale || !shift || !y || N <= 0 || D <= 0 || H <= 0 || W <= 0) return SSD3D_ERR_ARG;
  if (stride_d != 1 && stride_d != 2) return SSD3D_ERR_ARG;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const __nv_bfloat16* wp = static_cast<const __nv_bfloat16*>(w);
  const float floor = SSD3D_FLOOR(relu);
  if (x_is_bf16)
    return ssd3d::launch_stem<__nv_bfloat16>(x, wp, scale, shift, y, N, Cin, D, H, W, stride_d, floor, st);
  return ssd3d::launch_stem<float>(x, wp, scale, shift, y, N, Cin, D, H, W, stride_d, floor, st);
}

extern "C" int ssd3d_stem_conv_bn_relu_simt(const void* x, int x_is_bf16, const void* w, const float* scale,
                                            const float* shift, void* y, int N, int Cin, int D, int H, int W,
                                            int stride_d, void* stream) {
  return stem_simt(x, x_is_bf16, w, scale, shift, y, N, Cin, D, H, W, stride_d, 1, stream);
}

extern "C" int ssd3d_stem_conv_affine_simt(const void* x, int x_is_bf16, const void* w, const float* scale,
                                           const float* shift, void* y, int N, int Cin, int D, int H, int W,
                                           int stride_d, int relu, void* stream) {
  return stem_simt(x, x_is_bf16, w, scale, shift, y, N, Cin, D, H, W, stride_d, relu, stream);
}

// conv_dw_tma.cu: TMA halo-tile kernel for the large maps
int ssd3d_dwconv3d_tma(const void* x, const void* w, const float* scale, const float* shift, void* y, int N, int C,
                       int D, int H, int W, int stride, float floor, cudaStream_t st);

static int dwconv3d_direct(const void* x, const void* w, const float* scale, const float* shift, void* y, int N,
                           int C, int D, int H, int W, int stride, int relu, void* stream);

extern "C" int ssd3d_dwconv3d_affine(const void* x, const void* w, const float* scale, const float* shift, void* y,
                                     int N, int C, int D, int H, int W, int stride, int relu, void* stream) {
  if (!x || !w || !scale || !shift || !y || N <= 0 || D <= 0 || H <= 0 || W <= 0) return SSD3D_ERR_ARG;
  if (C <= 0 || (C & 7)) return SSD3D_ERR_ARG;
  if (stride != 1 && stride != 2) return SSD3D_ERR_ARG;
  const int rc = ssd3d_dwconv3d_tma(x, w, scale, shift, y, N, C, D, H, W, stride, SSD3D_FLOOR(relu),
                                    static_cast<cudaStream_t>(stream));
  if (rc != SSD3D_ERR_UNSUPPORTED) return rc;
  return dwconv3d_direct(x, w, scale, shift, y, N, C, D, H, W, stride, relu, stream);
}

extern "C" int ssd3d_dwconv3d_affine_direct(const void* x, const void* w, const float* scale, const float* shift,
                                            void* y, int N, int C, int D, int H, int W, int stride, int relu,
                                            void* stream) {
  if (!x || !w || !scale || !shift || !y || N <= 0 || D <= 0 || H <= 0 || W <= 0) return SSD3D_ERR_ARG;
  if (C <= 0 || (C & 7)) return SSD3D_ERR_ARG;
  if (stride != 1 && stride != 2) return SSD3D_ERR_ARG;
  return dwconv3d_direct(x, w, scale, shift, y, N, C, D, H, W, stride, relu, stream);
}

static int dwconv3d_direct(const void* x, const void* w, const float* scale, const float* shift, void* y, int N,
                           int C, int D, int H, int W, int stride, int relu, void* stream) {
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int Do = (D - 1) / stride + 1, Ho = (H - 1) / stride + 1, Wo = (W - 1) / stride + 1;
  const __nv_bfloat16* xp = static_cast<const __nv_bfloat16*>(x);
  const __nv_bfloat16* wp = static_cast<const __nv_bfloat16*>(w);
  __nv_bfloat16* yp = static_cast<__nv_bfloat16*>(y);
  const float floor = SSD3D_FLOOR(relu);
  // WT = 4 outputs per thread and 2 resident blocks/SM measured best on B200 (WT = 2 or a tighter register
  // cap were 2-70 % slower on every layer of the benchmark network)
  constexpr int WT = 4;
  const long long total = (long long)N * Do * Ho * ((Wo + WT - 1) / WT) * (C / 8);
  const unsigned blocks = (unsigned)((total + 255) / 256);
  if (stride == 1)
    SSD3D_LAUNCH_PDL((ssd3d::dwconv3d_kernel<1, WT>), dim3(blocks), dim3(256), 0, st, xp, wp, scale, shift, yp, N, C, D,
                     H, W, Do, Ho, Wo, total, floor);
  else
    SSD3D_LAUNCH_PDL((ssd3d::dwconv3d_kernel<2, WT>), dim3(blocks), dim3(256), 0, st, xp, wp, scale, shift, yp, N, C, D,
                     H, W, Do, Ho, Wo, total, floor);
  return SSD3D_OK;
}

extern "C" int ssd3d_dwconv3d_bn_relu(const void* x, const void* w, const float* scale, const float* shift, void* y,
                                      int N, int C, int D, int H, int W, int stride, void* stream) {
  return ssd3d_dwconv3d_affine(x, w, scale, shift, y, N, C, D, H, W, stride, 1, stream);
}
