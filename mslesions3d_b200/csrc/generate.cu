// Synthetic lesion volumes generated on the device (SURVEY.md 8f rank 2; generate_artificial_dataset.py:63-105):
// uniform noise in [0, 1), then n = randint(lo, hi) + 1 axis-aligned cubes of side randint(smin, smax) at a corner
// randint(0, dim - side) per axis, each adding 0.4 followed by a clip to [0, 1] (one clip per cube, as the
// reference's loop does), and the binary mask of the cubes.  The reference draws from numpy's MT19937 stream, whose
// state after `np.random.rand(D*H*W)` cannot be reached without producing all D*H*W doubles serially; here every
// value is a pure function of (seed, volume index, channel, voxel) through Philox4x32-10, so the volumes are
// produced in parallel where they are consumed.  Same DISTRIBUTION and the same construction, not the same
// stream: mslesions3d_b200/synthetic.py keeps the numpy generator for the reference-stream volumes (goldens), and
// oracle/philox_oracle.py restates this kernel in numpy for the bit-exact parity test.
//
//   counter = (pair index low, pair index high, volume index, stream | channel << 8),  key = (seed low, seed high)
//   stream 0: voxel noise, two doubles per call: u = ((a >> 5) * 2^26 + (b >> 6)) / 2^53   (numpy's random_sample)
//   stream 1: cube parameters of the volume: call 0 word 0 -> object count, call 1 + i -> {side, corner d, h, w}
//   randint(lo, hi) = lo + ((u32 * (hi - lo)) >> 32)                                       (multiply-shift)
#include "common.cuh"
#include "philox.cuh"

namespace ssd3d {

// one thread per volume: the cube list (side, corner d, corner h, corner w)
__global__ void gen_cubes_kernel(unsigned long long seed, long long first_idx, int N, int D, int H, int W, int num_lo,
                                 int num_hi, int size_lo, int size_hi, int max_cubes, int* __restrict__ cubes,
                                 int* __restrict__ n_cubes) {
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= N) return;
  const unsigned long long idx = (unsigned long long)(first_idx + n);
  const uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
  const uint32_t i0 = (uint32_t)idx;
  const Philox4 h = philox4x32_10(0u, 0u, i0, 1u, k0, k1);
  int count = randint_ms(h.v[0], num_lo, num_hi) + 1;          // generate_artificial_dataset.py:71-73
  if (count > max_cubes) count = max_cubes;
  n_cubes[n] = count;
  for (int i = 0; i < count; ++i) {
    const Philox4 r = philox4x32_10((uint32_t)(1 + i), 0u, i0, 1u, k0, k1);
    const int side = randint_ms(r.v[0], size_lo, size_hi);     // :75
    int* c = cubes + ((size_t)n * max_cubes + i) * 4;
    c[0] = side;
    c[1] = randint_ms(r.v[1], 0, D - side);                    // :80
    c[2] = randint_ms(r.v[2], 0, H - side);
    c[3] = randint_ms(r.v[3], 0, W - side);
  }
}

// thread = two consecutive voxels (one Philox call); grid.y = volume * C + channel
__global__ void __launch_bounds__(256) gen_volume_kernel(unsigned long long seed, long long first_idx, int C, int D,
                                                         int H, int W, int max_cubes, const int* __restrict__ cubes,
                                                         const int* __restrict__ n_cubes, float* __restrict__ out,
                                                         uint8_t* __restrict__ mask) {
  __shared__ int sc[64 * 4];
  __shared__ int scount;
  const int item = blockIdx.y, n = item / C, ch = item % C;
  if (threadIdx.x == 0) scount = n_cubes[n];
  __syncthreads();
  const int count = scount;
  for (int i = threadIdx.x; i < count * 4; i += blockDim.x) sc[i] = cubes[(size_t)n * max_cubes * 4 + i];
  __syncthreads();
  const long long vox = (long long)D * H * W;
  const long long pairs = (vox + 1) / 2;
  const uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
  const uint32_t i0 = (uint32_t)(unsigned long long)(first_idx + n);
  float* dst = out + (long long)item * vox;
  uint8_t* mk = (ch == 0 && mask) ? mask + (long long)n * vox : nullptr;
  for (long long pr = (long long)blockIdx.x * blockDim.x + threadIdx.x; pr < pairs; pr += (long long)gridDim.x * blockDim.x) {
    const Philox4 r = philox4x32_10((uint32_t)pr, (uint32_t)((unsigned long long)pr >> 32), i0, (uint32_t)ch << 8, k0, k1);
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      const long long v = 2 * pr + e;
      if (v >= vox) break;
      const uint32_t a = r.v[2 * e] >> 5, b = r.v[2 * e + 1] >> 6;
      double x = ((double)a * 67108864.0 + (double)b) * (1.0 / 9007199254740992.0);        // :68, np.random.rand
      const int w = (int)(v % W);
      const long long t = v / W;
      const int h = (int)(t % H), d = (int)(t / H);
      bool inside = false;
      for (int i = 0; i < count; ++i) {
        const int side = sc[4 * i], cd = sc[4 * i + 1], chh = sc[4 * i + 2], cw = sc[4 * i + 3];
        if (d >= cd && d < cd + side && h >= chh && h < chh + side && w >= cw && w < cw + side) {
          x = x + 0.4;                                                                     // :85
          x = x < 0.0 ? 0.0 : (x > 1.0 ? 1.0 : x);                                         // :86, clip per cube
          inside = true;
        }
      }
      dst[v] = (float)x;
      if (mk) mk[v] = inside ? 1 : 0;
    }
  }
}

}  // namespace ssd3d

using namespace ssd3d;

extern "C" int ssd3d_generate_volumes(uint64_t seed, int64_t first_idx, int N, int C, int D, int H, int W, int num_lo,
                                      int num_hi, int size_lo, int size_hi, int max_cubes, float* out_raw,
                                      uint8_t* mask, int32_t* cubes, int32_t* n_cubes, void* stream) {
  if (!out_raw || !cubes || !n_cubes || N <= 0 || C <= 0 || C > 255 || D <= 0 || H <= 0 || W <= 0) return SSD3D_ERR_ARG;
  if (num_hi <= num_lo || size_hi <= size_lo || size_lo < 1 || max_cubes < 1 || max_cubes > 64) return SSD3D_ERR_ARG;
  if (size_hi - 1 >= D || size_hi - 1 >= H || size_hi - 1 >= W) return SSD3D_ERR_ARG;      // randint(0, dim - side)
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  gen_cubes_kernel<<<(N + 63) / 64, 64, 0, st>>>((unsigned long long)seed, (long long)first_idx, N, D, H, W, num_lo,
                                                 num_hi, size_lo, size_hi, max_cubes, cubes, n_cubes);
  SSD3D_CHECK_LAUNCH();
  const long long pairs = ((long long)D * H * W + 1) / 2;
  long long bx = (pairs + 255) / 256;
  const long long cap = (long long)148 * 8;
  if (bx > cap) bx = cap;
  dim3 grid((unsigned)bx, (unsigned)(N * C));
  gen_volume_kernel<<<grid, 256, 0, st>>>((unsigned long long)seed, (long long)first_idx, C, D, H, W, max_cubes, cubes,
                                          n_cubes, out_raw, mask);
  SSD3D_CHECK_LAUNCH();
  return SSD3D_OK;
}
