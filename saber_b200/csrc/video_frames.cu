// saber_b200 — video frame loading: Pillow's 8-bit bicubic resize of uint8 RGB frames to S x S, then upstream's
// ImageNet normalisation through a lookup table (sam2/utils/misc.py::load_video_frames_from_jpg_images on the device).
//
// The arithmetic is Pillow's ImagingResample for 8-bit images (libImaging/Resample.c), reproduced exactly: 22-bit
// fixed-point weights (built on the host in float64), an int32 accumulator seeded with 2^21, `clip8(acc >> 22)` after
// each pass, the horizontal pass first over the source rows the vertical pass reads, a uint8 intermediate. The fp32
// output is lut[c][byte], so the kernel does no floating-point arithmetic and the frames are bit-identical to the
// host route by construction.
//
// Two kernels with an HBM intermediate: the intermediate is uint8 [N, hy, S, 3] (hy = the source rows the vertical
// taps reach), at most a quarter of the fp32 output's bytes for any frame no taller than 4 S.
#include "common.cuh"

namespace {

constexpr int kPrec = 22;  // Pillow PRECISION_BITS (32 - 8 - 2)

inline int grid_for(long long total, int block = 256, int cap = 148 * 16) {
  long long g = (total + block - 1) / block;
  if (g > cap) g = cap;
  if (g < 1) g = 1;
  return static_cast<int>(g);
}

__device__ __forceinline__ int clip8(int acc) {
  const int v = acc >> kPrec;
  return v < 0 ? 0 : (v > 255 ? 255 : v);
}

// Horizontal pass. src: [N, H, W, 3] u8; rows [y0, y0 + hy) of every frame -> tmp: [N, hy, S, 3] u8.
// bounds[o] = (xmin, n); weights[o * ksize + k] for k < n. One thread per output pixel (3 channels): the threads of a
// warp take consecutive output columns, so each tap's loads fall in one contiguous span of the source row.
__global__ void __launch_bounds__(256) frames_hpass_kernel(const uint8_t* __restrict__ src, int N, int H, int W, int y0,
                                                           int hy, int S, const int2* __restrict__ bounds,
                                                           const int* __restrict__ weights, int ksize,
                                                           uint8_t* __restrict__ tmp) {
  const long long total = static_cast<long long>(N) * hy * S;
  const long long row_bytes = static_cast<long long>(W) * 3;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int ox = static_cast<int>(i % S);
    const long long r = i / S;  // n * hy + row
    const long long n = r / hy, row = r - n * hy;
    const int2 b = __ldg(bounds + ox);
    const int* wk = weights + static_cast<long long>(ox) * ksize;
    const uint8_t* p = src + (n * H + y0 + row) * row_bytes + static_cast<long long>(b.x) * 3;
    int a0 = 1 << (kPrec - 1), a1 = a0, a2 = a0;
    for (int k = 0; k < b.y; ++k) {
      const int w = __ldg(wk + k);
      a0 += static_cast<int>(__ldg(p + 3 * k)) * w;
      a1 += static_cast<int>(__ldg(p + 3 * k + 1)) * w;
      a2 += static_cast<int>(__ldg(p + 3 * k + 2)) * w;
    }
    uint8_t* q = tmp + i * 3;
    q[0] = static_cast<uint8_t>(clip8(a0));
    q[1] = static_cast<uint8_t>(clip8(a1));
    q[2] = static_cast<uint8_t>(clip8(a2));
  }
}

// Vertical pass + normalisation. in: [N, rows, S, 3] u8 whose row 0 is source row y0 -> out: [N, 3, S, S] fp32,
// out[n, c, oy, ox] = lut[c * 256 + clip8(sum_k in[n, ymin + k - y0, ox, c] * w[oy, k])]. A skipped vertical pass is
// the one-tap identity table (ymin = oy, w = 2^22), which reproduces the byte exactly.
__global__ void __launch_bounds__(256) frames_vpass_lut_kernel(const uint8_t* __restrict__ in, int N, int rows, int y0,
                                                               int S, const int2* __restrict__ bounds,
                                                               const int* __restrict__ weights, int ksize,
                                                               const float* __restrict__ lut, float* __restrict__ out) {
  __shared__ float s_lut[3 * 256];
  for (int t = threadIdx.x; t < 3 * 256; t += blockDim.x) s_lut[t] = lut[t];
  __syncthreads();
  const long long plane = static_cast<long long>(S) * S;
  const long long total = static_cast<long long>(N) * plane;
  const long long row_bytes = static_cast<long long>(S) * 3;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long n = i / plane, pix = i - n * plane;
    const int oy = static_cast<int>(pix / S), ox = static_cast<int>(pix - static_cast<long long>(oy) * S);
    const int2 b = __ldg(bounds + oy);
    const int* wk = weights + static_cast<long long>(oy) * ksize;
    const uint8_t* p = in + (n * rows + (b.x - y0)) * row_bytes + static_cast<long long>(ox) * 3;
    int a0 = 1 << (kPrec - 1), a1 = a0, a2 = a0;
    for (int k = 0; k < b.y; ++k) {
      const int w = __ldg(wk + k);
      const uint8_t* pk = p + k * row_bytes;
      a0 += static_cast<int>(__ldg(pk)) * w;
      a1 += static_cast<int>(__ldg(pk + 1)) * w;
      a2 += static_cast<int>(__ldg(pk + 2)) * w;
    }
    float* o = out + n * 3 * plane + pix;
    o[0] = s_lut[clip8(a0)];
    o[plane] = s_lut[256 + clip8(a1)];
    o[2 * plane] = s_lut[512 + clip8(a2)];
  }
}

}  // namespace

// src: [N, H, W, 3] u8 frames of one size. x*: horizontal coefficients (S entries; null when W == S, the pass is
// skipped), y*: vertical coefficients (S entries; the one-tap identity when H == S). The horizontal pass covers source
// rows [y0, y0 + hy) into tmp [N, hy, S, 3] u8. lut: [3, 256] fp32. out: [N, 3, S, S] fp32.
extern "C" int sb_resample_frames_u8(const void* src, int N, int H, int W, int S, const int* xbounds,
                                     const int* xweights, int xk, const int* ybounds, const int* yweights, int yk,
                                     int y0, int hy, void* tmp, const float* lut, float* out, void* stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  SB_REQUIRE(src && out && lut && ybounds && yweights && N > 0 && H > 0 && W > 0 && S > 0 && yk > 0,
             "sb_resample_frames_u8: bad arguments");
  const uint8_t* vin = static_cast<const uint8_t*>(src);
  int vrows = H, vy0 = 0;
  if (xbounds) {
    SB_REQUIRE(xweights && tmp && xk > 0 && y0 >= 0 && hy > 0 && y0 + hy <= H,
               "sb_resample_frames_u8: bad horizontal pass arguments");
    frames_hpass_kernel<<<grid_for(static_cast<long long>(N) * hy * S), 256, 0, stream>>>(
        vin, N, H, W, y0, hy, S, reinterpret_cast<const int2*>(xbounds), xweights, xk, static_cast<uint8_t*>(tmp));
    SB_CHECK_LAUNCH();
    vin = static_cast<const uint8_t*>(tmp);
    vrows = hy;
    vy0 = y0;
  } else {
    SB_REQUIRE(W == S, "sb_resample_frames_u8: the horizontal pass is skipped only when W == S");
  }
  frames_vpass_lut_kernel<<<grid_for(static_cast<long long>(N) * S * S), 256, 0, stream>>>(
      vin, N, vrows, vy0, S, reinterpret_cast<const int2*>(ybounds), yweights, yk, lut, out);
  SB_CHECK_LAUNCH();
  return SB_OK;
}
