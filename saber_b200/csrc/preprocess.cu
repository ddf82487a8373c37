// saber_b200 — bandwidth kernels for the image side of the slice-wise path:
//   * SABER's 2-D slice preparation (REF saber/utils/preprocessing.py:4-81): local contrast with a
//     500-px box mean / variance (scipy.ndimage.uniform_filter, mode='reflect'), clip to +-3 sigma,
//     min-max to [0,1];
//   * upstream SAM2Transforms (sam2/utils/transforms.py as called from sam2_image_predictor.set_image,
//     reached from REF saber/adapters/sam2/amg.py:163): crop -> bilinear-antialias resize to 1024^2 ->
//     ImageNet mean/std normalise, written channel-major for the patch-embedding im2col;
//   * the slice-by-slice label stitch (REF saber/segmenters/propagation.py:181-186).
// fp32 expressions are written with explicit round-to-nearest intrinsics (no FMA contraction) so the
// numpy oracle evaluates the same expression tree.
#include "common.cuh"

namespace {

__device__ __forceinline__ int reflect_idx(int i, int n) {
  // scipy 'reflect' (half-sample symmetric): d c b a | a b c d | d c b a
  const int period = 2 * n;
  int j = i % period;
  if (j < 0) j += period;
  return j < n ? j : period - 1 - j;
}

// 1-D uniform filter along `axis` of a row-major [H, W] fp32 image; window [i - size/2, i + size - size/2 - 1]
// (scipy origin 0), double accumulation, fp32 result. square != 0 filters in*in (fp32 product).
constexpr int BOX_SEG = 32;
__global__ void __launch_bounds__(256)
box_filter_kernel(const float* __restrict__ in, float* __restrict__ out, int H, int W, int axis, int size,
                  int square) {
  const int len = axis == 0 ? H : W;      // extent along the filtered axis
  const int lines = axis == 0 ? W : H;    // number of independent lines
  const int nseg = (len + BOX_SEG - 1) / BOX_SEG;
  const long long total = static_cast<long long>(lines) * nseg;
  const int s1 = size / 2, s2 = size - s1 - 1;
  const double inv = 1.0 / static_cast<double>(size);
  for (long long t = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; t < total;
       t += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int line = static_cast<int>(t % lines);
    const int seg = static_cast<int>(t / lines);
    const long long base = axis == 0 ? line : static_cast<long long>(line) * W;
    const long long stride = axis == 0 ? W : 1;
    auto ld = [&](int i) -> double {
      const float v = in[base + static_cast<long long>(reflect_idx(i, len)) * stride];
      return static_cast<double>(square ? __fmul_rn(v, v) : v);
    };
    const int i0 = seg * BOX_SEG;
    double sum = 0.0;
    for (int l = -s1; l <= s2; ++l) sum += ld(i0 + l);
    const int i1 = min(len, i0 + BOX_SEG);
    for (int i = i0; i < i1; ++i) {
      out[base + static_cast<long long>(i) * stride] = static_cast<float>(sum * inv);
      sum += ld(i + 1 + s2) - ld(i - s1);
    }
  }
}

// contrast(): (x - mean) / (sqrt(max(sq - mean^2, 0)) + 1e-8) clipped to +-cutoff; also emits per-block
// min / max partials for the following min-max normalisation.
__global__ void __launch_bounds__(256)
contrast_kernel(const float* __restrict__ img, const float* __restrict__ mean, const float* __restrict__ sq,
                float* __restrict__ out, long long n, float cutoff, float* __restrict__ pmin,
                float* __restrict__ pmax) {
  float lo = INFINITY, hi = -INFINITY;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < n;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const float m = mean[i];
    const float var = fmaxf(__fsub_rn(sq[i], __fmul_rn(m, m)), 0.f);
    const float sd = __fsqrt_rn(var);
    float v = __fdiv_rn(__fsub_rn(img[i], m), __fadd_rn(sd, 1e-8f));
    v = fminf(fmaxf(v, -cutoff), cutoff);
    out[i] = v;
    lo = fminf(lo, v);
    hi = fmaxf(hi, v);
  }
  __shared__ float slo[8], shi[8];
  lo = -sb::warp_max(-lo);
  hi = sb::warp_max(hi);
  if ((threadIdx.x & 31) == 0) {
    slo[threadIdx.x >> 5] = lo;
    shi[threadIdx.x >> 5] = hi;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int k = 1; k < 8; ++k) {
      lo = fminf(lo, slo[k]);
      hi = fmaxf(hi, shi[k]);
    }
    pmin[blockIdx.x] = lo;
    pmax[blockIdx.x] = hi;
  }
}

// normalize(): (x - min) / (max - min + 1e-8), min/max reduced from the per-block partials.
__global__ void __launch_bounds__(256)
minmax_normalize_kernel(float* __restrict__ x, long long n, const float* __restrict__ pmin,
                        const float* __restrict__ pmax, int nparts) {
  float lo = INFINITY, hi = -INFINITY;
  for (int k = threadIdx.x; k < nparts; k += blockDim.x) {
    lo = fminf(lo, pmin[k]);
    hi = fmaxf(hi, pmax[k]);
  }
  __shared__ float slo[8], shi[8];
  __shared__ float s_min, s_den;
  lo = -sb::warp_max(-lo);
  hi = sb::warp_max(hi);
  if ((threadIdx.x & 31) == 0) {
    slo[threadIdx.x >> 5] = lo;
    shi[threadIdx.x >> 5] = hi;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int k = 1; k < 8; ++k) {
      lo = fminf(lo, slo[k]);
      hi = fmaxf(hi, shi[k]);
    }
    s_min = lo;
    s_den = __fadd_rn(__fsub_rn(hi, lo), 1e-8f);
  }
  __syncthreads();
  const float mn = s_min, den = s_den;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < n;
       i += static_cast<long long>(gridDim.x) * blockDim.x)
    x[i] = __fdiv_rn(__fsub_rn(x[i], mn), den);
}

// ATen upsample_bilinear2d_aa taps for output index i: [xmin, xmin+xsize), triangle weights, normalised.
constexpr int MAX_TAPS = 12;  // supports down-scaling up to ~5x
__device__ __forceinline__ void aa_taps(int i, int in_size, float scale, int& xmin, int& xsize, float* w) {
  const float support = scale >= 1.f ? scale : 1.f;
  const float invscale = scale >= 1.f ? __fdiv_rn(1.f, scale) : 1.f;
  const float center = __fmul_rn(scale, __fadd_rn(static_cast<float>(i), 0.5f));
  xmin = max(0, static_cast<int>(__fadd_rn(__fsub_rn(center, support), 0.5f)));
  xsize = min(in_size, static_cast<int>(__fadd_rn(__fadd_rn(center, support), 0.5f))) - xmin;
  xsize = min(xsize, MAX_TAPS);
  float total = 0.f;
  for (int j = 0; j < xsize; ++j) {
    const float a = __fmul_rn(__fadd_rn(__fsub_rn(static_cast<float>(j + xmin), center), 0.5f), invscale);
    const float v = fmaxf(0.f, __fsub_rn(1.f, fabsf(a)));
    w[j] = v;
    total = __fadd_rn(total, v);
  }
  for (int j = 0; j < xsize; ++j) w[j] = total != 0.f ? __fdiv_rn(w[j], total) : 0.f;
}

// img: [H, W, C] fp32 (C = 1 or 3; C = 1 is replicated to 3 channels). For each crop k (x0,y0,x1,y1):
// out[k, c, S, S] = (resize_aa(img[y0:y1, x0:x1, c]) - mean[c]) / std[c]. Horizontal pass first, then
// vertical, as ATen's CPU separable kernel orders them.
__global__ void __launch_bounds__(256)
resize_normalize_kernel(const float* __restrict__ img, int H, int W, int C, const int* __restrict__ crops,
                        int ncrops, int S, float m0, float m1, float m2, float s0, float s1, float s2,
                        float* __restrict__ out) {
  const long long total = static_cast<long long>(ncrops) * S * S;
  for (long long t = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; t < total;
       t += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int ox = static_cast<int>(t % S);
    const int oy = static_cast<int>((t / S) % S);
    const int k = static_cast<int>(t / (static_cast<long long>(S) * S));
    const int x0 = crops[4 * k + 0], y0 = crops[4 * k + 1];
    const int Wc = crops[4 * k + 2] - x0, Hc = crops[4 * k + 3] - y0;
    float acc[3] = {0.f, 0.f, 0.f};
    if (Wc == S && Hc == S) {
      const float* p = img + (static_cast<long long>(y0 + oy) * W + x0 + ox) * C;
      acc[0] = p[0];
      acc[1] = C == 3 ? p[1] : p[0];
      acc[2] = C == 3 ? p[2] : p[0];
    } else {
      float wx[MAX_TAPS], wy[MAX_TAPS];
      int xmin, xs, ymin, ys;
      aa_taps(ox, Wc, __fdiv_rn(static_cast<float>(Wc), static_cast<float>(S)), xmin, xs, wx);
      aa_taps(oy, Hc, __fdiv_rn(static_cast<float>(Hc), static_cast<float>(S)), ymin, ys, wy);
      for (int jy = 0; jy < ys; ++jy) {
        const float* row = img + (static_cast<long long>(y0 + ymin + jy) * W + x0 + xmin) * C;
        float h[3] = {0.f, 0.f, 0.f};
        for (int jx = 0; jx < xs; ++jx) {
          const float* p = row + jx * C;
          h[0] = __fadd_rn(h[0], __fmul_rn(p[0], wx[jx]));
          if (C == 3) {
            h[1] = __fadd_rn(h[1], __fmul_rn(p[1], wx[jx]));
            h[2] = __fadd_rn(h[2], __fmul_rn(p[2], wx[jx]));
          }
        }
        if (C != 3) h[1] = h[2] = h[0];
#pragma unroll
        for (int c = 0; c < 3; ++c) acc[c] = __fadd_rn(acc[c], __fmul_rn(h[c], wy[jy]));
      }
    }
    const long long plane = static_cast<long long>(S) * S;
    float* o = out + static_cast<long long>(k) * 3 * plane + static_cast<long long>(oy) * S + ox;
    o[0] = __fdiv_rn(__fsub_rn(acc[0], m0), s0);
    o[plane] = __fdiv_rn(__fsub_rn(acc[1], m1), s1);
    o[2 * plane] = __fdiv_rn(__fsub_rn(acc[2], m2), s2);
  }
}

// Label stitch of one slice: labels[y, x] = 1 + max{ k : bit (y,x) of mask order[k] is set } (0 if none);
// equals the sequential "masks3d[mask] = idx + 1" loop where later masks overwrite earlier ones.
__global__ void __launch_bounds__(256)
stitch_labels_kernel(const uint32_t* __restrict__ bits, const int* __restrict__ order, int m, int H, int W,
                     int WW, unsigned short* __restrict__ labels) {
  const int lane = threadIdx.x & 31;
  const long long nwords = static_cast<long long>(H) * WW;
  for (long long wi = (static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5; wi < nwords;
       wi += (static_cast<long long>(gridDim.x) * blockDim.x) >> 5) {
    const int y = static_cast<int>(wi / WW), wx = static_cast<int>(wi % WW);
    const int x = wx * 32 + lane;
    int label = 0;
    uint32_t unresolved = 0xffffffffu;
    for (int k = m - 1; k >= 0 && unresolved; --k) {
      const int src = order ? order[k] : k;
      const uint32_t w = __ldg(bits + static_cast<long long>(src) * nwords + wi);  // warp-uniform address
      if (label == 0 && ((w >> lane) & 1u)) label = k + 1;
      unresolved &= ~w;
    }
    if (x < W) labels[static_cast<long long>(y) * W + x] = static_cast<unsigned short>(label);
  }
}


// F.interpolate(x, (Ho, Wo), mode="bilinear", align_corners=False) on [N, Si, Si]-shaped planes
// (SAM2Transforms.postprocess_masks; video-resolution logits). Same fp32 expression tree as amg_post.cu.
__device__ __forceinline__ void bl_src_index(float scale, int dst, int in_size, int& i0, int& i1, float& l0,
                                             float& l1) {
  float s = __fmaf_rn(scale, __fadd_rn(static_cast<float>(dst), 0.5f), -0.5f);
  if (s < 0.f) s = 0.f;
  i0 = min(static_cast<int>(floorf(s)), in_size - 1);
  l1 = fminf(fmaxf(__fsub_rn(s, static_cast<float>(i0)), 0.f), 1.f);
  i1 = i0 + (i0 < in_size - 1 ? 1 : 0);
  l0 = __fsub_rn(1.f, l1);
}

__global__ void __launch_bounds__(256)
upsample_bilinear_kernel(const float* __restrict__ in, int N, int Hi, int Wi, int Ho, int Wo,
                         float* __restrict__ out) {
  const float scale_h = __fdiv_rn(static_cast<float>(Hi), static_cast<float>(Ho));
  const float scale_w = __fdiv_rn(static_cast<float>(Wi), static_cast<float>(Wo));
  const long long total = static_cast<long long>(N) * Ho * Wo;
  for (long long t = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; t < total;
       t += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int ox = static_cast<int>(t % Wo);
    const int oy = static_cast<int>((t / Wo) % Ho);
    const long long n = t / (static_cast<long long>(Wo) * Ho);
    const float* plane = in + n * Hi * Wi;
    int y0, y1, x0, x1;
    float ly0, ly1, lx0, lx1;
    bl_src_index(scale_h, oy, Hi, y0, y1, ly0, ly1);
    bl_src_index(scale_w, ox, Wi, x0, x1, lx0, lx1);
    const float v00 = plane[y0 * Wi + x0], v01 = plane[y0 * Wi + x1];
    const float v10 = plane[y1 * Wi + x0], v11 = plane[y1 * Wi + x1];
    const float t0 = __fmaf_rn(v00, lx0, __fmul_rn(v01, lx1));
    const float t1 = __fmaf_rn(v10, lx0, __fmul_rn(v11, lx1));
    out[t] = __fmaf_rn(t0, ly0, __fmul_rn(t1, ly1));
  }
}

// Decoder planes -> SAM2ImagePredictor's full-resolution output in one pass, with no intermediate buffer. Candidate c
// of P * cpp reads plane [c / cpp, token] of planes [P, 4, S, S]: token 1 + c % 3 for cpp = 3, otherwise sel[c] or 0
// (the candidate convention of amg_mask_post / amg_fill_lowres). It is up-sampled with upsample_bilinear_kernel's
// expression tree, so the logits are bit-identical to it, and out[c, Ho, Wo] gets the fp32 logits or the bool
// mask (value > thr). A thread owns UPS_RUN consecutive pixels of one row over `rows` rows: its x-taps are computed
// once and its y-taps once per row. Each row's run is stored with V-byte stores, V = gcd(row bytes, 16) (1 when that
// is 2): every row start, and the ragged tail of Wo % UPS_RUN pixels, is then a whole number of aligned V-byte words.
constexpr int UPS_RUN = 16;

template <int V, int NB>
__device__ __forceinline__ void store_run(unsigned char* dst, const uint32_t (&w)[NB / 4], int nbytes) {
#pragma unroll
  for (int b = 0; b < NB; b += V) {
    if (b < nbytes) {
      if constexpr (V == 16) {
        *reinterpret_cast<uint4*>(dst + b) = make_uint4(w[b / 4], w[b / 4 + 1], w[b / 4 + 2], w[b / 4 + 3]);
      } else if constexpr (V == 8) {
        *reinterpret_cast<uint2*>(dst + b) = make_uint2(w[b / 4], w[b / 4 + 1]);
      } else if constexpr (V == 4) {
        *reinterpret_cast<uint32_t*>(dst + b) = w[b / 4];
      } else {
        dst[b] = static_cast<unsigned char>(w[b / 4] >> (8 * (b % 4)));
      }
    }
  }
}

template <bool LOGITS, int V>
__global__ void __launch_bounds__(256)
upsample_select_kernel(const float* __restrict__ planes, int P, int S, const int* __restrict__ sel, int cpp, int Ho,
                       int Wo, int rows, float thr, unsigned char* __restrict__ out) {
  constexpr int E = LOGITS ? 4 : 1;  // output bytes per pixel
  constexpr int NB = UPS_RUN * E;
  const float scale_h = __fdiv_rn(static_cast<float>(S), static_cast<float>(Ho));
  const float scale_w = __fdiv_rn(static_cast<float>(S), static_cast<float>(Wo));
  const int runs = (Wo + UPS_RUN - 1) / UPS_RUN;
  const int bands = (Ho + rows - 1) / rows;
  const long long total = static_cast<long long>(P) * cpp * bands * runs;
  for (long long t = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; t < total;
       t += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int run = static_cast<int>(t % runs);
    const long long cb = t / runs;
    const int band = static_cast<int>(cb % bands);
    const int c = static_cast<int>(cb / bands);
    const int p = c / cpp;
    const int token = cpp == 3 ? 1 + c % 3 : (sel ? __ldg(sel + p) : 0);
    const float* plane = planes + (static_cast<long long>(p) * 4 + token) * S * S;
    const int x_begin = run * UPS_RUN;
    int xa[UPS_RUN];
    float lx0[UPS_RUN], lx1[UPS_RUN];
#pragma unroll
    for (int i = 0; i < UPS_RUN; ++i) {
      int x1;
      bl_src_index(scale_w, min(x_begin + i, Wo - 1), S, xa[i], x1, lx0[i], lx1[i]);  // x1 = min(xa + 1, S - 1)
    }
    const int nbytes = min(UPS_RUN, Wo - x_begin) * E;
    const int y_end = min(Ho, (band + 1) * rows);
    for (int oy = band * rows; oy < y_end; ++oy) {
      int y0, y1;
      float ly0, ly1;
      bl_src_index(scale_h, oy, S, y0, y1, ly0, ly1);
      const float* r0 = plane + y0 * S;
      const float* r1 = plane + y1 * S;
      uint32_t w[NB / 4];
#pragma unroll
      for (int i = 0; i < UPS_RUN; ++i) {
        const int x1 = min(xa[i] + 1, S - 1);
        const float t0 = __fmaf_rn(__ldg(r0 + xa[i]), lx0[i], __fmul_rn(__ldg(r0 + x1), lx1[i]));
        const float t1 = __fmaf_rn(__ldg(r1 + xa[i]), lx0[i], __fmul_rn(__ldg(r1 + x1), lx1[i]));
        const float v = __fmaf_rn(t0, ly0, __fmul_rn(t1, ly1));
        if constexpr (LOGITS) {
          w[i] = __float_as_uint(v);
        } else {
          const uint32_t bit = (v > thr ? 1u : 0u) << (8 * (i % 4));
          w[i / 4] = (i % 4 == 0) ? bit : (w[i / 4] | bit);
        }
      }
      store_run<V, NB>(out + ((static_cast<long long>(c) * Ho + oy) * Wo + x_begin) * E, w, nbytes);
    }
  }
}

inline int grid_for(long long total, int block = 256, int cap = 148 * 16) {
  long long g = (total + block - 1) / block;
  if (g > cap) g = cap;
  if (g < 1) g = 1;
  return static_cast<int>(g);
}

// (H,W,3) interleaved -> three planes, mixed over the channel axis: out[c'][p] = sum_c mix[c'][c] * f(img[p][c]),
// f = identity or square. This is the channel-axis pass of scipy.ndimage.uniform_filter on an (H,W,3) array
// (REF saber/utils/preprocessing.py:12-13 filters every axis of what it is given).
__global__ void __launch_bounds__(256)
rgb_mix_planar_kernel(const float* __restrict__ img, const float* __restrict__ mix, int square, long long npix,
                      float* __restrict__ out) {
  float m[9];
#pragma unroll
  for (int i = 0; i < 9; ++i) m[i] = __ldg(mix + i);
  for (long long p = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; p < npix;
       p += static_cast<long long>(gridDim.x) * blockDim.x) {
    float a = img[3 * p], b = img[3 * p + 1], c = img[3 * p + 2];
    if (square) {
      a *= a;
      b *= b;
      c *= c;
    }
    out[p] = m[0] * a + m[1] * b + m[2] * c;
    out[npix + p] = m[3] * a + m[4] * b + m[5] * c;
    out[2 * npix + p] = m[6] * a + m[7] * b + m[8] * c;
  }
}
__global__ void __launch_bounds__(256)
planar_to_hwc3_kernel(const float* __restrict__ planar, long long npix, float* __restrict__ out) {
  for (long long p = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; p < npix;
       p += static_cast<long long>(gridDim.x) * blockDim.x) {
    out[3 * p] = planar[p];
    out[3 * p + 1] = planar[npix + p];
    out[3 * p + 2] = planar[2 * npix + p];
  }
}

}  // namespace

// img [npix,3] fp32 -> out [3,npix] fp32 = mix (3x3 row-major, device) applied over the channel axis to img or img^2.
extern "C" int sb_rgb_mix_planar(const float* img, const float* mix, int square, long long npix, float* out,
                                 void* stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  SB_REQUIRE(img && mix && out && npix > 0, "sb_rgb_mix_planar: bad arguments");
  rgb_mix_planar_kernel<<<grid_for(npix), 256, 0, stream>>>(img, mix, square, npix, out);
  SB_CHECK_LAUNCH();
  return SB_OK;
}
extern "C" int sb_planar_to_hwc3(const float* planar, long long npix, float* out, void* stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  SB_REQUIRE(planar && out && npix > 0, "sb_planar_to_hwc3: bad arguments");
  planar_to_hwc3_kernel<<<grid_for(npix), 256, 0, stream>>>(planar, npix, out);
  SB_CHECK_LAUNCH();
  return SB_OK;
}

// scipy.ndimage.uniform_filter1d(in (optionally squared), size, axis, mode='reflect') on [H, W] fp32.
extern "C" int sb_box_filter(const float* in, float* out, int H, int W, int axis, int size, int square,
                             void* stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  SB_REQUIRE(H > 0 && W > 0 && size > 0 && (axis == 0 || axis == 1), "sb_box_filter: bad arguments");
  SB_REQUIRE(in != out, "sb_box_filter: in-place filtering is not supported");
  const int len = axis == 0 ? H : W, lines = axis == 0 ? W : H;
  const long long total = static_cast<long long>(lines) * ((len + BOX_SEG - 1) / BOX_SEG);
  box_filter_kernel<<<grid_for(total), 256, 0, stream>>>(in, out, H, W, axis, size, square);
  SB_CHECK_LAUNCH();
  return SB_OK;
}

// out = clip((img - mean) / (sqrt(max(sq - mean^2, 0)) + 1e-8), +-cutoff) then min-max to [0,1] in place.
// partials: workspace of 2 * 1024 floats.
extern "C" int sb_contrast_normalize(const float* img, const float* mean, const float* sq, float* out,
                                     long long n, float cutoff, float* partials, void* stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  SB_REQUIRE(n > 0, "sb_contrast_normalize: empty");
  const int g = grid_for(n, 256, 1024);
  contrast_kernel<<<g, 256, 0, stream>>>(img, mean, sq, out, n, cutoff, partials, partials + 1024);
  SB_CHECK_LAUNCH();
  minmax_normalize_kernel<<<grid_for(n), 256, 0, stream>>>(out, n, partials, partials + 1024, g);
  SB_CHECK_LAUNCH();
  return SB_OK;
}

// crops: device int32 [ncrops, 4] (x0, y0, x1, y1). out: [ncrops, 3, S, S] fp32.
extern "C" int sb_resize_normalize(const float* img, int H, int W, int C, const int* crops, int ncrops, int S,
                                   const float* mean3, const float* std3, float* out, void* stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  SB_REQUIRE(H > 0 && W > 0 && (C == 1 || C == 3) && ncrops > 0 && S > 0, "sb_resize_normalize: bad arguments");
  SB_REQUIRE(H <= 5 * S && W <= 5 * S, "sb_resize_normalize: down-scaling beyond 5x is not supported");
  const long long total = static_cast<long long>(ncrops) * S * S;
  resize_normalize_kernel<<<grid_for(total, 256, 148 * 32), 256, 0, stream>>>(
      img, H, W, C, crops, ncrops, S, mean3[0], mean3[1], mean3[2], std3[0], std3[1], std3[2], out);
  SB_CHECK_LAUNCH();
  return SB_OK;
}

// bits: [*, H, ceil(W/32)] packed masks; order: [m] mask indices (nullable = identity); labels: [H, W] u16.
extern "C" int sb_stitch_labels(const void* bits, const int* order, int m, int H, int W, void* labels,
                                void* stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  SB_REQUIRE(m >= 0 && H > 0 && W > 0 && m < 65535, "sb_stitch_labels: bad arguments (m=%d)", m);
  const int WW = (W + 31) / 32;
  const long long threads = static_cast<long long>(H) * WW * 32;
  stitch_labels_kernel<<<grid_for(threads, 256, 148 * 32), 256, 0, stream>>>(
      static_cast<const uint32_t*>(bits), order, m, H, W, WW, static_cast<unsigned short*>(labels));
  SB_CHECK_LAUNCH();
  return SB_OK;
}

// in: [N, Hi, Wi] fp32 -> out: [N, Ho, Wo] fp32, bilinear, align_corners=False (ATen semantics).
extern "C" int sb_upsample_bilinear(const float* in, int N, int Hi, int Wi, int Ho, int Wo, float* out,
                                    void* stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  SB_REQUIRE(N > 0 && Hi > 0 && Wi > 0 && Ho > 0 && Wo > 0, "sb_upsample_bilinear: bad sizes");
  const long long total = static_cast<long long>(N) * Ho * Wo;
  upsample_bilinear_kernel<<<grid_for(total, 256, 148 * 32), 256, 0, stream>>>(in, N, Hi, Wi, Ho, Wo, out);
  SB_CHECK_LAUNCH();
  return SB_OK;
}

// planes: [P, 4, S, S] fp32; sel: [P] int32 or null; cpp 3 (tokens 1..3) or 1 (sel, or token 0).
// out: [P * cpp, Ho, Wo] fp32 logits (logits != 0) or bool (value > thr), 16-byte aligned.
extern "C" int sb_upsample_select(const float* planes, int P, int S, const int* sel, int cpp, int Ho, int Wo, float thr,
                                  int logits, void* out, void* stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  SB_REQUIRE(planes && out && P > 0 && S > 0 && Ho > 0 && Wo > 0 && (cpp == 1 || cpp == 3),
             "sb_upsample_select: bad arguments");
  SB_REQUIRE((reinterpret_cast<uintptr_t>(out) & 15) == 0, "sb_upsample_select: out must be 16-byte aligned");
  const int E = logits ? 4 : 1;
  int V = 16;
  while ((static_cast<long long>(Wo) * E) % V) V >>= 1;
  const long long cands = static_cast<long long>(P) * cpp, runs = (Wo + UPS_RUN - 1) / UPS_RUN;
  // up to 8 rows per thread, fewer while that would leave the GPU short of threads (few candidates, small frames)
  int rows = 8;
  while (rows > 1 && cands * ((Ho + rows - 1) / rows) * runs < 148LL * 1024) rows >>= 1;
  const long long total = cands * ((Ho + rows - 1) / rows) * runs;
  const int grid = grid_for(total, 256, 148 * 32);
  unsigned char* o = static_cast<unsigned char*>(out);
#define SB_UPS_LAUNCH(L, VV) \
  upsample_select_kernel<L, VV><<<grid, 256, 0, stream>>>(planes, P, S, sel, cpp, Ho, Wo, rows, thr, o)
  if (logits) {
    switch (V) {
      case 16: SB_UPS_LAUNCH(true, 16); break;
      case 8: SB_UPS_LAUNCH(true, 8); break;
      default: SB_UPS_LAUNCH(true, 4); break;
    }
  } else {
    switch (V) {
      case 16: SB_UPS_LAUNCH(false, 16); break;
      case 8: SB_UPS_LAUNCH(false, 8); break;
      case 4: SB_UPS_LAUNCH(false, 4); break;
      default: SB_UPS_LAUNCH(false, 1); break;  // odd widths; a 2-byte variant spilled and gained nothing
    }
  }
#undef SB_UPS_LAUNCH
  SB_CHECK_LAUNCH();
  return SB_OK;
}
