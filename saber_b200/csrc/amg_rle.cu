// saber_b200 — run-length encoding of packed masks on the device: upstream SAM2's mask_to_rle_pytorch
// (sam2/utils/amg.py; SAM2AutomaticMaskGenerator output_mode "uncompressed_rle") and pycocotools' rleToString
// (maskApi.c; output_mode "coco_rle") on the bit-packed masks the AMG keeps, so that only the run lengths, not the
// dense [m, H, W] masks, leave the device.
//
// Input: int32 [*, H, WW], WW = ceil(W/32); pixel (y, x) of row k is bit x & 31 of word (k*H + y)*WW + (x >> 5). Bits
// past W in the last word are ignored. Pixels are read in column-major order (p = x*H + y). A transition is a p >= 1
// with pixel(p) != pixel(p - 1); it belongs to column p / H. The counts of a mask are a leading 0 when pixel 0 is set,
// then the distance between consecutive transitions (with 0 before the first and H*W after the last): T + 1 + lead
// counts for T transitions.
//
// One warp owns one word column (32 pixel columns) of one mask; lane c owns pixel column 32j + c. The warp reads 32 rows
// at a time (lane l: row 32r + l) and transposes the 32x32 bit block with shuffles, so that lane c holds 32 consecutive
// pixels of its column in one word: the transitions of 32 pixels are one xor with the word shifted by one row, their
// count one popc. Sizing writes per-column transition counts and last positions; a per-mask scan turns them into the
// column's first output index and the position of the transition before it, and the emit pass writes every count
// independently. The oracle twin is oracle/sam2_ref/amg.py (mask_to_rle) and oracle/sam2_ref/coco_rle.py.
#include "common.cuh"

namespace {

constexpr unsigned FULL = 0xffffffffu;
constexpr int RLE_WARPS = 8;  // word columns per CTA of the sizing / emit passes

// lane l holds row l of a 32x32 bit block (bit c = column c); returns column `lane` (bit l = row l)
__device__ __forceinline__ uint32_t transpose32(uint32_t x, int lane) {
  const uint32_t masks[5] = {0x0000FFFFu, 0x00FF00FFu, 0x0F0F0F0Fu, 0x33333333u, 0x55555555u};
#pragma unroll
  for (int i = 0; i < 5; ++i) {
    const int s = 16 >> i;
    const uint32_t m = masks[i];
    const uint32_t y = __shfl_xor_sync(FULL, x, s);
    x = (lane & s) ? (((y >> s) & m) | (x & ~m)) : ((x & m) | ((y & m) << s));
  }
  return x;
}

struct ColumnWalk {
  const uint32_t* mk;  // the mask's [H, WW] words
  int H, WW, j, lane;
  uint32_t colmask;    // valid columns of word j
  int x;               // pixel column of this lane
  bool valid;

  __device__ ColumnWalk(const uint32_t* bits, const int* sel, int k, int H_, int W, int WW_, int j_, int lane_)
      : H(H_), WW(WW_), j(j_), lane(lane_) {
    const int src = sel ? sel[k] : k;
    mk = bits + static_cast<long long>(src) * H * WW;
    colmask = (j == WW - 1 && (W & 31)) ? ((1u << (W & 31)) - 1u) : FULL;
    x = j * 32 + lane;
    valid = x < W;
  }
  // transition between the last pixel of column x - 1 and the first of column x
  __device__ bool cross() const {
    if (!valid || x == 0) return false;
    const uint32_t top = (__ldg(mk + j) >> lane) & 1u;
    const uint32_t bottom = lane > 0 ? (__ldg(mk + static_cast<long long>(H - 1) * WW + j) >> (lane - 1)) & 1u
                                     : __ldg(mk + static_cast<long long>(H - 1) * WW + j - 1) >> 31;
    return top != bottom;
  }
  // transitions inside the column at rows 32r .. 32r + 31 (bit b = row 32r + b); `carry` is the column's pixel at row
  // 32r - 1 and is advanced. Warp-uniform: every lane must call it.
  __device__ uint32_t chunk(int r, uint32_t& carry) const {
    const int y = r * 32 + lane;
    const uint32_t w = y < H ? (__ldg(mk + static_cast<long long>(y) * WW + j) & colmask) : 0u;
    const uint32_t t = transpose32(w, lane);
    if (r == 0) carry = t & 1u;  // row 0 has no predecessor inside the column
    const uint32_t rows = (r == (H - 1) / 32 && (H & 31)) ? ((1u << (H & 31)) - 1u) : FULL;
    const uint32_t e = (t ^ ((t << 1) | carry)) & rows;
    carry = t >> 31;
    return e;
  }
};

// colcnt[k, x] = transitions of column x, collast[k, x] = position of its last transition (0: none)
__global__ void __launch_bounds__(RLE_WARPS * 32)
rle_size_kernel(const uint32_t* __restrict__ bits, const int* __restrict__ sel, int H, int W, int WW,
                int* __restrict__ colcnt, int* __restrict__ collast) {
  const int k = blockIdx.x;
  const int j = blockIdx.y * RLE_WARPS + (threadIdx.x >> 5);
  if (j >= WW) return;  // warp-uniform
  const ColumnWalk cw(bits, sel, k, H, W, WW, j, threadIdx.x & 31);
  const int base = cw.x * H;
  int cnt = 0, last = 0;
  if (cw.cross()) {
    cnt = 1;
    last = base;
  }
  uint32_t carry = 0;
  for (int r = 0; r * 32 < H; ++r) {
    const uint32_t e = cw.chunk(r, carry);
    if (e) {
      cnt += __popc(e);
      last = base + r * 32 + 31 - __clz(e);
    }
  }
  if (cw.valid) {
    colcnt[static_cast<long long>(k) * W + cw.x] = cnt;
    collast[static_cast<long long>(k) * W + cw.x] = last;
  }
}

// inclusive block scan (blockDim.x a multiple of 32, at most 1024); *total receives the block's reduction
template <typename T, typename Op>
__device__ T block_scan(T v, T* sh, Op op, T identity, T* total) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const T u = __shfl_up_sync(FULL, v, o);
    if (lane >= o) v = op(v, u);
  }
  if (lane == 31) sh[warp] = v;
  __syncthreads();
  if (warp == 0) {
    T w = lane < nw ? sh[lane] : identity;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const T u = __shfl_up_sync(FULL, w, o);
      if (lane >= o) w = op(w, u);
    }
    sh[lane] = w;
  }
  __syncthreads();
  if (warp > 0) v = op(v, sh[warp - 1]);
  *total = sh[nw - 1];
  __syncthreads();
  return v;
}

struct Add {
  template <typename T>
  __device__ T operator()(T a, T b) const { return a + b; }
};
struct Max {
  __device__ int operator()(int a, int b) const { return a > b ? a : b; }
};

// per mask (one CTA each): colcnt / collast -> inclusive prefix sum / max over the columns, len[k] = T + 1 + lead
__global__ void __launch_bounds__(1024)
rle_scan_columns_kernel(const uint32_t* __restrict__ bits, const int* __restrict__ sel, int H, int W, int WW,
                        int* __restrict__ colcnt, int* __restrict__ collast, long long* __restrict__ len) {
  __shared__ int sh_sum[32], sh_max[32];
  const int k = blockIdx.x;
  int* cnt = colcnt + static_cast<long long>(k) * W;
  int* last = collast + static_cast<long long>(k) * W;
  int carry_sum = 0, carry_max = 0;
  for (int x0 = 0; x0 < W; x0 += blockDim.x) {
    const int x = x0 + threadIdx.x;
    int tot_sum, tot_max;
    const int s = block_scan(x < W ? cnt[x] : 0, sh_sum, Add(), 0, &tot_sum);
    const int mx = block_scan(x < W ? last[x] : 0, sh_max, Max(), 0, &tot_max);
    if (x < W) {
      cnt[x] = carry_sum + s;
      last[x] = max(carry_max, mx);
    }
    carry_sum += tot_sum;
    carry_max = max(carry_max, tot_max);
  }
  if (threadIdx.x == 0) {
    const int src = sel ? sel[k] : k;
    const int lead = bits[static_cast<long long>(src) * H * WW] & 1u;
    len[k] = static_cast<long long>(carry_sum) + 1 + lead;
  }
}

// off[0] = 0, off[1..m] = inclusive prefix sum of off[1..m] (in place; one CTA)
__global__ void __launch_bounds__(1024)
offsets_scan_kernel(long long* __restrict__ off, int m) {
  __shared__ long long sh[32];
  long long carry = 0;
  for (int i0 = 0; i0 < m; i0 += blockDim.x) {
    const int i = i0 + threadIdx.x;
    long long tot;
    const long long s = block_scan(i < m ? off[i + 1] : 0ll, sh, Add(), 0ll, &tot);
    if (i < m) off[i + 1] = carry + s;
    carry += tot;
  }
  if (threadIdx.x == 0) off[0] = 0;
}

__global__ void __launch_bounds__(RLE_WARPS * 32)
rle_counts_kernel(const uint32_t* __restrict__ bits, const int* __restrict__ sel, int H, int W, int WW,
                  const int* __restrict__ colcnt, const int* __restrict__ collast,
                  const long long* __restrict__ off, int* __restrict__ counts) {
  const int k = blockIdx.x;
  const int j = blockIdx.y * RLE_WARPS + (threadIdx.x >> 5);
  if (j >= WW) return;  // warp-uniform
  const ColumnWalk cw(bits, sel, k, H, W, WW, j, threadIdx.x & 31);
  const int lead = __ldg(cw.mk) & 1u;
  const long long row = static_cast<long long>(k) * W;
  long long o = off[k] + lead;
  int prev = 0;
  if (cw.valid && cw.x > 0) {
    o += colcnt[row + cw.x - 1];
    prev = collast[row + cw.x - 1];
  }
  if (cw.x == 0 && lead) counts[off[k]] = 0;
  const int base = cw.x * H;
  if (cw.cross()) {
    counts[o++] = base - prev;
    prev = base;
  }
  uint32_t carry = 0;
  for (int r = 0; r * 32 < H; ++r) {
    uint32_t e = cw.chunk(r, carry);
    if (!cw.valid) continue;
    while (e) {
      const int p = base + r * 32 + __ffs(e) - 1;
      e &= e - 1u;
      counts[o++] = p - prev;
      prev = p;
    }
  }
  if (cw.x == W - 1) counts[o] = H * W - prev;
}

// pycocotools rleToString: characters of count i of a mask
__device__ __forceinline__ int coco_chars(long long v, unsigned char* out) {
  int n = 0;
  bool more = true;
  while (more) {
    int c = static_cast<int>(v & 0x1f);
    v >>= 5;  // arithmetic
    more = (c & 0x10) ? v != -1 : v != 0;
    if (more) c |= 0x20;
    if (out) out[n] = static_cast<unsigned char>(c + 48);
    ++n;
  }
  return n;
}

__device__ __forceinline__ long long coco_delta(const int* cnts, long long i) {
  return static_cast<long long>(cnts[i]) - (i > 2 ? static_cast<long long>(cnts[i - 2]) : 0ll);
}

// len[k] = characters of mask k (one CTA per mask)
__global__ void __launch_bounds__(256)
coco_size_kernel(const int* __restrict__ counts, const long long* __restrict__ off, long long* __restrict__ len) {
  __shared__ long long sh[32];
  const int k = blockIdx.x;
  const int* c = counts + off[k];
  const long long n = off[k + 1] - off[k];
  long long s = 0;
  for (long long i = threadIdx.x; i < n; i += blockDim.x) s += coco_chars(coco_delta(c, i), nullptr);
  long long tot;
  block_scan(s, sh, Add(), 0ll, &tot);
  if (threadIdx.x == 0) len[k] = tot;
}

__global__ void __launch_bounds__(256)
coco_emit_kernel(const int* __restrict__ counts, const long long* __restrict__ off,
                 const long long* __restrict__ coff, unsigned char* __restrict__ chars) {
  __shared__ long long sh[32];
  const int k = blockIdx.x;
  const int* c = counts + off[k];
  const long long n = off[k + 1] - off[k];
  unsigned char* out = chars + coff[k];
  long long base = 0;
  for (long long i0 = 0; i0 < n; i0 += blockDim.x) {
    const long long i = i0 + threadIdx.x;
    const long long v = i < n ? coco_delta(c, i) : 0;
    const int len = i < n ? coco_chars(v, nullptr) : 0;
    long long tot;
    const long long incl = block_scan(static_cast<long long>(len), sh, Add(), 0ll, &tot);
    if (i < n) coco_chars(v, out + base + incl - len);
    base += tot;
  }
}

int check_frame(int m, int H, int W, const char* who) {
  SB_REQUIRE(m > 0 && H > 0 && W > 0, "%s: empty (m=%d H=%d W=%d)", who, m, H, W);
  SB_REQUIRE(static_cast<long long>(H) * W < (1ll << 31) - 1, "%s: H*W = %lld does not fit int32 counts", who,
             static_cast<long long>(H) * W);
  return SB_OK;
}

}  // namespace

extern "C" int sb_masks_rle_size(const void* bits, const int* sel, int m, int H, int W, int* ws, long long* offsets,
                                 void* stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  if (int rc = check_frame(m, H, W, "sb_masks_rle_size")) return rc;
  const int WW = (W + 31) / 32;
  int* colcnt = ws;
  int* collast = ws + static_cast<long long>(m) * W;
  rle_size_kernel<<<dim3(m, (WW + RLE_WARPS - 1) / RLE_WARPS), RLE_WARPS * 32, 0, stream>>>(
      static_cast<const uint32_t*>(bits), sel, H, W, WW, colcnt, collast);
  SB_CHECK_LAUNCH();
  const int scan_threads = W < 1024 ? (W + 31) / 32 * 32 : 1024;
  rle_scan_columns_kernel<<<m, scan_threads, 0, stream>>>(static_cast<const uint32_t*>(bits), sel, H, W, WW, colcnt, collast,
                                                  offsets + 1);
  SB_CHECK_LAUNCH();
  offsets_scan_kernel<<<1, 1024, 0, stream>>>(offsets, m);
  SB_CHECK_LAUNCH();
  return SB_OK;
}

extern "C" int sb_masks_rle_counts(const void* bits, const int* sel, int m, int H, int W, const int* ws,
                                   const long long* offsets, int* counts, void* stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  if (int rc = check_frame(m, H, W, "sb_masks_rle_counts")) return rc;
  const int WW = (W + 31) / 32;
  rle_counts_kernel<<<dim3(m, (WW + RLE_WARPS - 1) / RLE_WARPS), RLE_WARPS * 32, 0, stream>>>(
      static_cast<const uint32_t*>(bits), sel, H, W, WW, ws, ws + static_cast<long long>(m) * W, offsets, counts);
  SB_CHECK_LAUNCH();
  return SB_OK;
}

extern "C" int sb_masks_rle_coco_size(const int* counts, const long long* offsets, int m, long long* coco_offsets,
                                      void* stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  SB_REQUIRE(m > 0, "sb_masks_rle_coco_size: empty");
  coco_size_kernel<<<m, 256, 0, stream>>>(counts, offsets, coco_offsets + 1);
  SB_CHECK_LAUNCH();
  offsets_scan_kernel<<<1, 1024, 0, stream>>>(coco_offsets, m);
  SB_CHECK_LAUNCH();
  return SB_OK;
}

extern "C" int sb_masks_rle_coco(const int* counts, const long long* offsets, int m, const long long* coco_offsets,
                                 unsigned char* chars, void* stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  SB_REQUIRE(m > 0, "sb_masks_rle_coco: empty");
  coco_emit_kernel<<<m, 256, 0, stream>>>(counts, offsets, coco_offsets, chars);
  SB_CHECK_LAUNCH();
  return SB_OK;
}
