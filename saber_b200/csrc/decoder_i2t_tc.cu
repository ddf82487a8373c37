// saber_b200 — the fused "image attends to tokens" block of the SAM2 mask decoder on tcgen05 / TMEM / TMA.
//
// Upstream sam2/modeling/sam/transformer.py TwoWayAttentionBlock step 4:
// keys = norm4(keys + cross_attn_image_to_token(keys + pe, tokens + pe, tokens)), computed in one pass over the image
// stream with the per-prompt folded operands W1 [256 x 64], W2 [64 x 256] of decoder_fused.cu (the out-projection bias
// is folded into W2: every softmax row sums to 1 per head):
//     S = X W1 + qres . kts      (128-row tile: tcgen05.mma M128 N64 K256, accumulator in TMEM; the block-diagonal
//                                  positional term is 8 mma.sync steps per warp, added in registers)
//     P = per-head softmax(S)    (one thread per (row, column half); written to shared memory as the K-major,
//                                  128B-swizzled A operand of the second MMA)
//     O = P W2                   (tcgen05.mma M128 N256 K64, accumulator in TMEM)
//     keys_new = LN(X + O)       (two passes over TMEM; the residual is read from the TMA-staged X tile)
// Both GEMMs run on the tensor core so that W1 / W2 are read once per 128-row tile (an earlier mma.sync kernel re-read
// them from shared memory for every 16 rows and was shared-memory / latency bound at ~2.2 TB/s of HBM traffic); the
// SM's LSU bandwidth is left to the softmax / LayerNorm epilogue.
//
// CTA = one prompt x `tiles` consecutive 128-row tiles. Warp roles: warp 0 TMA producer (W1, W2 once; X tiles into a
// 2-deep ring), warp 1 MMA issuer, warp 2 TMEM allocator, warps 4-11 epilogue (thread = row x column half).
// TMEM: two 256-column O buffers; S of tile n lives in the first 64 columns of O buffer n & 1 (it is consumed before
// the second MMA of that tile overwrites the buffer). The epilogue is software-pipelined as
//     S(0); for n: LN1(n) [residual + statistics, frees the X slot], S(n+1), LN2(n) [normalise + store]
// so that the second MMA of tile n runs under LN2(n-1), the first MMA of tile n+1 under LN1(n), and the X tile n+2
// streams in under S(n+1) / LN2(n) / LN1(n+1).
#include "common.cuh"

namespace {

using bf16 = __nv_bfloat16;

constexpr int TC_THREADS = 384;
constexpr int TC_XBUF = 65536;                       // one X tile: 4 K-blocks x [128 rows x 128 B]
constexpr int TC_OFF_W1 = 2 * TC_XBUF;               // 4 K-blocks x [64 rows x 128 B]
constexpr int TC_OFF_W2 = TC_OFF_W1 + 32768;         // [256 rows x 128 B]
constexpr int TC_OFF_P = TC_OFF_W2 + 32768;          // [128 rows x 128 B]
constexpr int TC_OFF_STG = TC_OFF_P + 16384;         // 8 epilogue warps x 2 KB staging tiles
constexpr int TC_OFF_VEC = TC_OFF_STG + 8 * 2048;    // gamma[256], beta[256]
constexpr int TC_OFF_BAR = TC_OFF_VEC + 2048;        // mbarriers + TMEM base
constexpr int TC_SMEM = TC_OFF_BAR + 256;            // 231,680 B (limit 232,448)

struct I2TTCParams {
  const bf16* qres;   // [nq, 128] positional term of the query projection (shared by all prompts)
  const bf16* kts;    // [B, 8, 128] scaled token keys
  const float* gamma;
  const float* beta;
  float eps;
  bf16* out;          // [B*nq, 256]
  int nt, nq, tiles;  // tokens per prompt, image tokens per prompt, 128-row tiles per CTA
  int x_bstride;      // rows between the prompts' streams in x (0: one stream shared by all prompts)
};

__device__ __forceinline__ void mma_bf16_16816(float* c, const uint32_t* a, uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ uint4 lds128(uint32_t addr) {
  uint4 v;
  asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr));
  return v;
}
__device__ __forceinline__ void sts128(uint32_t addr, uint4 v) {
  asm volatile("st.shared.v4.u32 [%0], {%1,%2,%3,%4};" ::"r"(addr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
__device__ __forceinline__ void sts64(uint32_t addr, float a, float b) {
  asm volatile("st.shared.v2.f32 [%0], {%1,%2};" ::"r"(addr), "f"(a), "f"(b) : "memory");
}
// 32 rows x 64 B staging tile, 16-byte chunks XOR-swizzled: conflict-free for "thread = row" and for coalesced IO
__device__ __forceinline__ uint32_t swz64(int row, int chunk) {
  return static_cast<uint32_t>(row * 64 + ((chunk ^ ((row >> 1) & 3)) << 4));
}
__device__ __forceinline__ void prefetch_l1(const void* ptr) {
  asm volatile("prefetch.global.L1 [%0];" ::"l"(ptr));
}
__device__ __forceinline__ void pair_barrier(int q) {  // the two warps (column halves) that share 32 rows
  asm volatile("bar.sync %0, 64;" ::"r"(q + 2) : "memory");
}

__global__ void __launch_bounds__(TC_THREADS, 1)
i2t_tc_kernel(const __grid_constant__ CUtensorMap tmX, const __grid_constant__ CUtensorMap tmW1,
              const __grid_constant__ CUtensorMap tmW2, const I2TTCParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + TC_OFF_BAR);
  uint64_t* w_full = bars;            // 1
  uint64_t* x_full = bars + 1;        // 2
  uint64_t* x_empty = bars + 3;       // 2
  uint64_t* s_full = bars + 5;        // 2
  uint64_t* p_full = bars + 7;        // 1
  uint64_t* o_full = bars + 8;        // 2
  uint64_t* o_empty = bars + 10;      // 2
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(bars + 12);
  float* sVec = reinterpret_cast<float*>(smem + TC_OFF_VEC);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int b = blockIdx.y;
  const int row_base = blockIdx.x * p.tiles * 128;  // first image token of this CTA
  const int T = p.tiles;

  if ((sb::smem_u32(smem) & 1023u) != 0u) __trap();  // SW128 operand tiles need 1024-byte alignment
  if (warp == 0 && lane == 0) {
    sb::tma_prefetch_desc(&tmX);
    sb::tma_prefetch_desc(&tmW1);
    sb::tma_prefetch_desc(&tmW2);
  }
  if (warp == 1 && lane == 0) {
    sb::mbar_init(w_full, 1);
    for (int i = 0; i < 2; ++i) {
      sb::mbar_init(&x_full[i], 1);
      sb::mbar_init(&x_empty[i], 8);
      sb::mbar_init(&s_full[i], 1);
      sb::mbar_init(&o_full[i], 1);
      sb::mbar_init(&o_empty[i], 8);
    }
    sb::mbar_init(p_full, 8);
    sb::fence_barrier_init();
  }
  if (warp == 2) {
    sb::tmem_alloc(tmem_ptr, 512);
    sb::tmem_relinquish();
  }
  if (warp >= 4) {
    const int te = threadIdx.x - 128;
    sVec[te] = p.gamma[te];
    sVec[256 + te] = p.beta[te];
  }
  sb::tc_fence_before();
  __syncthreads();
  sb::tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      sb::mbar_arrive_expect_tx(w_full, 65536);
      for (int kb = 0; kb < 4; ++kb) sb::tma_load_2d(smem + TC_OFF_W1 + kb * 8192, &tmW1, w_full, kb * 64, b * 64);
      sb::tma_load_2d(smem + TC_OFF_W2, &tmW2, w_full, 0, b * 256);
      const int xrow0 = b * p.x_bstride + row_base;
      for (int n = 0; n < T; ++n) {
        const int buf = n & 1;
        if (n >= 2) sb::mbar_wait(&x_empty[buf], static_cast<uint32_t>(((n >> 1) - 1) & 1));
        sb::mbar_arrive_expect_tx(&x_full[buf], TC_XBUF);
        for (int kb = 0; kb < 4; ++kb)
          sb::tma_load_2d(smem + buf * TC_XBUF + kb * 16384, &tmX, &x_full[buf], kb * 64, xrow0 + n * 128);
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (warp-converged, one elected lane per tcgen05 instruction) =====================
    {
      constexpr uint32_t idesc1 = sb::umma_idesc_bf16(128, 64);
      constexpr uint32_t idesc2 = sb::umma_idesc_bf16(128, 256);
      const uint32_t sbase = sb::smem_u32(smem);
      auto issue_mma1 = [&](int m) {
        const int buf = m & 1;
        sb::mbar_wait(&x_full[buf], static_cast<uint32_t>((m >> 1) & 1));
        if (m >= 2) sb::mbar_wait(&o_empty[buf], static_cast<uint32_t>(((m >> 1) - 1) & 1));
        sb::tc_fence_after();
        const uint32_t d = tmem_base + static_cast<uint32_t>(buf * 256);
#pragma unroll
        for (int kb = 0; kb < 4; ++kb) {
          const uint64_t da = sb::umma_desc_k_sw128(sbase + buf * TC_XBUF + kb * 16384);
          const uint64_t db = sb::umma_desc_k_sw128(sbase + TC_OFF_W1 + kb * 8192);
#pragma unroll
          for (int k = 0; k < 4; ++k)
            if (sb::elect_one())
              sb::umma_bf16(d, da + static_cast<uint64_t>(2 * k), db + static_cast<uint64_t>(2 * k), idesc1,
                            static_cast<uint32_t>((kb | k) != 0));
        }
        if (sb::elect_one()) sb::umma_commit(&s_full[buf]);
        __syncwarp();
      };
      sb::mbar_wait(w_full, 0);
      issue_mma1(0);
      const uint64_t dp = sb::umma_desc_k_sw128(sbase + TC_OFF_P);
      const uint64_t dw2 = sb::umma_desc_k_sw128(sbase + TC_OFF_W2);
      for (int n = 0; n < T; ++n) {
        sb::mbar_wait(p_full, static_cast<uint32_t>(n & 1));
        sb::tc_fence_after();
        const uint32_t d = tmem_base + static_cast<uint32_t>((n & 1) * 256);
#pragma unroll
        for (int k = 0; k < 4; ++k)
          if (sb::elect_one())
            sb::umma_bf16(d, dp + static_cast<uint64_t>(2 * k), dw2 + static_cast<uint64_t>(2 * k), idesc2,
                          static_cast<uint32_t>(k != 0));
        if (sb::elect_one()) sb::umma_commit(&o_full[n & 1]);
        __syncwarp();
        if (n + 1 < T) issue_mma1(n + 1);
      }
    }
  } else if (warp >= 4) {
    // ===================== epilogue: thread = (row r of the tile, column half hf) =====================
    const int q = warp & 3;            // TMEM lane quadrant of this warp
    const int hf = (warp - 4) >> 2;    // column half: heads 4*hf..4*hf+3 of S, channels 128*hf.. of O
    const int r = q * 32 + lane;
    const int g = lane >> 2, q4 = lane & 3;
    const uint32_t tlane = static_cast<uint32_t>(q * 32) << 16;
    const uint32_t sbase = sb::smem_u32(smem);
    const uint32_t stg = sbase + TC_OFF_STG + (warp - 4) * 2048;
    const uint32_t stg_partner = sbase + TC_OFF_STG + ((warp - 4) ^ 4) * 2048;
    const int nt = p.nt;
    const bf16* ktsb = p.kts + static_cast<long long>(b) * 8 * 128;
    float mean = 0.f, rstd = 0.f;
    // token-key B fragments of this warp's 4 heads: constant for the whole CTA
    uint2 bk[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) bk[j] = __ldg(reinterpret_cast<const uint2*>(ktsb + g * 128 + (hf * 4 + j) * 16 + q4 * 4));
    // this lane's row of the positional-term matrix (128 B = heads 4*hf..4*hf+3): prefetched into L1 one stage ahead
    const bf16* qpf = p.qres + static_cast<long long>(row_base + q * 32 + lane) * 128 + hf * 64;
    prefetch_l1(qpf);

    auto s_stage = [&](int m) {
      const int buf = m & 1;
      // ---- positional term of this warp's 32 rows x 4 heads on mma.sync (one k16 step per head), through the staging
      // tile (fp32, two heads at a time) into "thread = row" order
      float pe[32];
      const bf16* qrow = p.qres + static_cast<long long>(row_base + m * 128 + q * 32) * 128 + q4 * 4;
#pragma unroll
      for (int hp = 0; hp < 2; ++hp) {
#pragma unroll
        for (int hh = 0; hh < 2; ++hh) {
          const int head = hf * 4 + hp * 2 + hh;
#pragma unroll
          for (int mt = 0; mt < 2; ++mt) {
            const uint2 alo = __ldg(reinterpret_cast<const uint2*>(qrow + (mt * 16 + g) * 128 + head * 16));
            const uint2 ahi = __ldg(reinterpret_cast<const uint2*>(qrow + (mt * 16 + g + 8) * 128 + head * 16));
            const uint32_t a[4] = {alo.x, ahi.x, alo.y, ahi.y};
            float c[4] = {0.f, 0.f, 0.f, 0.f};
            mma_bf16_16816(c, a, bk[hp * 2 + hh].x, bk[hp * 2 + hh].y);
            // rows mt*16+g / +8, columns hh*8 + 2*q4 (+1) of the 32 x 16 fp32 staging tile
            const int col = hh * 8 + 2 * q4;
            sts64(stg + swz64(mt * 16 + g, col >> 2) + (col & 3) * 4, c[0], c[1]);
            sts64(stg + swz64(mt * 16 + g + 8, col >> 2) + (col & 3) * 4, c[2], c[3]);
          }
        }
        __syncwarp();
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const uint4 v = lds128(stg + swz64(lane, j));
          pe[hp * 16 + 4 * j + 0] = __uint_as_float(v.x);
          pe[hp * 16 + 4 * j + 1] = __uint_as_float(v.y);
          pe[hp * 16 + 4 * j + 2] = __uint_as_float(v.z);
          pe[hp * 16 + 4 * j + 3] = __uint_as_float(v.w);
        }
        __syncwarp();
      }
      // ---- S from TMEM (first 64 columns of O buffer `buf`)
      sb::mbar_wait(&s_full[buf], static_cast<uint32_t>((m >> 1) & 1));
      sb::tc_fence_after();
      uint32_t v[32];
      const uint32_t ta = tmem_base + tlane + static_cast<uint32_t>(buf * 256 + hf * 32);
      sb::tmem_ld_32x16(ta, v);
      sb::tmem_ld_32x16(ta + 16, v + 16);
      sb::tmem_ld_wait();
      // ---- per-head softmax over the 8 token slots; P as bf16, one 16-byte chunk per head
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        float s[8];
        float mx = -INFINITY;
#pragma unroll
        for (int t = 0; t < 8; ++t) {
          s[t] = t < nt ? __uint_as_float(v[j * 8 + t]) + pe[j * 8 + t] : -INFINITY;
          mx = fmaxf(mx, s[t]);
        }
        float l = 0.f;
#pragma unroll
        for (int t = 0; t < 8; ++t) {
          s[t] = sb::fast_exp2(s[t] - mx);
          l += s[t];
        }
        const float inv = __fdividef(1.f, l);
        const int chunk = hf * 4 + j;
        sts128(sbase + TC_OFF_P + r * 128 + ((chunk ^ (r & 7)) << 4),
               make_uint4(sb::pack_bf16x2(s[0] * inv, s[1] * inv), sb::pack_bf16x2(s[2] * inv, s[3] * inv),
                          sb::pack_bf16x2(s[4] * inv, s[5] * inv), sb::pack_bf16x2(s[6] * inv, s[7] * inv)));
      }
      sb::tc_fence_before();
      sb::fence_proxy_async();  // P (generic-proxy stores) -> visible to the tensor core's async-proxy reads
      __syncwarp();
      if (lane == 0) sb::mbar_arrive(p_full);
    };

    s_stage(0);
#pragma unroll 1
    for (int n = 0; n < T; ++n) {
      const int buf = n & 1;
      const uint32_t to = tmem_base + tlane + static_cast<uint32_t>(buf * 256 + hf * 128);
      // ---------------- LN1(n): y = O + residual, row statistics, y parked back in TMEM ----------------
      if (n + 1 < T) prefetch_l1(qpf + static_cast<long long>(n + 1) * 128 * 128);
      sb::mbar_wait(&o_full[buf], static_cast<uint32_t>((n >> 1) & 1));
      sb::tc_fence_after();
      sb::mbar_wait(&x_full[buf], static_cast<uint32_t>((n >> 1) & 1));  // (already complete) TMA writes -> this thread
      float2 sum2 = make_float2(0.f, 0.f), sq2 = make_float2(0.f, 0.f);
#pragma unroll 1
      for (int c = 0; c < 4; ++c) {
        uint32_t v[32];
        sb::tmem_ld_32x16(to + c * 32, v);
        sb::tmem_ld_32x16(to + c * 32 + 16, v + 16);
        const uint32_t xrow = sbase + buf * TC_XBUF + (hf * 2 + (c >> 1)) * 16384 + r * 128;
        uint4 res[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) res[j] = lds128(xrow + ((((c & 1) * 4 + j) ^ (r & 7)) << 4));
        sb::tmem_ld_wait();
        float y[32];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const uint32_t w4[4] = {res[j].x, res[j].y, res[j].z, res[j].w};
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const float2 yy = sb::add2(make_float2(__uint_as_float(v[8 * j + 2 * e]), __uint_as_float(v[8 * j + 2 * e + 1])),
                                   make_float2(sb::bf16_lo(w4[e]), sb::bf16_hi(w4[e])));
            y[8 * j + 2 * e] = yy.x;
            y[8 * j + 2 * e + 1] = yy.y;
            sum2 = sb::add2(sum2, yy);
            sq2 = sb::fma2(yy, yy, sq2);
          }
        }
        sb::tmem_st_32x16(to + c * 32, reinterpret_cast<const uint32_t*>(y));
        sb::tmem_st_32x16(to + c * 32 + 16, reinterpret_cast<const uint32_t*>(y) + 16);
      }
      sb::tmem_st_wait();
      float sum = sum2.x + sum2.y, sumsq = sq2.x + sq2.y;
      __syncwarp();
      if (lane == 0) sb::mbar_arrive(&x_empty[buf]);  // residual consumed (the first MMA of this tile retired long ago)
      // statistics of the other column half (partner warp, same rows) through the staging tiles
      sts64(stg + lane * 8, sum, sumsq);
      pair_barrier(q);
      {
        float ps, pq;
        asm volatile("ld.shared.v2.f32 {%0,%1}, [%2];" : "=f"(ps), "=f"(pq) : "r"(stg_partner + lane * 8));
        sum += ps;
        sumsq += pq;
      }
      pair_barrier(q);  // both warps have read before the tiles are reused
      mean = sum * (1.f / 256.f);
      rstd = rsqrtf(fmaxf(sumsq * (1.f / 256.f) - mean * mean, 0.f) + p.eps);

      // ---------------- S(n+1): softmax of the next tile (its first MMA ran under LN1) ----------------
      if (n + 1 < T) s_stage(n + 1);

      // ---------------- LN2(n): normalise, bf16, coalesced store through the staging tile ----------------
      uint8_t* orow = reinterpret_cast<uint8_t*>(p.out + (static_cast<long long>(b) * p.nq + row_base + n * 128 + q * 32) * 256 +
                                                 hf * 128);
#pragma unroll 1
      for (int c = 0; c < 4; ++c) {
        uint32_t v[32];
        sb::tmem_ld_32x16(to + c * 32, v);
        sb::tmem_ld_32x16(to + c * 32 + 16, v + 16);
        sb::tmem_ld_wait();
        const float* ga = sVec + hf * 128 + c * 32;
        const float* be = sVec + 256 + hf * 128 + c * 32;
        uint32_t o16[16];
        const float2 rs2 = make_float2(rstd, rstd), nm2 = make_float2(-mean, -mean);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float4 g4 = *reinterpret_cast<const float4*>(ga + 4 * j);
          const float4 b4 = *reinterpret_cast<const float4*>(be + 4 * j);
          const float2 d0 = sb::add2(make_float2(__uint_as_float(v[4 * j + 0]), __uint_as_float(v[4 * j + 1])), nm2);
          const float2 d1 = sb::add2(make_float2(__uint_as_float(v[4 * j + 2]), __uint_as_float(v[4 * j + 3])), nm2);
          const float2 f01 = sb::fma2(d0, sb::mul2(rs2, make_float2(g4.x, g4.y)), make_float2(b4.x, b4.y));
          const float2 f23 = sb::fma2(d1, sb::mul2(rs2, make_float2(g4.z, g4.w)), make_float2(b4.z, b4.w));
          o16[2 * j] = sb::pack_bf16x2(f01.x, f01.y);
          o16[2 * j + 1] = sb::pack_bf16x2(f23.x, f23.y);
        }
#pragma unroll
        for (int j = 0; j < 4; ++j)
          sts128(stg + swz64(lane, j), make_uint4(o16[4 * j], o16[4 * j + 1], o16[4 * j + 2], o16[4 * j + 3]));
        __syncwarp();
#pragma unroll
        for (int t = 0; t < 4; ++t) {
          const int id = t * 32 + lane;
          const int row = id >> 2, ch = id & 3;
          *reinterpret_cast<uint4*>(orow + static_cast<long long>(row) * 512 + c * 64 + ch * 16) = lds128(stg + swz64(row, ch));
        }
        __syncwarp();
      }
      sb::tc_fence_before();
      __syncwarp();
      if (lane == 0) sb::mbar_arrive(&o_empty[buf]);
    }
  }

  sb::tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    sb::tc_fence_after();
    sb::tmem_dealloc(tmem_base, 512);
  }
}

}  // namespace

// keys_new = LayerNorm(keys + out_proj(softmax((keys Wq^T + qres) kt^T) vt)) for every prompt, one pass over the stream.
// x [batch*nq, 256] bf16 (or [nq, 256] shared by all prompts), qres [nq,128] bf16 (= image_pe Wq^T + bq), w1t
// [batch,64,256], w2t [batch,256,64] (out-projection bias folded in), kts [batch,8,128]: the outputs of sb_i2t_fold.
// out [batch*nq, 256] bf16 may alias x when x is per-prompt. nq must be a multiple of 256.
extern "C" int sb_i2t_block_tc(const void* x, int x_shared, const void* qres, const void* w1t, const void* w2t,
                               const void* kts, const float* gamma, const float* beta, float eps, void* out, int batch,
                               int nq, int nt, void* stream) {
  SB_REQUIRE(batch > 0 && nq > 0 && (nq % 256) == 0, "sb_i2t_block_tc: nq must be a positive multiple of 256 (got %d)", nq);
  SB_REQUIRE(nt >= 1 && nt <= 8, "sb_i2t_block_tc: nt must be in 1..8 (got %d)", nt);
  SB_REQUIRE(x && qres && w1t && w2t && kts && gamma && beta && out, "sb_i2t_block_tc: null operand");
  SB_REQUIRE(((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(qres) | reinterpret_cast<uintptr_t>(w1t) |
               reinterpret_cast<uintptr_t>(w2t) | reinterpret_cast<uintptr_t>(kts) | reinterpret_cast<uintptr_t>(out)) & 15) == 0,
             "sb_i2t_block_tc: operands must be 16-byte aligned");
  CUtensorMap tmX, tmW1, tmW2;
  SB_REQUIRE(!(x_shared && x == out), "sb_i2t_block_tc: a shared stream cannot be updated in place");
  int rc = sb_make_tmap_2d_bf16(&tmX, x, static_cast<uint64_t>(x_shared ? 1 : batch) * nq, 256, 256, 128, 64);
  if (rc != SB_OK) return rc;
  rc = sb_make_tmap_2d_bf16(&tmW1, w1t, static_cast<uint64_t>(batch) * 64, 256, 256, 64, 64);
  if (rc != SB_OK) return rc;
  rc = sb_make_tmap_2d_bf16(&tmW2, w2t, static_cast<uint64_t>(batch) * 256, 64, 64, 256, 64);
  if (rc != SB_OK) return rc;
  int sms = 148;
  {
    int dev = 0;
    if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  }
  // rows per CTA: one CTA per SM (TMEM + shared memory); fewest SM-waves x (rows + pipeline fill of ~1.5 tiles)
  int best_rows = 256;
  long long best_cost = -1;
  for (int rows = 2048; rows >= 256; rows >>= 1) {
    if (nq % rows) continue;
    const long long ctas = static_cast<long long>(batch) * (nq / rows);
    const long long waves = (ctas + sms - 1) / sms;
    const long long cost = waves * (rows + 192);
    if (best_cost < 0 || cost < best_cost) {
      best_cost = cost;
      best_rows = rows;
    }
  }
  I2TTCParams p;
  p.qres = static_cast<const bf16*>(qres);
  p.kts = static_cast<const bf16*>(kts);
  p.gamma = gamma;
  p.beta = beta;
  p.eps = eps;
  p.out = static_cast<bf16*>(out);
  p.nt = nt;
  p.nq = nq;
  p.tiles = best_rows / 128;
  p.x_bstride = x_shared ? 0 : nq;
  static SbPerDeviceOnce attr_once;
  if (attr_once.need()) {
    SB_CHECK_CUDA(cudaFuncSetAttribute(i2t_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, TC_SMEM));
    attr_once.mark();
  }
  i2t_tc_kernel<<<dim3(nq / best_rows, batch), TC_THREADS, TC_SMEM, reinterpret_cast<cudaStream_t>(stream)>>>(tmX, tmW1, tmW2, p);
  SB_CHECK_LAUNCH();
  return SB_OK;
}
