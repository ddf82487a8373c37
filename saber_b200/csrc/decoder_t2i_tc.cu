// saber_b200 — mask-decoder "tokens attend to image" attention on tcgen05 / TMEM / TMA.
//
// Upstream sam2/modeling/sam/transformer.py TwoWayAttentionBlock step 2 and final_attn_token_to_image, with the k / v
// projections folded onto the <= 8 tokens (decoder_fused.cu): flash attention with 64 query rows (8 heads x 8 token
// slots) whose keys AND values are the raw image stream x [4096, 256] of the prompt:
//     S = Q'' [x | kadd]^T     Q'' = [Wk_h^T q_{t,h} | block-diagonal q_{t,h}]  (64 x 384),  kadd = image_pe Wk^T + bk
//     O = softmax(S) x         (the value projection Wv / bv is applied afterwards on the 64 x 256 result)
// Both GEMMs are UMMAs with M = 64 (an earlier mma.sync kernel was bound by the legacy tensor path, 54 % of its
// 0.5 MMA/clk/SM, and by every warp re-loading the key tile from shared memory):
//   * QK^T: A = Q'' (K-major, resident), B = the TMA-staged key tile [64 keys x (256 + 128)] (K-major), D = S in TMEM
//   * PV  : A = P (bf16, written by the softmax warps as a K-major 128B-swizzled tile), B = the SAME key tile read as
//           an MN-major operand (N = 256 channels contiguous, K = keys), D = O in TMEM (fp32, 64 x 256)
// With M = 64 the accumulator rows live in lanes 0-15 of each TMEM lane quadrant: two softmax warps per quadrant, thread =
// (row, key half), exchange only the row maximum through shared memory. Rescaling of O is lazy (only when
// a row maximum grows by more than 2^8). CTA = (key split, prompt); unnormalised partials per split are merged and
// projected by t2i_unfold_kernel.
#include "common.cuh"

namespace {

using bf16 = __nv_bfloat16;

constexpr int TT_KT = 64;                               // keys per tile
constexpr int TT_STAGES = 3;
constexpr int TT_THREADS = 384;                         // warp 0 TMA, 1 MMA, 2 TMEM alloc, 4-11 softmax
constexpr int TT_KBLK = TT_KT * 128;                    // one K-block of a key tile: [64 keys x 128 B] = 8 KB
constexpr int TT_OFF_Q = 0;                             // 6 K-blocks x [64 rows x 128 B]
constexpr int TT_STAGE_BYTES = 6 * TT_KBLK;             // x: 4 K-blocks, kadd: 2 K-blocks
constexpr int TT_OFF_ST = 6 * 8192;
constexpr int TT_OFF_P = TT_OFF_ST + TT_STAGES * TT_STAGE_BYTES;   // 2 x [64 rows x 128 B]
constexpr int TT_OFF_BAR = TT_OFF_P + 2 * 8192;
constexpr int TT_OFF_XCH = TT_OFF_BAR + 256;            // row-max / row-sum exchange between the two column halves
constexpr int TT_SMEM = TT_OFF_XCH + 2048;

struct T2ITCParams {
  float* opart;   // [B, ns, 64, 256] unnormalised partial outputs
  float* ml;      // [B, ns, 2, 64] running max (log2 domain) and row sum
  int nk, ns, x_bstride;
};

// MN-major, 128-byte-swizzled shared-memory matrix descriptor: 128-byte rows hold 64 contiguous MN elements of one
// k index, 8 consecutive k indices form a 1024-byte swizzle atom; SBO = byte distance between 8-k groups, LBO = byte
// distance between 64-element atoms along MN (canonical layout ((8,n),(8,k)):((1,LBO),(8,SBO)) in 16-byte units).
__device__ __forceinline__ uint64_t umma_desc_mn_sw128(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3FFFF) >> 4);
  d |= static_cast<uint64_t>(lbo_bytes >> 4) << 16;
  d |= static_cast<uint64_t>(sbo_bytes >> 4) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(2) << 61;
  return d;
}
__device__ __forceinline__ void pair_barrier(int q) {  // the two warps (key halves) that share a TMEM lane quadrant
  asm volatile("bar.sync %0, 64;" ::"r"(q + 2) : "memory");
}
__device__ __forceinline__ void sts128(uint32_t addr, uint4 v) {
  asm volatile("st.shared.v4.u32 [%0], {%1,%2,%3,%4};" ::"r"(addr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

__global__ void __launch_bounds__(TT_THREADS, 1)
t2i_tc_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmX,
              const __grid_constant__ CUtensorMap tmKA, const T2ITCParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + TT_OFF_BAR);
  uint64_t* q_full = bars;             // 1
  uint64_t* st_full = bars + 1;        // 3
  uint64_t* st_empty = bars + 4;       // 3
  uint64_t* s_full = bars + 7;         // 2
  uint64_t* p_full = bars + 9;         // 2
  uint64_t* pv_done = bars + 11;       // 2
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(bars + 13);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int split = blockIdx.x, b = blockIdx.y;
  const int keys_per_split = p.nk / p.ns;
  const int key0 = split * keys_per_split;
  const int T = keys_per_split / TT_KT;

  if ((sb::smem_u32(smem) & 1023u) != 0u) __trap();
  if (warp == 0 && lane == 0) {
    sb::tma_prefetch_desc(&tmQ);
    sb::tma_prefetch_desc(&tmX);
    sb::tma_prefetch_desc(&tmKA);
  }
  if (warp == 1 && lane == 0) {
    sb::mbar_init(q_full, 1);
    for (int i = 0; i < TT_STAGES; ++i) {
      sb::mbar_init(&st_full[i], 1);
      sb::mbar_init(&st_empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      sb::mbar_init(&s_full[i], 1);
      sb::mbar_init(&p_full[i], 8);
      sb::mbar_init(&pv_done[i], 1);
    }
    sb::fence_barrier_init();
  }
  if (warp == 2) {
    sb::tmem_alloc(tmem_ptr, 512);
    sb::tmem_relinquish();
  }
  sb::tc_fence_before();
  __syncthreads();
  sb::tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;
  // TMEM columns: S buffers at [0,64) and [64,128); O at [128,384)

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      sb::mbar_arrive_expect_tx(q_full, 6 * 8192);
      for (int kb = 0; kb < 6; ++kb) sb::tma_load_2d(smem + TT_OFF_Q + kb * 8192, &tmQ, q_full, kb * 64, b * 64);
      const int xrow0 = b * p.x_bstride + key0;
      for (int t = 0; t < T; ++t) {
        const int s = t % TT_STAGES;
        if (t >= TT_STAGES) sb::mbar_wait(&st_empty[s], static_cast<uint32_t>((t / TT_STAGES - 1) & 1));
        uint8_t* dst = smem + TT_OFF_ST + s * TT_STAGE_BYTES;
        sb::mbar_arrive_expect_tx(&st_full[s], TT_STAGE_BYTES);
        for (int kb = 0; kb < 4; ++kb) sb::tma_load_2d(dst + kb * TT_KBLK, &tmX, &st_full[s], kb * 64, xrow0 + t * TT_KT);
        for (int kb = 0; kb < 2; ++kb)
          sb::tma_load_2d(dst + (4 + kb) * TT_KBLK, &tmKA, &st_full[s], kb * 64, key0 + t * TT_KT);
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    // The whole warp runs this role converged and one elected lane issues each tcgen05 instruction: inside a divergent
    // `if (lane == 0)` the compiler wraps every UMMA in an ELECT / BRA.U.ANY loop (~13 instructions and several R2UR
    // round trips per UMMA), which made the M = 64 UMMAs of this kernel issue-bound (the MMA thread never waited).
    {
      constexpr uint32_t idesc_qk = sb::umma_idesc_bf16(64, 64);
      constexpr uint32_t idesc_pv = sb::umma_idesc_bf16(64, 256) | (1u << 16);  // B operand MN-major
      const uint32_t sbase = sb::smem_u32(smem);
      auto issue_qk = [&](int t) {
        const int s = t % TT_STAGES;
        sb::mbar_wait(&st_full[s], static_cast<uint32_t>((t / TT_STAGES) & 1));
        sb::tc_fence_after();
        const uint32_t d = tmem_base + static_cast<uint32_t>((t & 1) * 64);
#pragma unroll
        for (int kb = 0; kb < 6; ++kb) {
          const uint64_t da = sb::umma_desc_k_sw128(sbase + TT_OFF_Q + kb * 8192);
          const uint64_t db = sb::umma_desc_k_sw128(sbase + TT_OFF_ST + s * TT_STAGE_BYTES + kb * TT_KBLK);
#pragma unroll
          for (int k = 0; k < 4; ++k)
            if (sb::elect_one())
              sb::umma_bf16(d, da + static_cast<uint64_t>(2 * k), db + static_cast<uint64_t>(2 * k), idesc_qk,
                            static_cast<uint32_t>((kb | k) != 0));
        }
        if (sb::elect_one()) sb::umma_commit(&s_full[t & 1]);
        __syncwarp();
      };
      sb::mbar_wait(q_full, 0);
      issue_qk(0);
      if (T > 1) issue_qk(1);
      for (int t = 0; t < T; ++t) {
        const int s = t % TT_STAGES;
        sb::mbar_wait(&p_full[t & 1], static_cast<uint32_t>((t >> 1) & 1));
        sb::tc_fence_after();
        const uint32_t d = tmem_base + 128u;
        const uint64_t da = sb::umma_desc_k_sw128(sbase + TT_OFF_P + (t & 1) * 8192);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          // 16 keys per step: two 8-key swizzle atoms (1024 B each) of every 64-channel K-block of the x tile
          const uint64_t db = umma_desc_mn_sw128(sbase + TT_OFF_ST + s * TT_STAGE_BYTES + k * 2048, TT_KBLK, 1024);
          if (sb::elect_one())
            sb::umma_bf16(d, da + static_cast<uint64_t>(2 * k), db, idesc_pv, static_cast<uint32_t>((t | k) != 0));
        }
        if (sb::elect_one()) {
          sb::umma_commit(&pv_done[t & 1]);
          sb::umma_commit(&st_empty[s]);
        }
        __syncwarp();
        if (t + 2 < T) issue_qk(t + 2);
      }
    }
  } else if (warp >= 4) {
    // ===================== online softmax =====================
    // With M = 64 the rows 16q..16q+15 live in lanes 0..15 of TMEM lane quadrant q. Two warps share a quadrant and
    // split the 64 keys of a tile (and the 256 columns of O): thread = (row, key half). The row maximum is exchanged
    // through shared memory, so both halves keep identical running maxima.
    const int q = warp & 3;
    const int hf = (warp - 4) >> 2;
    const bool active = lane < 16;
    const int r = q * 16 + (lane & 15);
    const uint32_t tlane = static_cast<uint32_t>(q * 32) << 16;
    const uint32_t sbase = sb::smem_u32(smem);
    float* xch = reinterpret_cast<float*>(smem + TT_OFF_XCH);  // [2 parities][2 halves][64 rows] maxima, then [2][64] sums
    float m = -INFINITY, l = 0.f;
#pragma unroll 1
    for (int t = 0; t < T; ++t) {
      sb::mbar_wait(&s_full[t & 1], static_cast<uint32_t>((t >> 1) & 1));
      sb::tc_fence_after();
      uint32_t v[32];
      const uint32_t ta = tmem_base + tlane + static_cast<uint32_t>((t & 1) * 64 + hf * 32);
      sb::tmem_ld_32x16(ta, v);
      sb::tmem_ld_32x16(ta + 16, v + 16);
      sb::tmem_ld_wait();
      float mx4[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) mx4[j] = __uint_as_float(v[j]);
#pragma unroll
      for (int j = 4; j < 32; ++j) mx4[j & 3] = fmaxf(mx4[j & 3], __uint_as_float(v[j]));
      float mx = fmaxf(fmaxf(mx4[0], mx4[1]), fmaxf(mx4[2], mx4[3]));
      if (active) xch[((t & 1) * 2 + hf) * 64 + r] = mx;
      pair_barrier(q);
      mx = fmaxf(mx, xch[((t & 1) * 2 + (hf ^ 1)) * 64 + r]);
      if (__any_sync(0xffffffffu, active && (mx > m + 8.f))) {
        // lazy rescale of O (rare): every previous PV has to be complete before O is touched; each half rescales its
        // 128 columns
        const float mn = fmaxf(m, mx);
        const float alpha = sb::fast_exp2(m - mn);  // m = -inf on the first tile -> 0 (O holds nothing yet)
        m = mn;
        l *= alpha;
        if (t > 0) {
          sb::mbar_wait(&pv_done[(t - 1) & 1], static_cast<uint32_t>(((t - 1) >> 1) & 1));
          sb::tc_fence_after();
          const uint32_t to = tmem_base + tlane + 128u + static_cast<uint32_t>(hf * 128);
#pragma unroll 1
          for (int c = 0; c < 8; ++c) {
            uint32_t o[16];
            sb::tmem_ld_32x16(to + c * 16, o);
            sb::tmem_ld_wait();
#pragma unroll
            for (int j = 0; j < 16; ++j) o[j] = __float_as_uint(__uint_as_float(o[j]) * alpha);
            sb::tmem_st_32x16(to + c * 16, o);
          }
          sb::tmem_st_wait();
        }
      }
      // P(t) overwrites the buffer the PV of tile t-2 read
      if (t >= 2) sb::mbar_wait(&pv_done[t & 1], static_cast<uint32_t>(((t >> 1) - 1) & 1));
      const uint32_t prow = sbase + TT_OFF_P + (t & 1) * 8192 + r * 128;
      const float2 nm2 = sb::splat2(-m);
      float2 l2[2] = {make_float2(0.f, 0.f), make_float2(0.f, 0.f)};
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        float2 e[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float2 d = sb::add2(make_float2(__uint_as_float(v[c * 8 + 2 * j]), __uint_as_float(v[c * 8 + 2 * j + 1])), nm2);
          e[j] = make_float2(sb::fast_exp2(d.x), sb::fast_exp2(d.y));
          l2[j & 1] = sb::add2(l2[j & 1], e[j]);
        }
        if (active)
          sts128(prow + (((hf * 4 + c) ^ (r & 7)) << 4),
                 make_uint4(sb::pack_bf16x2(e[0].x, e[0].y), sb::pack_bf16x2(e[1].x, e[1].y),
                            sb::pack_bf16x2(e[2].x, e[2].y), sb::pack_bf16x2(e[3].x, e[3].y)));
      }
      l += (l2[0].x + l2[0].y) + (l2[1].x + l2[1].y);
      sb::tc_fence_before();
      sb::fence_proxy_async();
      __syncwarp();
      if (lane == 0) sb::mbar_arrive(&p_full[t & 1]);
    }
    // ---- partial result of this split: unnormalised O (this half's 128 columns), running max and row sum
    if (active) xch[256 + hf * 64 + r] = l;
    pair_barrier(q);
    l += xch[256 + (hf ^ 1) * 64 + r];
    sb::mbar_wait(&pv_done[(T - 1) & 1], static_cast<uint32_t>(((T - 1) >> 1) & 1));
    sb::tc_fence_after();
    const long long pb = static_cast<long long>(b) * p.ns + split;
    float* orow = p.opart + (pb * 64 + r) * 256 + hf * 128;
    const uint32_t to = tmem_base + tlane + 128u + static_cast<uint32_t>(hf * 128);
#pragma unroll 1
    for (int c = 0; c < 8; ++c) {
      uint32_t o[16];
      sb::tmem_ld_32x16(to + c * 16, o);
      sb::tmem_ld_wait();
      if (active) {
#pragma unroll
        for (int j = 0; j < 4; ++j)
          *reinterpret_cast<uint4*>(orow + c * 16 + 4 * j) = make_uint4(o[4 * j], o[4 * j + 1], o[4 * j + 2], o[4 * j + 3]);
      }
    }
    if (active && hf == 0) {
      float* ml = p.ml + pb * 128;
      ml[r] = m;
      ml[64 + r] = l;
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

// internal launchers of decoder_fused.cu
int sb_internal_i2t_fold(const void* kt, long long kt_ld, const void* vt, long long vt_ld, const void* wq, const void* wo,
                         const float* bo, void* w1t, int w1_ld, int blockdiag, void* w2t, void* kts, int batch, int nt,
                         float scale, cudaStream_t stream);
int sb_internal_t2i_unfold(const float* opart, const float* ml, int ns, const void* wv, const float* bv, void* out,
                           long long out_ld, int batch, int nt, cudaStream_t stream);

extern "C" int sb_t2i_tc_splits(int batch, int nk) {
  // one CTA per SM (TMEM): enough (split, prompt) CTAs to fill 148 SMs a few times, each at least 8 tiles long
  int ns = batch >= 96 ? 4 : (batch >= 48 ? 8 : 16);
  while (ns > 1 && ((nk % (ns * TT_KT)) != 0 || nk / (ns * TT_KT) < 4)) ns >>= 1;
  return ns;
}

// Token -> image attention of the mask decoder straight on the image stream (see the header of this file).
// q [batch*nt, 128] bf16 (projected token queries incl. bias), x [batch*nk (nk when x_shared), 256] bf16, kadd [nk,128]
// bf16 (= image_pe Wk^T + bk), wk / wv [128,256] bf16 (the k_proj / v_proj weights), bv [128] fp32. Workspaces
// (caller-owned): qf [batch,64,384] bf16 (folded queries followed by the block-diagonal scaled queries), qs [batch,8,128]
// bf16, opart [batch,ns,64,256] fp32, ml [batch,ns,2,64] fp32 with ns = sb_t2i_tc_splits(batch, nk).
// out [batch*nt, 128] bf16 = the attention output before out_proj. nt <= 8, nk a multiple of 256.
extern "C" int sb_t2i_fold_attention_tc(const void* q, long long q_ld, const void* x, int x_shared, const void* kadd,
                                        const void* wk, const void* wv, const float* bv, void* qf, void* qs, float* opart,
                                        float* ml, void* out, long long out_ld, int batch, int nt, int nk, float scale,
                                        void* stream) {
  SB_REQUIRE(batch > 0 && nt >= 1 && nt <= 8, "sb_t2i_fold_attention_tc: nt must be in 1..8 (got %d)", nt);
  SB_REQUIRE(nk > 0 && (nk % 256) == 0, "sb_t2i_fold_attention_tc: nk must be a positive multiple of 256 (got %d)", nk);
  SB_REQUIRE(q && x && kadd && wk && wv && bv && qf && qs && opart && ml && out, "sb_t2i_fold_attention_tc: null operand");
  SB_REQUIRE(((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(kadd) | reinterpret_cast<uintptr_t>(qf) |
               reinterpret_cast<uintptr_t>(qs) | reinterpret_cast<uintptr_t>(wv) | reinterpret_cast<uintptr_t>(opart)) & 15) == 0,
             "sb_t2i_fold_attention_tc: operands must be 16-byte aligned");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const int ns = sb_t2i_tc_splits(batch, nk);
  int rc = sb_internal_i2t_fold(q, q_ld, nullptr, 0, wk, nullptr, nullptr, qf, 384, 1, nullptr, qs, batch, nt, scale, st);
  if (rc != SB_OK) return rc;
  CUtensorMap tmQ, tmX, tmKA;
  rc = sb_make_tmap_2d_bf16(&tmQ, qf, static_cast<uint64_t>(batch) * 64, 384, 384, 64, 64);
  if (rc != SB_OK) return rc;
  rc = sb_make_tmap_2d_bf16(&tmX, x, static_cast<uint64_t>(x_shared ? 1 : batch) * nk, 256, 256, TT_KT, 64);
  if (rc != SB_OK) return rc;
  rc = sb_make_tmap_2d_bf16(&tmKA, kadd, static_cast<uint64_t>(nk), 128, 128, TT_KT, 64);
  if (rc != SB_OK) return rc;
  static SbPerDeviceOnce attr_once;
  if (attr_once.need()) {
    SB_CHECK_CUDA(cudaFuncSetAttribute(t2i_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, TT_SMEM));
    attr_once.mark();
  }
  T2ITCParams p;
  p.opart = opart;
  p.ml = ml;
  p.nk = nk;
  p.ns = ns;
  p.x_bstride = x_shared ? 0 : nk;
  t2i_tc_kernel<<<dim3(ns, batch), TT_THREADS, TT_SMEM, st>>>(tmQ, tmX, tmKA, p);
  SB_CHECK_LAUNCH();
  return sb_internal_t2i_unfold(opart, ml, ns, wv, bv, out, out_ld, batch, nt, st);
}
