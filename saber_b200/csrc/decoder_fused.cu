// saber_b200 — per-prompt operand fold and key-split merge of the SAM2 mask decoder's fused attention blocks, shared by
// the two tcgen05 kernels (decoder_i2t_tc.cu, decoder_t2i_tc.cu).
//
// "Image attends to tokens" (upstream sam2/modeling/sam/transformer.py TwoWayAttentionBlock.forward, step 4):
//     q = keys + key_pe ; k = queries + query_pe ; v = queries
//     attn_out = cross_attn_image_to_token(q, k, v)          # 8 heads x 16, 4096 image queries, <= 8 token keys
//     keys = norm4(keys + attn_out)
// Unfused this is three passes over the per-prompt image stream [B, 4096, 256] (Q projection GEMM, few-keys attention,
// out-projection GEMM + LayerNorm: 5 x 2 MB of HBM traffic per prompt). Because a prompt has at most 8 tokens, both
// projections fold into per-prompt weights:
//     scores[i, (h,t)] = keys_i . (Wq_h^T kt_{t,h}) + qres_{i,h} . kt_{t,h}        qres = image_pe Wq^T + bq (weights only)
//     keys_new_i       = LN(keys_i + bo + sum_{h,t} p[i,(h,t)] (Wo_h vt_{t,h}))
// so the whole block is   S = X W1  ->  per-head softmax over 8 tokens  ->  O = P W2  ->  + residual, LayerNorm
// with W1 [256 x 64], W2 [64 x 256] per prompt: one read and one write of the image stream (2 x 2 MB per prompt).
// Every head's softmax row sums to 1, so bo / 8 added to each of the 64 (head, token) columns of W2 contributes exactly
// bo: the block needs no separate bias. i2t_fold_kernel builds W1, W2 and the scaled token keys; sb_i2t_block_tc runs
// the block.
//
// "Tokens attend to image" (step 2 and final_attn_token_to_image) folds the k / v projections onto the token side:
//     score[(h,t), j] = (Wk_h^T q_{t,h}) . x_j + q_{t,h} . kadd_{j,h}          kadd = image_pe Wk^T + bk (weights only)
//     out[t, h]       = Wv_h (sum_j p[(h,t), j] x_j) + bv_h                    (sum_j p = 1)
// i.e. flash attention with 64 query rows of width 256 whose keys AND values are the raw image stream x [4096, 256]:
// the stream is read once (2 MB per prompt) instead of being projected (read 2 MB, write 2 MB) and read again.
// i2t_fold_kernel builds the folded queries, sb_t2i_fold_attention_tc computes unnormalised partial results per key
// split, and t2i_unfold_kernel merges the splits and applies Wv / bv.
#include "common.cuh"

namespace {

using bf16 = __nv_bfloat16;

constexpr int I2T_C = 256;    // image stream width
constexpr int I2T_QD = 128;   // attention width (8 heads x 16)
constexpr int I2T_TOK = 8;    // token slots per head (padded with masked slots)
constexpr int I2T_NC = 64;    // (head, token) columns

// ------------------------------------------------------------------------------------------------
// Per-prompt folded operands. One block per prompt, 256 threads.
//   kts [B, 8, 128]  = scale*log2(e) * kt                     (zero rows for t >= nt)
//   w1t [B, 64, 256] : row (h*8+t), col c = scale*log2(e) * sum_d Wq[h*16+d, c] kt[t, h*16+d]
//   w2t [B, 256, 64] : row c, col (h*8+t) = bo[c] / 8 + sum_d Wo[c, h*16+d] vt[t, h*16+d]      (nullable)
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
i2t_fold_kernel(const bf16* __restrict__ kt, long long kt_ld, const bf16* __restrict__ vt, long long vt_ld,
                const bf16* __restrict__ wq /* [128,256] */, const bf16* __restrict__ wo /* [256,128] */,
                bf16* __restrict__ w1t, bf16* __restrict__ w2t, bf16* __restrict__ kts, int nt, float scale_log2,
                const float* __restrict__ bo /* out-projection bias folded into w2t (bo / 8 per column) */,
                int w1_ld /* row pitch of w1t (elements) */, int blockdiag /* w1t rows continue with the block-diagonal
                scaled keys in columns [256, 384): row (h,t) holds kts[t, h*16..h*16+15] at 256 + h*16 */) {
  // One block per (head, prompt, operand): blockIdx.z == 0 -> kts + w1t (from kt), 1 -> w2t (from vt). Each thread owns
  // one of the 256 channels and needs 16 weights: a single round of independent loads (the kernel is pure latency).
  __shared__ float sk[I2T_TOK][16];
  const int h = blockIdx.x, b = blockIdx.y, tid = threadIdx.x;
  const bool second = blockIdx.z == 1;
  const int c = tid;
  if (!second) {
    float w[16];
#pragma unroll
    for (int d = 0; d < 16; ++d) w[d] = __bfloat162float(wq[(h * 16 + d) * I2T_C + c]);
    if (tid < I2T_TOK * 16) {
      const int t = tid >> 4, d = tid & 15;
      const float v = t < nt ? __bfloat162float(kt[(static_cast<long long>(b) * nt + t) * kt_ld + h * 16 + d]) * scale_log2 : 0.f;
      sk[t][d] = v;
      kts[(static_cast<long long>(b) * I2T_TOK + t) * I2T_QD + h * 16 + d] = __float2bfloat16(v);
    }
    __syncthreads();
    float acc[I2T_TOK];
#pragma unroll
    for (int t = 0; t < I2T_TOK; ++t) acc[t] = 0.f;
#pragma unroll
    for (int d = 0; d < 16; ++d) {
#pragma unroll
      for (int t = 0; t < I2T_TOK; ++t) acc[t] = fmaf(w[d], sk[t][d], acc[t]);
    }
#pragma unroll
    for (int t = 0; t < I2T_TOK; ++t)
      w1t[(static_cast<long long>(b) * I2T_NC + h * 8 + t) * w1_ld + c] = __float2bfloat16(acc[t]);
    if (blockdiag) {
      for (int i = tid; i < I2T_TOK * I2T_QD; i += 256) {
        const int t = i >> 7, col = i & 127;
        w1t[(static_cast<long long>(b) * I2T_NC + h * 8 + t) * w1_ld + I2T_C + col] =
            __float2bfloat16((col >> 4) == h ? sk[t][col & 15] : 0.f);
      }
    }
  } else {
    const uint4 wa = *reinterpret_cast<const uint4*>(wo + c * I2T_QD + h * 16);
    const uint4 wb = *reinterpret_cast<const uint4*>(wo + c * I2T_QD + h * 16 + 8);
    // every head's softmax row sums to 1, so bo[c] / 8 added to all 64 (head, token) columns contributes exactly bo[c]
    const float bfold = bo[c] * 0.125f;
    if (tid < I2T_TOK * 16) {
      const int t = tid >> 4, d = tid & 15;
      sk[t][d] = t < nt ? __bfloat162float(vt[(static_cast<long long>(b) * nt + t) * vt_ld + h * 16 + d]) : 0.f;
    }
    __syncthreads();
    float acc[I2T_TOK];
#pragma unroll
    for (int t = 0; t < I2T_TOK; ++t) acc[t] = bfold;
    const uint32_t w8[8] = {wa.x, wa.y, wa.z, wa.w, wb.x, wb.y, wb.z, wb.w};
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const float w0 = sb::bf16_lo(w8[e]), w1 = sb::bf16_hi(w8[e]);
#pragma unroll
      for (int t = 0; t < I2T_TOK; ++t) {
        acc[t] = fmaf(w0, sk[t][2 * e], acc[t]);
        acc[t] = fmaf(w1, sk[t][2 * e + 1], acc[t]);
      }
    }
    *reinterpret_cast<uint4*>(w2t + (static_cast<long long>(b) * I2T_C + c) * I2T_NC + h * 8) =
        make_uint4(sb::pack_bf16x2(acc[0], acc[1]), sb::pack_bf16x2(acc[2], acc[3]), sb::pack_bf16x2(acc[4], acc[5]),
                   sb::pack_bf16x2(acc[6], acc[7]));
  }
}

// Merge the key splits and apply the value projection: a[b*nt + t, h*16+d] = bv[h*16+d] + sum_c Wv[h*16+d, c] O[(h,t), c]
// with O = sum_s 2^(m_s - m) O_s / sum_s 2^(m_s - m) l_s. One block per (head, prompt), 256 threads.
template <int NS>
__global__ void __launch_bounds__(256)
t2i_unfold_kernel(const float* __restrict__ opart, const float* __restrict__ ml, const bf16* __restrict__ wv /*[128,256]*/,
                  const float* __restrict__ bv, bf16* __restrict__ out, long long out_ld, int nt) {
  __shared__ float so[I2T_TOK][I2T_C + 4];
  __shared__ float sw[I2T_TOK][NS];  // per (token row, split) weight 2^(m_s - m) / L
  constexpr int ns = NS;
  const int h = blockIdx.x, b = blockIdx.y, tid = threadIdx.x;
  // partial rows of head h (8 tokens x NS splits, thread = channel), in groups of <= 4 splits (32 independent loads in
  // flight; the first group is issued before the split weights are known)
  constexpr int G = NS < 4 ? NS : 4;
  float v[G][I2T_TOK];
  const float* ob = opart + (static_cast<long long>(b) * ns * I2T_NC + h * 8) * I2T_C + tid;
#pragma unroll
  for (int s = 0; s < G; ++s)
#pragma unroll
    for (int t = 0; t < I2T_TOK; ++t) v[s][t] = __ldg(ob + (static_cast<long long>(s) * I2T_NC + t) * I2T_C);
  if (tid < I2T_TOK) {
    const int row = h * 8 + tid;
    float mm[NS], ll[NS];
    float m = -INFINITY;
#pragma unroll
    for (int s = 0; s < NS; ++s) {
      const float* q = ml + (static_cast<long long>(b) * ns + s) * 2 * I2T_NC;
      mm[s] = q[row];
      ll[s] = q[I2T_NC + row];
      m = fmaxf(m, mm[s]);
    }
    float L = 0.f;
#pragma unroll
    for (int s = 0; s < NS; ++s) {
      mm[s] = sb::fast_exp2(mm[s] - m);
      L = fmaf(mm[s], ll[s], L);
    }
    const float inv = 1.f / L;
#pragma unroll
    for (int s = 0; s < NS; ++s) sw[tid][s] = mm[s] * inv;
  }
  __syncthreads();
  float part[I2T_TOK];
#pragma unroll
  for (int t = 0; t < I2T_TOK; ++t) part[t] = 0.f;
#pragma unroll
  for (int g0 = 0; g0 < NS; g0 += G) {
    if (g0 > 0) {
#pragma unroll
      for (int s = 0; s < G; ++s)
#pragma unroll
        for (int t = 0; t < I2T_TOK; ++t) v[s][t] = __ldg(ob + (static_cast<long long>(g0 + s) * I2T_NC + t) * I2T_C);
    }
#pragma unroll
    for (int s = 0; s < G; ++s)
#pragma unroll
      for (int t = 0; t < I2T_TOK; ++t) part[t] = fmaf(sw[t][g0 + s], v[s][t], part[t]);
  }
#pragma unroll
  for (int t = 0; t < I2T_TOK; ++t) so[t][tid] = part[t];
  // 8 tokens x 16 dims = 128 outputs, two threads (channel halves) each
  const int half = tid & 1, d = (tid >> 1) & 15, t = tid >> 5;
  const bf16* wrow = wv + (h * 16 + d) * I2T_C + half * 128;
  __syncthreads();
  // the 64 KB weight matrix is shared by every block (L1 / L2 hits): loaded four 16-byte pieces at a time so that the
  // kernel stays at ~48 registers (holding all 16 pieces next to the NS x 8 partial rows capped it at 2 blocks per SM)
  float acc = 0.f;
#pragma unroll
  for (int c32 = 0; c32 < 4; ++c32) {
    uint4 w8[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) w8[j] = __ldg(reinterpret_cast<const uint4*>(wrow + (c32 * 4 + j) * 8));
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float* ov = &so[t][half * 128 + (c32 * 4 + j) * 8];
      acc = fmaf(sb::bf16_lo(w8[j].x), ov[0], acc);
      acc = fmaf(sb::bf16_hi(w8[j].x), ov[1], acc);
      acc = fmaf(sb::bf16_lo(w8[j].y), ov[2], acc);
      acc = fmaf(sb::bf16_hi(w8[j].y), ov[3], acc);
      acc = fmaf(sb::bf16_lo(w8[j].z), ov[4], acc);
      acc = fmaf(sb::bf16_hi(w8[j].z), ov[5], acc);
      acc = fmaf(sb::bf16_lo(w8[j].w), ov[6], acc);
      acc = fmaf(sb::bf16_hi(w8[j].w), ov[7], acc);
    }
  }
  acc += __shfl_xor_sync(0xffffffffu, acc, 1);
  if (half == 0 && t < nt)
    out[(static_cast<long long>(b) * nt + t) * out_ld + h * 16 + d] = __float2bfloat16(acc + bv[h * 16 + d]);
}

}  // namespace

// ---- internal launchers shared with decoder_t2i_tc.cu ----------------------------------------------------------------
int sb_internal_i2t_fold(const void* kt, long long kt_ld, const void* vt, long long vt_ld, const void* wq, const void* wo,
                         const float* bo, void* w1t, int w1_ld, int blockdiag, void* w2t, void* kts, int batch, int nt,
                         float scale, cudaStream_t stream) {
  i2t_fold_kernel<<<dim3(8, batch, w2t ? 2 : 1), 256, 0, stream>>>(
      static_cast<const bf16*>(kt), kt_ld, static_cast<const bf16*>(vt), vt_ld, static_cast<const bf16*>(wq),
      static_cast<const bf16*>(wo), static_cast<bf16*>(w1t), static_cast<bf16*>(w2t), static_cast<bf16*>(kts), nt,
      scale * 1.4426950408889634f, bo, w1_ld, blockdiag);
  SB_CHECK_LAUNCH();
  return SB_OK;
}

int sb_internal_t2i_unfold(const float* opart, const float* ml, int ns, const void* wv, const float* bv, void* out,
                           long long out_ld, int batch, int nt, cudaStream_t st) {
  const bf16* w = static_cast<const bf16*>(wv);
  bf16* o = static_cast<bf16*>(out);
  if (ns == 16)
    t2i_unfold_kernel<16><<<dim3(8, batch), 256, 0, st>>>(opart, ml, w, bv, o, out_ld, nt);
  else if (ns == 8)
    t2i_unfold_kernel<8><<<dim3(8, batch), 256, 0, st>>>(opart, ml, w, bv, o, out_ld, nt);
  else if (ns == 4)
    t2i_unfold_kernel<4><<<dim3(8, batch), 256, 0, st>>>(opart, ml, w, bv, o, out_ld, nt);
  else if (ns == 2)
    t2i_unfold_kernel<2><<<dim3(8, batch), 256, 0, st>>>(opart, ml, w, bv, o, out_ld, nt);
  else if (ns == 1)
    t2i_unfold_kernel<1><<<dim3(8, batch), 256, 0, st>>>(opart, ml, w, bv, o, out_ld, nt);
  else {
    sb_set_error("t2i unfold: unsupported split count %d", ns);
    return SB_ERR_ARG;
  }
  SB_CHECK_LAUNCH();
  return SB_OK;
}

// Per-prompt folded operands of sb_i2t_block_tc (see the header of this file). kt / vt [B*nt, 128] bf16 (the projected
// token keys / values of cross_attn_image_to_token), wq [128,256] / wo [256,128] bf16 (its q_proj / out_proj weights),
// bo [256] fp32 (its out_proj bias, folded into w2t). Outputs: w1t [B,64,256], w2t [B,256,64], kts [B,8,128] bf16.
extern "C" int sb_i2t_fold(const void* kt, long long kt_ld, const void* vt, long long vt_ld, const void* wq, const void* wo,
                           const float* bo, void* w1t, void* w2t, void* kts, int batch, int nt, float scale, void* stream) {
  SB_REQUIRE(batch > 0 && nt >= 1 && nt <= I2T_TOK, "sb_i2t_fold: nt must be in 1..%d (got %d)", I2T_TOK, nt);
  SB_REQUIRE(kt && vt && wq && wo && bo && w1t && w2t && kts, "sb_i2t_fold: null operand");
  SB_REQUIRE(((reinterpret_cast<uintptr_t>(wo) | reinterpret_cast<uintptr_t>(w2t)) & 15) == 0, "sb_i2t_fold: wo / w2t must be 16-byte aligned");
  return sb_internal_i2t_fold(kt, kt_ld, vt, vt_ld, wq, wo, bo, w1t, I2T_C, 0, w2t, kts, batch, nt, scale,
                              reinterpret_cast<cudaStream_t>(stream));
}
