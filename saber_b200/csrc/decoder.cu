// saber_b200 — SAM2 prompt-encoder / mask-decoder glue kernels (everything that is not a GEMM,
// LayerNorm or attention): point-prompt token assembly with random-Fourier positional encoding,
// the fused mask-prompt down-scaling convs, the m2m pass's per-prompt image stream, the IoU gate and
// the dynamic-multimask-via-stability selection. (The transposed-conv up-scaling stages are fused
// into the GEMM epilogues of gemm_tcgen05.cu.)
// Restates sam2/modeling/sam/prompt_encoder.py and mask_decoder.py (SURVEY §8a U2/U3; HF
// modeling_sam2.py:712-856, 859-1296) as called from REF saber/adapters/sam2/automask.py:66-78.
#include "common.cuh"

namespace {

constexpr float kTwoPi = 6.283185307179586f;

// tokens[b, 0..5] = (obj_score_token, iou_token, mask_tokens[0..3]); tokens[b, 6 + p] = point p's
// embedding; last = padding point (label -1) when pad != 0. coords are in model-input pixels.
__global__ void __launch_bounds__(256)
prompt_tokens_kernel(const float* __restrict__ coords, const int* __restrict__ labels, int B, int Np,
                     int pad, const float* __restrict__ gauss /*[2,128]*/,
                     const float* __restrict__ point_emb /*[4,256]*/,
                     const float* __restrict__ not_a_point /*[256]*/,
                     const float* __restrict__ out_tokens /*[6,256]*/, float inv_size,
                     float* __restrict__ tokens, int Nt) {
  const int b = blockIdx.x;
  const int c = threadIdx.x;  // 0..255
  float* tb = tokens + static_cast<long long>(b) * Nt * 256;
  for (int t = 0; t < 6; ++t) tb[t * 256 + c] = out_tokens[t * 256 + c];
  const int f = c & 127;
  for (int p = 0; p < Np + (pad ? 1 : 0); ++p) {
    float x = 0.f, y = 0.f;
    int label = -1;
    if (p < Np) {
      x = coords[(static_cast<long long>(b) * Np + p) * 2 + 0];
      y = coords[(static_cast<long long>(b) * Np + p) * 2 + 1];
      label = labels[static_cast<long long>(b) * Np + p];
    }
    // (coord + 0.5) / size -> [0,1] -> [-1,1] -> @ gaussian -> * 2pi -> [sin | cos]
    const float nx = 2.f * ((x + 0.5f) * inv_size) - 1.f;
    const float ny = 2.f * ((y + 0.5f) * inv_size) - 1.f;
    const float proj = kTwoPi * (nx * gauss[f] + ny * gauss[128 + f]);
    float v = (c < 128) ? sinf(proj) : cosf(proj);
    if (label == -1)
      v = not_a_point[c];
    else if (label >= 0 && label < 4)
      v += point_emb[label * 256 + c];
    tb[(6 + p) * 256 + c] = v;
  }
}

// Fused mask_downscaling[0..5]: Conv2d(1->4,k2,s2) + LN2d(4) + GELU + Conv2d(4->16,k2,s2) + LN2d(16)
// + GELU. in: [B, S, S] fp32 (S = 256) -> out: [B*(S/4)^2, 16] bf16 token-major.
__global__ void __launch_bounds__(256)
mask_downscale_kernel(const float* __restrict__ in, int B, int S, int cpp, float clampv,
                      const float* __restrict__ w1,
                      const float* __restrict__ b1, const float* __restrict__ g1,
                      const float* __restrict__ be1, const float* __restrict__ w2,
                      const float* __restrict__ b2, const float* __restrict__ g2,
                      const float* __restrict__ be2, __nv_bfloat16* __restrict__ out) {
  __shared__ float sw1[16], sb1[4], sg1[4], sbe1[4], sw2[256], sb2[16], sg2[16], sbe2[16];
  for (int i = threadIdx.x; i < 256; i += blockDim.x) sw2[i] = w2[i];
  if (threadIdx.x < 16) {
    sw1[threadIdx.x] = w1[threadIdx.x];
    sb2[threadIdx.x] = b2[threadIdx.x];
    sg2[threadIdx.x] = g2[threadIdx.x];
    sbe2[threadIdx.x] = be2[threadIdx.x];
  }
  if (threadIdx.x < 4) {
    sb1[threadIdx.x] = b1[threadIdx.x];
    sg1[threadIdx.x] = g1[threadIdx.x];
    sbe1[threadIdx.x] = be1[threadIdx.x];
  }
  __syncthreads();
  const int T = S / 4;
  const long long total = static_cast<long long>(B) * T * T;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int tx = static_cast<int>(i % T), ty = static_cast<int>((i / T) % T);
    const int b = static_cast<int>(i / (static_cast<long long>(T) * T));
    // cpp == 3: mask prompt b is token 1 + b % 3 of prompt b / 3 in a [*, 4, S, S] decoder output (m2m pass)
    const long long pl = cpp == 3 ? static_cast<long long>(b / 3) * 4 + 1 + b % 3 : b;
    const float* src = in + (pl * S + ty * 4) * S + tx * 4;
    float h1[2][2][4];  // [py][px][channel] after conv1 + LN + GELU
#pragma unroll
    for (int py = 0; py < 2; ++py)
#pragma unroll
      for (int px = 0; px < 2; ++px) {
        float a00 = src[(py * 2 + 0) * S + px * 2 + 0], a01 = src[(py * 2 + 0) * S + px * 2 + 1];
        float a10 = src[(py * 2 + 1) * S + px * 2 + 0], a11 = src[(py * 2 + 1) * S + px * 2 + 1];
        if (clampv > 0.f) {  // upstream clamps the low-res logits fed back as mask prompts to +-32
          a00 = fminf(fmaxf(a00, -clampv), clampv);
          a01 = fminf(fmaxf(a01, -clampv), clampv);
          a10 = fminf(fmaxf(a10, -clampv), clampv);
          a11 = fminf(fmaxf(a11, -clampv), clampv);
        }
        float c[4], mean = 0.f;
#pragma unroll
        for (int o = 0; o < 4; ++o) {
          c[o] = sb1[o] + sw1[o * 4 + 0] * a00 + sw1[o * 4 + 1] * a01 + sw1[o * 4 + 2] * a10 +
                 sw1[o * 4 + 3] * a11;
          mean += c[o];
        }
        mean *= 0.25f;
        float var = 0.f;
#pragma unroll
        for (int o = 0; o < 4; ++o) var += (c[o] - mean) * (c[o] - mean);
        const float rstd = rsqrtf(var * 0.25f + 1e-6f);
#pragma unroll
        for (int o = 0; o < 4; ++o)
          h1[py][px][o] = sb::gelu_erf((c[o] - mean) * rstd * sg1[o] + sbe1[o]);
      }
    float c2[16], mean = 0.f;
#pragma unroll
    for (int o = 0; o < 16; ++o) {
      float acc = sb2[o];
#pragma unroll
      for (int ci = 0; ci < 4; ++ci)
#pragma unroll
        for (int py = 0; py < 2; ++py)
#pragma unroll
          for (int px = 0; px < 2; ++px) acc += sw2[((o * 4 + ci) * 2 + py) * 2 + px] * h1[py][px][ci];
      c2[o] = acc;
      mean += acc;
    }
    mean *= (1.f / 16.f);
    float var = 0.f;
#pragma unroll
    for (int o = 0; o < 16; ++o) var += (c2[o] - mean) * (c2[o] - mean);
    const float rstd = rsqrtf(var * (1.f / 16.f) + 1e-6f);
    uint32_t packed[8];
#pragma unroll
    for (int o = 0; o < 16; o += 2) {
      const float v0 = sb::gelu_erf((c2[o] - mean) * rstd * sg2[o] + sbe2[o]);
      const float v1 = sb::gelu_erf((c2[o + 1] - mean) * rstd * sg2[o + 1] + sbe2[o + 1]);
      packed[o >> 1] = sb::pack_bf16x2(v0, v1);
    }
    uint4* dst = reinterpret_cast<uint4*>(out + i * 16);
    dst[0] = make_uint4(packed[0], packed[1], packed[2], packed[3]);
    dst[1] = make_uint4(packed[4], packed[5], packed[6], packed[7]);
  }
}


// keys[b*T + t, n] = bf16(image_embed[t, n] + bias[n] + sum_c ds[b*T + t, c] * w[n, c])   (n < 256, c < 16):
// mask_downscaling[6] (1x1 conv 16 -> 256) plus the dense-prompt add of the mask decoder (src = image_embeddings +
// dense_prompt_embeddings), i.e. the per-prompt image stream of the m2m pass, written once. The K = 16 contraction is
// exactly one mma.sync.m16n8k16 step per 16 tokens x 8 channels (a CUDA-core version needs 128 FMA instructions per
// token and is instruction-bound at ~6x the store time): the 16 x 256 weights live in registers as B fragments, the
// accumulators are initialised with image_embed + bias (fp32, loaded once per token tile and reused for `PPW`
// prompts), and the bf16 result is staged through a per-warp shared-memory tile so that every global store
// instruction writes one full 512-byte row. The kernel is bound by the 512 B it stores per token.
constexpr int MEK_PPW = 8;     // prompts per warp (reuse of the image_embed tile held in registers)
constexpr int MEK_PITCH = 528; // staged row pitch (bytes): odd multiple of 16

__device__ __forceinline__ void mek_mma(float* c, const uint32_t* a, uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%10,%11,%12,%13};"
      : "=f"(c[0]), "=f"(c[1]), "=f"(c[2]), "=f"(c[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1), "f"(c[4]), "f"(c[5]), "f"(c[6]), "f"(c[7]));
}

__global__ void __launch_bounds__(128)
mask_embed_keys_kernel(const __nv_bfloat16* __restrict__ ds, const float* __restrict__ w /*[256,16]*/,
                       const float* __restrict__ bias, const float* __restrict__ image_embed /*[T,256]*/, int T,
                       int nprompts, __nv_bfloat16* __restrict__ keys) {
  __shared__ __align__(16) uint8_t stage[4][16 * MEK_PITCH];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, q4 = lane & 3;
  const int tile = blockIdx.x * 4 + warp;  // 16-token tile of the image grid
  const int tok0 = tile * 16;
  if (tok0 >= T) return;
  // The k index is permuted identically on A and B (MMA k = 2*q4+e <-> dim 4*q4+e, MMA k = 8+2*q4+e <-> dim 4*q4+2+e),
  // so the A fragment of a token row is one 8-byte load; the B fragments of a channel half stay in registers.
  uint8_t* st = stage[warp];
  const int b_begin = blockIdx.y * MEK_PPW;
  const int b_end = min(nprompts, b_begin + MEK_PPW);
#pragma unroll 1
  for (int half = 0; half < 2; ++half) {  // channels [128*half, 128*half + 128): keeps init + accumulators at 64 + 64 regs
    uint32_t wb[16][2];
#pragma unroll
    for (int n = 0; n < 16; ++n) {
      const float4 w4 = __ldg(reinterpret_cast<const float4*>(w + (half * 128 + n * 8 + g) * 16 + q4 * 4));
      wb[n][0] = sb::pack_bf16x2(w4.x, w4.y);
      wb[n][1] = sb::pack_bf16x2(w4.z, w4.w);
    }
    float init[16][4];
#pragma unroll
    for (int n = 0; n < 16; ++n) {
      const int c = half * 128 + n * 8 + 2 * q4;
      const float2 bb = __ldg(reinterpret_cast<const float2*>(bias + c));
      const float2 e0 = __ldg(reinterpret_cast<const float2*>(image_embed + static_cast<size_t>(tok0 + g) * 256 + c));
      const float2 e1 = __ldg(reinterpret_cast<const float2*>(image_embed + static_cast<size_t>(tok0 + g + 8) * 256 + c));
      init[n][0] = e0.x + bb.x;
      init[n][1] = e0.y + bb.y;
      init[n][2] = e1.x + bb.x;
      init[n][3] = e1.y + bb.y;
    }
#pragma unroll 1
    for (int b = b_begin; b < b_end; ++b) {
      const size_t row0 = static_cast<size_t>(b) * T + tok0;
      const uint2 alo = *reinterpret_cast<const uint2*>(ds + (row0 + g) * 16 + q4 * 4);
      const uint2 ahi = *reinterpret_cast<const uint2*>(ds + (row0 + g + 8) * 16 + q4 * 4);
      const uint32_t a[4] = {alo.x, ahi.x, alo.y, ahi.y};
#pragma unroll
      for (int n = 0; n < 16; ++n) {
        float c[8] = {0.f, 0.f, 0.f, 0.f, init[n][0], init[n][1], init[n][2], init[n][3]};
        mek_mma(c, a, wb[n][0], wb[n][1]);
        const int col = n * 8 + 2 * q4;
        *reinterpret_cast<uint32_t*>(st + g * MEK_PITCH + col * 2) = sb::pack_bf16x2(c[0], c[1]);
        *reinterpret_cast<uint32_t*>(st + (g + 8) * MEK_PITCH + col * 2) = sb::pack_bf16x2(c[2], c[3]);
      }
      __syncwarp();
      // 16 rows x 256 B (this half): two rows per warp instruction, 16 B per lane
      uint8_t* dst = reinterpret_cast<uint8_t*>(keys + row0 * 256 + half * 128);
#pragma unroll
      for (int it = 0; it < 8; ++it) {
        const int r = it * 2 + (lane >> 4);
        *reinterpret_cast<uint4*>(dst + static_cast<size_t>(r) * 512 + (lane & 15) * 16) =
            *reinterpret_cast<const uint4*>(st + r * MEK_PITCH + (lane & 15) * 16);
      }
      __syncwarp();
    }
  }
}

// AMG m2m pass: which prompts can still pass `iou > thresh` whatever dynamic_multimask_via_stability picks? The output
// IoU of a prompt is ious[b][0] or max(ious[b][1..3]), so max over the four is an upper bound: prompts below it are
// discarded by SAM2AutomaticMaskGenerator's pred_iou_thresh filter without their masks ever being looked at
// (automatic_mask_generator.py _process_batch: keep = data["iou_preds"] > pred_iou_thresh), and the up-scaling GEMMs
// skip them. Ordered compaction (ascending prompt index) by one block; list [B], count [1].
__global__ void __launch_bounds__(1024)
iou_gate_kernel(const float* __restrict__ ious /*[B,4]*/, int B, float thresh, int* __restrict__ list,
                int* __restrict__ count) {
  __shared__ int warp_tot[32];
  __shared__ int base_s;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (threadIdx.x == 0) base_s = 0;
  __syncthreads();
  for (int b0 = 0; b0 < B; b0 += blockDim.x) {
    const int b = b0 + threadIdx.x;
    bool pass = false;
    if (b < B) {
      const float4 v = __ldg(reinterpret_cast<const float4*>(ious) + b);
      pass = fmaxf(fmaxf(v.x, v.y), fmaxf(v.z, v.w)) > thresh;
    }
    const unsigned m = __ballot_sync(0xffffffffu, pass);
    if (lane == 0) warp_tot[warp] = __popc(m);
    __syncthreads();
    int off = base_s;
    for (int w = 0; w < warp; ++w) off += warp_tot[w];
    if (pass) list[off + __popc(m & ((1u << lane) - 1u))] = b;
    __syncthreads();
    if (threadIdx.x == 0) {
      int t = 0;
      for (int w = 0; w < static_cast<int>(blockDim.x >> 5); ++w) t += warp_tot[w];
      base_s += t;
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) *count = base_s;
}

// dynamic_multimask_via_stability (single-mask output): per prompt, stability of mask token 0 =
// count(logit > delta) / count(logit > -delta) (1 when the union is empty); if >= thresh keep token 0
// else the best-IoU token among 1..3 (first max). Writes the chosen token index and IoU.
__global__ void __launch_bounds__(1024)
select_mask_kernel(const float* __restrict__ masks /*[B,4,HW]*/, const float* __restrict__ ious /*[B,4]*/,
                   int HW, float delta, float thresh, int* __restrict__ sel_idx,
                   float* __restrict__ sel_iou) {
  const int b = blockIdx.x;
  const float* m0 = masks + static_cast<long long>(b) * 4 * HW;
  int ci = 0, cu = 0;
  // one plane (256 KB at 256^2) per block: 16-byte loads, four in flight per thread (the counts are integers, so the
  // summation order is free)
  const int n4 = ((reinterpret_cast<uintptr_t>(m0) & 15) == 0) ? (HW >> 2) : 0;
  const float4* m4 = reinterpret_cast<const float4*>(m0);
  int i = threadIdx.x;
  for (; i + 3 * static_cast<int>(blockDim.x) < n4; i += 4 * blockDim.x) {
    float4 v[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) v[u] = __ldg(m4 + i + u * blockDim.x);
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      ci += (v[u].x > delta) + (v[u].y > delta) + (v[u].z > delta) + (v[u].w > delta);
      cu += (v[u].x > -delta) + (v[u].y > -delta) + (v[u].z > -delta) + (v[u].w > -delta);
    }
  }
  for (; i < n4; i += blockDim.x) {
    const float4 v = __ldg(m4 + i);
    ci += (v.x > delta) + (v.y > delta) + (v.z > delta) + (v.w > delta);
    cu += (v.x > -delta) + (v.y > -delta) + (v.z > -delta) + (v.w > -delta);
  }
  for (int j = n4 * 4 + threadIdx.x; j < HW; j += blockDim.x) {
    const float v = m0[j];
    ci += v > delta;
    cu += v > -delta;
  }
  __shared__ int si[32], su[32];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    ci += __shfl_xor_sync(0xffffffffu, ci, o);
    cu += __shfl_xor_sync(0xffffffffu, cu, o);
  }
  if ((threadIdx.x & 31) == 0) {
    si[threadIdx.x >> 5] = ci;
    su[threadIdx.x >> 5] = cu;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    int ti = 0, tu = 0;
    for (int k = 0; k < static_cast<int>(blockDim.x >> 5); ++k) {
      ti += si[k];
      tu += su[k];
    }
    const float stab = tu > 0 ? static_cast<float>(ti) / static_cast<float>(tu) : 1.0f;
    int idx = 0;
    if (!(stab >= thresh)) {
      idx = 1;
      float best = ious[b * 4 + 1];
      for (int k = 2; k < 4; ++k)
        if (ious[b * 4 + k] > best) {
          best = ious[b * 4 + k];
          idx = k;
        }
    }
    sel_idx[b] = idx;
    sel_iou[b] = ious[b * 4 + idx];
  }
}

inline int blocks_for(long long threads_needed, int block = 256, int cap = 148 * 16) {
  long long g = (threads_needed + block - 1) / block;
  if (g > cap) g = cap;
  if (g < 1) g = 1;
  return static_cast<int>(g);
}

}  // namespace

extern "C" int sb_prompt_tokens(const float* coords, const int* labels, int B, int Np, int pad,
                                const float* gauss, const float* point_emb, const float* not_a_point,
                                const float* out_tokens, int image_size, float* tokens, void* stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  SB_REQUIRE(B > 0 && Np >= 0, "sb_prompt_tokens: bad sizes");
  const int Nt = 6 + Np + (pad ? 1 : 0);
  prompt_tokens_kernel<<<B, 256, 0, stream>>>(coords, labels, B, Np, pad, gauss, point_emb,
                                              not_a_point, out_tokens, 1.0f / image_size, tokens, Nt);
  SB_CHECK_LAUNCH();
  return SB_OK;
}

extern "C" int sb_mask_downscale(const float* in, int B, int S, int cpp, float clampv, const float* w1,
                                 const float* b1,
                                 const float* g1, const float* be1, const float* w2, const float* b2,
                                 const float* g2, const float* be2, void* out, void* stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  SB_REQUIRE(B > 0 && S % 4 == 0 && (cpp == 1 || cpp == 3), "sb_mask_downscale: bad sizes");
  const long long total = static_cast<long long>(B) * (S / 4) * (S / 4);
  mask_downscale_kernel<<<blocks_for(total), 256, 0, stream>>>(
      in, B, S, cpp, clampv, w1, b1, g1, be1, w2, b2, g2, be2, static_cast<__nv_bfloat16*>(out));
  SB_CHECK_LAUNCH();
  return SB_OK;
}

extern "C" int sb_mask_embed_keys(const void* ds, const float* w, const float* bias, const float* image_embed, int T,
                                  long long ntok, void* keys, void* stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  SB_REQUIRE(ds && w && bias && image_embed && keys && T > 0 && ntok > 0 && ntok < (1ll << 31),
             "sb_mask_embed_keys: bad arguments");
  SB_REQUIRE((T % 16) == 0 && (ntok % T) == 0, "sb_mask_embed_keys: T must be a multiple of 16 and ntok a multiple of T");
  const int nprompts = static_cast<int>(ntok / T);
  dim3 grid((T / 16 + 3) / 4, (nprompts + MEK_PPW - 1) / MEK_PPW);
  mask_embed_keys_kernel<<<grid, 128, 0, stream>>>(
      static_cast<const __nv_bfloat16*>(ds), w, bias, image_embed, T, nprompts, static_cast<__nv_bfloat16*>(keys));
  SB_CHECK_LAUNCH();
  return SB_OK;
}

extern "C" int sb_select_mask(const float* masks, const float* ious, int B, int HW, float delta,
                              float thresh, int* sel_idx, float* sel_iou, void* stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  SB_REQUIRE(B > 0 && HW > 0, "sb_select_mask: bad sizes");
  select_mask_kernel<<<B, 1024, 0, stream>>>(masks, ious, HW, delta, thresh, sel_idx, sel_iou);
  SB_CHECK_LAUNCH();
  return SB_OK;
}

extern "C" int sb_iou_gate(const float* ious4, int B, float thresh, int* list, int* count, void* stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  SB_REQUIRE(B > 0 && ious4 && list && count, "sb_iou_gate: bad arguments");
  SB_REQUIRE((reinterpret_cast<uintptr_t>(ious4) & 15) == 0, "sb_iou_gate: ious must be 16-byte aligned");
  iou_gate_kernel<<<1, 1024, 0, stream>>>(ious4, B, thresh, list, count);
  SB_CHECK_LAUNCH();
  return SB_OK;
}
