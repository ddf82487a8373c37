/* saber_b200 — C ABI of libsaber_b200.so (sm_100a CUDA kernels of SABER's SAM2 slice-wise hot path).
 *
 * The reference (chanzuckerberg/saber) is pure Python and has no FFI of its own: its plugin seam for this
 * path is the `sam2` package API (build_sam2 / SAM2ImagePredictor / SAM2AutomaticMaskGenerator, bound at
 * REF saber/adapters/sam2/automask.py:55-78, REF saber/adapters/sam2/predictor.py:24-26,
 * REF saber/classifier/models/SAM2.py:45-46). `saber_b200.sam2` re-implements that Python surface; every
 * arithmetic operation underneath it is one of the entry points below, reached through ctypes
 * (saber_b200/lib.py). Each entry point names the reference / upstream computation it replaces.
 *
 * Conventions
 *  - plain pointers and sizes only; all data pointers are DEVICE pointers unless marked [host];
 *  - the caller owns every buffer (the library allocates nothing persistent), `stream` is a cudaStream_t;
 *  - launches are asynchronous on `stream`; return value 0 = OK, negative = error (-1 CUDA, -2 bad argument,
 *    -3 unsupported device, -4 driver entry point); sb_last_error() returns the per-thread message;
 *  - no global mutable state besides per-process caches of function attributes: safe for SABER's
 *    one-thread-per-GPU GPUPool (REF saber/utils/parallelization.py:155) and one-process-per-GPU NCCL mode;
 *  - "bf16" buffers are __nv_bfloat16, row-major with the stated pitch in ELEMENTS.
 */
#ifndef SABER_B200_H
#define SABER_B200_H
#ifdef __cplusplus
extern "C" {
#endif

/* ---- runtime ---------------------------------------------------------------------------------------- */
const char* sb_last_error(void);
int sb_version(void);
int sb_device_sm_count(void);           /* SM count of the current device (148 on B200) */
int sb_require_sm100(void);             /* fails unless the current device is compute capability 10.x */

/* ---- tensor-core kernels (tcgen05 / TMEM / TMA) ----------------------------------------------------- */
/* out[M,N] = act(alpha * A[M,K] @ W[N,K]^T + bias[N]) + residual[m % res_mod (or m), N].
 * Replaces torch.nn.Linear / 1x1 Conv2d / ConvTranspose2d(k2,s2) (cuBLASLt / cuDNN) inside upstream sam2:
 * Hiera qkv/proj/mlp (sam2/modeling/backbones/hieradet.py), FpnNeck laterals, mask-decoder projections.
 * act: 0 none, 1 GELU(erf), 2 ReLU, 3 sigmoid. flags: bit0 out is fp32 (else bf16), bit1 residual is fp32.
 * force_bn: 0 = choose the kernel and tile N automatically (products with M >= 4096 and N >= 128 run on CTA pairs:
 * tcgen05.mma.cta_group::2 over 256 x {128,192,256} pair tiles with a TMA-store epilogue); 64 / 128 / 192 / 256 = that
 * tile N on the single-CTA kernel; -128 / -192 / -256 = that pair-tile N. */
int sb_gemm_bf16(const void* A, long long lda, const void* W, long long ldw, void* out, long long ldo, int M, int N,
                 int K, const float* bias, int act, const void* residual, long long ldr, int res_mod, int flags,
                 float alpha, int force_bn, void* stream);
/* Diagnostic: device array of 8 u64 clock counters that every following sb_gemm_bf16 launch adds to (NULL = off):
 * producer / MMA / epilogue wait and work clocks summed over CTAs (see csrc/gemm_tcgen05.cu). */
int sb_gemm_set_prof(unsigned long long* counters);
/* out[M,N] = LayerNorm_N(A @ W^T + bias + residual) * gamma + beta in one kernel (N <= 256, N % 16 == 0): the
 * "keys = norm4(keys + cross_attn_image_to_token(...))" step of sam2/modeling/sam/transformer.py TwoWayAttentionBlock. */
int sb_gemm_ln(const void* A, long long lda, const void* W, long long ldw, void* out, long long ldo, int M, int N, int K,
               const float* bias, const void* residual, long long ldr, int res_mod, int flags, const float* gamma,
               const float* beta, float eps, void* stream);
/* mask_decoder.py output_upscaling[0..2]: ConvTranspose2d(256->64,k2,s2) + feat_s1 skip + LayerNorm2d + GELU, fused */
int sb_gemm_upscale1(const void* A, long long lda, const void* W, long long ldw, int B, int gh, int gw,
                     const float* bias, const float* feat_s1, long long skip_bstride, const float* gamma,
                     const float* beta, float eps, void* u1, const int* plist, const int* pcount, void* stream);
/* output_upscaling[3..4] + (hyper_in @ upscaled_embedding): ConvTranspose2d(64->32,k2,s2) + feat_s0 + GELU + dot with the
 * prompt's 4 hyper-network vectors -> masks [B,4,2gh,2gw] fp32, fused */
int sb_gemm_upscale2(const void* A, long long lda, const void* W, long long ldw, int B, int gh, int gw,
                     const float* bias, const float* feat_s0, long long skip_bstride, const float* hyper, float* masks,
                     const int* plist, const int* pcount, void* stream);
/* Both up-scaling stages take an optional device-side prompt list (plist [<= B] int32, *pcount entries; NULL = all B):
 * only the listed prompts are processed, the other prompts' rows of u1 / masks are left untouched. sb_iou_gate builds
 * the list of the AMG m2m pass: prompts with max(ious[b][0..3]) > thresh, the only ones that can survive
 * SAM2AutomaticMaskGenerator's pred_iou_thresh filter (sam2/automatic_mask_generator.py _process_batch), in ascending
 * order. */
int sb_iou_gate(const float* ious4, int B, float thresh, int* list, int* count, void* stream);
/* Plain batched multi-head attention (mask-decoder two-way transformer: sam2/modeling/sam/transformer.py
 * Attention.forward -> F.scaled_dot_product_attention). q [batch*nq, heads*hd], k/v [batch*nk, heads*hd]. */
int sb_attention(const void* q, long long q_ld, const void* k, long long k_ld, const void* v, long long v_ld, void* o,
                 long long o_ld, int batch, int heads, int hd, int nq, int nk, float scale, int q_shared,
                 int kv_shared, void* stream);
/* sb_attention with an additive key term shared by all batch entries (scores = q (k[b] + k_add)^T): the mask decoder's
 * token -> image attention, k_add = image_pe @ Wk^T + bk ([nk, heads*hd] bf16) */
int sb_attention_kadd(const void* q, long long q_ld, const void* k, long long k_ld, const void* k_add, long long k_add_ld,
                      const void* v, long long v_ld, void* o, long long o_ld, int batch, int heads, int hd, int nq,
                      int nk, float scale, int kv_shared, void* stream);
/* Mask-decoder image -> token attention (TwoWayAttentionBlock.cross_attn_image_to_token; 8 heads x 16, <= 16 keys per
 * prompt) as a stream over the query matrix; q_add [nq,128] fp32 (nullable) is the query projection's positional term
 * (image_pe @ Wq^T + bq), shared by all prompts, added before the scores. */
int sb_attention_few_keys(const void* q, long long q_ld, const float* q_add, const void* k, long long k_ld, const void* v,
                          long long v_ld, void* o, long long o_ld, int batch, int nq, int nk, float scale, int q_shared,
                          void* stream);
/* Fused TwoWayAttentionBlock step 4 (sam2/modeling/sam/transformer.py: `keys = norm4(keys + cross_attn_image_to_token(
 * q=keys+key_pe, k=queries+query_pe, v=queries))`) for prompts with <= 8 tokens. sb_i2t_fold folds the q / out
 * projections and the out-projection bias bo [256] fp32 into per-prompt operands (kts [B,8,128], w1t [B,64,256],
 * w2t [B,256,64], all bf16) from the projected token keys / values kt, vt [B*nt,128] bf16; sb_i2t_block_tc then makes
 * one pass over the image stream x [B*nq,256] bf16 (or [nq,256] when x_shared) on tcgen05 / TMEM / TMA (128-row tiles,
 * both GEMMs as UMMA, softmax + LayerNorm in the epilogue warps): scores, per-head softmax, out projection, residual,
 * LayerNorm. qres [nq,128] bf16 = image_pe Wq^T + bq is shared by all prompts. out [B*nq,256] bf16 may alias a
 * per-prompt x. */
int sb_i2t_fold(const void* kt, long long kt_ld, const void* vt, long long vt_ld, const void* wq, const void* wo,
                const float* bo, void* w1t, void* w2t, void* kts, int batch, int nt, float scale, void* stream);
int sb_i2t_block_tc(const void* x, int x_shared, const void* qres, const void* w1t, const void* w2t, const void* kts,
                    const float* gamma, const float* beta, float eps, void* out, int batch, int nq, int nt, void* stream);
/* Mask-decoder "tokens attend to image" (TwoWayAttentionBlock step 2, final_attn_token_to_image) for prompts with <= 8
 * tokens, computed straight on the image stream x [batch*nk (nk when x_shared), 256] bf16 without materialising K / V:
 * the k / v projections (wk, wv [128,256] bf16, bv [128] fp32; kadd [nk,128] bf16 = image_pe Wk^T + bk) fold onto the
 * token side. q [batch*nt,128] bf16 are the projected token queries; out [batch*nt,128] bf16 is the attention output
 * before out_proj. Runs on tcgen05 / TMEM / TMA (csrc/decoder_t2i_tc.cu): QK^T and PV as M = 64 UMMAs, the TMA-staged key
 * tile is the K-major B operand of QK^T and the MN-major B operand of PV. Caller-owned workspaces: qf [batch,64,384]
 * bf16, qs [batch,8,128] bf16, opart [batch,ns,64,256] fp32, ml [batch,ns,2,64] fp32 with ns = sb_t2i_tc_splits(batch, nk). */
int sb_t2i_tc_splits(int batch, int nk);
int sb_t2i_fold_attention_tc(const void* q, long long q_ld, const void* x, int x_shared, const void* kadd, const void* wk,
                             const void* wv, const float* bv, void* qf, void* qs, float* opart, float* ml, void* out,
                             long long out_ld, int batch, int nt, int nk, float scale, void* stream);
/* Hiera MultiScaleAttention over a fused qkv buffer [B*H*W, 3*heads*hd]: window partition (with upstream's zero
 * padding of ragged windows), optional 2x2 max-pool of q, SDPA, window unpartition — hieradet.py
 * MultiScaleBlock.forward / MultiScaleAttention.forward. ws >= max(H,W) = global attention. */
int sb_window_attention(const void* qkv, const float* qkv_bias, void* o, int batch, int H, int W, int heads, int hd,
                        int ws, int pool, float scale, void* stream);
/* The same op for hiera-L's head_dim 72 without q-pooling on tcgen05 / TMEM with TMA loads and a TMA tensor store
 * (16 x 16 windows and the global blocks of stage 3; sb_window_attention routes here by default). Returns -3
 * (unsupported) for other window shapes. */
int sb_hiera_attention_tc(const void* qkv, void* out, int batch, int H, int W, int heads, int ws, float scale,
                          void* stream);
/* Instrumented build (tools/attn_probe.py): prof [num_sms][16] int64 per-CTA clock sums per pipeline role. */
int sb_hiera_attention_tc_prof(const void* qkv, void* out, int batch, int H, int W, int heads, int ws, float scale,
                               long long* prof, void* stream);

/* ---- token-major bandwidth kernels of the encoder / decoder ----------------------------------------- */
int sb_layernorm(const void* in, long long ld_in, int in_f32, void* out, long long ld_out, int out_f32,
                 const float* gamma, const float* beta, int M, int C, float eps, int act, void* stream);
int sb_im2col_k7s4(const float* img, void* cols, int B, int Cin, int S, int Kp, void* stream); /* PatchEmbed 7x7 s4 p3 */

/* ---- fp32 validation mode (SB_VALIDATE_FP32; BASELINE north_star "1e-4 in the fp32 validation mode") -------------- */
/* x (fp32) split into three bf16 parts, K-concatenated into the operand of a 6-term split product: a GEMM of the role-0
 * (activation: [h h h m m l]) and role-1 (weight: [h m l h m h]) outputs with K' = 6K on sb_gemm_bf16 reproduces the
 * fp32 product to ~2^-24: the production tcgen05 kernel is the one validated. out [M, 6K] bf16, pitch ldo. */
int sb_split3_bf16(const float* x, long long ldx, int M, int K, int role, void* out, long long ldo, void* stream);
/* fp32 twin of sb_window_attention (hieradet.py MultiScaleAttention in torch fp32): CUDA cores, one block per query. */
int sb_window_attention_f32(const float* qkv, const float* qkv_bias, float* o, int batch, int H, int W, int heads,
                            int hd, int ws, int pool, float scale, void* stream);
int sb_im2col_k7s4_f32(const float* img, float* cols, int B, int Cin, int S, int Kp, void* stream);
/* fp32 twin of sb_attention / sb_attention_kadd (k_add may be NULL) */
int sb_attention_f32(const float* q, long long q_ld, const float* k, long long k_ld, const float* k_add, long long ka_ld,
                     const float* v, long long v_ld, float* o, long long o_ld, int batch, int heads, int hd, int nq,
                     int nk, float scale, int q_shared, int kv_shared, void* stream);
int sb_rope_apply_f32(const float* x, long long ld_in, float* out, long long ld_out, long long rows, int C,
                      int rows_per_batch, int n_rope, int ntok, const float* cos_sin, void* stream);
int sb_gelu_exact_f32(float* x, long long n, void* stream); /* erff GELU in place (the fused epilogue form is 4e-4) */
int sb_maxpool2x2(const void* in, void* out, int is_f32, int B, int H, int W, int C, void* stream); /* hieradet do_pool */
int sb_add_upsample2x(float* dst, const float* src, int B, int H, int W, int C, void* stream);   /* FpnNeck top-down */
int sb_nhwc_to_nchw(const void* in, int in_f32, void* out, int out_f32, int B, int HW, int C, const float* chan_add,
                    void* stream);
int sb_nchw_to_nhwc(const void* in, int in_f32, void* out, int out_f32, int B, int HW, int C, void* stream);
int sb_add_cast(const void* a, int a_f32, const float* b, long long b_mod, void* out, int out_f32, long long n,
                void* stream);

/* ---- prompt encoder / mask decoder glue (sam2/modeling/sam/prompt_encoder.py, mask_decoder.py) ------- */
int sb_prompt_tokens(const float* coords, const int* labels, int B, int Np, int pad, const float* gauss,
                     const float* point_emb, const float* not_a_point, const float* out_tokens, int image_size,
                     float* tokens, void* stream);
/* mask_downscaling[0..5] fused. cpp == 3: `in` is a decoder output [B/3,4,S,S] whose tokens 1..3 are the B mask
 * prompts (AMG m2m refinement); clampv > 0 clamps to +-clampv (upstream clamps low-res logits to +-32). */
int sb_mask_downscale(const float* in, int B, int S, int cpp, float clampv, const float* w1, const float* b1,
                      const float* g1, const float* be1, const float* w2, const float* b2, const float* g2,
                      const float* be2, void* out, void* stream);
/* mask_downscaling[6] (1x1 conv 16->256) + `src = image_embeddings + dense_prompt_embeddings` of the mask decoder:
 * keys[b*T+t] = bf16(image_embed[t] + bias + ds[b*T+t] @ w^T); ds [ntok,16] bf16, w [256,16] fp32, image_embed [T,256] */
int sb_mask_embed_keys(const void* ds, const float* w, const float* bias, const float* image_embed, int T, long long ntok,
                       void* keys, void* stream);
int sb_upscale1_post(const void* g1, const float* feat_s1, long long s1_batch_stride, const float* gamma,
                     const float* beta, int B, int h, int w, void* u1, void* stream);
int sb_upscale2_mask(const void* g2, const float* feat_s0, long long s0_batch_stride, const float* hyper, int B,
                     int H1, int W1, float* masks, void* stream);
/* MaskDecoder._dynamic_multimask_via_stability (delta 0.05, thresh 0.98 set by build_sam2(apply_postprocessing)) */
int sb_select_mask(const float* masks, const float* ious, int B, int HW, float delta, float thresh, int* sel_idx,
                   float* sel_iou, void* stream);

/* ---- automatic-mask-generation post-processing: integer / indexing, bit-exact ------------------------ */
/* For n candidates (planes [*,4,S,S], ious4 [*,4]; candidate i = prompt i/cpp, token sel[i] or 1 + i%3 or 0):
 * bilinear up-sampling to the crop (SAM2Transforms.postprocess_masks), pred-IoU filter, stability score
 * (sam2/utils/amg.py calculate_stability_score), threshold, box (batched_mask_to_box), near-crop-edge filter
 * (is_box_near_crop_edge), uncrop + bit-pack into the full frame. Outputs are written at index i. geom_dev (optional,
 * device int[5] = {Hc, Wc, x0, y0, base}) overrides the crop geometry and offsets the outputs by `base` entries, so a
 * captured CUDA graph can be replayed for every crop / prompt batch. */
int sb_amg_mask_post(const float* planes, const float* ious4, const int* sel, int cpp, int n, int S, int Hc, int Wc,
                     int x0, int y0, int H, int W, float pred_iou_thresh, float mask_thresh, float stab_offset,
                     float stab_thresh, unsigned char* keep, float* stability, float* iou_out, int* bbox, int* area,
                     void* bits, const int* geom_dev, void* stream);
int sb_compact_keep(const unsigned char* keep, int base, int n, int* cand, int* count, void* stream);
/* torchvision.ops.nms semantics (upstream batched_nms per crop and across crops); list lengths are device ints. */
int sb_nms_dev(const int* bbox, const float* scores, const int* cand, const int* n_ptr, int n_cap, float iou_thresh,
               int* order, void* mask_ws, int* out_list, int* out_count, void* stream);
/* pairwise |mask_i & mask_j| for REF saber/segmenters/utils.py:5-86 remove_duplicate_masks */
int sb_pair_intersections(const void* bits, const int* bbox, const int* area, int m, int H, int W,
                          double area_ratio_thresh, int* inter, void* stream);
int sb_unpack_bits(const void* bits, const int* sel, int m, int H, int W, unsigned char* out, void* stream);
int sb_gather_rows(const void* src, const int* sel, int m, long long row_words, void* dst, void* stream);
/* REF saber/segmenters/propagation.py:181-186: masks3d[mask] = idx + 1 in list order (later masks win) */
int sb_stitch_labels(const void* bits, const int* order, int m, int H, int W, void* labels, void* stream);
/* REF saber/segmenters/utils.py:88-131 separate_masks: 26-connected components (scipy.ndimage.label numbering),
 * components < min_vol voxels dropped, compact relabel. labels: uint32 [Z,Y,X]; aux: Z*Y*X int32 workspace;
 * chunk_ws: ceil(Z*Y*X/2048)+1 int32 workspace whose last element receives the component count. */
int sb_ccl3d_26(const void* vol, int elem_bytes, int Z, int Y, int X, int min_vol, void* labels, int* aux,
                int* chunk_ws, void* stream);
/* The same with the connectivity as an argument (6 = scipy.ndimage.label's default structure, 26) and, optionally, the
 * voxel count of every surviving component (sizes_out[id - 1]): the connected-component steps of the membrane-refinement
 * workflow (REF saber/analysis/refine_membranes.py:136-249). */
int sb_ccl3d(const void* vol, int elem_bytes, int Z, int Y, int X, int min_vol, int conn, void* labels, int* aux,
             int* chunk_ws, int* sizes_out, void* stream);

/* ---- image-side bandwidth kernels -------------------------------------------------------------------- */
/* scipy.ndimage.uniform_filter1d(mode='reflect') along one axis — REF saber/utils/preprocessing.py:13-14 */
int sb_box_filter(const float* in, float* out, int H, int W, int axis, int size, int square, void* stream);
/* REF saber/utils/preprocessing.py:15-18,36 contrast + clip + min-max; partials: 2048-float workspace */
int sb_contrast_normalize(const float* img, const float* mean, const float* sq, float* out, long long n,
                          float cutoff, float* partials, void* stream);
/* (H,W,3) inputs of prepare(): the reference's uniform_filter also runs along the channel axis (REF saber/utils/
 * preprocessing.py:12-13 on a 3-D array) = a constant 3x3 mix; img [npix,3] -> out [3,npix] (of img or img^2), and back. */
int sb_rgb_mix_planar(const float* img, const float* mix, int square, long long npix, float* out, void* stream);
int sb_planar_to_hwc3(const float* planar, long long npix, float* out, void* stream);
/* SAM2Transforms: crop -> Resize(S, bilinear, antialias) -> Normalize(mean, std). mean3/std3 are [host]. */
int sb_resize_normalize(const float* img, int H, int W, int C, const int* crops, int ncrops, int S,
                        const float* mean3, const float* std3, float* out, void* stream);
/* F.interpolate(bilinear, align_corners=False): SAM2Transforms.postprocess_masks / video-resolution logits */
int sb_upsample_bilinear(const float* in, int N, int Hi, int Wi, int Ho, int Wo, float* out, void* stream);

/* ---- z-axis propagation: memory attention / memory encoder / tracking glue (upstream sam2_video_predictor.py, ----
 * modeling/{memory_attention,memory_encoder,sam2_base}.py, reached from REF saber/adapters/sam2/predictor.py:164-202) */
/* axial RoPE (position_encoding.py apply_rotary_enc): rows r < n_rope of each batch entry are rotated with the
 * frequencies of token r % ntok (rope_k_repeat), the rest (object-pointer tokens) are copied. cos_sin: [ntok, C/2, 2]. */
int sb_rope_apply(const void* x, long long ld_in, int in_f32, void* out, long long ld_out, long long rows, int C,
                  int rows_per_batch, int n_rope, int ntok, const float* cos_sin, void* stream);
/* MaskDownSampler stage: Conv2d(k3,s2,p1) + LayerNorm2d + GELU on NHWC; stage 0: 1->4 (fp32 in; in_xf 1 = sigmoid(v)*
 * xf_scale+xf_bias, 2 = (v>0)*xf_scale+xf_bias: SAM2Base._encode_new_memory), 1: 4->16, 2: 16->64 (bf16 in). bf16 out. */
int sb_conv3x3s2_ln_gelu(const void* in, int stage, int B, int Hi, int Wi, const float* w, const float* bias,
                         const float* gamma, const float* beta, float eps, int in_xf, float xf_scale, float xf_bias,
                         void* out, void* stream);
int sb_im2col_3x3s2(const void* in, int B, int Hi, int Wi, int C, void* cols, void* stream);
/* CXBlock: depth-wise Conv2d(256,k7,p3) + LayerNorm on NHWC fp32 -> bf16 */
int sb_dwconv7_ln(const float* in, int B, int H, int W, int C, const float* w, const float* bias, const float* gamma,
                  const float* beta, float eps, void* out, void* stream);
/* maskmem_features + (score <= 0) * no_obj_embed_spatial, stored as bf16 (sam2_video_predictor.py) */
int sb_add_vec_cond(const float* x, const float* score, const float* vec, int B, long long rows_per_batch, int C,
                    void* out, void* stream);
/* SAM2Base._forward_sam_heads: best-IoU multimask choice (or `sel`), object-score gate (-1024), output token */
int sb_track_select(const float* masks, const float* ious, const float* obj, const float* hs, const int* sel,
                    int multimask, int B, int Nt, int S, float* low_res, float* token, int* best, void* stream);
int sb_objptr_mix(float* ptr, const float* cond, const float* no_obj_ptr, int B, int C, void* stream);
/* sam2/utils/misc.py fill_holes_in_mask_scores (8-connected background components of area <= max_area -> +0.1).
 * ws: B*2*S*S int32 workspace */
int sb_fill_holes(const float* in, float* out, int B, int S, int max_area, int* ws, void* stream);
int sb_threshold_affine(const float* in, float thr, float scale, float bias, long long n, float* out, void* stream);
int sb_conv4x4s4(const float* in, int B, int S, const float* w, const float* bias, float* out, void* stream); /* SAM2Base.mask_downsample */
/* REF saber/adapters/sam2/predictor.py:289-297: per-frame label stitch (threshold > 0, skimage order-0 resize to (H,W),
 * later objects overwrite earlier ones). logits [N,Sv,Sv] fp32, ids int32 [N], labels uint16 [H,W] updated in place. */
int sb_stitch_objects(const float* logits, const int* ids, int N, int Sv, int H, int W, void* labels, void* stream);
int sb_slice_any(const void* vol, int Z, long long n, unsigned char* any, void* stream);     /* REF :321 `.any()` */
int sb_erase_label(void* labels, long long n, int id, void* stream);                          /* REF :345-346 */

/* ---- whole-tomogram bandwidth kernels of the 3-D path (REF saber/adapters/preprocessing.py, saber/filters/gaussian.py) */
int sb_minmax(const float* in, long long n, float* mm, float* partials, void* stream);  /* mm[0]=min, mm[1]=max (device) */
/* out = ((in - mm[0]) / ((mm[1] - mm[0]) + eps)) * a + b: normalize_tomogram (REF adapters/preprocessing.py:72-76: eps 0,
 * a 2, b -1) and preprocessing.normalize (REF utils/preprocessing.py:20-37: eps 1e-8, a 1, b 0) */
int sb_minmax_affine(const float* in, long long n, const float* mm, float eps, float a, float b, float* out, void* stream);
/* skimage.transform.resize(order=1, mode='reflect') of each z-slice = scipy zoom(grid_mode, mirror), then a*v+b
 * (REF adapters/preprocessing.py:21,59) */
int sb_zoom_linear_mirror(const float* in, int Z, int Hi, int Wi, int Ho, int Wo, float a, float b, float* out,
                          void* stream);
/* the anti-aliasing Gaussian skimage applies before down-sampling (scipy gaussian_filter, mode='mirror'); axis 1=y, 2=x */
int sb_gauss1d_mirror(const float* in, int Z, int H, int W, int axis, const double* weights, int r, float* out,
                      void* stream);
int sb_gaussian_z(const float* in, int Z, long long plane, const float* w, int ks, float* out, void* stream); /* REF filters/gaussian.py:17-74 */
int sb_mean_z(const float* in, long long plane, int z0, int z1, float* out, void* stream); /* REF utils/preprocessing.py:39-66 */

/* ---- expert classifier (REF saber/classifier/models/{predictor,SAM2}.py, classifier/datasets/RandMaskCrop.py) ------- */
int sb_mean_std(const float* in, long long n, float* ms, double* ws, void* stream);   /* monai NormalizeIntensity stats */
int sb_standardize(const float* in, long long n, const float* ms, float* out, void* stream);
int sb_mask_bbox(const unsigned char* masks, int N, int H, int W, int* bbox, void* stream); /* (ymin,ymax,xmin,xmax) | -1 */
/* crop_and_resize_adaptive: crop geom[n] = (top,left,h,w) -> bilinear (image) / nearest (mask) resize to SxS + mask area */
int sb_crop_resize(const float* img, const unsigned char* masks, const int* geom, int N, int H, int W, int S,
                   float* out_img, unsigned char* out_mask, int* area, void* stream);
/* SAM2Classifier.apply_mask_to_features: [feat*m | feat*(1-m)] with m nearest-resized to the GxG embedding grid */
int sb_mask_features(const float* feat, const unsigned char* mask, int B, int G, int S, int C, void* out, void* stream);
int sb_prelu(const void* in, int in_f32, long long n, float slope, void* out, void* stream);
int sb_im2col_3x3s1(const void* in, int B, int H, int W, int C, void* cols, void* stream);
int sb_mean_tokens(const void* in, int B, int T, int C, float* out, void* stream);     /* adaptive_avg_pool2d(1,1) */
int sb_softmax_rows(const float* in, int B, int C, float* out, void* stream);

/* ---- label-volume filters next to the path: fast_3d_gaussian_smoothing (REF saber/filters/masks.py:230-309, -------
 * gaussian.py:76-138) and ball morphology (REF saber/analysis/refine_membranes.py:100-117,274-333) */
int sb_label_equals(const void* vol, int elem_bytes, long long n, unsigned int label, float* out,
                    unsigned long long* count, void* stream);
int sb_corr1d_zero(const float* in, int Z, int Y, int X, int axis, const float* w, int ks, float* out, void* stream);
int sb_threshold_label(const float* sm, long long n, float thr, int label, unsigned char* result, void* stream);
int sb_morph_ball(const unsigned char* in, int Z, int Y, int X, int r, int op, unsigned char* out, void* stream);
/* the same with the full (2r+1)^3 cube (scipy binary_erosion(structure=ones((3,3,3))), REF refine_membranes.py:172) */
int sb_morph_cube(const unsigned char* in, int Z, int Y, int X, int r, int op, unsigned char* out, void* stream);

/* ---- Fourier-space rescale and band-pass (SURVEY 8f row 2) -------------------------------------------------------------
 * REF saber/filters/downsample.py:67-129,153-204 (FourierRescale3D / 2D) and saber/filters/tomograms.py:67-184 (Filter3D).
 * A 3-D transform is three sb_fft_lines passes (x rows, y columns, z columns); see csrc/fft.cu. */
int sb_fft_twiddles(int n, void* tw, void* stream);
int sb_fft_lines(const void* in, void* out, const void* tw, int n, int m, int rows_mode, long long lines, int batch,
                 int in_real, int out_mode, int inverse, float scale, int crop, int start, const float* bandpass, int D,
                 int H, int W, void* stream);
int sb_bandpass_volume(int D, int H, int W, const float* bandpass, float* out, void* stream);

/* ---- organelle / membrane refinement workflow (SURVEY 8f row 3; REF saber/analysis/refine_membranes.py:120-548) ------
 * dtype codes of label / mask volumes: 0 uint8, 1 int16, 2 uint16, 3 int32, 4 int64, 5 float32. */
/* _trim_edges + (> 0): REF :120-135,142 (incl. the empty-slice quirks of `[t:-t]` for t == 0 and t >= size // 2) */
int sb_trim_binarize(const void* vol, int dtype, int Z, int Y, int X, int zt, int xyt, unsigned char* out, void* stream);
/* present[z] = any(vol[z]): REF :466 */
int sb_z_any(const unsigned char* vol, int Z, long long plane, unsigned char* present, void* stream);
/* table[(cap + 1) x 8] = {min z,y,x, max z,y,x, count, -} per label on slices with present[z] (nullable); table[7] != 0
 * when a label exceeds cap. One pass instead of REF :251-272,470,489-495 (clone + nonzero per organelle, torch.unique). */
int sb_label_bbox(const void* vol, int dtype, int Z, int Y, int X, const unsigned char* present, int cap, int* table,
                  void* stream);
/* out[roi] = vol == label (label < 0: vol != 0), zero on slices without present[z] (nullable): REF :363-364 */
int sb_roi_binarize(const void* vol, int dtype, int Z, int Y, int X, int z0, int y0, int x0, int dz, int dy, int dx,
                    long long label, const unsigned char* present, unsigned char* out, void* stream);
/* vol[roi][mask] = value: REF :431-438 and convert_to_3d_labels :548-573 */
int sb_roi_paste(void* vol, int dtype, int Z, int Y, int X, int z0, int y0, int x0, int dz, int dy, int dx,
                 const unsigned char* mask, long long value, void* stream);
/* dst[src > 0] = src[src > 0]: one step of convert_to_3d_labels, REF :548-573 */
int sb_overlay_nonzero(void* dst, const void* src, int dtype, long long n, void* stream);
/* op 0: a & b, 1: a | b, 2: a & ~b on {0,1} bytes */
int sb_mask_logic(const unsigned char* a, const unsigned char* b, long long n, int op, unsigned char* out, void* stream);
/* mode 0: labels > 0 (REF :202-222); mode 1: the largest component, first among equals (REF :224-249) */
int sb_label_select(const int* labels, long long n, const int* sizes, const int* count, int mode, int* which,
                    unsigned char* out, void* stream);
/* components whose overlap with mask exceeds ratio x size: REF :160-199 */
int sb_label_keep_ratio(const int* labels, const unsigned char* mask, long long n, const int* sizes, int* overlap,
                        int capacity, double ratio, unsigned char* out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SABER_B200_H */
