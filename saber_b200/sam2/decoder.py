"""B200 executor of the SAM2 prompt encoder + mask decoder (two-way transformer, transposed-conv
up-scaling with high-res skips, hyper-network mask heads, IoU and object-score heads).

Token-major layout throughout: decoder tokens ``[B*Nt, 256]`` (fp32 residual stream), image stream
``[B*4096, 256]``. Constant terms are folded at load time: the image positional encoding is pushed
through the K/Q projections once (``pe @ W^T + b`` becomes the GEMM's broadcast residual), and the
first AMG pass — where the dense prompt is the same ``no_mask_embed`` for every point — computes
the layer-0 image-side projections once per image and shares them across the prompt batch
(results equal upstream up to fp reassociation; SURVEY §7 "algorithmic redundancy").
Restates sam2/modeling/sam/{prompt_encoder,mask_decoder,transformer}.py (SURVEY §8a U2/U3).
"""
from __future__ import annotations

import math
from typing import Dict, Optional, Tuple

import torch

from .. import ops
from . import arch

_BF16, _F32 = torch.bfloat16, torch.float32
NT_IMG = 4096  # 64 x 64 image tokens


def _dense_pe(gauss: torch.Tensor, size: int = 64) -> torch.Tensor:
    """PositionEmbeddingRandom.forward((64,64)) -> [4096, 256] fp32 (weights-only constant)."""
    g = gauss.float()
    grid = torch.ones((size, size), dtype=torch.float32)
    y = (grid.cumsum(0) - 0.5) / size
    x = (grid.cumsum(1) - 0.5) / size
    coords = 2 * torch.stack([x, y], dim=-1) - 1
    proj = 2 * math.pi * (coords @ g)
    return torch.cat([proj.sin(), proj.cos()], dim=-1).reshape(size * size, -1)


class MaskDecoder:
    def __init__(self, sd: Dict[str, torch.Tensor], device, dynamic_multimask_via_stability: bool = True):
        dev = self.device = torch.device(device)
        md, pe = "sam_mask_decoder.", "sam_prompt_encoder."
        self.dynamic_multimask_via_stability = dynamic_multimask_via_stability
        self.stab_delta, self.stab_thresh = 0.05, 0.98

        def w16(t):  # bf16 GEMM operand (fp32 in the validation mode)
            return ops.weight(t, dev)

        def f32(t):
            return t.to(dev, _F32).contiguous()

        self.out_tokens = f32(torch.cat([sd[md + "obj_score_token.weight"], sd[md + "iou_token.weight"],
                                         sd[md + "mask_tokens.weight"]], dim=0))
        gauss = sd[pe + "pe_layer.positional_encoding_gaussian_matrix"]
        self.gauss = f32(gauss)
        self.point_emb = f32(torch.cat([sd[pe + f"point_embeddings.{i}.weight"] for i in range(4)], dim=0))
        self.not_a_point = f32(sd[pe + "not_a_point_embed.weight"].reshape(-1))
        self.no_mask_embed = f32(sd[pe + "no_mask_embed.weight"].reshape(-1))
        self.md_w = [f32(sd[pe + "mask_downscaling.0.weight"].reshape(-1)), f32(sd[pe + "mask_downscaling.0.bias"]),
                     f32(sd[pe + "mask_downscaling.1.weight"]), f32(sd[pe + "mask_downscaling.1.bias"]),
                     f32(sd[pe + "mask_downscaling.3.weight"].reshape(-1)), f32(sd[pe + "mask_downscaling.3.bias"]),
                     f32(sd[pe + "mask_downscaling.4.weight"]), f32(sd[pe + "mask_downscaling.4.bias"])]
        self.md6_w = f32(sd[pe + "mask_downscaling.6.weight"].reshape(256, 16))
        self.md6_b = f32(sd[pe + "mask_downscaling.6.bias"])
        image_pe = _dense_pe(gauss)  # [4096, 256] fp32 on CPU
        self.image_pe = f32(image_pe)

        def attn_w(prefix):
            # keys: qw/qb/kw/kb/vw/vb/outw/outb
            return {f"{k}{p[0]}": sd[f"{prefix}.{k}_proj.{p}"].float()
                    for k in ("q", "k", "v", "out") for p in ("weight", "bias")}

        self.layers = []
        for l in range(2):
            b = f"{md}transformer.layers.{l}."
            sa, t2i, i2t = attn_w(b + "self_attn"), attn_w(b + "cross_attn_token_to_image"), attn_w(b + "cross_attn_image_to_token")
            L = {}
            if l == 0:
                L["sa_qkv_w"] = w16(torch.cat([sa["qw"], sa["kw"], sa["vw"]], 0))
                L["sa_qkv_b"] = f32(torch.cat([sa["qb"], sa["kb"], sa["vb"]], 0))
            else:
                L["sa_qk_w"] = w16(torch.cat([sa["qw"], sa["kw"]], 0))
                L["sa_qk_b"] = f32(torch.cat([sa["qb"], sa["kb"]], 0))
                L["sa_v_w"], L["sa_v_b"] = w16(sa["vw"]), f32(sa["vb"])
            L["sa_o_w"], L["sa_o_b"] = w16(sa["outw"]), f32(sa["outb"])
            L["t2i_q_w"], L["t2i_q_b"] = w16(t2i["qw"]), f32(t2i["qb"])
            L["t2i_kv_w"] = w16(torch.cat([t2i["kw"], t2i["vw"]], 0))
            # k = (keys + pe) Wk^T + bk: the pe term (weights only) is added inside the attention kernel as a second MMA
            # (scores = q k^T + q k_add^T), so the big K|V GEMM carries a plain bias and no broadcast residual
            L["t2i_kv_b"] = f32(torch.cat([torch.zeros(128), t2i["vb"]]))
            L["t2i_v_b"] = f32(t2i["vb"])
            L["t2i_k_add"] = w16(image_pe @ t2i["kw"].t() + t2i["kb"])  # [4096, 128]
            L["t2i_o_w"], L["t2i_o_b"] = w16(t2i["outw"]), f32(t2i["outb"])
            L["i2t_q_w"] = w16(i2t["qw"])
            L["i2t_q_res"] = f32(image_pe @ i2t["qw"].t() + i2t["qb"])  # [4096, 128]
            L["i2t_q_res16"] = w16(image_pe @ i2t["qw"].t() + i2t["qb"])
            L["i2t_k_w"], L["i2t_k_b"] = w16(i2t["kw"]), f32(i2t["kb"])
            L["i2t_v_w"], L["i2t_v_b"] = w16(i2t["vw"]), f32(i2t["vb"])
            L["i2t_o_w"], L["i2t_o_b"] = w16(i2t["outw"]), f32(i2t["outb"])
            L["mlp1_w"], L["mlp1_b"] = w16(sd[b + "mlp.layers.0.weight"]), f32(sd[b + "mlp.layers.0.bias"])
            L["mlp2_w"], L["mlp2_b"] = w16(sd[b + "mlp.layers.1.weight"]), f32(sd[b + "mlp.layers.1.bias"])
            for k in (1, 2, 3, 4):
                L[f"n{k}w"], L[f"n{k}b"] = f32(sd[b + f"norm{k}.weight"]), f32(sd[b + f"norm{k}.bias"])
            self.layers.append(L)
        fa = attn_w(md + "transformer.final_attn_token_to_image")
        self.fa_q_w, self.fa_q_b = w16(fa["qw"]), f32(fa["qb"])
        self.fa_kv_w = w16(torch.cat([fa["kw"], fa["vw"]], 0))
        self.fa_kv_b = f32(torch.cat([torch.zeros(128), fa["vb"]]))
        self.fa_v_b = f32(fa["vb"])
        self.fa_k_add = w16(image_pe @ fa["kw"].t() + fa["kb"])
        self.fa_o_w, self.fa_o_b = w16(fa["outw"]), f32(fa["outb"])
        self.nf_w, self.nf_b = f32(sd[md + "transformer.norm_final_attn.weight"]), f32(sd[md + "transformer.norm_final_attn.bias"])
        # transposed convs as GEMMs: out column = (dy*2+dx)*Cout + co
        w1 = sd[md + "output_upscaling.0.weight"].float()  # [ci=256, co=64, 2, 2]
        self.up1_w = w16(w1.permute(2, 3, 1, 0).reshape(256, 256))
        self.up1_b = f32(sd[md + "output_upscaling.0.bias"].float().repeat(4))
        self.up_ln_w, self.up_ln_b = f32(sd[md + "output_upscaling.1.weight"]), f32(sd[md + "output_upscaling.1.bias"])
        w2 = sd[md + "output_upscaling.3.weight"].float()  # [ci=64, co=32, 2, 2]
        self.up2_w = w16(w2.permute(2, 3, 1, 0).reshape(128, 64))
        self.up2_b = f32(sd[md + "output_upscaling.3.bias"].float().repeat(4))

        def mlp3(prefix):
            return [(w16(sd[f"{prefix}.layers.{k}.weight"]), f32(sd[f"{prefix}.layers.{k}.bias"])) for k in range(3)]

        self.hyper = [mlp3(md + f"output_hypernetworks_mlps.{i}") for i in range(4)]
        self.iou_head = mlp3(md + "iou_prediction_head")
        self.obj_head = mlp3(md + "pred_obj_score_head")

    # ------------------------------------------------------------------
    def prompt_tokens(self, coords: torch.Tensor, labels: torch.Tensor, pad: bool = True) -> torch.Tensor:
        """coords [B, Np, 2] fp32 in model-input pixels, labels [B, Np] int32 -> tokens [B, Nt, 256] fp32."""
        return ops.prompt_tokens(coords, labels, self.gauss, self.point_emb, self.not_a_point, self.out_tokens,
                                 arch.IMAGE_SIZE, pad)

    def _mlp3(self, a: torch.Tensor, head, last_act=ops.ACT_NONE, out: Optional[torch.Tensor] = None):
        h = ops.gemm(a, head[0][0], head[0][1], act=ops.ACT_RELU)
        h = ops.gemm(h, head[1][0], head[1][1], act=ops.ACT_RELU)
        return ops.gemm(h, head[2][0], head[2][1], act=last_act, out_dtype=_F32, out=out)

    def _upscale_validate(self, keys, s0, s1, hyper, B, kb):
        """fp32 validation route of output_upscaling + the hyper-network product, unfused: transposed convolutions as
        split-product GEMMs (column = (dy, dx, channel)), pixel shuffle by tensor views (data movement only), skip adds,
        LayerNorm2d and exact GELU through the stand-alone kernels, one small GEMM per prompt for the mask logits."""
        if kb == 1:
            keys = keys.repeat(B, 1)
        g1 = ops.gemm(keys, self.up1_w, self.up1_b, out_dtype=_F32)  # [B*4096, 4*64]
        u = g1.view(B, 64, 64, 2, 2, 64).permute(0, 1, 3, 2, 4, 5).reshape(B * 16384, 64).contiguous()
        u = ops.add_cast(u, s1.contiguous(), _F32)  # + feat_s1 (broadcast over the prompts)
        u = ops.layernorm(u, self.up_ln_w, self.up_ln_b, 1e-6, _F32)
        u = ops.gelu_exact_(u)
        g2 = ops.gemm(u, self.up2_w, self.up2_b, out_dtype=_F32)  # [B*16384, 4*32]
        z = g2.view(B, 128, 128, 2, 2, 32).permute(0, 1, 3, 2, 4, 5).reshape(B * 65536, 32).contiguous()
        z = ops.gelu_exact_(ops.add_cast(z, s0.contiguous(), _F32))
        masks = torch.empty((B, 4, 256, 256), dtype=_F32, device=self.device)
        for b in range(B):
            m = ops.gemm(z[b * 65536:(b + 1) * 65536], hyper[b].contiguous(), None, out_dtype=_F32)  # [65536, 4]
            masks[b] = m.t().reshape(4, 256, 256)
        return masks

    def forward(self, image_embed: torch.Tensor, s0: torch.Tensor, s1: torch.Tensor, tokens: torch.Tensor,
                mask_input: Optional[torch.Tensor] = None, multimask_output: bool = True,
                mask_clamp: float = 0.0, iou_gate: Optional[float] = None, zero_fill: bool = False):
        """image_embed [4096,256] fp32 (one image shared by the B prompts) or [B*4096,256] fp32 (one conditioned
        embedding per prompt: the video predictor's memory-attention output), s0 [65536,32] fp32, s1 [16384,64] fp32
        (one image, token-major);
        tokens [B, Nt, 256] fp32; mask_input [B, 256, 256] fp32, or a previous decoder output
        [B/3, 4, 256, 256] whose multimask tokens 1..3 are the B mask prompts (AMG m2m), or None;
        mask_clamp > 0 clamps the mask prompt to +-mask_clamp (upstream clamps low-res logits to +-32).

        iou_gate (AMG m2m pass): prompts whose four predicted IoUs are all <= iou_gate cannot pass the caller's
        ``iou > pred_iou_thresh`` filter whichever token the stability rule selects, so the up-scaling stages (a third
        of the pass) skip them; their ``masks`` entries are uninitialised (zero with ``zero_fill``).

        Returns dict: masks [B,4,256,256] fp32 (all four tokens), ious [B,4], obj [B,1], hs [B,Nt,256]
        and, per upstream's output selection, ``sel`` describing which tokens are "the output":
        multimask -> tokens 1..3; single -> token 0 or the dynamic-stability choice (sel_idx, sel_iou).
        """
        B, Nt, _ = tokens.shape
        val = ops.VALIDATE_FP32  # fp32 validation mode: the unfused route through GEMM + generic attention + LayerNorm
        if val and mask_input is not None:
            raise NotImplementedError("fp32 validation mode covers point / box prompts (the mask-prompt convolutions "
                                      "exist in bf16 only)")
        fuse8 = Nt <= 8 and not val
        query_pe = tokens.reshape(B * Nt, 256)
        queries = query_pe
        per_prompt = image_embed.shape[0] != NT_IMG
        assert image_embed.shape[0] == (B * NT_IMG if per_prompt else NT_IMG)
        shared = mask_input is None and not per_prompt
        if mask_input is None:
            keys_f32 = ops.add_cast(image_embed, self.no_mask_embed, _F32)  # [4096,256] or [B*4096,256]
            keys = ops.add_cast(keys_f32, None, _BF16)
        else:
            assert not per_prompt, "mask prompts with per-prompt image embeddings are not on the path"
            ds = ops.mask_downscale(mask_input.contiguous(), self.md_w, mask_clamp)  # [B*4096,16]
            assert ds.shape[0] == B * NT_IMG, (ds.shape, B)
            # per-prompt image stream (image_embed + dense mask embedding) kept in bf16: it is re-normalised by
            # norm4 right after the first block, and an fp32 copy would be 805 MB per 192 prompts
            keys = ops.mask_embed_keys(ds, self.md6_w, self.md6_b, image_embed)
            keys_f32 = keys
        kb = 1 if shared else B  # batch entries of the image stream

        for l, L in enumerate(self.layers):
            # ---- token self-attention
            if l == 0:
                qkv = ops.gemm(ops.add_cast(queries, None, _BF16), L["sa_qkv_w"], L["sa_qkv_b"])
                a = ops.attention(qkv[:, 0:256], qkv[:, 256:512], qkv[:, 512:768], B, 8, Nt, Nt)
                queries = ops.gemm(a, L["sa_o_w"], L["sa_o_b"], out_dtype=_F32)
            else:
                qk = ops.gemm(ops.add_cast(queries, query_pe, _BF16), L["sa_qk_w"], L["sa_qk_b"])
                v = ops.gemm(ops.add_cast(queries, None, _BF16), L["sa_v_w"], L["sa_v_b"])
                a = ops.attention(qk[:, 0:256], qk[:, 256:512], v, B, 8, Nt, Nt)
                queries = ops.gemm(a, L["sa_o_w"], L["sa_o_b"], residual=queries, out_dtype=_F32)
            queries = ops.layernorm(queries, L["n1w"], L["n1b"], 1e-5, _F32)
            # ---- tokens attend to image
            q = ops.gemm(ops.add_cast(queries, query_pe, _BF16), L["t2i_q_w"], L["t2i_q_b"])
            if fuse8:  # k / v projections folded onto the tokens: the image stream is read once, K|V never exist
                a = ops.t2i_fold_attention(q, keys, L["t2i_k_add"], L["t2i_kv_w"][0:128], L["t2i_kv_w"][128:256],
                                           L["t2i_v_b"], B, Nt, NT_IMG, x_shared=(kb == 1))
            else:
                kv = ops.gemm(keys, L["t2i_kv_w"], L["t2i_kv_b"])
                a = ops.attention_kadd(q, kv[:, 0:128], L["t2i_k_add"], kv[:, 128:256], B, 8, Nt, NT_IMG,
                                       kv_shared=(kb == 1))
            queries = ops.gemm(a, L["t2i_o_w"], L["t2i_o_b"], residual=queries, out_dtype=_F32)
            queries = ops.layernorm(queries, L["n2w"], L["n2b"], 1e-5, _F32)
            # ---- token MLP
            hdn = ops.gemm(ops.add_cast(queries, None, _BF16), L["mlp1_w"], L["mlp1_b"], act=ops.ACT_RELU)
            queries = ops.gemm(hdn, L["mlp2_w"], L["mlp2_b"], residual=queries, out_dtype=_F32)
            queries = ops.layernorm(queries, L["n3w"], L["n3b"], 1e-5, _F32)
            # ---- image attends to tokens
            kt = ops.gemm(ops.add_cast(queries, query_pe, _BF16), L["i2t_k_w"], L["i2t_k_b"])
            vt = ops.gemm(ops.add_cast(queries, None, _BF16), L["i2t_v_w"], L["i2t_v_b"])
            # q = keys @ Wq^T; its positional term (image_pe @ Wq^T + bq) is added inside the attention kernel, so the
            # big GEMM has no residual stream to gather
            if fuse8:
                # <= 8 tokens per prompt: q projection, attention, out projection, residual and norm4 in ONE pass over
                # the image stream, with the projections folded into per-prompt operands (csrc/decoder_fused.cu) and
                # both GEMMs on tcgen05 (csrc/decoder_i2t_tc.cu). A stream shared by all prompts (layer 0 of the first
                # pass) is read through the same tensor map by every prompt; a per-prompt stream is private to this
                # call (built above from the image embedding) and is updated in place.
                w1t, w2t, kts = ops.i2t_fold(kt, vt, L["i2t_q_w"], L["i2t_o_w"], B, Nt, bo=L["i2t_o_b"])
                keys = ops.i2t_block_tc(keys, L["i2t_q_res16"], w1t, w2t, kts, L["n4w"], L["n4b"], 1e-5, B, NT_IMG, Nt,
                                        out=(None if kb == 1 else keys), x_shared=(kb == 1))
                keys_f32, kb = keys, B
                continue
            if Nt <= 16 and not val:
                qi = ops.gemm(keys, L["i2t_q_w"], None)
                a = ops.attention_few_keys(qi, L["i2t_q_res"], kt, vt, B, NT_IMG, Nt, q_shared=(kb == 1))  # [B*4096,128]
            else:  # many prompt points per object: generic flash kernel
                qi = ops.gemm(keys, L["i2t_q_w"], None, residual=L["i2t_q_res"], res_mod=NT_IMG)
                a = ops.attention(qi, kt, vt, B, 8, NT_IMG, Nt, q_shared=(kb == 1))
            # keys = norm4(keys + out_proj(attn)) fused in the GEMM epilogue (no fp32 round trip of the image stream)
            keys = ops.gemm_ln(a, L["i2t_o_w"], L["i2t_o_b"], keys_f32, L["n4w"], L["n4b"], 1e-5,
                               res_mod=(NT_IMG if kb == 1 else 0))
            keys_f32 = keys  # bf16 residual from here on (immediately re-normalised)
            kb = B
        # ---- final token -> image attention
        q = ops.gemm(ops.add_cast(queries, query_pe, _BF16), self.fa_q_w, self.fa_q_b)
        if fuse8:
            a = ops.t2i_fold_attention(q, keys, self.fa_k_add, self.fa_kv_w[0:128], self.fa_kv_w[128:256], self.fa_v_b, B,
                                       Nt, NT_IMG, x_shared=(kb == 1))
        else:
            kv = ops.gemm(keys, self.fa_kv_w, self.fa_kv_b)
            a = ops.attention_kadd(q, kv[:, 0:128], self.fa_k_add, kv[:, 128:256], B, 8, Nt, NT_IMG, kv_shared=(kb == 1))
        queries = ops.gemm(a, self.fa_o_w, self.fa_o_b, residual=queries, out_dtype=_F32)
        hs = ops.layernorm(queries, self.nf_w, self.nf_b, 1e-5, _F32)  # [B*Nt,256]
        # ---- IoU head first: it decides (iou_gate) which prompts need their masks at all
        hs16 = ops.add_cast(hs, None, _BF16).view(B, Nt * 256)
        ious = self._mlp3(hs16[:, 256:512], self.iou_head, last_act=ops.ACT_SIGMOID)  # [B,4]
        plist = ops.iou_gate(ious, iou_gate) if (iou_gate is not None and not val) else None
        # ---- up-scaling + hyper-network masks
        hyper = torch.empty((B, 4, 32), dtype=_F32, device=self.device)
        hv = hyper.view(B, 128)
        for i in range(4):
            self._mlp3(hs16[:, (2 + i) * 256:(3 + i) * 256], self.hyper[i], out=hv[:, i * 32:(i + 1) * 32])
        if val:
            masks = self._upscale_validate(keys, s0, s1, hyper, B, kb)
        else:
            u1 = ops.gemm_upscale1(keys, self.up1_w, self.up1_b, s1, 0, self.up_ln_w, self.up_ln_b, B, 64, 64, plist=plist)
            masks = ops.gemm_upscale2(u1, self.up2_w, self.up2_b, s0, 0, hyper, B, 128, 128, plist=plist,
                                      zero_fill=zero_fill)  # [B,4,256,256]
            del u1
        obj = self._mlp3(hs16[:, 0:256], self.obj_head)  # [B,1]
        out = {"masks": masks, "ious": ious, "obj": obj, "hs": hs.view(B, Nt, 256)}
        if not multimask_output:
            if self.dynamic_multimask_via_stability:
                out["sel_idx"], out["sel_iou"] = ops.select_mask(masks, ious, self.stab_delta, self.stab_thresh)
            else:
                out["sel_idx"], out["sel_iou"] = None, None  # token 0
        return out
