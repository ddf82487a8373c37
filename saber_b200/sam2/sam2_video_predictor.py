"""Drop-in for ``sam2.sam2_video_predictor.SAM2VideoPredictor`` (as returned by ``build_sam2_video_predictor``) on the
B200 kernels — the surface REF saber/adapters/sam2/predictor.py binds:

  ``maskmem_tpos_enc`` (re-assigned, REF :31-32), ``num_maskmem`` (REF :33-34), ``image_size`` (:101), ``device``,
  ``sam_mask_decoder.register_forward_hook`` (hook reads ``output[3]``, REF :278,284),
  ``_get_image_feature(state, frame_idx=, batch_size=)`` (:114,152), ``add_new_mask`` (:164-169),
  ``propagate_in_video`` -> ``(frame_idx, obj_ids, logits [N,1,Hv,Wv])`` (:196-202), ``reset_state``,
  ``add_new_points_or_box`` (:171-180), ``clear_all_prompts_in_frame`` / ``remove_object`` (:358-366).
  The inference-state dict is the one SABER builds itself (REF :130-150).

B200 design (SURVEY §7 "device-resident batched state machine"): all objects tracked in a frame run as ONE batch
through memory attention -> mask decoder -> memory encoder (upstream loops objects with batch 1); the per-object
memory bank (bf16 ``[4096,64]`` features, fp32 object pointers, low-res scores) never leaves the device; every frame is
encoded once and its features stay cached (upstream keeps one frame and re-encodes the volume for every pass). The
forward hook still fires once per object per frame with ``output[3]`` shaped ``[1,1]``.
Restates sam2/sam2_video_predictor.py + sam2/modeling/sam2_base.py (SURVEY §8a U6-U10, Appendix A4).
"""
from __future__ import annotations

import os
from typing import Any, Callable, Dict, List, Optional, Tuple

import numpy as np
import torch

from .. import ops
from . import arch
from .build_sam import SAM2Model, _load_state_dict
from .memory import MemoryAttention, MemoryEncoder, sine_pe_1d

_BF16, _F32, _I32 = torch.bfloat16, torch.float32, torch.int32
NT = 4096
NO_OBJ_SCORE = -1024.0


class _HookHandle:
    def __init__(self, hooks: list, fn):
        self._hooks, self._fn = hooks, fn

    def remove(self):
        if self._fn in self._hooks:
            self._hooks.remove(self._fn)


class _DecoderModule:
    """``predictor.sam_mask_decoder``: the B200 mask-decoder executor behind torch's forward-hook interface."""

    def __init__(self, exec_):
        self.exec = exec_
        self._hooks: List[Callable] = []
        # resident alternative to a forward hook: when set to a callable it receives the DEVICE tensor of object scores
        # [B,1] of every decoder call (no host copy, no synchronisation); SAM2Adapter.segment_volume_device uses it so
        # that the host can run ahead of the GPU across frames. Forward hooks (the reference's interface) still work.
        self.device_sink: Optional[Callable] = None

    def register_forward_hook(self, fn):
        self._hooks.append(fn)
        return _HookHandle(self._hooks, fn)

    def fire(self, masks, ious, tokens, obj_scores):
        """One hook call per batch entry with upstream's output tuple (masks, iou_pred, sam_tokens_out,
        object_score_logits); the scores are brought to the host once for the whole batch."""
        if self.device_sink is not None:
            self.device_sink(obj_scores.detach().reshape(-1, 1))
        if not self._hooks:
            return
        host = obj_scores.detach().reshape(-1, 1).cpu()
        for i in range(host.shape[0]):
            out = (masks[i:i + 1], ious[i:i + 1], tokens[i:i + 1], host[i:i + 1])
            for fn in list(self._hooks):
                fn(self, (), out)


class SAM2VideoPredictor(SAM2Model):
    def __init__(self, cfg, state_dict, device="cuda", dynamic_multimask_via_stability=True, num_maskmem=7,
                 fill_hole_area=8, binarize_mask_from_pts_for_mem_enc=True):
        self.fill_hole_area = fill_hole_area
        self.binarize_mask_from_pts_for_mem_enc = binarize_mask_from_pts_for_mem_enc
        self.max_obj_ptrs_in_encoder = 16
        self.mem_attn: Optional[MemoryAttention] = None
        self.mem_enc: Optional[MemoryEncoder] = None
        self.sam_mask_decoder: Optional[_DecoderModule] = None
        self._const_cache: Dict[Any, Any] = {}
        self.max_encode_batch = int(os.environ.get("SB_ENCODE_BATCH", "8"))  # crops / frames per encoder pass
        # A tracking step is ~175 launches of mostly small kernels: run eagerly it is bound by the host (25 us per launch,
        # 4.5 ms per frame with one object). Steps whose memory layout is in steady state (all 15 object pointers present)
        # are captured once per (layout, batch) into a CUDA graph and replayed; SB_PROP_GRAPH=0 keeps everything eager.
        self.use_cuda_graph = os.environ.get("SB_PROP_GRAPH", "1") != "0"
        self._step_graphs: Dict[Any, Any] = {}
        super().__init__(cfg, state_dict, device=device, dynamic_multimask_via_stability=dynamic_multimask_via_stability,
                         num_maskmem=num_maskmem)

    # ---- attributes SABER re-assigns: `maskmem_tpos_enc` is a registered nn.Parameter (REF saber/adapters/sam2/
    # predictor.py:31-32 slices it and assigns a new torch.nn.Parameter) and `num_maskmem` a plain attribute (:33-34);
    # every constant derived from them is cached under a key that includes both.
    def _tpos(self) -> torch.Tensor:
        return self._parameters["maskmem_tpos_enc"].detach().cpu().float()

    def _tpos_key(self):
        p = self._parameters["maskmem_tpos_enc"]
        return (p.data_ptr(), tuple(p.shape), int(self.num_maskmem))

    def _build_executors(self, dev):
        super()._build_executors(dev)
        sd = {k: v.cpu() for k, v in self.upstream_state_dict().items()}
        with torch.cuda.device(dev):
            self.mem_attn = MemoryAttention(sd, dev)
            self.mem_enc = MemoryEncoder(sd, dev)
            self.sam_mask_decoder = _DecoderModule(self.decoder)
            self.k_no_obj_ptr = sd["no_obj_ptr"].reshape(-1).to(dev, _F32).contiguous()
            self.objptr_mlp = [(sd[f"obj_ptr_proj.layers.{k}.weight"].to(dev, _BF16).contiguous(),
                                sd[f"obj_ptr_proj.layers.{k}.bias"].to(dev, _F32).contiguous()) for k in range(3)]
            self.mask_ds_w = sd["mask_downsample.weight"].reshape(16).to(dev, _F32).contiguous()
            self.mask_ds_b = sd["mask_downsample.bias"].reshape(1).to(dev, _F32).contiguous()
            self._tpos_proj = (sd["obj_ptr_tpos_proj.weight"].float(), sd["obj_ptr_tpos_proj.bias"].float())
        self._const_cache.clear()

    # ---- constants that depend on (re-assignable) maskmem_tpos_enc / num_maskmem ------------------
    def _spatial_key_pos(self, t_pos: int) -> List[torch.Tensor]:
        """Per layer [4096,256]: k_proj(maskmem_pos_enc + maskmem_tpos_enc[num_maskmem - t_pos - 1]) positional term."""
        key = ("spatial", t_pos, self._tpos_key())
        if key not in self._const_cache:
            tpos = self._tpos()[self.num_maskmem - t_pos - 1].reshape(1, -1)  # [1,64]
            self._const_cache[key] = self.mem_attn.key_pos_term(self.mem_enc.pos + tpos)
        return self._const_cache[key]

    def _ptr_key_pos(self, t_diffs: Tuple[int, ...], num_frames: int) -> List[torch.Tensor]:
        """Per layer [4*len(t_diffs), 256]: positional term of the object-pointer tokens (signed temporal distance)."""
        key = ("ptr", t_diffs, num_frames)
        if key not in self._const_cache:
            t_diff_max = min(num_frames, self.max_obj_ptrs_in_encoder) - 1
            pos = torch.tensor(t_diffs, dtype=torch.float32)
            pe = sine_pe_1d(pos / t_diff_max, arch.HIDDEN)
            w, b = self._tpos_proj
            pe = pe @ w.t() + b  # [n,64]
            pe = pe.repeat_interleave(arch.HIDDEN // arch.MEM_DIM, dim=0)
            self._const_cache[key] = self.mem_attn.key_pos_term(pe)
        return self._const_cache[key]

    # ---- frame features ------------------------------------------------------------------------------
    @torch.no_grad()
    def encode_frames(self, inference_state, frame_ids=None) -> None:
        """Phase A (SURVEY §8e): encode frames in batches and keep their features resident (bf16 is not needed: a
        300-slice tomogram is 5 GB of fp32 features in 180 GB of HBM)."""
        self._require_gpu()
        st = inference_state
        ids = [f for f in (range(st["num_frames"]) if frame_ids is None else frame_ids) if f not in st["cached_features"]]
        for k0 in range(0, len(ids), self.max_encode_batch):
            chunk = ids[k0:k0 + self.max_encode_batch]
            x = torch.stack([st["images"][f] for f in chunk]).to(self.device, _F32).contiguous()
            out = self.encoder.forward(x)
            for j, f in enumerate(chunk):
                st["cached_features"][f] = {
                    "feat": out["feat"][j * NT:(j + 1) * NT], "s1": out["s1"][j * 16384:(j + 1) * 16384],
                    "s0": out["s0"][j * 65536:(j + 1) * 65536]}

    def _frame(self, st, frame_idx) -> Dict[str, torch.Tensor]:
        c = st["cached_features"].get(frame_idx)
        if c is None or "feat" not in c:
            self.encode_frames(st, [frame_idx])
            c = st["cached_features"][frame_idx]
        if "pix_proj" not in c:
            c["pix_proj"] = self.mem_enc.project_pix(c["feat"])
        return c

    @torch.no_grad()
    def _get_image_feature(self, inference_state, frame_idx=0, batch_size=1):
        """Upstream returns (image, backbone_out, vision_feats, vision_pos, feat_sizes); SABER discards the result
        (REF :114,152) — this warms the feature cache and returns the token-major features of the frame."""
        c = self._frame(inference_state, frame_idx)
        return c

    # ---- object bookkeeping (upstream dict layout) ---------------------------------------------------------
    def _obj_id_to_idx(self, st, obj_id):
        idx = st["obj_id_to_idx"].get(obj_id, None)
        if idx is not None:
            return idx
        idx = len(st["obj_id_to_idx"])
        st["obj_id_to_idx"][obj_id] = idx
        st["obj_idx_to_id"][idx] = obj_id
        st["obj_ids"] = list(st["obj_id_to_idx"])
        st["point_inputs_per_obj"][idx] = {}
        st["mask_inputs_per_obj"][idx] = {}
        st["output_dict_per_obj"][idx] = {"cond_frame_outputs": {}, "non_cond_frame_outputs": {}}
        st["temp_output_dict_per_obj"][idx] = {"cond_frame_outputs": {}, "non_cond_frame_outputs": {}}
        st["frames_tracked_per_obj"][idx] = {}
        return idx

    def _get_obj_num(self, st):
        return len(st["obj_idx_to_id"])

    # ---- prompting -------------------------------------------------------------------------------------------
    def _mask_to_model_res(self, mask) -> torch.Tensor:
        """bool/float (H,W) mask -> [1024,1024] fp32 {0,1} on the device (bilinear-antialias resize + >= 0.5)."""
        if isinstance(mask, torch.Tensor):
            m = mask.to(self.device)
        else:
            m = torch.from_numpy(np.ascontiguousarray(mask)).to(self.device)
        m = (m != 0).to(_F32).contiguous()  # torch.tensor(mask, dtype=torch.bool).float()
        assert m.dim() == 2
        H, W = m.shape
        S = self.image_size
        if (H, W) != (S, S):
            crops = torch.tensor([[0, 0, W, H]], dtype=_I32, device=self.device)
            r = ops.resize_normalize(m, crops, S, mean=(0.0, 0.0, 0.0), std=(1.0, 1.0, 1.0))[0, 0].contiguous()
            m = ops.threshold_affine(r, 0.5, 1.0, 0.0)
        return m

    @torch.no_grad()
    def add_new_mask(self, inference_state, frame_idx, obj_id, mask):
        self._require_gpu()
        st = inference_state
        obj_idx = self._obj_id_to_idx(st, obj_id)
        mi = self._mask_to_model_res(mask)  # [S,S] {0,1}
        st["mask_inputs_per_obj"][obj_idx][frame_idx] = mi
        st["point_inputs_per_obj"][obj_idx].pop(frame_idx, None)
        tracked = st["frames_tracked_per_obj"][obj_idx]
        is_init_cond_frame = frame_idx not in tracked
        key = "cond_frame_outputs" if is_init_cond_frame else "non_cond_frame_outputs"
        st["temp_output_dict_per_obj"][obj_idx][key][frame_idx] = self._use_mask_as_output(st, frame_idx, mi)
        # consolidated video-resolution scores of every object on this frame (upstream's return value)
        return frame_idx, st["obj_ids"], self._consolidated_video_res(st, frame_idx, is_init_cond_frame)

    def _use_mask_as_output(self, st, frame_idx, mask_inputs: torch.Tensor) -> Dict[str, Any]:
        """SAM2Base._use_mask_as_output for one object: scores = mask*20-10, low-res = antialiased x1/4, pointer from a
        decoder call prompted with mask_downsample(mask); memory is encoded later (preflight)."""
        S = self.image_size
        c = self._frame(st, frame_idx)
        hi = ops.threshold_affine(mask_inputs, 0.5, 20.0, -10.0)  # mask in {0,1} -> {-10, +10}
        crops = torch.tensor([[0, 0, S, S]], dtype=_I32, device=self.device)
        low = ops.resize_normalize(hi, crops, S // 4, mean=(0.0, 0.0, 0.0), std=(1.0, 1.0, 1.0))[0, 0:1].contiguous()
        prompt = ops.conv4x4s4(mask_inputs.view(1, S, S), self.mask_ds_w, self.mask_ds_b)  # [1,256,256]
        dec = self.decoder
        coords = torch.zeros((1, 1, 2), dtype=_F32, device=self.device)
        labels = torch.full((1, 1), -1, dtype=_I32, device=self.device)
        tokens = dec.prompt_tokens(coords, labels)
        out = dec.forward(c["feat"], c["s0"], c["s1"], tokens, prompt, multimask_output=False)
        self.sam_mask_decoder.fire(out["masks"][:, 0:1], out["ious"][:, 0:1], out["hs"][:, 2:3], out["obj"])
        _, tok, _ = ops.track_select(out["masks"], out["ious"], out["obj"].reshape(-1).contiguous(), out["hs"].contiguous(),
                                     out.get("sel_idx"), False)
        ptr = self._obj_ptr(tok, out["obj"].reshape(-1).contiguous())
        # torch.any(mask > 0) on a {0,1} mask == any non-zero bit pattern
        appear = ops.slice_any(mask_inputs.view(torch.int16).view(1, S, 2 * S)).to(_F32)
        score = ops.threshold_affine(appear, 0.5, 20.0, -10.0)
        ptr = ops.objptr_mix_(ptr, score, self.k_no_obj_ptr)
        if self.fill_hole_area > 0:  # sam2_video_predictor._run_single_frame_inference fills holes on every path
            low = ops.fill_holes(low, self.fill_hole_area)
        return {"maskmem_features": None, "maskmem_pos_enc": None, "pred_masks": low.view(1, 1, S // 4, S // 4),
                "obj_ptr": ptr, "object_score_logits": score.view(1, 1)}

    def _obj_ptr(self, token: torch.Tensor, obj_scores: torch.Tensor) -> torch.Tensor:
        h = ops.gemm(ops.add_cast(token.contiguous(), None, _BF16), *self.objptr_mlp[0], act=ops.ACT_RELU)
        h = ops.gemm(h, *self.objptr_mlp[1], act=ops.ACT_RELU)
        ptr = ops.gemm(h, *self.objptr_mlp[2], out_dtype=_F32)
        return ops.objptr_mix_(ptr, obj_scores, self.k_no_obj_ptr)

    # ---- propagation ------------------------------------------------------------------------------------------
    @torch.no_grad()
    def propagate_in_video_preflight(self, inference_state):
        st = inference_state
        B = self._get_obj_num(st)
        if B == 0:
            raise RuntimeError("No input points or masks are provided for any object; please add inputs first.")
        for i in range(B):
            obj_out = st["output_dict_per_obj"][i]
            obj_tmp = st["temp_output_dict_per_obj"][i]
            for is_cond in (False, True):
                key = "cond_frame_outputs" if is_cond else "non_cond_frame_outputs"
                for frame_idx, out in obj_tmp[key].items():
                    if out["maskmem_features"] is None:
                        c = self._frame(st, frame_idx)
                        out["maskmem_features"] = self.mem_enc.forward(
                            c["pix_proj"], out["pred_masks"].view(1, 256, 256), out["object_score_logits"].reshape(-1),
                            binarize=self.binarize_mask_from_pts_for_mem_enc)
                        out["maskmem_pos_enc"] = True
                    obj_out[key][frame_idx] = out
                obj_tmp[key].clear()
            if len(obj_out["cond_frame_outputs"]) == 0:
                raise RuntimeError(f"No input points or masks are provided for object id {st['obj_idx_to_id'][i]}; "
                                   "please add inputs first.")
            for frame_idx in obj_out["cond_frame_outputs"]:
                obj_out["non_cond_frame_outputs"].pop(frame_idx, None)

    def _memory_plan(self, obj_out, frame_idx, num_frames, reverse):
        """Which stored outputs form the memory of `frame_idx` for one object (SAM2Base._prepare_memory_conditioned_
        features): returns (signature, spatial [(t_pos, out)], pointers [(t_diff, out)])."""
        cond = obj_out["cond_frame_outputs"]
        spatial = [(0, f, out) for f, out in cond.items()]
        for t_pos in range(1, self.num_maskmem):
            t_rel = self.num_maskmem - t_pos
            if t_rel == 1:
                prev = frame_idx + t_rel if reverse else frame_idx - t_rel
            elif not reverse:
                prev = (frame_idx - 2) - (t_rel - 2)
            else:
                prev = (frame_idx + 2) + (t_rel - 2)
            out = obj_out["non_cond_frame_outputs"].get(prev)
            if out is not None:
                spatial.append((t_pos, prev, out))
        sign = -1 if reverse else 1
        ptrs = [((frame_idx - f) * sign, f, out) for f, out in cond.items() if (f >= frame_idx if reverse else f <= frame_idx)]
        for t_diff in range(1, min(num_frames, self.max_obj_ptrs_in_encoder)):
            t = frame_idx + t_diff if reverse else frame_idx - t_diff
            if t < 0 or t >= num_frames:
                break
            out = obj_out["non_cond_frame_outputs"].get(t)
            if out is not None:
                ptrs.append((t_diff, t, out))
        sig = (tuple(tp for tp, _, _ in spatial), tuple(td for td, _, _ in ptrs))
        return sig, spatial, ptrs

    def _assemble_memory(self, memory: torch.Tensor, objs: List[int], plans) -> None:
        """Fill memory [B, Nk, 64] bf16: per object the spatial memories, then the object pointers (4 tokens each). Stored
        outputs of one tracking step are views of ONE [B*4096,64] / [B,256] tensor per group (`_batch` entry), so a
        slot that every object of this batch fills from the same earlier step is ONE copy instead of B."""
        B = len(objs)
        first = plans[objs[0]]
        n_sp, n_pt = len(first[1]), len(first[2])
        off = 0
        for k in range(n_sp + n_pt):
            is_sp = k < n_sp
            outs = [plans[i][1][k][2] if is_sp else plans[i][2][k - n_sp][2] for i in objs]
            width = NT if is_sp else 4
            b0 = outs[0].get("_batch")
            if b0 is not None and b0["objs"] == tuple(objs) and all(o.get("_batch") is b0 for o in outs):
                src = b0["mem"].view(B, NT, 64) if is_sp else b0["ptr"].view(B, 4, 64)
                memory[:, off:off + width] = src  # (fp32 pointers -> bf16 storage cast)
            else:
                for bi, out in enumerate(outs):
                    memory[bi, off:off + width] = out["maskmem_features"] if is_sp else out["obj_ptr"].view(4, 64)
            off += width

    def _layout_pos(self, st, sig):
        """Key positional term of a memory layout, per layer [Nk, 256]: spatial slots + pointer tokens (weights-only
        constants). The pointer part depends on the temporal distances — the conditioning frame's distance changes
        every frame — so the term lives in ONE buffer per layout STRUCTURE (which slots, how many pointers): the spatial
        rows are written once, the 4 * n_ptr pointer rows are refreshed per call (stream-ordered before their consumer).
        A CUDA graph of the step can therefore bake the buffer addresses."""
        t_pos_list, t_diff_list = sig
        ck = ("layout", tuple(t_pos_list), len(t_diff_list), st["num_frames"], self._tpos_key())
        buf = self._const_cache.get(ck)
        if buf is None:
            parts = [self._spatial_key_pos(tp) for tp in t_pos_list]
            n_sp = sum(p[0].shape[0] for p in parts)
            n_pt = 4 * len(t_diff_list)
            ref = parts[0][0] if parts else self._ptr_key_pos(tuple(t_diff_list), st["num_frames"])[0]
            buf = [torch.empty((n_sp + n_pt, ref.shape[1]), dtype=ref.dtype, device=ref.device) for _ in range(4)]
            for l in range(4):
                off = 0
                for p_ in parts:
                    buf[l][off:off + p_[l].shape[0]] = p_[l]
                    off += p_[l].shape[0]
            self._const_cache[ck] = buf
        if t_diff_list:
            # pointer rows from a per-distance table on the device (built once per video length); only the rows whose
            # distance changed since the last call are rewritten — in steady state that is the conditioning frame's
            # pointer alone: 4 small device copies per frame, no host matmul / H2D copy on the frame path
            table = self._ptr_pos_table(st["num_frames"])
            last = self._const_cache.setdefault(ck + ("last",), [None] * len(t_diff_list))
            n_sp = buf[0].shape[0] - 4 * len(t_diff_list)
            for j, td in enumerate(t_diff_list):
                if last[j] != td:
                    for l in range(4):
                        buf[l][n_sp + 4 * j:n_sp + 4 * j + 4] = table[l][td]
                    last[j] = td
        return buf

    def _ptr_pos_table(self, num_frames: int) -> List[torch.Tensor]:
        """Per layer [num_frames, 4, 256]: positional term of an object pointer at temporal distance t (0 .. num_frames-1)."""
        key = ("ptr_table", num_frames)
        if key not in self._const_cache:
            per = self._ptr_key_pos(tuple(range(num_frames)), num_frames)  # per layer [4 * num_frames, 256]
            self._const_cache[key] = [p_.view(num_frames, 4, -1).contiguous() for p_ in per]
        return self._const_cache[key]

    def _conditioned_features(self, st, c, objs: List[int], sig, plans) -> torch.Tensor:
        """Memory attention for a batch of objects that share the memory layout `sig` (SAM2Base._prepare_memory_
        conditioned_features for a non-initial frame) -> [B*4096, 256] fp32."""
        B = len(objs)
        t_pos_list, t_diff_list = sig
        n_ptr_tok = 4 * len(t_diff_list)
        Nk = NT * len(t_pos_list) + n_ptr_tok
        memory = torch.empty((B, Nk, 64), dtype=_BF16, device=self.device)
        self._assemble_memory(memory, objs, plans)
        pos_k = self._layout_pos(st, sig)
        return self.mem_attn.forward(c["feat"], memory.view(B * Nk, 64), pos_k, n_ptr_tok, B)  # [B*4096,256]

    def _step_body(self, feat, s0, s1, pix_proj, memory, pos_k, n_ptr_tok, B):
        """The device work of one tracking step on given inputs (memory attention -> mask decoder -> selection ->
        object pointer -> memory encoder -> hole filling). No host synchronisation: capturable."""
        Nk = memory.shape[1]
        pix = self.mem_attn.forward(feat, memory.view(B * Nk, 64), pos_k, n_ptr_tok, B)
        dec = self.decoder
        coords = torch.zeros((B, 1, 2), dtype=_F32, device=self.device)
        labels = torch.full((B, 1), -1, dtype=_I32, device=self.device)
        tokens = dec.prompt_tokens(coords, labels)
        out = dec.forward(pix, s0, s1, tokens, None, multimask_output=True)
        obj = out["obj"].reshape(-1).contiguous()
        low, tok, _ = ops.track_select(out["masks"], out["ious"], obj, out["hs"].contiguous(), None, True)
        ptr = self._obj_ptr(tok, obj)
        mem = self.mem_enc.forward(pix_proj, low, obj, binarize=False)  # is_mask_from_pts = False
        pred = ops.fill_holes(low, self.fill_hole_area) if self.fill_hole_area > 0 else low
        return {"masks": out["masks"], "ious": out["ious"], "hs": out["hs"], "obj_raw": out["obj"], "obj": obj, "ptr": ptr,
                "mem": mem, "pred": pred}

    def _step_graph(self, st, sig, B):
        """CUDA graph of `_step_body` for the steady-state layout `sig` and batch B (static input / output buffers)."""
        key = (tuple(sig[0]), len(sig[1]), B, st["num_frames"], self._tpos_key())
        g = self._step_graphs.get(key)
        if g is not None:
            return g
        dev = self.device
        t_pos_list, t_diff_list = sig
        n_ptr_tok = 4 * len(t_diff_list)
        Nk = NT * len(t_pos_list) + n_ptr_tok
        g = {"feat": torch.zeros((NT, 256), dtype=_F32, device=dev), "s0": torch.zeros((65536, 32), dtype=_F32, device=dev),
             "s1": torch.zeros((16384, 64), dtype=_F32, device=dev), "pix_proj": None,
             "memory": torch.zeros((B, Nk, 64), dtype=_BF16, device=dev), "n_ptr_tok": n_ptr_tok}
        self._step_graphs[key] = g
        return g

    def _track_group(self, st, frame_idx, objs: List[int], sig, plans, reverse) -> Dict[int, Dict[str, Any]]:
        """One tracking step for a batch of objects that share the memory layout `sig`."""
        B = len(objs)
        c = self._frame(st, frame_idx)
        pos_k = self._layout_pos(st, sig)
        t_pos_list, t_diff_list = sig
        n_ptr_tok = 4 * len(t_diff_list)
        steady = len(t_diff_list) >= self.max_obj_ptrs_in_encoder - 1 or len(t_diff_list) >= st["num_frames"] - 2
        use_graph = (self.use_cuda_graph and steady and not self.sam_mask_decoder._hooks
                     and not torch.cuda.is_current_stream_capturing())
        if use_graph:
            g = self._step_graph(st, sig, B)
            if g["pix_proj"] is None:
                g["pix_proj"] = torch.zeros_like(c["pix_proj"])
            g["feat"].copy_(c["feat"])
            g["s0"].copy_(c["s0"])
            g["s1"].copy_(c["s1"])
            g["pix_proj"].copy_(c["pix_proj"])
            self._assemble_memory(g["memory"], objs, plans)
            if "graph" not in g:
                args = (g["feat"], g["s0"], g["s1"], g["pix_proj"], g["memory"], pos_k, n_ptr_tok, B)
                main = torch.cuda.current_stream()
                side = torch.cuda.Stream(device=self.device)
                side.wait_stream(main)
                with torch.cuda.stream(side):
                    self._step_body(*args)  # warm-up: function attributes, constant caches
                main.wait_stream(side)
                torch.cuda.synchronize()
                n0 = ops.launch_count
                graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(graph, capture_error_mode="thread_local"):
                    g["out"] = self._step_body(*args)
                g["launches"] = ops.launch_count - n0
                ops.launch_count = n0
                g["graph"] = graph
            g["graph"].replay()
            ops.launch_count += g["launches"]
            o = g["out"]
            # results are stored across frames: copy them out of the graph's static buffers (one clone per tensor)
            r = {k: o[k].clone() for k in ("obj", "ptr", "mem", "pred")}
            self.sam_mask_decoder.fire(o["masks"][:, 1:4], o["ious"][:, 1:4], o["hs"][:, 3:6], o["obj_raw"])
        else:
            memory = torch.empty((B, NT * len(t_pos_list) + n_ptr_tok, 64), dtype=_BF16, device=self.device)
            self._assemble_memory(memory, objs, plans)
            r = self._step_body(c["feat"], c["s0"], c["s1"], c["pix_proj"], memory, pos_k, n_ptr_tok, B)
            self.sam_mask_decoder.fire(r["masks"][:, 1:4], r["ious"][:, 1:4], r["hs"][:, 3:6], r["obj_raw"])
        obj, ptr, mem, pred = r["obj"], r["ptr"], r["mem"], r["pred"]
        batch = {"objs": tuple(objs), "mem": mem, "ptr": ptr}
        res = {}
        for bi, i in enumerate(objs):
            res[i] = {"maskmem_features": mem[bi * NT:(bi + 1) * NT], "maskmem_pos_enc": True,
                      "pred_masks": pred[bi].view(1, 1, 256, 256), "obj_ptr": ptr[bi:bi + 1],
                      "object_score_logits": obj[bi].view(1, 1), "_batch": batch}
        return res

    @torch.no_grad()
    def propagate_in_video(self, inference_state, start_frame_idx=None, max_frame_num_to_track=None, reverse=False):
        self._require_gpu()
        st = inference_state
        self.propagate_in_video_preflight(st)
        obj_ids = st["obj_ids"]
        num_frames = st["num_frames"]
        B = self._get_obj_num(st)
        if start_frame_idx is None:
            start_frame_idx = min(t for d in st["output_dict_per_obj"].values() for t in d["cond_frame_outputs"])
        if max_frame_num_to_track is None:
            max_frame_num_to_track = num_frames
        if reverse:
            end = max(start_frame_idx - max_frame_num_to_track, 0)
            order = range(start_frame_idx, end - 1, -1) if start_frame_idx > 0 else []
        else:
            end = min(start_frame_idx + max_frame_num_to_track, num_frames - 1)
            order = range(start_frame_idx, end + 1)
        vh, vw = st["video_height"], st["video_width"]
        for frame_idx in order:
            low = torch.empty((B, 256, 256), dtype=_F32, device=self.device)
            groups: Dict[Any, List[int]] = {}
            plans = {}
            for i in range(B):
                obj_out = st["output_dict_per_obj"][i]
                if frame_idx in obj_out["cond_frame_outputs"]:
                    low[i] = obj_out["cond_frame_outputs"][frame_idx]["pred_masks"].view(256, 256)
                else:
                    plans[i] = self._memory_plan(obj_out, frame_idx, num_frames, reverse)
                    groups.setdefault(plans[i][0], []).append(i)
            for sig, objs in groups.items():
                res = self._track_group(st, frame_idx, objs, sig, plans, reverse)
                for i in objs:
                    st["output_dict_per_obj"][i]["non_cond_frame_outputs"][frame_idx] = res[i]
                    low[i] = res[i]["pred_masks"].view(256, 256)
            for i in range(B):
                st["frames_tracked_per_obj"][i][frame_idx] = {"reverse": reverse}
            video_res = ops.upsample_bilinear(low, vh, vw).view(B, 1, vh, vw)
            yield frame_idx, obj_ids, video_res

    # ---- state ------------------------------------------------------------------------------------------------
    @torch.inference_mode()
    def init_state(self, video_path, offload_video_to_cpu=False, offload_state_to_cpu=False, async_loading_frames=False):
        """Upstream's ``init_state`` on a folder of JPEG frames (``video_io.load_video_frames``): the inference-state
        dict with frame 0's features warmed. ``storage_device`` is the host with ``offload_state_to_cpu``, as upstream
        reports it; the memory bank stays on the device either way (the outputs do not depend on it)."""
        from .video_io import load_video_frames
        self._require_gpu()
        images, video_height, video_width = load_video_frames(video_path, self.image_size, offload_video_to_cpu,
                                                              async_loading_frames=async_loading_frames,
                                                              compute_device=self.device)
        storage = torch.device("cpu") if offload_state_to_cpu else self.device
        return self.new_inference_state(images, video_height, video_width, offload_video_to_cpu, offload_state_to_cpu,
                                        self.device, storage)

    def new_inference_state(self, images, video_height, video_width, offload_video_to_cpu, offload_state_to_cpu,
                            device, storage_device) -> Dict[str, Any]:
        """Upstream's inference-state dict (same keys, same value types) over ``images`` [N,3,S,S] or a lazy frame
        list, with frame 0's features warmed through ``_get_image_feature`` as upstream's ``init_state`` does."""
        from collections import OrderedDict
        st = {"images": images, "num_frames": len(images), "offload_video_to_cpu": offload_video_to_cpu,
              "offload_state_to_cpu": offload_state_to_cpu, "video_height": video_height, "video_width": video_width,
              "device": device, "storage_device": storage_device, "point_inputs_per_obj": {}, "mask_inputs_per_obj": {},
              "cached_features": {}, "constants": {}, "obj_id_to_idx": OrderedDict(), "obj_idx_to_id": OrderedDict(),
              "obj_ids": [], "output_dict_per_obj": {}, "temp_output_dict_per_obj": {}, "frames_tracked_per_obj": {}}
        self._get_image_feature(st, frame_idx=0, batch_size=1)
        return st

    @torch.no_grad()
    def reset_state(self, inference_state):
        s = inference_state
        for k in ("obj_id_to_idx", "obj_idx_to_id", "obj_ids", "point_inputs_per_obj", "mask_inputs_per_obj",
                  "output_dict_per_obj", "temp_output_dict_per_obj", "frames_tracked_per_obj"):
            s[k].clear()

    # ---- point / box prompts, prompt removal, object removal (forwarded by REF saber/adapters/sam2/predictor.py:171-180,
    # 358-366; restates sam2_video_predictor.SAM2VideoPredictor.{add_new_points_or_box, clear_all_prompts_in_frame,
    # remove_object}) --------------------------------------------------------------------------------------------
    def _consolidated_video_res(self, st, frame_idx, is_cond: bool) -> torch.Tensor:
        """_consolidate_temp_output_across_obj(consolidate_at_video_res=True) + _get_orig_video_res_output."""
        key = "cond_frame_outputs" if is_cond else "non_cond_frame_outputs"
        B = self._get_obj_num(st)
        vh, vw = st["video_height"], st["video_width"]
        low = torch.full((B, 256, 256), NO_OBJ_SCORE, dtype=_F32, device=self.device)
        for i in range(B):
            out = st["temp_output_dict_per_obj"][i][key].get(frame_idx)
            if out is None:
                out = st["output_dict_per_obj"][i]["cond_frame_outputs"].get(frame_idx)
            if out is None:
                out = st["output_dict_per_obj"][i]["non_cond_frame_outputs"].get(frame_idx)
            if out is not None:
                low[i] = out["pred_masks"].view(256, 256)
        return ops.upsample_bilinear(low, vh, vw).view(B, 1, vh, vw)

    @torch.no_grad()
    def add_new_points_or_box(self, inference_state, frame_idx, obj_id, points=None, labels=None, clear_old_points=True,
                              normalize_coords=True, box=None):
        self._require_gpu()
        st = inference_state
        obj_idx = self._obj_id_to_idx(st, obj_id)
        point_inputs_per_frame = st["point_inputs_per_obj"][obj_idx]
        if (points is not None) != (labels is not None):
            raise ValueError("points and labels must be provided together")
        if points is None and box is None:
            raise ValueError("at least one of points or box must be provided as input")
        pts = torch.zeros(0, 2, dtype=_F32) if points is None else torch.as_tensor(points, dtype=_F32).cpu()
        lbl = torch.zeros(0, dtype=_I32) if labels is None else torch.as_tensor(labels, dtype=_I32).cpu()
        if pts.dim() == 2:
            pts = pts.unsqueeze(0)
        if lbl.dim() == 1:
            lbl = lbl.unsqueeze(0)
        if box is not None:
            if not clear_old_points:
                raise ValueError("cannot add box without clearing old points, since box prompt must be provided before "
                                 "any point prompt (please use clear_old_points=True instead)")
            bc = torch.as_tensor(box, dtype=_F32).cpu().reshape(1, 2, 2)
            pts = torch.cat([bc, pts], dim=1)
            lbl = torch.cat([torch.tensor([[2, 3]], dtype=_I32), lbl], dim=1)
        if normalize_coords:
            pts = pts / torch.tensor([st["video_width"], st["video_height"]], dtype=_F32)
        pts = pts * self.image_size
        old = None if clear_old_points else point_inputs_per_frame.get(frame_idx)
        if old is not None:
            pts = torch.cat([old["point_coords"].cpu(), pts], dim=1)
            lbl = torch.cat([old["point_labels"].cpu(), lbl], dim=1)
        point_inputs = {"point_coords": pts.to(self.device).contiguous(), "point_labels": lbl.to(self.device).contiguous()}
        point_inputs_per_frame[frame_idx] = point_inputs
        st["mask_inputs_per_obj"][obj_idx].pop(frame_idx, None)
        tracked = st["frames_tracked_per_obj"][obj_idx]
        is_init_cond_frame = frame_idx not in tracked
        reverse = False if is_init_cond_frame else tracked[frame_idx]["reverse"]
        obj_out = st["output_dict_per_obj"][obj_idx]
        obj_tmp = st["temp_output_dict_per_obj"][obj_idx]
        is_cond = is_init_cond_frame  # add_all_frames_to_correct_as_cond = False
        key = "cond_frame_outputs" if is_cond else "non_cond_frame_outputs"
        prev = obj_tmp[key].get(frame_idx)
        if prev is None:
            prev = obj_out["cond_frame_outputs"].get(frame_idx)
            if prev is None:
                prev = obj_out["non_cond_frame_outputs"].get(frame_idx)
        prev_logits = prev["pred_masks"].view(1, 256, 256) if prev is not None and prev["pred_masks"] is not None else None
        obj_tmp[key][frame_idx] = self._point_step(st, obj_out, frame_idx, is_init_cond_frame, point_inputs, reverse,
                                                   prev_logits)
        return frame_idx, st["obj_ids"], self._consolidated_video_res(st, frame_idx, is_cond)

    def _point_step(self, st, obj_out, frame_idx, is_init_cond_frame, point_inputs, reverse, prev_logits):
        """SAM2Base.track_step for one object with point inputs (run_mem_encoder=False): the frame embedding is
        `feat + no_mem_embed` on an initial conditioning frame, otherwise conditioned on the object's memory; the
        previous prediction on the frame (clamped to +-32) is the dense mask prompt; multimask output for <= 1 point."""
        c = self._frame(st, frame_idx)
        if is_init_cond_frame:
            pix = ops.add_cast(c["feat"], self.no_mem_embed_vec, _F32)
        else:
            plan = self._memory_plan(obj_out, frame_idx, st["num_frames"], reverse)
            pix = self._conditioned_features(st, c, [0], plan[0], {0: plan})
        npts = int(point_inputs["point_labels"].shape[1])
        multimask = 0 <= npts <= 1  # multimask_min_pt_num = 0, multimask_max_pt_num = 1 (SAM2.1 configs)
        dec = self.decoder
        tokens = dec.prompt_tokens(point_inputs["point_coords"], point_inputs["point_labels"])
        out = dec.forward(pix, c["s0"], c["s1"], tokens, prev_logits, multimask_output=multimask,
                          mask_clamp=(32.0 if prev_logits is not None else 0.0))
        obj = out["obj"].reshape(-1).contiguous()
        if multimask:
            self.sam_mask_decoder.fire(out["masks"][:, 1:4], out["ious"][:, 1:4], out["hs"][:, 3:6], out["obj"])
        else:
            self.sam_mask_decoder.fire(out["masks"][:, 0:1], out["ious"][:, 0:1], out["hs"][:, 2:3], out["obj"])
        low, tok, _ = ops.track_select(out["masks"], out["ious"], obj, out["hs"].contiguous(), out.get("sel_idx"), multimask)
        ptr = self._obj_ptr(tok, obj)
        pred = ops.fill_holes(low, self.fill_hole_area) if self.fill_hole_area > 0 else low
        return {"maskmem_features": None, "maskmem_pos_enc": None, "pred_masks": pred.view(1, 1, 256, 256),
                "obj_ptr": ptr, "object_score_logits": obj.view(1, 1)}

    @torch.no_grad()
    def clear_all_prompts_in_frame(self, inference_state, frame_idx, obj_id, need_output=True):
        st = inference_state
        obj_idx = self._obj_id_to_idx(st, obj_id)
        st["point_inputs_per_obj"][obj_idx].pop(frame_idx, None)
        st["mask_inputs_per_obj"][obj_idx].pop(frame_idx, None)
        tmp = st["temp_output_dict_per_obj"]
        tmp[obj_idx]["cond_frame_outputs"].pop(frame_idx, None)
        tmp[obj_idx]["non_cond_frame_outputs"].pop(frame_idx, None)
        obj_out = st["output_dict_per_obj"][obj_idx]
        out = obj_out["cond_frame_outputs"].pop(frame_idx, None)
        if out is not None:  # no inputs left on the frame: its output is downgraded to a non-conditioning one
            obj_out["non_cond_frame_outputs"][frame_idx] = out
            st["frames_tracked_per_obj"][obj_idx].pop(frame_idx, None)
        if not need_output:
            return None
        is_cond = any(frame_idx in d["cond_frame_outputs"] for d in tmp.values())
        return frame_idx, st["obj_ids"], self._consolidated_video_res(st, frame_idx, is_cond)

    @torch.no_grad()
    def remove_object(self, inference_state, obj_id, strict=False, need_output=True):
        st = inference_state
        old_idx = st["obj_id_to_idx"].get(obj_id, None)
        updated_frames = []
        if old_idx is None:
            if not strict:
                return st["obj_ids"], updated_frames
            raise RuntimeError(f"Cannot remove object id {obj_id} as it doesn't exist. "
                               f"All existing object ids: {st['obj_ids']}.")
        if len(st["obj_id_to_idx"]) == 1:
            self.reset_state(st)
            return st["obj_ids"], updated_frames
        input_frames = set(st["point_inputs_per_obj"][old_idx]) | set(st["mask_inputs_per_obj"][old_idx])
        for frame_idx in input_frames:
            self.clear_all_prompts_in_frame(st, frame_idx, obj_id, need_output=False)
        old_obj_ids = st["obj_ids"]
        old_inds = list(range(len(old_obj_ids)))
        remain = [k for k in old_inds if k != old_idx]
        new_obj_ids = [old_obj_ids[k] for k in remain]
        new_inds = list(range(len(new_obj_ids)))
        old_to_new = dict(zip(remain, new_inds))
        st["obj_id_to_idx"] = dict(zip(new_obj_ids, new_inds))
        st["obj_idx_to_id"] = dict(zip(new_inds, new_obj_ids))
        st["obj_ids"] = new_obj_ids
        for name in ("point_inputs_per_obj", "mask_inputs_per_obj", "output_dict_per_obj", "temp_output_dict_per_obj",
                     "frames_tracked_per_obj"):
            container = st[name]
            kept = []
            for k in old_inds:
                v = container.pop(k)
                if k in old_to_new:
                    kept.append((old_to_new[k], v))
            container.update(kept)
        if need_output:
            tmp = st["temp_output_dict_per_obj"]
            for frame_idx in input_frames:
                is_cond = any(frame_idx in d["cond_frame_outputs"] for d in tmp.values())
                updated_frames.append((frame_idx, self._consolidated_video_res(st, frame_idx, is_cond)))
        return st["obj_ids"], updated_frames


def build_sam2_video_predictor(config_file, ckpt_path=None, device="cuda", mode="eval", hydra_overrides_extra=None,
                               apply_postprocessing=True, vos_optimized=False, seed: int = 0, state_dict=None,
                               allow_random_init: bool = False, **kwargs) -> SAM2VideoPredictor:
    """Same call shape as upstream ``sam2.build_sam.build_sam2_video_predictor`` (REF saber/adapters/sam2/
    predictor.py:24-26); applies upstream's overrides: binarize_mask_from_pts_for_mem_enc, fill_hole_area=8 and (with
    apply_postprocessing) dynamic multimask via stability."""
    cfg = arch.resolve(config_file)
    sd = state_dict if state_dict is not None else _load_state_dict(cfg, ckpt_path, seed,
                                                                    allow_random_init=allow_random_init)
    model = SAM2VideoPredictor(cfg, sd, device=device, dynamic_multimask_via_stability=bool(apply_postprocessing),
                               fill_hole_area=8, binarize_mask_from_pts_for_mem_enc=True)
    if mode == "eval":
        model.eval()
    return model
