"""Drop-in for ``sam2.sam2_image_predictor.SAM2ImagePredictor`` on the B200 kernels.

Surface used by the reference: ``SAM2ImagePredictor(model)``, ``.model``, ``.set_image_batch(list of
(H,W,3) float32 arrays)``, ``._features["image_embed"]`` ``[B,256,64,64]`` and
``._features["high_res_feats"]`` (REF saber/classifier/models/SAM2.py:46-51,145-151), plus the
``set_image`` / ``_predict`` pair the automatic mask generator drives (upstream
sam2/automatic_mask_generator.py), and upstream's interactive ``predict`` / ``predict_batch`` with point, box and mask
prompts. Restates sam2/sam2_image_predictor.py + sam2/utils/transforms.py
(SURVEY §8a U4): float input is not rescaled, Resize(1024^2) is bilinear with antialias, ImageNet
mean/std, ``no_mem_embed`` is added to the lowest-resolution feature.
"""
from __future__ import annotations

import os
from typing import Dict, List, Optional, Sequence, Union

import numpy as np
import torch

from .. import ops
from . import arch

_F32 = torch.float32
ImageLike = Union[np.ndarray, torch.Tensor]


class _Features(dict):
    """``_features`` dict: token-major device features are authoritative; the NCHW views the reference
    reads (``image_embed``, ``high_res_feats``) are materialised on first access."""

    def __init__(self, feat, s0, s1, batch):
        super().__init__()
        self.tok = {"embed": feat, "s0": s0, "s1": s1}
        self.batch = batch

    def __missing__(self, key):
        B = self.batch
        if key == "image_embed":
            v = ops.nhwc_to_nchw(self.tok["embed"], B, 4096, _F32).view(B, 256, 64, 64)
        elif key == "high_res_feats":
            v = [ops.nhwc_to_nchw(self.tok["s0"], B, 65536, _F32).view(B, 32, 256, 256),
                 ops.nhwc_to_nchw(self.tok["s1"], B, 16384, _F32).view(B, 64, 128, 128)]
        else:
            raise KeyError(key)
        self[key] = v
        return v


class SAM2ImagePredictor:
    def __init__(self, sam_model, mask_threshold: float = 0.0, max_hole_area: float = 0.0,
                 max_sprinkle_area: float = 0.0, **kwargs):
        self.model = sam_model
        self.mask_threshold = mask_threshold
        # SAM2Transforms.postprocess_masks: fill holes / remove sprinkles of the low-res planes before up-sampling
        self.max_hole_area = max_hole_area
        self.max_sprinkle_area = max_sprinkle_area
        self.resolution = sam_model.image_size
        self._bb_feat_sizes = [(256, 256), (128, 128), (64, 64)]
        self.max_encode_batch = int(os.environ.get("SB_ENCODE_BATCH", "24"))  # crops per encoder pass (all 21 AMG crops at once)
        self.reset_predictor()

    @property
    def device(self):
        return self.model.device

    def reset_predictor(self) -> None:
        self._is_image_set = False
        self._features: Optional[_Features] = None
        self._orig_hw: Optional[List[tuple]] = None
        self._is_batch = False

    # ------------------------------------------------------------------
    def _to_device_image(self, image: ImageLike) -> torch.Tensor:
        """(H,W,3) / (H,W) uint8 or float -> contiguous fp32 CUDA tensor (uint8 is divided by 255 as ToTensor does)."""
        if isinstance(image, np.ndarray):
            t = torch.from_numpy(np.ascontiguousarray(image))
        else:
            t = image
        if t.dtype == torch.uint8:
            t = t.to(self.device, non_blocking=True).float() / 255.0  # host-format conversion, not model arithmetic
        else:
            t = t.to(self.device, dtype=_F32, non_blocking=True)
        assert t.dim() in (2, 3) and (t.dim() == 2 or t.shape[2] == 3), f"expected HxW or HxWx3 image, got {tuple(t.shape)}"
        return t.contiguous()

    @torch.no_grad()
    def encode_crops(self, image: torch.Tensor, crops: torch.Tensor) -> _Features:
        """Encode ``crops`` (int32 [n,4] xyxy, device) of one device image; returns token-major features."""
        self.model._require_gpu()
        n = crops.shape[0]
        feats, s0s, s1s = [], [], []
        for k0 in range(0, n, self.max_encode_batch):
            kb = min(self.max_encode_batch, n - k0)
            x = ops.resize_normalize(image, crops[k0:k0 + kb].contiguous(), self.resolution)
            out = self.model.encoder.forward(x)
            del x
            feats.append(ops.add_cast(out["feat"], self.model.no_mem_embed_vec, _F32))
            s0s.append(out["s0"])
            s1s.append(out["s1"])
        cat = (lambda xs: xs[0] if len(xs) == 1 else torch.cat(xs, 0))
        return _Features(cat(feats), cat(s0s), cat(s1s), n)

    @torch.no_grad()
    def set_image(self, image: ImageLike) -> None:
        self.reset_predictor()
        img = self._to_device_image(image)
        H, W = img.shape[:2]
        self._orig_hw = [(H, W)]
        crops = torch.tensor([[0, 0, W, H]], dtype=torch.int32, device=self.device)
        self._features = self.encode_crops(img, crops)
        self._is_image_set = True

    @torch.no_grad()
    def set_image_batch(self, image_list: Sequence[ImageLike]) -> None:
        self.reset_predictor()
        assert isinstance(image_list, (list, tuple)) and len(image_list) > 0
        self._orig_hw = []
        parts = []
        for im in image_list:
            img = self._to_device_image(im)
            H, W = img.shape[:2]
            self._orig_hw.append((H, W))
            crops = torch.tensor([[0, 0, W, H]], dtype=torch.int32, device=self.device)
            parts.append(self.encode_crops(img, crops))
        if len(parts) == 1:
            self._features = parts[0]
        else:
            self._features = _Features(torch.cat([p.tok["embed"] for p in parts], 0),
                                       torch.cat([p.tok["s0"] for p in parts], 0),
                                       torch.cat([p.tok["s1"] for p in parts], 0), len(parts))
        self._is_image_set = True
        self._is_batch = True

    def get_image_embedding(self) -> torch.Tensor:
        if not self._is_image_set:
            raise RuntimeError("An image must be set with .set_image(...) to generate an embedding.")
        return self._features["image_embed"]

    # ------------------------------------------------------------------
    def _transform_coords(self, coords: torch.Tensor, normalize: bool, orig_hw) -> torch.Tensor:
        """SAM2Transforms.transform_coords: [..., 2] xy in original-image pixels with ``normalize`` (else already in
        [0, 1]) -> model-input pixels, in fp32 as upstream evaluates it."""
        if normalize:
            h, w = orig_hw
            coords = coords.clone()
            coords[..., 0] = coords[..., 0] / w
            coords[..., 1] = coords[..., 1] / h
        return coords * self.resolution

    def _prep_prompts(self, point_coords, point_labels, box, mask_logits, normalize_coords, img_idx=-1):
        """Upstream ``_prep_prompts``: numpy / tensor prompts -> device tensors in model-input pixels."""
        unnorm_coords, labels, unnorm_box, mask_input = None, None, None, None
        hw = self._orig_hw[img_idx]
        if point_coords is not None:
            assert point_labels is not None, "point_labels must be supplied if point_coords is supplied."
            coords = torch.as_tensor(point_coords, dtype=_F32).cpu()
            unnorm_coords = self._transform_coords(coords, normalize_coords, hw).to(self.device)
            labels = torch.as_tensor(point_labels, dtype=torch.int32).to(self.device)
            if unnorm_coords.dim() == 2:
                unnorm_coords, labels = unnorm_coords[None, ...], labels[None, ...]
        if box is not None:
            b = torch.as_tensor(box, dtype=_F32).cpu()
            unnorm_box = self._transform_coords(b.reshape(-1, 2, 2), normalize_coords, hw).to(self.device)  # Bx2x2
        if mask_logits is not None:
            mask_input = torch.as_tensor(mask_logits, dtype=_F32).to(self.device)
            if mask_input.dim() == 3:
                mask_input = mask_input[None, :, :, :]
        return mask_input, unnorm_coords, labels, unnorm_box

    @staticmethod
    def _to_numpy(masks, ious, low):
        # bool masks cross to the host as bytes and are widened there: a quarter of the fp32 copy
        m = masks.squeeze(0).cpu().numpy()
        return m.astype(np.float32) if m.dtype == np.bool_ else m, ious.squeeze(0).cpu().numpy(), low.squeeze(0).cpu().numpy()

    def predict(self, point_coords: Optional[np.ndarray] = None, point_labels: Optional[np.ndarray] = None,
                box: Optional[np.ndarray] = None, mask_input: Optional[np.ndarray] = None, multimask_output: bool = True,
                return_logits: bool = False, normalize_coords: bool = True):
        """Upstream ``SAM2ImagePredictor.predict``: point (xy + labels 1 / 0), box (xyxy) and mask (low-res logits
        [1, 256, 256]) prompts for the image of ``set_image``. N prompts come as [N, k, 2] / [N, k] points, [N, 4] boxes
        or [N, 1, 256, 256] masks. Returns float32 numpy (masks [C,H,W], ious [C], low-res logits [C,256,256]; with N > 1
        prompts [N,C,H,W], [N,C], [N,C,256,256]); C is 3 with ``multimask_output``, else 1."""
        if not self._is_image_set:
            raise RuntimeError("An image must be set with .set_image(...) before mask prediction.")
        mask_input, coords, labels, box = self._prep_prompts(point_coords, point_labels, box, mask_input,
                                                             normalize_coords)
        return self._to_numpy(*self._predict(coords, labels, box, mask_input, multimask_output,
                                             return_logits=return_logits))

    def predict_batch(self, point_coords_batch: Optional[List[np.ndarray]] = None,
                      point_labels_batch: Optional[List[np.ndarray]] = None, box_batch: Optional[List[np.ndarray]] = None,
                      mask_input_batch: Optional[List[np.ndarray]] = None, multimask_output: bool = True,
                      return_logits: bool = False, normalize_coords: bool = True):
        """Upstream ``SAM2ImagePredictor.predict_batch``: one prompt set per image of ``set_image_batch`` (each list,
        when given, has one entry per image, which may be None); returns three lists of ``predict``'s outputs."""
        assert self._is_batch, "This function should only be used when in batched mode"
        if not self._is_image_set:
            raise RuntimeError("An image must be set with .set_image_batch(...) before mask prediction.")
        num_images = self._features.batch
        for name, lst in (("point_coords_batch", point_coords_batch), ("point_labels_batch", point_labels_batch),
                          ("box_batch", box_batch), ("mask_input_batch", mask_input_batch)):
            assert lst is None or len(lst) == num_images, f"{name} must have one entry per image ({num_images})"
        all_masks, all_ious, all_low = [], [], []
        for img_idx in range(num_images):
            pick = (lambda lst: lst[img_idx] if lst is not None else None)
            mask_input, coords, labels, box = self._prep_prompts(pick(point_coords_batch), pick(point_labels_batch),
                                                                 pick(box_batch), pick(mask_input_batch),
                                                                 normalize_coords, img_idx=img_idx)
            m, i, low = self._to_numpy(*self._predict(coords, labels, box, mask_input, multimask_output,
                                                      return_logits=return_logits, img_idx=img_idx))
            all_masks.append(m)
            all_ious.append(i)
            all_low.append(low)
        return all_masks, all_ious, all_low

    @torch.no_grad()
    def _predict(self, point_coords: Optional[torch.Tensor], point_labels: Optional[torch.Tensor],
                 boxes: Optional[torch.Tensor] = None, mask_input: Optional[torch.Tensor] = None,
                 multimask_output: bool = True, return_logits: bool = False, img_idx: int = -1):
        """point_coords [B,Np,2] fp32 and boxes [B,4] / [B,2,2] (model-input pixels), point_labels [B,Np] int, mask_input
        [B,1,256,256] low-res logits (or one for all B prompts). Returns (masks, iou_predictions, low_res_masks) shaped
        like upstream: masks are the low-res logits bilinearly up-sampled to the original size, thresholded unless
        return_logits, in one kernel."""
        if not self._is_image_set:
            raise RuntimeError("An image must be set with .set_image(...) before mask prediction.")
        dec = self.model.decoder
        B = self._features.batch
        k = img_idx % B
        tok = self._features.tok
        emb = tok["embed"][k * 4096:(k + 1) * 4096]
        s0 = tok["s0"][k * 65536:(k + 1) * 65536]
        s1 = tok["s1"][k * 16384:(k + 1) * 16384]
        coords = None if point_coords is None else point_coords.to(self.device, _F32)
        labels = None if point_coords is None else point_labels.to(self.device, torch.int32)
        if boxes is not None:  # box corners go in front of the points, labelled 2 and 3 (upstream concat_points)
            bc = boxes.to(self.device, _F32).reshape(-1, 2, 2)
            bl = torch.tensor([[2, 3]], dtype=torch.int32, device=self.device).repeat(bc.shape[0], 1)
            coords = bc if coords is None else torch.cat([bc, coords], dim=1)
            labels = bl if labels is None else torch.cat([bl, labels], dim=1)
        mi = None
        if mask_input is not None:
            mi = mask_input.to(self.device, _F32).reshape(-1, 256, 256)
        if coords is None:  # no sparse prompt: the decoder runs on its 6 output tokens alone
            n = 1 if mi is None else mi.shape[0]
            tokens = dec.prompt_tokens(torch.zeros((n, 0, 2), dtype=_F32, device=self.device),
                                       torch.zeros((n, 0), dtype=torch.int32, device=self.device), pad=False)
        else:
            tokens = dec.prompt_tokens(coords.contiguous(), labels.contiguous())
        P = tokens.shape[0]
        if mi is not None:
            if mi.shape[0] != P:  # one mask for all prompts: upstream broadcasts its dense embedding
                assert mi.shape[0] == 1, f"{mi.shape[0]} mask inputs for {P} prompts"
                mi = mi.expand(P, 256, 256)
            mi = mi.contiguous()
        out = dec.forward(emb, s0, s1, tokens, mi, multimask_output=multimask_output)
        sel = None if multimask_output else out.get("sel_idx")
        cpp = 3 if multimask_output else 1
        if multimask_output:  # the planes upstream returns: tokens 1..3, the dynamic choice, or token 0
            low, ious = out["masks"][:, 1:4], out["ious"][:, 1:4]
        elif sel is not None:
            low, ious = out["masks"][torch.arange(P, device=self.device), sel.long()].unsqueeze(1), out["sel_iou"].unsqueeze(1)
        else:
            low, ious = out["masks"][:, 0:1], out["ious"][:, 0:1]
        H, W = self._orig_hw[k]
        up_in = out["masks"]
        if self.max_hole_area > 0 or self.max_sprinkle_area > 0:
            # the fill writes a separate buffer: low_res_masks (the m2m mask input) stay unfilled, as upstream returns them
            up_in = ops.amg_fill_lowres(out["masks"], out["ious"], sel, cpp, P * cpp, 0.0, self.mask_threshold,
                                        self.max_hole_area, self.max_sprinkle_area)
        masks = ops.upsample_select(up_in, sel, cpp, H, W, self.mask_threshold, logits=return_logits)
        low = low.clamp(-32.0, 32.0)
        return masks, ious, low
