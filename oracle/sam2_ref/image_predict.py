"""ORACLE (test infrastructure only). Restatement of upstream sam2/sam2_image_predictor.py's interactive surface, which
the restatement in image_predictor.py (the set_image / _predict pair SABER's path uses) stops short of:

* ``SAM2Transforms.transform_boxes``, and ``postprocess_masks`` with max_hole_area / max_sprinkle_area above 0, the fill
  being small_regions.fill_holes_and_sprinkles (scipy labelling in place of get_connected_components);
* ``SAM2ImagePredictor._prep_prompts``, ``predict``, ``predict_batch``, and ``_predict`` with box prompts (box corners
  merged in front of the points with labels 2 and 3).

Everything else (the image transform, set_image / set_image_batch, the features) is image_predictor.py's.
"""
from __future__ import annotations

import torch

from . import image_predictor as base
from .small_regions import fill_holes_and_sprinkles


class SAM2Transforms(base.SAM2Transforms):
    def transform_boxes(self, boxes, normalize=False, orig_hw=None):
        return self.transform_coords(boxes.reshape(-1, 2, 2), normalize, orig_hw)

    def postprocess_masks(self, masks, orig_hw):
        masks = masks.float()
        if self.max_hole_area > 0 or self.max_sprinkle_area > 0:
            masks = fill_holes_and_sprinkles(masks, self.mask_threshold, self.max_hole_area, self.max_sprinkle_area)
        return super().postprocess_masks(masks, orig_hw)


class SAM2ImagePredictor(base.SAM2ImagePredictor):
    def __init__(self, sam_model, mask_threshold=0.0, max_hole_area=0.0, max_sprinkle_area=0.0):
        super().__init__(sam_model, mask_threshold, max_hole_area, max_sprinkle_area)
        self._transforms = SAM2Transforms(self.model.image_size, mask_threshold, max_hole_area, max_sprinkle_area)

    def predict(self, point_coords=None, point_labels=None, box=None, mask_input=None, multimask_output=True,
                return_logits=False, normalize_coords=True):
        if not self._is_image_set:
            raise RuntimeError("An image must be set with .set_image(...) before mask prediction.")
        mask_input, unnorm_coords, labels, unnorm_box = self._prep_prompts(point_coords, point_labels, box, mask_input,
                                                                           normalize_coords)
        masks, iou_predictions, low_res_masks = self._predict(unnorm_coords, labels, unnorm_box, mask_input,
                                                              multimask_output, return_logits=return_logits)
        return (masks.squeeze(0).float().detach().cpu().numpy(), iou_predictions.squeeze(0).float().detach().cpu().numpy(),
                low_res_masks.squeeze(0).float().detach().cpu().numpy())

    def _prep_prompts(self, point_coords, point_labels, box, mask_logits, normalize_coords, img_idx=-1):
        unnorm_coords, labels, unnorm_box, mask_input = None, None, None, None
        if point_coords is not None:
            assert point_labels is not None, "point_labels must be supplied if point_coords is supplied."
            point_coords = torch.as_tensor(point_coords, dtype=torch.float, device=self.device)
            unnorm_coords = self._transforms.transform_coords(point_coords, normalize=normalize_coords,
                                                              orig_hw=self._orig_hw[img_idx])
            labels = torch.as_tensor(point_labels, dtype=torch.int, device=self.device)
            if len(unnorm_coords.shape) == 2:
                unnorm_coords, labels = unnorm_coords[None, ...], labels[None, ...]
        if box is not None:
            box = torch.as_tensor(box, dtype=torch.float, device=self.device)
            unnorm_box = self._transforms.transform_boxes(box, normalize=normalize_coords,
                                                          orig_hw=self._orig_hw[img_idx])  # Bx2x2
        if mask_logits is not None:
            mask_input = torch.as_tensor(mask_logits, dtype=torch.float, device=self.device)
            if len(mask_input.shape) == 3:
                mask_input = mask_input[None, :, :, :]
        return mask_input, unnorm_coords, labels, unnorm_box

    def predict_batch(self, point_coords_batch=None, point_labels_batch=None, box_batch=None, mask_input_batch=None,
                      multimask_output=True, return_logits=False, normalize_coords=True):
        assert self._is_batch, "This function should only be used when in batched mode"
        if not self._is_image_set:
            raise RuntimeError("An image must be set with .set_image_batch(...) before mask prediction.")
        num_images = len(self._features["image_embed"])
        all_masks, all_ious, all_low_res_masks = [], [], []
        for img_idx in range(num_images):
            point_coords = point_coords_batch[img_idx] if point_coords_batch is not None else None
            point_labels = point_labels_batch[img_idx] if point_labels_batch is not None else None
            box = box_batch[img_idx] if box_batch is not None else None
            mask_input = mask_input_batch[img_idx] if mask_input_batch is not None else None
            mask_input, unnorm_coords, labels, unnorm_box = self._prep_prompts(point_coords, point_labels, box,
                                                                               mask_input, normalize_coords,
                                                                               img_idx=img_idx)
            masks, iou_predictions, low_res_masks = self._predict(unnorm_coords, labels, unnorm_box, mask_input,
                                                                  multimask_output, return_logits=return_logits,
                                                                  img_idx=img_idx)
            all_masks.append(masks.squeeze(0).float().detach().cpu().numpy())
            all_ious.append(iou_predictions.squeeze(0).float().detach().cpu().numpy())
            all_low_res_masks.append(low_res_masks.squeeze(0).float().detach().cpu().numpy())
        return all_masks, all_ious, all_low_res_masks

    @torch.no_grad()
    def _predict(self, point_coords, point_labels, boxes=None, mask_input=None, multimask_output=True,
                 return_logits=False, img_idx=-1):
        if not self._is_image_set:
            raise RuntimeError("An image must be set with .set_image(...) before mask prediction.")
        concat_points = (point_coords, point_labels) if point_coords is not None else None
        if boxes is not None:  # box corners go in front of the points (upstream merges them into concat_points)
            box_coords = boxes.reshape(-1, 2, 2)
            box_labels = torch.tensor([[2, 3]], dtype=torch.int, device=boxes.device).repeat(boxes.size(0), 1)
            if concat_points is not None:
                concat_points = (torch.cat([box_coords, concat_points[0]], dim=1),
                                 torch.cat([box_labels, concat_points[1]], dim=1))
            else:
                concat_points = (box_coords, box_labels)
        sparse, dense = self.model.sam_prompt_encoder(points=concat_points, boxes=None, masks=mask_input)
        batched_mode = concat_points is not None and concat_points[0].shape[0] > 1
        high_res = [lvl[img_idx].unsqueeze(0) for lvl in self._features["high_res_feats"]]
        low_res_masks, iou_predictions, _, _ = self.model.sam_mask_decoder(
            image_embeddings=self._features["image_embed"][img_idx].unsqueeze(0),
            image_pe=self.model.sam_prompt_encoder.get_dense_pe(),
            sparse_prompt_embeddings=sparse, dense_prompt_embeddings=dense,
            multimask_output=multimask_output, repeat_image=batched_mode, high_res_features=high_res)
        masks = self._transforms.postprocess_masks(low_res_masks, self._orig_hw[img_idx])
        low_res_masks = torch.clamp(low_res_masks, -32.0, 32.0)
        if not return_logits:
            masks = masks > self.mask_threshold
        return masks, iou_predictions, low_res_masks
