"""B200 twin of REF saber/adapters/sam2/{predictor,automask,amg}.py — the SAM2 adapter SABER's segmenters
drive. Same class / method names and return types; the arithmetic underneath is the sm_100a kernel path.

* ``build_amg``                         REF saber/adapters/sam2/automask.py:49-86
* ``FilteredSAM2MaskGenerator``         REF saber/adapters/sam2/amg.py:139-201 (min/max area + relative box filters)
* ``SAM2Adapter.segment_image_2d``      REF saber/adapters/sam2/predictor.py:48-70
* ``SAM2Adapter.segment_image_2d_device`` resident variant (CUDA slice in, DeviceMasks out) used by the
  slice-wise segmenter so masks never leave the GPU.
"""
from __future__ import annotations

import os

from typing import Any, Dict, List, Optional

import numpy as np
import torch

from ..sam2.automatic_mask_generator import DeviceMasks, SAM2AutomaticMaskGenerator
from ..sam2.build_sam import build_sam2
from ..utils import preprocessing as prep
from .base import BaseAdapter, SAM2AdapterConfig, cfgAMG

_CFG_TO_ARCH = {"tiny": "tiny", "small": "small", "base": "base_plus", "large": "large"}


def filter_masks_by_area(anns: List[Dict[str, Any]], min_area: Optional[int] = None,
                         max_area: Optional[int] = None) -> List[Dict[str, Any]]:
    if min_area is None and max_area is None:
        return anns
    out = []
    for ann in anns:
        area = ann.get("area", 0)
        if (min_area is None or area >= min_area) and (max_area is None or area <= max_area):
            out.append(ann)
    return out


def filter_masks_by_relative_box_size(anns, max_rel_box_size=None, min_rel_box_size=None, image_height=None,
                                      image_width=None):
    if max_rel_box_size is None and min_rel_box_size is None:
        return anns
    if image_height is None or image_width is None:
        raise ValueError("image_height and image_width must be provided for relative size filtering")
    out = []
    for ann in anns:
        bbox = ann.get("bbox", None)
        if bbox is None:
            continue
        _, _, w, h = bbox
        rw, rh = w / image_width, h / image_height
        ok = True
        if max_rel_box_size is not None:
            ok = ok and rw < max_rel_box_size and rh < max_rel_box_size
        if min_rel_box_size is not None:
            ok = ok and rw > min_rel_box_size and rh > min_rel_box_size
        if ok:
            out.append(ann)
    return out


class FilteredSAM2MaskGenerator:
    def __init__(self, base_generator, min_rel_box_size=None, max_rel_box_size=None, min_area_filter=None,
                 max_area_filter=None):
        self.base_generator = base_generator
        self.max_rel_box_size = max_rel_box_size
        self.min_rel_box_size = min_rel_box_size
        self.min_area_filter = min_area_filter
        self.max_area_filter = max_area_filter

    def _filter(self, anns, hw):
        anns = filter_masks_by_relative_box_size(anns, self.max_rel_box_size, self.min_rel_box_size, hw[0], hw[1])
        return filter_masks_by_area(anns, self.min_area_filter, self.max_area_filter)

    def generate(self, image) -> List[Dict[str, Any]]:
        return self._filter(self.base_generator.generate(image), image.shape[:2])

    def generate_device(self, image):
        """Resident variant: (DeviceMasks, kept record list); each record carries ``index`` into the DeviceMasks."""
        dm = self.base_generator.generate_device(image)
        recs = self.base_generator.records(dm)
        for i, r in enumerate(recs):
            r["index"] = i
        return dm, self._filter(recs, dm.hw)

    def set_filters(self, min_rel_box_size=None, max_rel_box_size=None, min_area_filter=None):
        if min_rel_box_size is not None:
            self.min_rel_box_size = min_rel_box_size
        if max_rel_box_size is not None:
            self.max_rel_box_size = max_rel_box_size
        if min_area_filter is not None:
            self.min_area_filter = min_area_filter

    def __getattr__(self, name):
        return getattr(self.base_generator, name)


def build_amg(amg_params: Dict[str, Any], min_mask_area: int, device="cuda", checkpoint: Optional[str] = None,
              seed: int = 0, model=None, allow_random_init: bool = False):
    """REF saber/adapters/sam2/automask.py:49-86: build_sam2(apply_postprocessing=True) + AMG + area filter. The
    checkpoint is resolved as the reference does (pretrained_weights.get_sam2_checkpoint); a missing file raises unless
    random initialisation was allowed explicitly."""
    if model is None:
        model = build_sam2(_CFG_TO_ARCH[amg_params["sam2_cfg"]], checkpoint, device=device,
                           apply_postprocessing=True, seed=seed, allow_random_init=allow_random_init)
        model.eval()
    gen = SAM2AutomaticMaskGenerator(
        model=model, points_per_side=amg_params["npoints"], points_per_batch=amg_params["points_per_batch"],
        pred_iou_thresh=amg_params["pred_iou_thresh"], stability_score_thresh=amg_params["stability_score_thresh"],
        stability_score_offset=amg_params["stability_score_offset"], crop_n_layers=amg_params["crop_n_layers"],
        box_nms_thresh=amg_params["box_nms_thresh"],
        crop_n_points_downscale_factor=amg_params["crop_n_points_downscale_factor"],
        use_m2m=amg_params["use_m2m"], multimask_output=amg_params["multimask_output"])
    return FilteredSAM2MaskGenerator(base_generator=gen, min_area_filter=min_mask_area)


class SAM2Adapter(BaseAdapter):
    def __init__(self, config: SAM2AdapterConfig, device: str = "cuda"):
        if config.num_maskmem > 7:
            raise ValueError("num_maskmem must be less than 7")
        self._config = config
        self.device = torch.device(device)
        self.frame_metrics: Dict[int, Dict[int, Dict[str, Any]]] = {}
        self._vol_shape = None
        self.inference_state = None
        self._current_frame = None
        self._mask_generator = None
        self.predictor = None  # video predictor: built on first volume call
        # multi-GPU propagation (one process per GPU): "zslab" = frames and features stay on the rank that owns the
        # z-slab, the memory-bank halo is relayed to the neighbour (north_star); "objects" = features all-gathered,
        # tracked objects sharded over the ranks (round-1 scheme, kept for A/B measurements)
        self.prop_shard = os.environ.get("SB_PROP_SHARD", "zslab")
        self.relay_stats = None

    # ------------------------------------------------------------------ 2-D segmentation
    def _amg(self):
        if self._mask_generator is None:
            if self._config.amg_cfg is not None:
                amg_dict = self._config.amg_cfg.dict()
            else:
                amg_dict = cfgAMG(sam2_cfg=self._config.cfg).dict()
            self._mask_generator = build_amg(amg_dict, self._config.min_mask_area, device=self.device,
                                             checkpoint=self._config.checkpoint, seed=self._config.seed,
                                             allow_random_init=getattr(self._config, "allow_random_init", False))
        return self._mask_generator

    @torch.inference_mode()
    def segment_image_2d(self, image: np.ndarray, text_prompt: str = None, threshold: float = None):
        """REF :48-70: prepare (to RGB when the input is a grayscale slice; an (H,W,3) input keeps its channels) -> AMG."""
        out_rgb = True if image.ndim == 2 else False
        if image.ndim not in (2, 3) or (image.ndim == 3 and image.shape[2] != 3):
            raise ValueError("segment_image_2d expects an (H,W) slice or an (H,W,3) image")
        x = (image.to(self.device, torch.float32) if isinstance(image, torch.Tensor) else
             torch.from_numpy(np.ascontiguousarray(image, dtype=np.float32)).to(self.device))
        x = prep.prepare(x, to_rgb=out_rgb)
        return self._amg().generate(x)

    @torch.inference_mode()
    def segment_image_2d_device(self, image: torch.Tensor):
        """CUDA (H,W) slice -> (DeviceMasks, filtered record list); nothing but the records leaves the GPU."""
        assert image.is_cuda and image.dim() == 2
        x = prep.prepare_device(image)
        return self._amg().generate_device(x)

    # ------------------------------------------------------------------ 3-D (z-axis memory propagation)
    def _video(self):
        """Video predictor built on first use (REF saber/adapters/sam2/predictor.py:24-34 builds it in __init__; the
        slice-wise path never needs it). maskmem_tpos_enc is truncated and num_maskmem set exactly as the reference."""
        if self.predictor is None:
            from ..sam2.sam2_video_predictor import build_sam2_video_predictor
            p = build_sam2_video_predictor(_CFG_TO_ARCH[self._config.cfg], self._config.checkpoint, device=self.device,
                                           vos_optimized=False, seed=self._config.seed,
                                           allow_random_init=getattr(self._config, "allow_random_init", False))
            maskmem = p.maskmem_tpos_enc[:self._config.num_maskmem]
            p.maskmem_tpos_enc = torch.nn.Parameter(maskmem, requires_grad=False)
            p.num_maskmem = self._config.num_maskmem
            self.predictor = p
        return self.predictor

    @torch.inference_mode()
    def set_volume(self, tomogram, offload_video_to_cpu: bool = False) -> None:
        """REF :76-84. `tomogram`: numpy (Z,Y,X) or a CUDA tensor (stays on the device)."""
        self._vol_shape = tuple(tomogram.shape)
        self.frame_metrics = {}
        self.inference_state = self.create_inference_state_from_tomogram(tomogram)

    @torch.inference_mode()
    def create_inference_state_from_tomogram(self, tomogram, offload_video_to_cpu: bool = False,
                                             offload_state_to_cpu: bool = False) -> Dict[str, Any]:
        """REF :90-116 with TomogramPreprocessor (REF saber/adapters/preprocessing.py:16-76) on the device:
        global min-max to [-1,1], per-slice skimage-style resize to 1024^2, `2x - 1`. The three RGB channels are
        identical, so `images` is a stride-0 view [Z,3,S,S] of one [Z,S,S] plane stack (3x less HBM than the
        reference's materialised tensor). Every frame is encoded here, once, in batches (Phase A)."""
        from .. import ops
        p = self._video()
        vol = (tomogram if isinstance(tomogram, torch.Tensor) else
               torch.from_numpy(np.ascontiguousarray(tomogram, dtype=np.float32)))
        vol = vol.to(self.device, dtype=torch.float32).contiguous()
        mm = ops.minmax(vol)
        vol = ops.minmax_affine(vol, mm, 0.0, 2.0, -1.0)  # normalize_tomogram
        S = p.image_size
        planes = ops.skimage_resize_stack(vol, S, 2.0, -1.0)  # load_grayscale_image_array: resize, then 2*x - 1
        del vol
        if self._config.light_modality:  # REF adapters/preprocessing.py:66-68: rescale the frames to [0, 255]
            planes = ops.minmax_affine(planes, ops.minmax(planes), 0.0, 255.0, 0.0)
        images = planes[:, None].expand(-1, 3, -1, -1)
        state = self._create_empty_inference_state(images, S, S, offload_video_to_cpu, offload_state_to_cpu)
        from .. import dist as sbdist
        world, rank = sbdist.world_rank()
        if world == 1:
            p.encode_frames(state)
        else:  # Phase A (SURVEY §8e): every rank encodes its z-slab once, then the cached features are exchanged
            z0, z1 = sbdist.zslab_range(len(images), rank, world)
            p.encode_frames(state, list(range(z0, z1)))
            if 0 not in range(z0, z1):
                state["cached_features"].pop(0, None)  # frame 0 was warmed above on every rank; slab owner is authoritative
            if self.prop_shard != "zslab":  # object sharding: every rank needs every frame
                sbdist.exchange_frame_features(state["cached_features"], len(images))
        return state

    def _create_empty_inference_state(self, images, video_height, video_width, offload_video_to_cpu=False,
                                      offload_state_to_cpu=False) -> Dict[str, Any]:
        """REF :118-154 (same keys); the state lives on the adapter's device."""
        return self._video().new_inference_state(images, video_height, video_width, offload_video_to_cpu,
                                                 offload_state_to_cpu, self.device, self.device)

    def add_new_mask(self, frame_idx: int, obj_id: int, mask, inference_state=None):
        state = inference_state or self.inference_state
        return self._video().add_new_mask(inference_state=state, frame_idx=frame_idx, obj_id=obj_id, mask=mask)

    def add_new_points_or_box(self, frame_idx: int, obj_id: int, inference_state=None, **kwargs):
        state = inference_state or self.inference_state
        return self._video().add_new_points_or_box(inference_state=state, frame_idx=frame_idx, obj_id=obj_id, **kwargs)

    @torch.inference_mode()
    def propagate_in_video(self, start_frame_idx, max_frame_num_to_track=None, reverse=False, inference_state=None):
        """REF :186-206: yields (frame_idx, obj_ids, low_res_masks, video_res_masks, obj_scores=None)."""
        state = inference_state or self.inference_state
        for frame_idx, obj_ids, logits in self._video().propagate_in_video(
                state, start_frame_idx=start_frame_idx, max_frame_num_to_track=max_frame_num_to_track, reverse=reverse):
            yield frame_idx, obj_ids, logits, logits, None

    @staticmethod
    def _normalize_masks(masks) -> List[Any]:
        """REF :208-230; CUDA tensors are kept on the device (the seed masks of the resident path)."""
        if masks is None:
            return []
        if isinstance(masks, torch.Tensor):
            return [masks[i].squeeze() for i in range(masks.shape[0])]
        if isinstance(masks, np.ndarray) and masks.ndim >= 3:
            return [np.squeeze(masks[i]).astype(np.float32) for i in range(masks.shape[0])]
        out = []
        for m in masks:
            if isinstance(m, dict):
                m = m["segmentation"]
            out.append(m.squeeze() if isinstance(m, torch.Tensor) else np.squeeze(np.asarray(m)).astype(np.float32))
        return out

    @torch.inference_mode()
    def segment_volume_device(self, start_frame_idx: int, masks=None, vol_shape=None, max_frame_num_to_track=None,
                              min_presence_score: float = 0.5, inference_state=None, group=None) -> torch.Tensor:
        """REF :232-348 with the label volume kept on the device: returns CUDA int16 (uint16 payload) [Z,H,W].
        Under torch.distributed (one process per GPU) the tracked objects are sharded over the ranks (object k ->
        rank k % world); label volumes are merged with an element-wise max (= "higher object id wins") after each
        pass and the hook log is merged into the single-process order, so every rank returns the same volume as a
        single GPU would."""
        from .. import dist as sbdist
        from .. import ops
        from ..filters import estimate_thickness
        world, rank = sbdist.world_rank(group)
        state = inference_state or self.inference_state
        if state is None:
            raise RuntimeError("Call set_volume() before segment_volume().")
        if vol_shape is None:
            vol_shape = self._vol_shape
        if vol_shape is None:
            raise RuntimeError("vol_shape required when inference_state is passed explicitly.")
        Z, H, W = vol_shape
        p = self._video()
        mask_list = self._normalize_masks(masks)
        if world > 1 and self.prop_shard == "zslab":
            return self._segment_volume_relay(start_frame_idx, mask_list, (Z, H, W), max_frame_num_to_track,
                                              min_presence_score, state, group)
        k = 0  # index among the non-empty seeds (the objects that are actually tracked)
        n_local = 0
        for obj_id, mask in enumerate(mask_list, start=1):
            if float(mask.max()) == 0:
                continue
            if k % world == rank:
                self.add_new_mask(frame_idx=start_frame_idx, obj_id=obj_id, mask=mask, inference_state=state)
                n_local += 1
            k += 1
        self._current_frame = None
        captured: Dict[Any, list] = {}

        # The reference registers a forward hook that copies output[3] to the host on every decoder call (REF :277-284):
        # one synchronisation per object and frame. Same bookkeeping here (scores filed under `_current_frame` at call
        # time, incl. the off-by-one of SURVEY 3.3), but the score tensors stay on the device until both passes are done.
        pending = []  # (frame key at call time, device tensor [B,1])
        p.sam_mask_decoder.device_sink = lambda scores: pending.append((self._current_frame, scores.clone()))
        self.frame_metrics = {}
        vol_masks = torch.zeros((Z, H, W), dtype=torch.int16, device=self.device)

        def _apply(frame_idx, obj_ids, mask_logits):
            ids = torch.tensor([int(o) for o in obj_ids], dtype=torch.int32, device=self.device)
            ops.stitch_objects_(mask_logits[:, 0].contiguous(), ids, vol_masks[frame_idx])

        def _frames(reverse):
            """Frame schedule of one pass; a rank without objects still walks it (its hook log stays empty)."""
            if n_local > 0:
                yield from self.propagate_in_video(start_frame_idx=start_frame_idx,
                                                   max_frame_num_to_track=max_frame_num_to_track, reverse=reverse,
                                                   inference_state=state)

        for frame_idx, obj_ids, mask_logits, _, _ in _frames(False):
            self._current_frame = frame_idx
            _apply(frame_idx, obj_ids, mask_logits)
        # which slices the forward pass filled ON ANY RANK: a Z-element flag vector crosses the ranks, not the label volume
        # (round 1 all-reduced the whole volume here and again after the backward pass)
        nonempty = sbdist.allreduce_any(ops.slice_any(vol_masks), group).cpu().numpy()  # one D2H of Z flags
        for frame_idx, obj_ids, mask_logits, _, _ in _frames(True):
            self._current_frame = frame_idx
            if not nonempty[frame_idx]:
                _apply(frame_idx, obj_ids, mask_logits)
        sbdist.allreduce_max_labels(vol_masks, group)
        p.sam_mask_decoder.device_sink = None
        for key, scores in pending:  # one D2H per call group, after the fact; per-object order as the hook would see it
            host = scores.to(torch.float32).cpu().numpy()
            for i in range(host.shape[0]):
                captured.setdefault(key, []).append(host[i:i + 1])
        if world > 1:
            import torch.distributed as tdist
            logs = [None] * world
            tdist.all_gather_object(logs, ({f: [float(v) for s_ in sc for v in s_.flatten()] for f, sc in captured.items()},
                                           n_local), group=group)
            merged = sbdist.merge_captured_scores([l[0] for l in logs], [l[1] for l in logs])
            captured = {f: [np.asarray(v, dtype=np.float32)] for f, v in merged.items()}
        nMasks = len(mask_list)
        self.frame_scores = np.zeros([Z, nMasks])
        if nMasks > 0:
            for fidx, scores in captured.items():
                if fidx is None:
                    continue
                vals = np.concatenate([s.flatten() for s in scores])
                n = min(len(vals), nMasks)
                self.frame_scores[fidx, :n] = vals[:n]
            bounds = estimate_thickness.fit_organelle_boundaries(self.frame_scores, plot=False)
            for fidx in range(Z):
                self.frame_metrics[fidx] = {}
                for mi in range(nMasks):
                    ps = float(bounds[fidx, mi])
                    self.frame_metrics[fidx][mi + 1] = {"presence_score": ps}
                    if ps < min_presence_score:
                        ops.erase_label_(vol_masks[fidx], mi + 1)
        return vol_masks

    def _presence_filter(self, vol_masks, captured, n_masks, Z, min_presence_score):
        """REF :300-348: per-frame object scores -> fitted presence curves -> labels below the threshold erased."""
        from .. import ops
        from ..filters import estimate_thickness
        self.frame_scores = np.zeros([Z, n_masks])
        if n_masks > 0:
            for fidx, scores in captured.items():
                if fidx is None:
                    continue
                vals = np.concatenate([np.asarray(s_, dtype=np.float32).flatten() for s_ in scores])
                n = min(len(vals), n_masks)
                self.frame_scores[fidx, :n] = vals[:n]
            bounds = estimate_thickness.fit_organelle_boundaries(self.frame_scores, plot=False)
            for fidx in range(Z):
                self.frame_metrics[fidx] = {}
                for mi in range(n_masks):
                    ps = float(bounds[fidx, mi])
                    self.frame_metrics[fidx][mi + 1] = {"presence_score": ps}
                    if ps < min_presence_score:
                        ops.erase_label_(vol_masks[fidx], mi + 1)
        return vol_masks

    def _segment_volume_relay(self, start, mask_list, vol_shape, max_frame_num_to_track, min_presence_score, state, group):
        """segment_volume with the frames sharded by z-slab (saber_b200/dist.py relay_propagate): this rank holds the
        features of its own slab only, tracks only its own frames, and the memory-bank halo (~0.5 MB per object) is
        handed to the neighbouring rank at each slab boundary; label slabs are all-gathered at the end. Every rank
        returns the single-GPU label volume, bit for bit."""
        import torch.distributed as tdist
        from .. import dist as sbdist
        from .. import ops
        if max_frame_num_to_track is not None:
            raise NotImplementedError("z-slab relay tracks the whole volume (max_frame_num_to_track=None)")
        world, rank = sbdist.world_rank(group)
        Z, H, W = vol_shape
        p = self._video()
        obj_ids = [oid for oid, m in enumerate(mask_list, start=1) if float(m.max()) != 0]
        self._current_frame = None
        self._relay_pass = 0
        pending = []  # (pass, frame key at call time, device scores [B,1])
        p.sam_mask_decoder.device_sink = lambda sc: pending.append((self._relay_pass, self._current_frame, sc.clone()))
        self.frame_metrics = {}
        vol_masks = torch.zeros((Z, H, W), dtype=torch.int16, device=self.device)
        nonempty = {}

        def seed_fn():
            for oid in obj_ids:
                self.add_new_mask(frame_idx=start, obj_id=oid, mask=mask_list[oid - 1], inference_state=state)

        def set_key(k, pass_id):
            self._current_frame = k
            self._relay_pass = pass_id

        def on_frame(pass_id, frame_idx, ids, logits):
            if pass_id == 1 and frame_idx not in nonempty:  # only the seed slice can have been filled by the forward pass
                nonempty[frame_idx] = bool(ops.slice_any(vol_masks[frame_idx:frame_idx + 1]).item()) if frame_idx == start else False
            if pass_id == 0 or not nonempty[frame_idx]:
                idt = torch.tensor([int(o) for o in ids], dtype=torch.int32, device=self.device)
                ops.stitch_objects_(logits[:, 0].contiguous(), idt, vol_masks[frame_idx])

        stats = {"bytes_sent": 0, "frames": 0}
        if obj_ids:
            stats = sbdist.relay_propagate(p, state, obj_ids, start, Z, seed_fn, on_frame, set_key, self.device, group)
        p.sam_mask_decoder.device_sink = None
        sbdist.allgather_label_slabs(vol_masks, Z, group)
        mine = [(ps, key, [float(v) for v in sc.to(torch.float32).cpu().numpy().flatten()]) for ps, key, sc in pending]
        logs = [None] * world
        tdist.all_gather_object(logs, mine, group=group)
        captured: Dict[Any, list] = {}
        for ps in (0, 1):  # single-process order: forward-pass calls first, then the backward pass; a (pass, key) pair
            for r in range(world):  # lives on exactly one rank
                for q, key, vals in logs[r]:
                    if q == ps:
                        captured.setdefault(key, []).extend(np.asarray([v], dtype=np.float32) for v in vals)
        self.relay_stats = stats
        return self._presence_filter(vol_masks, captured, len(mask_list), Z, min_presence_score)

    @torch.inference_mode()
    def segment_volume(self, start_frame_idx: int, masks=None, vol_shape=None, max_frame_num_to_track=None,
                       min_presence_score: float = 0.5, inference_state=None) -> np.ndarray:
        """REF :232-348: bidirectional propagation with hook-captured presence scores -> (Z,H,W) uint16."""
        v = self.segment_volume_device(start_frame_idx, masks, vol_shape, max_frame_num_to_track, min_presence_score,
                                       inference_state)
        return v.cpu().numpy().view(np.uint16)

    def reset_state(self, inference_state=None) -> None:
        state = inference_state or self.inference_state
        if state is not None and self.predictor is not None:
            self.predictor.reset_state(state)

    def clear_all_prompts_in_frame(self, *args, **kwargs):
        return self._video().clear_all_prompts_in_frame(*args, **kwargs)

    def remove_object(self, *args, **kwargs):
        return self._video().remove_object(*args, **kwargs)
