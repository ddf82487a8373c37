"""Drop-in for ``sam2.automatic_mask_generator.SAM2AutomaticMaskGenerator`` on the B200 kernels.

Binding site in the reference: REF saber/adapters/sam2/automask.py:66-78 (constructor keywords) and
REF saber/adapters/sam2/amg.py:163 (``generate(image) -> list[dict]`` with keys segmentation, area,
bbox, predicted_iou, point_coords, stability_score, crop_box). Restates upstream
sam2/automatic_mask_generator.py + sam2/utils/amg.py (SURVEY §3.4 / §8a U5).

B200 design: the whole image — all crops, both decoder passes, the integer post-processing, per-crop
NMS and the cross-crop NMS — runs device-resident on one stream without a host synchronisation.
Every candidate mask owns a fixed *slot* (crop-major, point-major, mask-minor: upstream's
concatenation order); kernels write per-slot records (keep flag, IoU, stability, box, area) and
bit-packed full-frame masks; candidate lists and their lengths stay in device memory. The fp32
full-resolution logits upstream materialises per batch never exist. One synchronisation at the end
fetches the survivor count. With ``min_mask_region_area > 0`` the decoder planes are hole / sprinkle filled on the
device before the post-processing (inside the captured graphs), and the survivors go through upstream's
postprocess_small_regions on their packed masks, with a second synchronisation for the new count. With
``output_mode`` "uncompressed_rle" / "coco_rle" the survivors are run-length encoded on the device and only the encodings
are copied to the host; "binary_mask" unpacks them to dense bool masks.
"""
from __future__ import annotations

import math
import os
from dataclasses import dataclass
from itertools import product
from typing import Any, Dict, List, Optional, Tuple

import numpy as np
import torch

from .. import ops
from .sam2_image_predictor import SAM2ImagePredictor

_F32, _I32, _U8 = torch.float32, torch.int32, torch.uint8


# ---------------------------------------------------------------------------------------------
# geometry (host, float64 numpy exactly as upstream sam2/utils/amg.py evaluates it)
# ---------------------------------------------------------------------------------------------
def build_point_grid(n_per_side: int) -> np.ndarray:
    offset = 1 / (2 * n_per_side)
    side = np.linspace(offset, 1 - offset, n_per_side)
    xs = np.tile(side[None, :], (n_per_side, 1))
    ys = np.tile(side[:, None], (1, n_per_side))
    return np.stack([xs, ys], axis=-1).reshape(-1, 2)


def build_all_layer_point_grids(n_per_side: int, n_layers: int, scale_per_layer: int) -> List[np.ndarray]:
    return [build_point_grid(int(n_per_side / (scale_per_layer ** i))) for i in range(n_layers + 1)]


def generate_crop_boxes(im_size: Tuple[int, int], n_layers: int, overlap_ratio: float):
    im_h, im_w = im_size
    short = min(im_h, im_w)
    boxes, layers = [[0, 0, im_w, im_h]], [0]
    for layer in range(n_layers):
        per_side = 2 ** (layer + 1)
        overlap = int(overlap_ratio * short * (2 / per_side))
        cw = int(math.ceil((overlap * (per_side - 1) + im_w) / per_side))
        ch = int(math.ceil((overlap * (per_side - 1) + im_h) / per_side))
        xs = [int((cw - overlap) * i) for i in range(per_side)]
        ys = [int((ch - overlap) * i) for i in range(per_side)]
        for x0, y0 in product(xs, ys):
            boxes.append([x0, y0, min(x0 + cw, im_w), min(y0 + ch, im_h)])
            layers.append(layer + 1)
    return boxes, layers


@dataclass
class _CropPlan:
    box: Tuple[int, int, int, int]
    layer: int
    base: int                 # first slot of this crop
    n_points: int
    points_crop: torch.Tensor   # [n,2] fp32 host: grid * (Wc, Hc), crop frame (upstream data["points"] before uncrop)
    points_full: torch.Tensor   # [n,2] fp32 host: uncrop_points
    in_points: torch.Tensor     # [n,1,2] fp32 device: model-input pixel coordinates
    labels: torch.Tensor        # [n,1] int32 device (ones)
    geom_dev: torch.Tensor = None  # [n_batches, 8] int32 device: (Hc, Wc, x0, y0, slot base of the batch, 0, 0, 0)


@dataclass
class _ImagePlan:
    hw: Tuple[int, int]
    crops: List[_CropPlan]
    crops_dev: torch.Tensor     # [ncrops,4] int32 device
    n_slots: int
    cpp: int                    # candidate masks per point
    score2: torch.Tensor        # [n_slots] fp32 device: 1 / crop area (cross-crop NMS score)
    slot_crop: np.ndarray       # [n_slots] crop index of each slot


@dataclass
class DeviceMasks:
    """AMG result kept on the device: survivors in upstream's output order."""
    hw: Tuple[int, int]
    count: int
    slots: torch.Tensor         # [m] int32 slot ids
    bits: torch.Tensor          # [m, H, ceil(W/32)] int32 packed masks
    bbox: torch.Tensor          # [m,4] int32 xyxy (inclusive max)
    area: torch.Tensor          # [m] int32
    iou: torch.Tensor           # [m] fp32
    stability: torch.Tensor     # [m] fp32
    plan: Any = None


class SAM2AutomaticMaskGenerator:
    def __init__(self, model, points_per_side: Optional[int] = 32, points_per_batch: int = 64,
                 pred_iou_thresh: float = 0.8, stability_score_thresh: float = 0.95,
                 stability_score_offset: float = 1.0, mask_threshold: float = 0.0, box_nms_thresh: float = 0.7,
                 crop_n_layers: int = 0, crop_nms_thresh: float = 0.7, crop_overlap_ratio: float = 512 / 1500,
                 crop_n_points_downscale_factor: int = 1, point_grids: Optional[List[np.ndarray]] = None,
                 min_mask_region_area: int = 0, output_mode: str = "binary_mask", use_m2m: bool = False,
                 multimask_output: bool = True, **kwargs) -> None:
        if (points_per_side is None) == (point_grids is None):
            raise ValueError("Exactly one of points_per_side or point_grid must be provided.")
        if output_mode not in ("binary_mask", "uncompressed_rle", "coco_rle"):
            raise ValueError(f"Unknown output_mode {output_mode}.")
        self.point_grids = (build_all_layer_point_grids(points_per_side, crop_n_layers, crop_n_points_downscale_factor)
                            if point_grids is None else point_grids)
        self.predictor = SAM2ImagePredictor(model, max_hole_area=min_mask_region_area,
                                            max_sprinkle_area=min_mask_region_area)
        self.points_per_batch = points_per_batch
        self.pred_iou_thresh = pred_iou_thresh
        self.stability_score_thresh = stability_score_thresh
        self.stability_score_offset = stability_score_offset
        self.mask_threshold = mask_threshold
        self.box_nms_thresh = box_nms_thresh
        self.crop_n_layers = crop_n_layers
        self.crop_nms_thresh = crop_nms_thresh
        self.crop_overlap_ratio = crop_overlap_ratio
        self.crop_n_points_downscale_factor = crop_n_points_downscale_factor
        self.min_mask_region_area = min_mask_region_area
        self.output_mode = output_mode
        self.use_m2m = use_m2m
        self.multimask_output = multimask_output
        # candidates per m2m decoder call (multiple of 3 so whole prompts stay together); results do not depend on it
        # Execution batch: `points_per_batch` is upstream's memory knob (64 points -> 192 m2m prompts per decoder call); the
        # results do not depend on it, and each decoder call costs ~100 latency-bound token-side launches, so the B200 path
        # runs SB_AMG_BATCH_MULT x points_per_batch points per call where a crop has that many (180 GB of HBM).
        self.exec_ppb = points_per_batch * max(1, int(os.environ.get("SB_AMG_BATCH_MULT", "2")))
        self.m2m_batch = 3 * self.exec_ppb
        # test hook: when a list, every post-processing call appends (crop, base, n, cpp, planes, ious4, sel) host copies
        self.capture: Optional[list] = None
        self.capture_compact = False
        self.use_cuda_graph = True
        # independent prompt batches in flight (one CUDA graph instance + stream each)
        self.graph_lanes = int(os.environ.get("SB_GRAPH_LANES", "4"))
        # m2m pass: skip the mask up-scaling of prompts whose predicted IoUs cannot pass pred_iou_thresh (results are
        # identical: upstream computes those masks and then drops them unseen); SB_M2M_GATE=0 computes everything
        self.m2m_gate = os.environ.get("SB_M2M_GATE", "1") != "0"
        self.phase_ms: Optional[Dict[str, float]] = None  # set to {} to accumulate encode / decode+post / total ms
        self._graphs: Dict[Tuple[int, int], Any] = {}
        self._plans: Dict[Tuple[int, int], _ImagePlan] = {}
        self._ws: Dict[Tuple[int, int], Dict[str, torch.Tensor]] = {}

    @property
    def device(self):
        return self.predictor.device

    # ------------------------------------------------------------------
    def _plan(self, hw: Tuple[int, int]) -> _ImagePlan:
        if hw in self._plans:
            return self._plans[hw]
        H, W = hw
        dev = self.device
        res = float(self.predictor.resolution)
        boxes, layers = generate_crop_boxes(hw, self.crop_n_layers, self.crop_overlap_ratio)
        cpp = 3 if self.multimask_output else 1
        crops, base = [], 0
        for box, layer in zip(boxes, layers):
            x0, y0, x1, y1 = box
            wc, hc = x1 - x0, y1 - y0
            pts64 = self.point_grids[layer] * np.array([hc, wc])[None, ::-1]
            pts = torch.as_tensor(pts64, dtype=_F32)
            inp = pts.clone()
            inp[..., 0] = inp[..., 0] / wc
            inp[..., 1] = inp[..., 1] / hc
            inp = inp * res
            full = pts + torch.tensor([[x0, y0]])
            n = pts.shape[0]
            ppb = self.exec_ppb
            geom = torch.tensor([[hc, wc, x0, y0, base + b0 * cpp, 0, 0, 0] for b0 in range(0, n, ppb)], dtype=_I32)
            crops.append(_CropPlan(tuple(box), layer, base, n, pts, full,
                                   inp[:, None, :].contiguous().to(dev),
                                   torch.ones((n, 1), dtype=_I32, device=dev), geom.to(dev)))
            base += n * cpp
        cb = torch.tensor(boxes, dtype=_F32)
        crop_score = 1 / ((cb[:, 2] - cb[:, 0]) * (cb[:, 3] - cb[:, 1]))
        slot_crop = np.concatenate([np.full(c.n_points * cpp, i, dtype=np.int64) for i, c in enumerate(crops)])
        plan = _ImagePlan(hw, crops, torch.tensor(boxes, dtype=_I32, device=dev), base, cpp,
                          crop_score[torch.from_numpy(slot_crop)].contiguous().to(dev), slot_crop)
        self._plans[hw] = plan
        return plan

    def _workspace(self, plan: _ImagePlan) -> Dict[str, torch.Tensor]:
        if plan.hw in self._ws:
            return self._ws[plan.hw]
        H, W = plan.hw
        N, dev = plan.n_slots, self.device
        nmax = max(N, 64)
        ws = dict(
            keep=torch.zeros((N,), dtype=_U8, device=dev), stab=torch.zeros((N,), dtype=_F32, device=dev),
            iou=torch.zeros((N,), dtype=_F32, device=dev), bbox=torch.zeros((N, 4), dtype=_I32, device=dev),
            area=torch.zeros((N,), dtype=_I32, device=dev),
            bits=torch.empty((N, H, (W + 31) // 32), dtype=_I32, device=dev),
            cand=torch.empty((nmax,), dtype=_I32, device=dev), order=torch.empty((nmax,), dtype=_I32, device=dev),
            nms_mask=torch.empty((nmax * ((nmax + 63) // 64),), dtype=torch.int64, device=dev),
            list1=torch.empty((nmax,), dtype=_I32, device=dev), list2=torch.empty((nmax,), dtype=_I32, device=dev),
            counts=torch.zeros((4,), dtype=_I32, device=dev),  # [cand, list1, list2, small-region survivors]
        )
        if self.min_mask_region_area > 0:
            ws.update(region_box=torch.zeros((N, 4), dtype=_I32, device=dev),
                      region_score=torch.zeros((N,), dtype=_F32, device=dev),
                      region_ws=ops.small_regions_workspace(H, W, dev))
        self._ws[plan.hw] = ws
        return ws

    # ------------------------------------------------------------------
    @torch.no_grad()
    def generate_device(self, image) -> DeviceMasks:
        """AMG of one image ((H,W) / (H,W,3), numpy or CUDA tensor) with results left on the device."""
        pred = self.predictor
        img = pred._to_device_image(image)
        hw = (int(img.shape[0]), int(img.shape[1]))
        H, W = hw
        plan = self._plan(hw)
        ws = self._workspace(plan)
        dec = pred.model.decoder
        counts = ws["counts"]
        counts.zero_()
        n_cand, n_l1, n_l2 = counts[0:1], counts[1:2], counts[2:3]
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)] if self.phase_ms is not None else None
        if ev:
            ev[0].record()
        feats = pred.encode_crops(img, plan.crops_dev)
        if ev:
            ev[1].record()
        tok = feats.tok
        ppb = self.exec_ppb
        for k, crop in enumerate(plan.crops):
            x0, y0, x1, y1 = crop.box
            emb = tok["embed"][k * 4096:(k + 1) * 4096]
            s0 = tok["s0"][k * 65536:(k + 1) * 65536]
            s1 = tok["s1"][k * 16384:(k + 1) * 16384]
            main = torch.cuda.current_stream()
            use_graph = self.use_cuda_graph and self.capture is None
            graphs = {}  # batch size -> captured lanes whose input buffers hold this crop's features
            nb = 0
            for p0 in range(0, crop.n_points, ppb):
                pb = min(ppb, crop.n_points - p0)
                base = crop.base + p0 * plan.cpp
                graph = None
                if use_graph and (pb == ppb or pb == self.points_per_batch):
                    if pb not in graphs:
                        g = self._batch_graph(plan, ws, pb)
                        if g is not None:
                            g["emb"].copy_(emb)
                            g["s0"].copy_(s0)
                            g["s1"].copy_(s1)
                            for lane in g["lanes"]:
                                lane["stream"].wait_stream(main)
                        graphs[pb] = g
                    graph = graphs[pb]
                if graph is not None:
                    # prompt batches are independent (disjoint slot ranges): replay them round-robin on the lanes'
                    # streams so that the latency-bound token-side launches of one batch overlap the bandwidth-bound
                    # image-stream kernels of another
                    lane = graph["lanes"][nb % len(graph["lanes"])]
                    nb += 1
                    with torch.cuda.stream(lane["stream"]):
                        lane["coords"].copy_(crop.in_points[p0:p0 + pb])
                        lane["geom"].copy_(crop.geom_dev[p0 // ppb])
                        lane["g"].replay()
                    ops.launch_count += lane["launches"]
                else:
                    for g in graphs.values():
                        if g is not None:
                            for lane in g["lanes"]:
                                main.wait_stream(lane["stream"])
                    self._process_batch(k, crop.in_points[p0:p0 + pb], crop.labels[p0:p0 + pb], emb, s0, s1, plan, ws,
                                        crop.box, base, None)
            for g in graphs.values():
                if g is not None:
                    for lane in g["lanes"]:
                        main.wait_stream(lane["stream"])
            n_crop = crop.n_points * plan.cpp
            ops.compact_keep(ws["keep"], crop.base, n_crop, ws["cand"], n_cand)
            ops.nms_dev(ws["bbox"], ws["iou"], ws["cand"], n_cand, n_crop, self.box_nms_thresh, ws["order"],
                        ws["nms_mask"], ws["list1"], n_l1)
        if len(plan.crops) > 1:
            ops.nms_dev(ws["bbox"], plan.score2, ws["list1"], n_l1, plan.n_slots, self.crop_nms_thresh, ws["order"],
                        ws["nms_mask"], ws["list2"], n_l2)
            final_list, final_count = ws["list2"], n_l2
        else:
            final_list, final_count = ws["list1"], n_l1
        if ev:
            ev[2].record()
        m = int(final_count.item())  # the one host synchronisation of the image
        if ev:
            self.phase_ms["encode"] = self.phase_ms.get("encode", 0.0) + ev[0].elapsed_time(ev[1])
            self.phase_ms["decode_post_nms"] = self.phase_ms.get("decode_post_nms", 0.0) + ev[1].elapsed_time(ev[2])
            self.phase_ms["images"] = self.phase_ms.get("images", 0) + 1
        if self.min_mask_region_area > 0 and m > 0:
            final_list, m = self._small_regions(ws, W, final_list, final_count, m)
        slots = final_list[:m].clone()
        return DeviceMasks(hw, m, slots, ops.gather_rows(ws["bits"], slots, m),
                           ops.gather_rows(ws["bbox"], slots, m), ops.gather_rows(ws["area"], slots, m),
                           ops.gather_rows(ws["iou"].view(_I32), slots, m).view(_F32),
                           ops.gather_rows(ws["stab"].view(_I32), slots, m).view(_F32), plan)

    def _small_regions(self, ws, W, lst, count, m):
        """Upstream postprocess_small_regions on the m survivors lst[0..m): hole / island removal in place on their
        packed masks (new box and area where a mask changed), then NMS with score 1.0 for unchanged and 0.0 for changed
        masks and the boxes of the cleaned masks. Returns the kept slots in NMS keep order and their count."""
        ops.amg_small_regions(ws["bits"], lst, m, W, self.min_mask_region_area, ws["region_box"], ws["area"],
                              ws["region_score"], ws["bbox"], ws["region_ws"])
        out = ws["list1"] if lst is ws["list2"] else ws["list2"]
        n_out = ws["counts"][3:4]
        ops.nms_dev(ws["region_box"], ws["region_score"], lst, count, m, max(self.box_nms_thresh, self.crop_nms_thresh),
                    ws["order"], ws["nms_mask"], out, n_out)
        return out, int(n_out.item())

    def _process_batch(self, k, coords, labels, emb, s0, s1, plan, ws, box, base, geom_dev):
        """One batch of point prompts of crop k: decoder (+ m2m refinement) + integer post-processing into the
        image-level slot arrays. With ``geom_dev`` the crop geometry / slot base are read on the device (graph replay)."""
        dec = self.predictor.model.decoder
        x0, y0, x1, y1 = box
        pb = coords.shape[0]
        tokens = dec.prompt_tokens(coords, labels)
        out = dec.forward(emb, s0, s1, tokens, None, multimask_output=self.multimask_output)
        geom = ((y1 - y0, x1 - x0), (x0, y0), plan.hw, self.pred_iou_thresh, self.mask_threshold,
                self.stability_score_offset, self.stability_score_thresh, ws["keep"], ws["stab"], ws["iou"],
                ws["bbox"], ws["area"], ws["bits"])
        if self.use_m2m:
            # every candidate mask of the first pass is refined with itself as the mask prompt
            if self.multimask_output:
                tokens2 = tokens.repeat_interleave(3, dim=0)
                mask_in, step = out["masks"], max(3, self.m2m_batch - self.m2m_batch % 3)
            else:
                tokens2 = tokens
                mask_in, step = self._select_planes(out, pb), max(1, self.m2m_batch)
            ncand = tokens2.shape[0]
            for c0 in range(0, ncand, step):
                cbn = min(step, ncand - c0)
                mi = mask_in[c0 // 3:(c0 + cbn) // 3] if self.multimask_output else mask_in[c0:c0 + cbn]
                gate = self.pred_iou_thresh if (self.m2m_gate and self.pred_iou_thresh > 0.0) else None
                out2 = dec.forward(emb, s0, s1, tokens2[c0:c0 + cbn].contiguous(), mi, multimask_output=False,
                                   mask_clamp=32.0, iou_gate=gate, zero_fill=self.capture is not None)
                self._post(k, out2["masks"], out2["ious"], out2.get("sel_idx"), 1, cbn, geom, base + c0,
                           geom_dev, c0)
        else:
            sel = None if self.multimask_output else out.get("sel_idx")
            self._post(k, out["masks"], out["ious"], sel, plan.cpp, pb * plan.cpp, geom, base, geom_dev, 0)

    def _batch_graph(self, plan, ws, ppb):
        """CUDA graph of one prompt batch of `ppb` points: the ~250 small launches of the two decoder passes are replayed
        with one host call; crop features, point coordinates and crop geometry are graph inputs."""
        key = (plan.hw, ppb)
        if key in self._graphs:
            return self._graphs[key]
        dev = self.device
        if self.use_m2m and self.m2m_batch < (3 if self.multimask_output else 1) * ppb:
            self._graphs[key] = None  # m2m split into several post calls with different bases: keep it eager
            return None
        st = dict(emb=torch.zeros((4096, 256), dtype=_F32, device=dev), s0=torch.zeros((65536, 32), dtype=_F32, device=dev),
                  s1=torch.zeros((16384, 64), dtype=_F32, device=dev), lanes=[])
        crop0 = plan.crops[0]
        for _ in range(max(1, int(self.graph_lanes))):
            lane = dict(coords=torch.zeros((ppb, 1, 2), dtype=_F32, device=dev),
                        labels=torch.ones((ppb, 1), dtype=_I32, device=dev), geom=torch.zeros((8,), dtype=_I32, device=dev),
                        stream=torch.cuda.Stream(device=dev))
            lane["geom"].copy_(crop0.geom_dev[0])
            lane["coords"].copy_(crop0.in_points[:ppb])

            def body(lane=lane):
                self._process_batch(0, lane["coords"], lane["labels"], st["emb"], st["s0"], st["s1"], plan, ws, crop0.box,
                                    0, lane["geom"])

            side = lane["stream"]
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                body()  # warm-up: sets function attributes, loads modules
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            n0 = ops.launch_count
            g = torch.cuda.CUDAGraph()
            # thread-local capture mode: SABER's GPUPool drives one GPU per THREAD of one process (REF saber/utils/
            # parallelization.py:95-155); in the default global mode an allocation by another worker thread during this
            # capture would invalidate it
            with torch.cuda.graph(g, capture_error_mode="thread_local"):
                body()
            lane["launches"] = ops.launch_count - n0
            ops.launch_count = n0
            lane["g"] = g
            st["lanes"].append(lane)
        self._graphs[key] = st
        return st

    def _post(self, crop_idx, planes, ious4, sel, cpp, n, geom, base, geom_dev=None, sub_base=0):
        assert geom_dev is None or sub_base == 0
        pred = self.predictor
        post_planes = planes
        if pred.max_hole_area > 0 or pred.max_sprinkle_area > 0:
            # into a separate buffer: the m2m pass reads the unfilled first-pass planes, as upstream's low_res_masks
            post_planes = ops.amg_fill_lowres(planes, ious4, sel, cpp, n, self.pred_iou_thresh, pred.mask_threshold,
                                              pred.max_hole_area, pred.max_sprinkle_area)
        ops.amg_mask_post(post_planes, ious4, sel, cpp, n, *geom, base, geom_dev)
        if self.capture is not None:
            if self.capture_compact:  # only the plane post-processing reads per candidate (config-1-sized captures)
                prompt = torch.arange(n, device=planes.device) // cpp
                token = (sel.long()[prompt] if sel is not None else
                         (1 + torch.arange(n, device=planes.device) % 3 if cpp == 3 else torch.zeros_like(prompt)))
                pl = planes[prompt, token].cpu().numpy()
            else:
                pl = planes.cpu().numpy()
            self.capture.append(dict(crop=crop_idx, base=base, n=n, cpp=cpp, planes=pl,
                                     ious4=ious4.cpu().numpy(), sel=None if sel is None else sel.cpu().numpy()))

    @staticmethod
    def _select_planes(out, pb):
        """single-mask first pass: the [P,256,256] planes upstream would return (token 0 or dynamic choice)."""
        masks = out["masks"]
        if out.get("sel_idx") is not None:
            return masks[torch.arange(pb, device=masks.device), out["sel_idx"].long()].contiguous()
        return masks[:, 0].contiguous()

    # ------------------------------------------------------------------
    def records(self, dm: DeviceMasks) -> List[Dict[str, Any]]:
        """Host-side records (everything except the segmentation) of a DeviceMasks result."""
        plan = dm.plan
        m = dm.count
        if m == 0:
            return []
        slots = dm.slots.cpu().numpy()
        bbox = dm.bbox.cpu().numpy()
        area = dm.area.cpu().numpy()
        iou = dm.iou.cpu().numpy()
        stab = dm.stability.cpu().numpy()
        recs = []
        for i in range(m):
            s = int(slots[i])
            k = int(plan.slot_crop[s])
            crop = plan.crops[k]
            p = (s - crop.base) // plan.cpp
            x0, y0, x1, y1 = (int(v) for v in bbox[i])
            cx0, cy0, cx1, cy1 = crop.box
            recs.append({
                "area": int(area[i]),
                "bbox": [x0, y0, x1 - x0, y1 - y0],
                "predicted_iou": float(iou[i]),
                "point_coords": [crop.points_full[p].numpy().tolist()],
                "stability_score": float(stab[i]),
                "crop_box": [cx0, cy0, cx1 - cx0, cy1 - cy0],
            })
        return recs

    @torch.no_grad()
    def generate(self, image) -> List[Dict[str, Any]]:
        """Upstream-compatible result: list of dicts with host (numpy / python) values."""
        dm = self.generate_device(image)
        recs = self.records(dm)
        if dm.count == 0:
            return []
        if self.output_mode == "binary_mask":
            seg = ops.unpack_bits(dm.bits, None, dm.count, dm.hw[1]).cpu().numpy()
        else:
            seg = self._rle_segmentations(dm)
        for i, r in enumerate(recs):
            r["segmentation"] = seg[i]
        return [{"segmentation": r["segmentation"], "area": r["area"], "bbox": r["bbox"],
                 "predicted_iou": r["predicted_iou"], "point_coords": r["point_coords"],
                 "stability_score": r["stability_score"], "crop_box": r["crop_box"]} for r in recs]

    def _rle_segmentations(self, dm: DeviceMasks) -> List[Dict[str, Any]]:
        """Segmentations of output_mode "uncompressed_rle" (upstream mask_to_rle_pytorch) and "coco_rle" (pycocotools'
        rleToString, which upstream's coco_encode_rle calls), run-length encoded on the device from the packed masks:
        only the encodings are copied to the host."""
        H, W = dm.hw
        data, off = ops.masks_to_rle(dm.bits, None, dm.count, W, coco=self.output_mode == "coco_rle")
        data, off = data.cpu().numpy(), off.cpu().tolist()
        if self.output_mode == "coco_rle":
            text = data.tobytes().decode("ascii")
            return [{"size": [H, W], "counts": text[a:b]} for a, b in zip(off[:-1], off[1:])]
        return [{"size": [H, W], "counts": data[a:b].tolist()} for a, b in zip(off[:-1], off[1:])]
