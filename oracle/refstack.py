"""TEST INFRASTRUCTURE — runs the UNMODIFIED reference Python (``$SABER_REFERENCE_DIR/saber``, a checkout of the
original SABER project; it is not part of this repository).

The reference's own modules for the hot path (``saber.adapters.sam2.predictor``, ``saber.segmenters.{base,tomo,
propagation}``, ``saber.adapters.preprocessing`` ...) import third-party packages that are absent here (``sam2``,
``skimage``, ``matplotlib``, ``mrcfile``, ``zarr``, ``copick``, ``monai``, ``rich_click``). ``install()`` puts
  * empty stub modules in ``sys.modules`` for the ones the path never calls (a call raises),
  * a functional ``skimage.transform.resize`` (the restatement ``oracle.saber_ref.skimage_resize``, SURVEY A1),
  * a ``sam2`` package: either the fp32 CPU restatement ``oracle.sam2_ref`` or a caller-supplied fake,
and adds ``REF_ROOT`` to ``sys.path`` so that ``import saber...`` resolves to the reference's files, unchanged.
Everything here is used by ``oracle/make_golden_refstack.py`` (which writes the committed fixtures) and by tests that
skip when ``SABER_REFERENCE_DIR`` does not point at such a checkout; the tests that compare with the fixtures need no
reference.
"""
from __future__ import annotations

import importlib
import importlib.machinery
import os
import sys
import types
from typing import Any, Dict, List, Optional

import numpy as np
import torch

REF_ROOT = os.environ.get("SABER_REFERENCE_DIR", "")


def available() -> bool:
    return bool(REF_ROOT) and os.path.isfile(os.path.join(REF_ROOT, "saber", "adapters", "sam2", "predictor.py"))


class _Stub(types.ModuleType):
    def __getattr__(self, name):
        if name.startswith("__"):
            raise AttributeError(name)
        m = _Stub(self.__name__ + "." + name)
        m.__spec__ = importlib.machinery.ModuleSpec(m.__name__, None)
        m.__path__ = []
        sys.modules[m.__name__] = m
        setattr(self, name, m)
        return m

    def __call__(self, *a, **k):
        raise RuntimeError(f"stubbed dependency {self.__name__} was called on the reference path")


_STUBBED = ("mrcfile", "matplotlib", "matplotlib.pyplot", "matplotlib.colors", "matplotlib.patches", "matplotlib.widgets",
            "matplotlib.cm", "matplotlib.figure", "skimage", "skimage.transform", "skimage.measure", "skimage.morphology",
            "zarr", "copick", "copick_utils", "rich_click", "monai", "monai.transforms", "starfile", "ome_zarr", "napari",
            "pyqtgraph", "PyQt5", "PIL", "tifffile", "nibabel", "h5py", "hyperspy", "hyperspy.api", "rsciio", "imageio",
            "kornia", "torchmetrics", "lightning", "torch_ema", "multiprocess")


def _stub(name: str) -> types.ModuleType:
    m = _Stub(name)
    m.__spec__ = importlib.machinery.ModuleSpec(name, None)
    m.__path__ = []
    sys.modules[name] = m
    if "." in name:
        parent, child = name.rsplit(".", 1)
        setattr(sys.modules[parent], child, m)
    return m


def install(sam2_package: Optional[Dict[str, types.ModuleType]] = None) -> None:
    """Make ``import saber...`` work on the reference's files. ``sam2_package``: {"sam2.build_sam": module, ...} to serve
    as the ``sam2`` package; default = the oracle restatement (``oracle.sam2_ref``)."""
    if not available():
        raise RuntimeError("set SABER_REFERENCE_DIR to a checkout of the original SABER project")
    for name in _STUBBED:
        if name in sys.modules:
            continue
        try:
            importlib.import_module(name)
            continue
        except Exception:
            pass
        _stub(name)
    # functional restatements of the two third-party calls that ARE on the path
    from oracle import saber_ref
    skt = sys.modules["skimage.transform"]
    if isinstance(skt, _Stub):
        skt.resize = lambda image, output_shape, order=None, anti_aliasing=None, **kw: saber_ref.skimage_resize(
            image, output_shape, order=order, anti_aliasing=anti_aliasing)
    if sam2_package is None:
        from oracle.sam2_ref import amg as o_amg, image_predictor as o_img, sam2_base as o_base, video_predictor as o_vid
        build = types.ModuleType("sam2.build_sam")
        build.build_sam2 = o_base.build_sam2
        build.build_sam2_video_predictor = o_vid.build_sam2_video_predictor
        sam2_package = {"sam2.build_sam": build, "sam2.sam2_image_predictor": o_img, "sam2.automatic_mask_generator": o_amg,
                        "sam2.sam2_video_predictor": o_vid}
    root = types.ModuleType("sam2")
    root.__path__ = []
    sys.modules["sam2"] = root
    for name, mod in sam2_package.items():
        sys.modules[name] = mod
        setattr(root, name.split(".", 1)[1], mod)
    if REF_ROOT not in sys.path:
        sys.path.insert(0, REF_ROOT)
    # the reference resolves checkpoints by downloading them: no network here, random-init weights of the named config
    pw = importlib.import_module("saber.pretrained_weights")
    pw.get_sam2_checkpoint = lambda cfg: (cfg, None)
    io = importlib.import_module("saber.utils.io")
    io.get_available_devices = lambda deviceID=None: torch.device("cpu")


def uninstall() -> None:
    """Drop the reference's modules and the sam2 alias again (tests that import saber_b200 twins afterwards)."""
    for name in [n for n in sys.modules if n == "saber" or n.startswith("saber.") or n == "sam2" or n.startswith("sam2.")]:
        del sys.modules[name]
    if REF_ROOT in sys.path:
        sys.path.remove(REF_ROOT)


# ---------------------------------------------------------------------------------------------------------------------
# Deterministic fakes behind the reference's seams (shared by the golden generator and the tests of the twins)
# ---------------------------------------------------------------------------------------------------------------------
def synth_masks(hw, n, seed) -> List[Dict[str, Any]]:
    """n elliptical mask dicts with the keys SABER reads (segmentation, area, bbox XYWH, predicted_iou, stability_score,
    point_coords, crop_box); masks 2k and 2k+1 are near-duplicates (exercises remove_duplicate_masks)."""
    H, W = hw
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:H, 0:W]
    out = []
    for i in range(n):
        if i % 2 == 1 and out:
            prev = out[-1]["_geom"]
            cy, cx, ry, rx = prev[0], prev[1], prev[2] * 0.99, prev[3]
        else:
            cy, cx = rng.uniform(0.15 * H, 0.85 * H), rng.uniform(0.15 * W, 0.85 * W)
            ry, rx = rng.uniform(0.04 * H, 0.2 * H), rng.uniform(0.04 * W, 0.2 * W)
        seg = ((yy - cy) / ry) ** 2 + ((xx - cx) / rx) ** 2 <= 1.0
        ys, xs = np.nonzero(seg)
        bbox = [int(xs.min()), int(ys.min()), int(xs.max() - xs.min()), int(ys.max() - ys.min())] if len(ys) else [0, 0, 0, 0]
        out.append({"segmentation": seg, "area": int(seg.sum()), "bbox": bbox,
                    "predicted_iou": float(np.round(rng.uniform(0.7, 1.0), 3)),
                    "stability_score": float(np.round(rng.uniform(0.92, 1.0), 3)),
                    "point_coords": [[float(cx), float(cy)]], "crop_box": [0, 0, W, H], "_geom": (cy, cx, ry, rx)})
    for m in out:
        del m["_geom"]
    return out


class FakeAdapter:
    """Stands in for ``SAM2Adapter`` behind ``get_adapter`` so that the segmenters' orchestration can be compared
    between the reference's classes and the twins: canned AMG lists, a canned propagation result that depends only on
    the arguments, and a log of every call."""

    def __init__(self, seed: int = 0, n_masks: int = 6):
        self.seed, self.n_masks = seed, n_masks
        self.calls: List[tuple] = []
        self._k = 0
        self.frame_metrics = {}

    @staticmethod
    def _np(a):
        if isinstance(a, torch.Tensor):
            a = a.detach().cpu().numpy()
        return np.asarray(a)

    def segment_image_2d(self, image, text_prompt=None, threshold=None, **kw):
        img = self._np(image)
        self.calls.append(("segment_image_2d", tuple(img.shape[:2]), float(img.mean()), float(img.std()), text_prompt,
                           tuple(sorted(kw))))
        self._k += 1
        masks = synth_masks(img.shape[:2], self.n_masks, self.seed + self._k)
        if self._k % 3 == 0:
            return []  # an empty slab now and then (REF tomo.py:123-124, propagation.py:111-112)
        return masks

    def set_volume(self, tomogram, offload_video_to_cpu: bool = False):
        v = self._np(tomogram)
        self.calls.append(("set_volume", tuple(v.shape), float(v.mean()), float(v.std())))

    def segment_volume(self, start_frame_idx, masks=None, vol_shape=None, max_frame_num_to_track=None,
                       min_presence_score=0.5, inference_state=None):
        ms = [self._np(m["segmentation"] if isinstance(m, dict) else m).astype(bool) for m in masks]
        self.calls.append(("segment_volume", int(start_frame_idx), len(ms), [int(m.sum()) for m in ms],
                           tuple(int(v) for v in vol_shape), max_frame_num_to_track, float(min_presence_score)))
        Z, H, W = (int(v) for v in vol_shape)
        out = np.zeros((Z, H, W), np.uint16)
        span = Z if max_frame_num_to_track is None else int(max_frame_num_to_track)
        for i, m in enumerate(ms):
            z0, z1 = max(0, start_frame_idx - min(span, 2 + i)), min(Z, start_frame_idx + min(span, 3 + i) + 1)
            out[z0:z1][:, m] = i + 1
        return out

    def reset_state(self, inference_state=None):
        self.calls.append(("reset_state",))


class ReplayPredictor(torch.nn.Module):
    """A ``sam2`` video predictor that replays a canned stream (per pass: hook scores and yielded logits) — drives the
    reference's ``SAM2Adapter.segment_volume`` (REF saber/adapters/sam2/predictor.py:232-348) without a network."""

    def __init__(self, image_size: int = 64):
        super().__init__()
        self.image_size = image_size
        self.num_maskmem = 7
        self.maskmem_tpos_enc = torch.nn.Parameter(torch.zeros(7, 1, 1, 64))
        self.sam_mask_decoder = _Decoder()
        self.passes: Dict[bool, list] = {False: [], True: []}
        self.added: List[int] = []
        self.add_scores: Dict[int, float] = {}

    @property
    def device(self):
        return torch.device("cpu")

    def _get_image_feature(self, inference_state, frame_idx=0, batch_size=1):
        return None

    def add_new_mask(self, inference_state, frame_idx, obj_id, mask):
        self.added.append(int(obj_id))
        # upstream calls the mask decoder once per prompted object (the object pointer): the hook fires
        self.sam_mask_decoder(torch.tensor([[self.add_scores.get(int(obj_id), 10.0)]]))
        return frame_idx, list(self.added), None

    def propagate_in_video(self, state, start_frame_idx=None, max_frame_num_to_track=None, reverse=False):
        for ev in self.passes[bool(reverse)]:
            if ev[0] == "hook":
                self.sam_mask_decoder(torch.tensor([[ev[1]]]))
            else:
                yield ev[1], ev[2], ev[3]

    def reset_state(self, state):
        self.added = []


class _Decoder(torch.nn.Module):
    def forward(self, score):
        return (None, None, None, score)


def synth_stream(Z: int, n_obj: int, start: int, size: int, seed: int):
    """Canned propagation stream: per pass, for every frame first one hook call per object (its object score), then the
    yielded logits [n_obj,1,size,size] (smooth blobs that fade with |z - start|). The object scores form a bump around
    the start frame so that fit_organelle_boundaries has something to fit."""
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:size, 0:size].astype(np.float32)
    cen = rng.uniform(0.25 * size, 0.75 * size, (n_obj, 2))
    rad = rng.uniform(0.1 * size, 0.25 * size, n_obj)
    width = rng.uniform(0.15 * Z, 0.45 * Z, n_obj)
    passes = {False: [], True: []}
    for rev in (False, True):
        frames = range(start, -1, -1) if rev else range(start, Z)
        for f in frames:
            logits = np.empty((n_obj, 1, size, size), np.float32)
            for o in range(n_obj):
                fade = np.exp(-0.5 * ((f - start) / width[o]) ** 2)
                score = float(12.0 * fade - 4.0 + 0.3 * rng.normal())
                passes[rev].append(("hook", score))
                d = np.sqrt((yy - cen[o, 0]) ** 2 + (xx - cen[o, 1]) ** 2)
                logits[o, 0] = 6.0 * (rad[o] * (0.3 + 0.7 * fade) - d) + 0.5 * rng.normal(size=(size, size)).astype(np.float32)
            passes[rev].append(("yield", f, list(range(1, n_obj + 1)), torch.from_numpy(logits)))
    return passes
