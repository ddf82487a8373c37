"""Generates tests/golden/refstack_*.npz by running the reference's OWN, UNMODIFIED hot-path Python
(``oracle/refstack.py`` supplies stubs for its absent third-party imports):

  refstack_adapter_replay.npz — ``saber.adapters.sam2.SAM2Adapter.{set_volume, segment_volume}`` (REF adapters/sam2/
      predictor.py:76-154, 232-348; preprocessing REF adapters/preprocessing.py:16-76) driven by a replayed predictor
      stream (``refstack.ReplayPredictor``): hook timing, stitch precedence, backward-fills-empty-slices, nearest resize,
      presence filtering -> label volumes + presence scores. Pins ``oracle.saber_ref.segment_volume`` and, through it,
      the twin adapter (GPU test "given identical logits").
  refstack_segmenters.npz — ``saber.segmenters.{base.saber2D, tomo.tomoSegmenter, tomo.multiDepthTomoSegmenter,
      propagation.propagationSegmenter}`` (REF segmenters/base.py:84-232,265-280, tomo.py:33-139,206-254,
      propagation.py:41-189) with ``get_adapter`` returning ``refstack.FakeAdapter``: outputs + the log of adapter calls.
      The GPU tests run the twins (``saber_b200.segmenters``) behind the same fake adapter and must reproduce both.

Run with SABER_REFERENCE_DIR pointing at a checkout of the original SABER project:  python -m oracle.make_golden_refstack
"""
from __future__ import annotations

import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")
sys.path.insert(0, ROOT)

from oracle import refstack  # noqa: E402

ADAPTER_CASES = [
    # name, Z, (H, W), image_size, n_obj, start, stream seed, zero-seed index (or -1), min_presence
    ("resize", 12, (40, 48), 64, 3, 5, 1, -1, 0.5),
    ("native", 10, (64, 64), 64, 2, 4, 2, -1, 0.5),
    ("zero_seed", 12, (40, 48), 64, 3, 6, 3, 1, 0.5),
    ("no_filter", 9, (33, 47), 64, 2, 0, 4, -1, -1e9),
]


def adapter_case(P, SAM2AdapterConfig, name, Z, hw, size, n_obj, start, seed, zero_idx, min_presence):
    rp = refstack.ReplayPredictor(size)
    P.build_sam2_video_predictor = lambda *a, **k: rp
    ad = P.SAM2Adapter(SAM2AdapterConfig(cfg="tiny"), device="cpu")
    vol = np.random.default_rng(100 + seed).normal(size=(Z,) + hw).astype(np.float32)
    ad.set_volume(vol)
    images = ad.inference_state["images"].numpy()
    rp.passes = refstack.synth_stream(Z, n_obj, start, size, seed)
    seeds = [m["segmentation"].astype(np.float32) for m in refstack.synth_masks(hw, n_obj, 200 + seed)]
    if zero_idx >= 0:
        seeds[zero_idx][:] = 0
    out = ad.segment_volume(start, masks=seeds, vol_shape=(Z,) + hw, min_presence_score=min_presence)
    pres = np.array([[ad.frame_metrics[f][o + 1]["presence_score"] for o in range(n_obj)] for f in range(Z)])
    return {f"{name}_labels": out, f"{name}_presence": pres, f"{name}_added": np.array(rp.added),
            f"{name}_images_mean": np.array([images.mean(), images.std(), images.min(), images.max()]),
            f"{name}_images0": images[0, 0, ::7, ::7].copy(),
            f"{name}_maskmem_rows": np.array(rp.maskmem_tpos_enc.shape[0])}


def segmenter_cases(vol):
    """Runs the reference's segmenter classes behind FakeAdapter. Returns ({name: array}, {name: call log})."""
    import saber.segmenters.base as B
    import saber.segmenters.propagation as PR
    import saber.segmenters.tomo as T
    from saber.adapters.base import SAM2AdapterConfig
    outs, logs = {}, {}

    def make(cls, seed, **kw):
        fake = refstack.FakeAdapter(seed=seed)
        B.get_adapter = lambda cfg, device: fake
        seg = cls(deviceID=0, cfg=SAM2AdapterConfig(cfg="tiny"), **kw)
        return seg, fake

    s, f = make(T.tomoSegmenter, 10, min_mask_area=20)
    outs["tomo_vol"] = s.segment_vol(vol, 4, zSlice=None)
    outs["tomo_image0"] = np.asarray(s.image0)
    logs["tomo_vol"] = f.calls
    s, f = make(T.tomoSegmenter, 11, min_mask_area=20)
    outs["tomo_vol_z"] = s.segment_vol(vol, 3, zSlice=5)
    logs["tomo_vol_z"] = f.calls
    s, f = make(T.multiDepthTomoSegmenter, 12, min_mask_area=10)
    outs["multidepth"] = s.segment(vol, 3, num_slabs=3, delta_z=5)
    logs["multidepth"] = f.calls
    s, f = make(PR.propagationSegmenter, 13, min_mask_area=20)
    outs["prop_single"] = s.segment(vol, ini_depth=4, nframes=3, target_class=1)
    logs["prop_single"] = f.calls
    s, f = make(PR.propagationSegmenter, 14, min_mask_area=20)
    outs["prop_slice_by_slice"] = s.slice_by_slice(vol, None)
    logs["prop_slice_by_slice"] = f.calls
    s, f = make(B.saber2D, 15, min_mask_area=20, window_size=48, overlap_ratio=0.25)
    masks = s.segment_image(vol[3], display=False, use_sliding_window=True)
    outs["sliding_window"] = np.stack([m["segmentation"] for m in masks]).astype(np.uint8)
    outs["sliding_window_bbox"] = np.array([m["bbox"] for m in masks])
    logs["sliding_window"] = f.calls

    # multiclass_segment (REF propagation.py:121-161) with a canned classifier
    class FakeClassifier:
        def batch_predict(self, image, masks, batchsize):
            n = len(masks)
            rng = np.random.default_rng(int(masks.reshape(n, -1).sum()) % 1000)
            p = rng.uniform(0.05, 1.0, (n, 3)).astype(np.float32)
            return p / p.sum(1, keepdims=True)

    fake = refstack.FakeAdapter(seed=16)
    B.get_adapter = lambda cfg, device: fake
    cfg = SAM2AdapterConfig(cfg="tiny")
    seg = PR.propagationSegmenter(deviceID=0, cfg=cfg, min_mask_area=20)
    seg.classifier, seg.batchsize = FakeClassifier(), 32
    outs["prop_multiclass"] = seg.segment(vol, ini_depth=5, nframes=2, target_class=0)
    logs["prop_multiclass"] = fake.calls
    return outs, logs


def _jsonable(calls):
    return [[(list(x) if isinstance(x, tuple) else x) for x in c] for c in calls]


def main():
    os.makedirs(GOLD, exist_ok=True)
    refstack.install()
    import saber.adapters.sam2.predictor as P
    from saber.adapters.base import SAM2AdapterConfig
    out = {}
    for case in ADAPTER_CASES:
        out.update(adapter_case(P, SAM2AdapterConfig, *case))
    np.savez_compressed(os.path.join(GOLD, "refstack_adapter_replay.npz"), **out)
    from saber_b200 import synth
    vol = synth.make_tomogram((16, 64, 80), seed=31, n_ellipsoids=6).numpy()
    outs, logs = segmenter_cases(vol)
    np.savez_compressed(os.path.join(GOLD, "refstack_segmenters.npz"), logs=json.dumps({k: _jsonable(v) for k, v in logs.items()}),
                        **outs)
    for k, v in outs.items():
        print(k, v.shape, v.dtype, int(v.max()))
    print("calls:", {k: len(v) for k, v in logs.items()})


if __name__ == "__main__":
    main()
