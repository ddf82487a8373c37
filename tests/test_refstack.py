"""Boundary / parity chain for the SABER-owned Python of the hot path (SURVEY 8a R5-R7, R9, R12):

  reference's own code (run by oracle/make_golden_refstack.py, fixtures committed)
      == oracle restatement (oracle/saber_ref.py)            -- CPU tests below, anywhere
      == the unmodified reference re-run live                 -- CPU tests below, when SABER_REFERENCE_DIR is set
      == saber_b200 twins behind the same fake adapter        -- GPU tests below (the twins have no CPU path)

The twin adapter itself is tied to the restatement on the GPU "given identical logits" (tests/test_gpu_video.py).
"""
import json
import os

import numpy as np
import pytest
import torch

from oracle import refstack, saber_ref
from oracle.make_golden_refstack import ADAPTER_CASES


def _adapter_inputs(Z, hw, size, n_obj, start, seed, zero_idx):
    vol = np.random.default_rng(100 + seed).normal(size=(Z,) + hw).astype(np.float32)
    seeds = [m["segmentation"].astype(np.float32) for m in refstack.synth_masks(hw, n_obj, 200 + seed)]
    if zero_idx >= 0:
        seeds[zero_idx][:] = 0
    rp = refstack.ReplayPredictor(size)
    rp.passes = refstack.synth_stream(Z, n_obj, start, size, seed)
    return vol, seeds, rp


@pytest.mark.parametrize("case", ADAPTER_CASES, ids=lambda c: c[0])
def test_oracle_adapter_restatement_matches_reference_golden(golden_dir, case):
    """oracle.saber_ref.{segment_volume, load_grayscale_image_array, normalize_tomogram} reproduce what the reference's
    SAM2Adapter produced on the same replayed predictor stream: label volume bit-exact, presence scores to 1e-9."""
    name, Z, hw, size, n_obj, start, seed, zero_idx, min_presence = case
    g = np.load(os.path.join(golden_dir, "refstack_adapter_replay.npz"))
    vol, seeds, rp = _adapter_inputs(Z, hw, size, n_obj, start, seed, zero_idx)
    images, vh, vw = saber_ref.load_grayscale_image_array(saber_ref.normalize_tomogram(vol), size)
    assert (vh, vw) == (size, size)  # REF adapters/preprocessing.py:24: read from the resized image
    np.testing.assert_allclose(np.array([images.mean(), images.std(), images.min(), images.max()]),
                               g[f"{name}_images_mean"], rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(images[0, 0, ::7, ::7], g[f"{name}_images0"], rtol=0, atol=1e-6)
    labels, frame_scores, metrics = saber_ref.segment_volume(rp, None, start, seeds, (Z,) + hw,
                                                             min_presence_score=min_presence)
    np.testing.assert_array_equal(labels, g[f"{name}_labels"])
    pres = np.array([[metrics[f][o + 1]["presence_score"] for o in range(n_obj)] for f in range(Z)])
    np.testing.assert_allclose(pres, g[f"{name}_presence"], rtol=1e-9, atol=1e-12)
    assert rp.added == list(g[f"{name}_added"])
    assert int(g[f"{name}_maskmem_rows"]) == 2  # REF predictor.py:31-34 truncated the parameter to num_maskmem rows


@pytest.mark.skipif(not refstack.available(), reason="needs SABER_REFERENCE_DIR: a checkout of the original SABER project")
def test_reference_stack_live_equals_committed_goldens(golden_dir, tmp_path, monkeypatch):
    """Re-runs oracle/make_golden_refstack.py (the unmodified reference Python) and compares with the committed files:
    the fixtures are what the reference produces, not what this repo wishes it produced."""
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    code = ("import oracle.make_golden_refstack as m, sys; m.GOLD = sys.argv[1]; m.main()")
    subprocess.run([sys.executable, "-c", code, str(tmp_path)], check=True, cwd=root, capture_output=True, timeout=600)
    for fn in ("refstack_adapter_replay.npz", "refstack_segmenters.npz"):
        a, b = np.load(os.path.join(golden_dir, fn)), np.load(os.path.join(tmp_path, fn))
        assert sorted(a.files) == sorted(b.files)
        for k in a.files:
            if a[k].dtype.kind in "US":
                assert str(a[k]) == str(b[k]), k
            elif a[k].dtype.kind == "f":
                np.testing.assert_allclose(a[k], b[k], rtol=1e-12, atol=0, err_msg=k)
            else:
                np.testing.assert_array_equal(a[k], b[k], err_msg=k)


def test_segmenter_goldens_are_consistent_with_the_oracle(golden_dir):
    """The reference-run segmenter fixtures against the oracle's restatements of their integer stages: the multi-depth /
    single-segment outputs are separate_masks of a binary union, slice_by_slice is separate_masks of the stitched slices."""
    g = np.load(os.path.join(golden_dir, "refstack_segmenters.npz"))
    logs = json.loads(str(g["logs"]))
    # tomoSegmenter.segment_vol: slab AMG -> set_volume -> segment_volume(start = Z // 2) -> reset_state
    kinds = [c[0] for c in logs["tomo_vol"]]
    assert kinds == ["segment_image_2d", "set_volume", "segment_volume", "reset_state"]
    assert logs["tomo_vol"][2][1] == 8 and logs["tomo_vol_z"][2][1] == 5
    assert logs["tomo_vol"][2][6] == 0.5  # filter_threshold -> min_presence_score
    for name in ("multidepth", "prop_single", "prop_slice_by_slice"):
        v = g[name]
        assert v.dtype == np.uint32
        np.testing.assert_array_equal(saber_ref.separate_masks((v > 0).astype(np.uint16), 0) > 0, v > 0)
    # propagationSegmenter seeds every ini_depth slices starting at 2 with nframes forwarded
    starts = [c[1] for c in logs["prop_single"] if c[0] == "segment_volume"]
    assert starts and all((s - 2) % 4 == 0 for s in starts)
    assert all(c[5] == 3 for c in logs["prop_single"] if c[0] == "segment_volume")


# ---------------------------------------------------------------------------------------------------------------------
# GPU: the twins behind the same fake adapter
# ---------------------------------------------------------------------------------------------------------------------
def _twin(cls, seed, monkeypatch, **kw):
    from saber_b200.adapters.base import SAM2AdapterConfig
    from saber_b200.segmenters import base as B
    fake = refstack.FakeAdapter(seed=seed)
    monkeypatch.setattr(B, "get_adapter", lambda cfg, device: fake)
    seg = cls(deviceID=0, cfg=SAM2AdapterConfig(cfg="tiny", allow_random_init=True), **kw)
    return seg, fake


def _assert_calls_equal(got, want):
    """Call logs: integer / string fields exact, image statistics (float) to 1e-4 (GPU fp32 vs numpy)."""
    assert len(got) == len(want), ([c[0] for c in got], [c[0] for c in want])
    for a, b in zip(got, want):
        assert a[0] == b[0]
        for x, y in zip(a[1:], b[1:]):
            if isinstance(x, tuple):
                x = list(x)
            if isinstance(y, float) or isinstance(x, float):
                assert x == pytest.approx(y, rel=1e-4, abs=1e-5), (a, b)
            else:
                assert x == y, (a, b)


@pytest.fixture(scope="module")
def seg_gold(golden_dir):
    g = np.load(os.path.join(golden_dir, "refstack_segmenters.npz"))
    from saber_b200 import synth
    vol = synth.make_tomogram((16, 64, 80), seed=31, n_ellipsoids=6).numpy()
    return g, json.loads(str(g["logs"])), vol


@pytest.mark.gpu
def test_tomo_segmenter_twin_matches_reference_run(seg_gold, monkeypatch):
    from saber_b200.segmenters.tomo import multiDepthTomoSegmenter, tomoSegmenter
    g, logs, vol = seg_gold
    s, f = _twin(tomoSegmenter, 10, monkeypatch, min_mask_area=20)
    out = s.segment_vol(vol, 4, zSlice=None)
    np.testing.assert_array_equal(out, g["tomo_vol"])
    np.testing.assert_allclose(s.image0.cpu().numpy(), g["tomo_image0"], rtol=0, atol=2e-5)
    _assert_calls_equal(f.calls, logs["tomo_vol"])
    s, f = _twin(tomoSegmenter, 11, monkeypatch, min_mask_area=20)
    np.testing.assert_array_equal(s.segment_vol(vol, 3, zSlice=5), g["tomo_vol_z"])
    _assert_calls_equal(f.calls, logs["tomo_vol_z"])
    s, f = _twin(multiDepthTomoSegmenter, 12, monkeypatch, min_mask_area=10)
    out = s.segment(vol, 3, num_slabs=3, delta_z=5)
    assert out.dtype == np.uint32
    np.testing.assert_array_equal(out, g["multidepth"])
    _assert_calls_equal(f.calls, logs["multidepth"])


@pytest.mark.gpu
def test_propagation_segmenter_twin_matches_reference_run(seg_gold, monkeypatch):
    from saber_b200.segmenters.propagation import propagationSegmenter
    g, logs, vol = seg_gold
    s, f = _twin(propagationSegmenter, 13, monkeypatch, min_mask_area=20)
    out = s.segment(vol, ini_depth=4, nframes=3, target_class=1)
    np.testing.assert_array_equal(out, g["prop_single"])
    _assert_calls_equal(f.calls, logs["prop_single"])

    class FakeClassifier:
        def batch_predict(self, image, masks, batchsize):
            n = len(masks)
            rng = np.random.default_rng(int(masks.reshape(n, -1).sum()) % 1000)
            p = rng.uniform(0.05, 1.0, (n, 3)).astype(np.float32)
            return p / p.sum(1, keepdims=True)

    s, f = _twin(propagationSegmenter, 16, monkeypatch, min_mask_area=20)
    s.classifier, s.batchsize = FakeClassifier(), 32
    out = s.segment(vol, ini_depth=5, nframes=2, target_class=0)
    np.testing.assert_array_equal(out, g["prop_multiclass"])
    _assert_calls_equal(f.calls, logs["prop_multiclass"])


@pytest.mark.gpu
def test_saber2d_sliding_window_twin_matches_reference_run(seg_gold, monkeypatch):
    from saber_b200.segmenters.base import saber2D
    g, logs, vol = seg_gold
    s, f = _twin(saber2D, 15, monkeypatch, min_mask_area=20, window_size=48, overlap_ratio=0.25)
    masks = s.segment_image(vol[3], display=False, use_sliding_window=True)
    np.testing.assert_array_equal(np.stack([m["segmentation"] for m in masks]).astype(np.uint8), g["sliding_window"])
    np.testing.assert_array_equal(np.array([m["bbox"] for m in masks]), g["sliding_window_bbox"])
    _assert_calls_equal(f.calls, logs["sliding_window"])
