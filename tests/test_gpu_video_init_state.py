"""-m gpu: ``SAM2VideoPredictor.init_state`` on JPEG folders and the frame kernel behind it.

* ``ops.resample_frames_u8`` equals the oracle's fixed-point restatement of Pillow's resize + upstream's normalisation
  with ``torch.equal``, at frame sizes that exercise both passes, each pass skipped, and 1 to 65 frames per call;
* ``init_state`` on folders written here (seeded synthetic frames saved as JPEG with PIL) gives ``images`` equal, bit
  for bit, to the oracle restatement of upstream's ``load_video_frames``, in the synchronous, offloaded and async modes;
* end to end at hiera-tiny: point, box, refinement-click and mask prompts, then propagation both ways, against the
  fp32 oracle predictor built from its own ``init_state`` (tolerances of tests/test_gpu_configs.py).
"""
import os

import numpy as np
import pytest
import torch
from PIL import Image

pytestmark = pytest.mark.gpu
S = 1024
SIZES = [(96, 120), (480, 854), (1080, 1920), (1024, 1024), (1, 1), (3000, 4000), (1024, 700), (700, 1024),
         (2000, 1024), (37, 2500)]


def rel_l2(a, b):
    a, b = a.float().cpu(), b.float().cpu()
    return ((a - b).norm() / (b.norm() + 1e-12)).item()


def _frame(rng, h, w):
    """A smooth colour field with a few discs and noise: JPEG-compressible, with edges for the model to see."""
    yy, xx = np.mgrid[0:h, 0:w].astype(np.float32)
    img = np.stack([128 + 60 * np.sin(xx / (w / 3 + 1) + c) * np.cos(yy / (h / 2 + 1) - c) for c in range(3)], -1)
    for _ in range(4):
        cy, cx, r = rng.uniform(0, h), rng.uniform(0, w), rng.uniform(0.05, 0.25) * min(h, w)
        img[((yy - cy) ** 2 + (xx - cx) ** 2) <= r * r] = rng.uniform(0, 255, 3)
    img += rng.normal(0, 6, img.shape)
    return np.clip(img, 0, 255).astype(np.uint8)


def _write_folder(path, sizes, seed):
    os.makedirs(path)
    rng = np.random.default_rng(seed)
    for i, (h, w) in enumerate(sizes):
        Image.fromarray(_frame(rng, h, w)).save(os.path.join(path, f"{i:05d}.jpg"), quality=90)
    return str(path)


@pytest.fixture(scope="module")
def folders(tmp_path_factory):
    root = tmp_path_factory.mktemp("video_init_state")
    return {"480x854": _write_folder(root / "a", [(480, 854)] * 4, 1),
            "1024": _write_folder(root / "b", [(1024, 1024)] * 3, 2),
            "mixed": _write_folder(root / "c", [(480, 854), (360, 640), (360, 640), (480, 854), (360, 640)], 3)}


@pytest.fixture(scope="module")
def luts():
    from saber_b200 import ops
    from saber_b200.sam2 import video_io
    ops.require_b200()
    return video_io.normalize_lut().cuda(), video_io.normalize_lut(float64_path=True).cuda()


@pytest.mark.parametrize("hw", SIZES)
def test_kernel_equals_oracle(hw, luts):
    from oracle.sam2_ref import video_io as ovio
    from saber_b200 import ops
    frames = np.random.default_rng(hw[0] + 3 * hw[1]).integers(0, 256, (2,) + hw + (3,), dtype=np.uint8)
    x = torch.from_numpy(frames).cuda()
    got = ops.resample_frames_u8(x, S, luts[0])
    assert torch.equal(got.cpu(), ovio.normalized_frames(frames, S))
    got64 = ops.resample_frames_u8(x[1:], S, luts[1])
    assert torch.equal(got64.cpu(), ovio.normalized_frames(frames[1:], S, float64_path=True))


def test_kernel_frames_per_call_1_to_65(luts):
    from oracle.sam2_ref import video_io as ovio
    from saber_b200 import ops
    frames = np.random.default_rng(5).integers(0, 256, (65, 37, 53, 3), dtype=np.uint8)
    want = ovio.normalized_frames(frames, S)
    x = torch.from_numpy(frames).cuda()
    for n in range(1, 66):
        out = torch.full((n, 3, S, S), float("nan"), device="cuda")
        ops.resample_frames_u8(x[:n].contiguous(), S, luts[0], out=out)
        assert torch.equal(out.cpu(), want[:n]), n


@pytest.fixture(scope="module")
def predictors():
    from oracle.sam2_ref.video_io import build_sam2_video_predictor as oracle_build
    from saber_b200.sam2 import arch
    from saber_b200.sam2.sam2_video_predictor import build_sam2_video_predictor
    sd = dict(arch.random_state_dict("tiny", seed=0))
    for k in list(sd):  # realistic logit range, separated IoU / object-score heads (as tests/test_gpu_configs.py)
        if "output_hypernetworks_mlps" in k and ".layers.2." in k:
            sd[k] = sd[k] * 30.0
    sd["sam_mask_decoder.iou_prediction_head.layers.2.bias"] = torch.tensor([0.0, -1.0, 1.0, 0.0])
    sd["sam_mask_decoder.pred_obj_score_head.layers.2.bias"] = torch.tensor([1.5])
    ours = build_sam2_video_predictor("tiny", None, device="cuda:0", state_dict=sd)
    orc = oracle_build("tiny", None, device="cpu", state_dict=sd)
    for m in (ours, orc):
        m.fill_hole_area = 0  # discontinuous in the logits; checked bit-exactly on identical inputs elsewhere
    return ours, orc


@pytest.mark.parametrize("name", ["480x854", "1024", "mixed"])
def test_init_state_images_equal_upstream_loading(folders, predictors, name):
    from oracle.sam2_ref import video_io as ovio
    ours = predictors[0]
    want, vh, vw = ovio.load_video_frames(folders[name], S, True, compute_device=torch.device("cpu"))
    st = ours.init_state(folders[name])
    assert st["images"].is_cuda and st["images"].dtype == torch.float32
    assert torch.equal(st["images"].cpu(), want)
    assert (st["video_height"], st["video_width"], st["num_frames"]) == (vh, vw, len(want))
    assert 0 in st["cached_features"]
    off = ours.init_state(folders[name], offload_video_to_cpu=True, offload_state_to_cpu=True)
    assert off["images"].device.type == "cpu" and torch.equal(off["images"], want)
    assert off["storage_device"] == torch.device("cpu") and off["offload_state_to_cpu"] and off["offload_video_to_cpu"]


@pytest.mark.parametrize("offload", [False, True])
def test_async_loading_equals_upstream_cast(folders, predictors, offload):
    from oracle.sam2_ref import video_io as ovio
    ours = predictors[0]
    folder = folders["mixed"]
    lazy_want, vh, vw = ovio.load_video_frames(folder, S, True, async_loading_frames=True,
                                               compute_device=torch.device("cpu"))
    st = ours.init_state(folder, offload_video_to_cpu=offload, async_loading_frames=True)
    lazy = st["images"]
    assert (st["video_height"], st["video_width"]) == (vh, vw) == (480, 854)
    assert len(lazy) == len(lazy_want) == st["num_frames"] == 5
    lazy.thread.join(timeout=120)
    lazy_want.thread.join(timeout=120)
    assert not lazy.thread.is_alive()
    for n in range(len(lazy)):
        img = lazy[n]
        assert img.dtype == torch.float32 and img.device.type == ("cpu" if offload else "cuda")
        assert torch.equal(img.cpu(), lazy_want[n].float()), n


def test_async_loading_error_is_raised_from_getitem(tmp_path):
    from saber_b200.sam2 import video_io
    folder = _write_folder(tmp_path / "v", [(64, 80)] * 3, 4)
    with open(os.path.join(folder, "00002.jpg"), "wb") as f:
        f.write(b"not a jpeg")
    lazy, vh, vw = video_io.load_video_frames(folder, S, False, async_loading_frames=True,
                                              compute_device=torch.device("cuda:0"))
    assert (vh, vw) == (64, 80)
    lazy.thread.join(timeout=60)
    with pytest.raises(RuntimeError, match="Failure in frame loading thread"):
        lazy[0]


def _prompt_and_track(p, st):
    H, W = st["video_height"], st["video_width"]
    yy, xx = np.mgrid[0:H, 0:W]
    mask = (((yy - 300) / 90) ** 2 + ((xx - 600) / 140) ** 2 <= 1)
    calls = [("pts", dict(frame_idx=0, obj_id=1, points=[[400.0, 240.0]], labels=[1])),
             ("pts", dict(frame_idx=0, obj_id=2, box=[150.0, 80.0, 520.0, 400.0])),
             ("pts", dict(frame_idx=0, obj_id=1, points=[[330.0, 170.0]], labels=[0], clear_old_points=False)),
             ("mask", dict(frame_idx=2, obj_id=3, mask=mask))]
    outs = []
    for kind, kw in calls:
        if kind == "pts":
            outs.append(p.add_new_points_or_box(st, **kw))
        else:
            outs.append(p.add_new_mask(st, **kw))
    fwd = list(p.propagate_in_video(st, start_frame_idx=0))
    bwd = list(p.propagate_in_video(st, start_frame_idx=2, reverse=True))
    return outs, fwd, bwd


def test_end_to_end_from_init_state_matches_oracle(folders, predictors):
    ours, orc = predictors
    folder = folders["480x854"]
    st = ours.init_state(folder)
    ost = orc.init_state(folder)
    assert st.keys() == ost.keys()
    for k in st:
        assert type(st[k]) is type(ost[k]), k
    assert (st["video_height"], st["video_width"], st["num_frames"]) == (480, 854, 4)
    assert torch.equal(st["images"].cpu(), ost["images"])
    prompts_a, fwd_a, bwd_a = _prompt_and_track(ours, st)
    prompts_b, fwd_b, bwd_b = _prompt_and_track(orc, ost)
    for (f1, ids1, v1), (f2, ids2, v2) in zip(prompts_a, prompts_b):
        assert (f1, list(ids1)) == (f2, list(ids2)) and tuple(v1.shape) == tuple(v2.shape)
        present = (v2 > -1000).flatten(1).any(1)
        assert torch.equal((v1.cpu() > -1000).flatten(1).any(1), present)
        assert rel_l2(v1.cpu()[present].clamp(-64, 64), v2[present].clamp(-64, 64)) < 2e-2, f1
    for a, b in ((fwd_a, fwd_b), (bwd_a, bwd_b)):
        assert [x[0] for x in a] == [x[0] for x in b] and [list(x[1]) for x in a] == [list(x[1]) for x in b]
        for (fa, _, la), (_, _, lb) in zip(a, b):
            assert tuple(la.shape) == tuple(lb.shape) == (3, 1, 480, 854)
            r = rel_l2(la.clamp(-64, 64), lb.clamp(-64, 64))
            agree = ((la.cpu() > 0) == (lb > 0)).float().mean().item()
            print(f"frame {fa}: rel_l2={r:.4f} sign agreement={agree:.5f}")
            # every propagated frame has at least one object tracked from memory (recurrence on top of the prompt step)
            assert r < 3e-2, (fa, r)
            assert agree > 0.995, (fa, agree)
