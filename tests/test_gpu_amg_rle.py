"""-m gpu: run-length encoding on the device. The kernels bit for bit against the oracle's mask_to_rle and COCO encoder
on packed masks (ragged widths, odd heights, 1x1 frames, empty / full / first-pixel / last-pixel masks, the maximum
H*W + 1 counts, garbage in the padding bits, a row selection, one and hundreds of masks), and the AMG's
"uncompressed_rle" / "coco_rle" output modes against its binary output on the same image."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def pack(masks, rng=None):
    """bool [m, H, W] -> int32 [m, H, ceil(W/32)]; with rng the bits past W are random"""
    m, H, W = masks.shape
    WW = (W + 31) // 32
    pad = np.zeros((m, H, WW * 32), bool)
    pad[:, :, :W] = masks
    if rng is not None:
        pad[:, :, W:] = rng.uniform(size=(m, H, WW * 32 - W)) < 0.5
    return np.packbits(pad, axis=-1, bitorder="little").view("<u4").view(np.int32).reshape(m, H, WW)


def edge_masks(H, W, rng):
    first = np.zeros((H, W), bool)
    first[0, 0] = True
    last = np.zeros((H, W), bool)
    last[-1, -1] = True
    alt = (np.arange(H * W) % 2 == 0).reshape(W, H).T  # column-major alternation from a set pixel: H*W + 1 counts
    yy, xx = np.mgrid[0:H, 0:W]
    blob = ((yy - H / 2) / max(H / 3, 1)) ** 2 + ((xx - W / 3) / max(W / 4, 1)) ** 2 < 1
    return np.stack([np.zeros((H, W), bool), np.ones((H, W), bool), first, last, alt, blob,
                     rng.uniform(size=(H, W)) < 0.5, rng.uniform(size=(H, W)) < 0.02])


def check(masks, got_counts, got_off, got_chars, got_coff):
    from oracle.sam2_ref import amg as up
    from oracle.sam2_ref.coco_rle import counts_to_string
    counts, off = got_counts.cpu().numpy(), got_off.cpu().numpy()
    chars, coff = got_chars.cpu().numpy().tobytes().decode("ascii"), got_coff.cpu().numpy()
    assert len(off) == len(coff) == len(masks) + 1
    assert off[-1] == len(counts) and coff[-1] == len(chars)
    for i, mk in enumerate(masks):
        want = up.mask_to_rle(mk)["counts"]
        assert counts[off[i]:off[i + 1]].tolist() == want, f"mask {i}"
        assert chars[coff[i]:coff[i + 1]] == counts_to_string(want), f"mask {i}"


def run(bits, sel, m, W):
    from saber_b200 import ops
    counts, off = ops.masks_to_rle(bits, sel, m, W)
    chars, coff = ops.masks_to_rle(bits, sel, m, W, coco=True)
    return counts, off, chars, coff


@pytest.mark.parametrize("hw", [(1, 1), (1, 33), (7, 1), (31, 927), (33, 1000), (300, 517), (1024, 1024), (96, 2085)])
def test_rle_kernels_match_oracle(hw):
    H, W = hw
    rng = np.random.default_rng(H * 7919 + W)
    masks = edge_masks(H, W, rng)
    bits = torch.from_numpy(pack(masks, rng)).cuda()
    check(masks, *run(bits, None, len(masks), W))


def test_rle_kernels_single_mask_and_max_counts():
    H, W = 37, 45
    alt = (np.arange(H * W) % 2 == 0).reshape(W, H).T[None]
    bits = torch.from_numpy(pack(alt, np.random.default_rng(1))).cuda()
    counts, off, chars, coff = run(bits, None, 1, W)
    assert int(off[1]) == H * W + 1
    check(alt, counts, off, chars, coff)


def test_rle_kernels_row_selection_hundreds_of_masks():
    H, W = 129, 200
    rng = np.random.default_rng(5)
    n = 300
    yy, xx = np.mgrid[0:H, 0:W]
    masks = []
    for i in range(n):
        if i % 3 == 0:
            masks.append(rng.uniform(size=(H, W)) < rng.uniform(0.01, 0.9))
        else:
            cy, cx, ry, rx = rng.uniform(0, H), rng.uniform(0, W), rng.uniform(2, H / 2), rng.uniform(2, W / 2)
            masks.append(((yy - cy) / ry) ** 2 + ((xx - cx) / rx) ** 2 < 1)
    masks = np.stack(masks)
    bits = torch.from_numpy(pack(masks, rng)).cuda()
    perm = rng.permutation(n)[:257].astype(np.int32)
    sel = torch.from_numpy(perm).cuda()
    check(masks[perm], *run(bits, sel, len(perm), W))
    # the first m rows without a selection
    check(masks[:100], *run(bits, None, 100, W))


def test_rle_zero_masks():
    from saber_b200 import ops
    bits = torch.zeros((4, 8, 1), dtype=torch.int32, device="cuda")
    counts, off = ops.masks_to_rle(bits, None, 0, 20)
    assert counts.numel() == 0 and off.tolist() == [0]


# ---------------------------------------------------------------------------------------------- AMG output modes
@pytest.fixture(scope="module")
def tiny():
    from saber_b200.sam2 import arch
    from saber_b200.sam2.build_sam import build_sam2
    sd = arch.random_state_dict("tiny", seed=0)
    for k in list(sd):  # realistic logit range, as tests/test_gpu_amg.py::tiny
        if "output_hypernetworks_mlps" in k and ".layers.2." in k:
            sd[k] = sd[k] * 30.0
    return build_sam2("tiny", None, device="cuda", state_dict=sd, apply_postprocessing=True)


AMG_KW = dict(points_per_side=8, crop_n_layers=1, crop_n_points_downscale_factor=2, box_nms_thresh=0.95,
              stability_score_offset=0.7, pred_iou_thresh=0.3, stability_score_thresh=0.2, use_m2m=True,
              multimask_output=True)


@pytest.mark.parametrize("min_area", [0, 25])
def test_amg_rle_output_modes_match_binary(tiny, min_area):
    from oracle.sam2_ref import amg as up
    from oracle.sam2_ref.coco_rle import coco_decode_rle
    from saber_b200 import synth
    from saber_b200.sam2.automatic_mask_generator import SAM2AutomaticMaskGenerator
    from saber_b200.utils import preprocessing as prep
    img = prep.prepare(synth.make_tomogram((1, 300, 517), seed=2, n_ellipsoids=10)[0].numpy(), to_rgb=True)
    res = {}
    for mode in ("binary_mask", "uncompressed_rle", "coco_rle"):
        gen = SAM2AutomaticMaskGenerator(tiny, min_mask_region_area=min_area, output_mode=mode, **AMG_KW)
        res[mode] = gen.generate(img)
    binary = res["binary_mask"]
    assert len(binary) > 0
    for mode in ("uncompressed_rle", "coco_rle"):
        got = res[mode]
        assert len(got) == len(binary)
        for i, (g, b) in enumerate(zip(got, binary)):
            assert list(g) == list(b), (mode, i)  # same keys in the same order
            seg = g["segmentation"]
            assert seg["size"] == [300, 517]
            if mode == "coco_rle":
                assert isinstance(seg["counts"], str)
                rle = coco_decode_rle(seg)
            else:
                assert isinstance(seg["counts"], list) and all(type(c) is int for c in seg["counts"])
                rle = seg
            np.testing.assert_array_equal(up.rle_to_mask(rle), b["segmentation"], err_msg=f"{mode} mask {i}")
            assert g["area"] == up.area_from_rle(rle) == b["area"], (mode, i)
            for key in ("bbox", "predicted_iou", "point_coords", "stability_score", "crop_box"):
                assert g[key] == b[key], (mode, i, key)


def test_unknown_output_mode_raises():
    from saber_b200.sam2.automatic_mask_generator import SAM2AutomaticMaskGenerator
    with pytest.raises(ValueError):
        SAM2AutomaticMaskGenerator(None, output_mode="foo")
