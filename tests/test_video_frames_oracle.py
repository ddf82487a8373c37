"""CPU: the fixed-point restatement of Pillow's bicubic resize (the device kernel's reference) equals Pillow bit for bit,
the product's coefficient tables equal the restatement's, and the JPEG-folder rules of ``load_video_frames`` are
upstream's."""
import os

import numpy as np
import pytest
from PIL import Image

from oracle.sam2_ref import video_io as ovio
from saber_b200 import ops
from saber_b200.sam2 import video_io

SIZES = [(96, 120), (480, 854), (1080, 1920), (1024, 1024), (1, 1), (3000, 4000), (1024, 700), (700, 1024),
         (2000, 1024), (37, 2500)]


@pytest.mark.parametrize("hw", SIZES)
def test_fixed_point_resize_equals_pillow(hw):
    img = np.random.default_rng(hw[0] * 7 + hw[1]).integers(0, 256, hw + (3,), dtype=np.uint8)
    want = np.asarray(Image.fromarray(img).resize((1024, 1024)))
    np.testing.assert_array_equal(ovio.pillow_resize_u8(img, 1024), want)


@pytest.mark.parametrize("hw", [(1024, 333), (1024, 1500), (64, 1024), (1800, 1024)])
def test_fixed_point_resize_with_one_axis_at_size(hw):
    img = np.random.default_rng(hw[1]).integers(0, 256, hw + (3,), dtype=np.uint8)
    want = np.asarray(Image.fromarray(img).resize((1024, 1024)))
    np.testing.assert_array_equal(ovio.pillow_resize_u8(img, 1024), want)


@pytest.mark.parametrize("mode", ["L", "CMYK"])
def test_grayscale_and_cmyk_jpegs_after_convert(tmp_path, mode):
    rng = np.random.default_rng(3)
    chans = {"L": 1, "CMYK": 4}[mode]
    arr = rng.integers(0, 256, (150, 211, chans), dtype=np.uint8)
    Image.fromarray(arr[..., 0] if chans == 1 else arr, mode).save(tmp_path / "0.jpg", quality=90)
    with Image.open(tmp_path / "0.jpg") as im:
        assert im.mode == mode
        rgb = np.asarray(im.convert("RGB"))
        want = np.asarray(im.convert("RGB").resize((1024, 1024)))
    np.testing.assert_array_equal(ovio.pillow_resize_u8(rgb, 1024), want)
    got, h, w = video_io._decode(str(tmp_path / "0.jpg"))
    np.testing.assert_array_equal(got, rgb)
    assert (h, w) == (150, 211)


@pytest.mark.parametrize("n_in", [1, 37, 96, 120, 480, 700, 854, 1080, 1920, 2000, 2500, 3000, 4000])
def test_product_coefficients_equal_restatement(n_in):
    kk, bounds = ovio.pillow_coeffs(n_in, 1024)
    b, w = ops.pillow_bicubic_coeffs(n_in, 1024)
    np.testing.assert_array_equal(b, np.array(bounds))
    np.testing.assert_array_equal(w, kk)


def test_normalize_luts_follow_upstream_arithmetic():
    import torch
    v = torch.from_numpy(np.arange(256, dtype=np.uint8)[None, None, :].repeat(3, 0) / 255.0)  # [3,1,256] float64
    mean = torch.tensor(ovio.IMG_MEAN, dtype=torch.float32)[:, None, None]
    std = torch.tensor(ovio.IMG_STD, dtype=torch.float32)[:, None, None]
    sync = (v.float() - mean) / std  # images[n] = float64 frame (cast to fp32); images -= mean; images /= std
    x = v.clone()
    x -= mean
    x /= std  # async path: in place on the float64 frame
    assert torch.equal(video_io.normalize_lut(), sync[:, 0])
    assert torch.equal(video_io.normalize_lut(float64_path=True), x.float()[:, 0])
    assert not torch.equal(video_io.normalize_lut(), video_io.normalize_lut(float64_path=True))


def _touch(folder, names):
    for n in names:
        Image.new("RGB", (8, 6)).save(os.path.join(folder, n), format="JPEG")


def test_folder_rules(tmp_path):
    _touch(tmp_path, ["10.jpg", "2.JPEG", "1.jpeg", "003.JPG", "4.png", "5.bmp"])
    (tmp_path / "notes.txt").write_text("x")
    got = [os.path.basename(p) for p in video_io.jpeg_frame_paths(str(tmp_path))]
    assert got == ["1.jpeg", "2.JPEG", "003.JPG", "10.jpg"]
    frame_names = [p for p in os.listdir(tmp_path) if os.path.splitext(p)[-1] in [".jpg", ".jpeg", ".JPG", ".JPEG"]]
    frame_names.sort(key=lambda p: int(os.path.splitext(p)[0]))
    assert got == frame_names  # upstream's own expression
    _touch(tmp_path, ["cover.jpg"])
    with pytest.raises(ValueError):
        video_io.jpeg_frame_paths(str(tmp_path))
    empty = tmp_path / "empty"
    empty.mkdir()
    _touch(empty, ["0.png"])
    with pytest.raises(RuntimeError, match="no images found in"):
        video_io.load_video_frames(str(empty), 1024, False)


@pytest.mark.parametrize("src", ["clip.mp4", "clip.MP4", b"\x00\x00\x00\x18ftypmp42"])
def test_mp4_input_is_not_built(tmp_path, src):
    path = str(tmp_path / src) if isinstance(src, str) else src
    with pytest.raises(NotImplementedError, match="MP4"):
        video_io.load_video_frames(path, 1024, False)


@pytest.mark.parametrize("src", ["frames_missing", "video.avi", 7])
def test_other_inputs_are_rejected_as_upstream(tmp_path, src):
    path = str(tmp_path / src) if isinstance(src, str) else src
    with pytest.raises(NotImplementedError, match="Only MP4 video and JPEG folder are supported at this moment"):
        video_io.load_video_frames(path, 1024, False)
