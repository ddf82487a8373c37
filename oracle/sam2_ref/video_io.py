"""ORACLE (test infrastructure only). Restatement of upstream sam2's JPEG-folder video loading (sam2/utils/misc.py:
load_video_frames, load_video_frames_from_jpg_images, _load_img_as_tensor, AsyncVideoFrameLoader) on PIL, of
``SAM2VideoPredictor.init_state`` (sam2/sam2_video_predictor.py) on the oracle predictor, and a numpy int64
restatement of Pillow's 8-bit bicubic resize (libImaging/Resample.c) that the device kernel reproduces.
"""
from __future__ import annotations

import math
import os
from collections import OrderedDict
from threading import Thread

import numpy as np
import torch
from PIL import Image

from .sam2_base import _load
from .video_predictor import SAM2VideoPredictor as _OracleVideoPredictor

IMG_MEAN = (0.485, 0.456, 0.406)
IMG_STD = (0.229, 0.224, 0.225)


# ---- Pillow's ImagingResample for 8-bit images, BICUBIC (a = -0.5), 22-bit fixed point -----------------------------
PRECISION_BITS = 22


def _bicubic(x):
    a = -0.5
    if x < 0.0:
        x = -x
    if x < 1.0:
        return ((a + 2.0) * x - (a + 3.0)) * x * x + 1
    if x < 2.0:
        return (((x - 5) * x + 8) * x - 4) * a
    return 0.0


def pillow_coeffs(n_in: int, n_out: int):
    """precompute_coeffs + normalize_coeffs_8bpc: per output index (xmin, n) and the int weights [n_out, ksize]."""
    scale = n_in / n_out
    fs = max(scale, 1.0)
    support = 2.0 * fs
    ksize = int(math.ceil(support)) * 2 + 1
    kk = np.zeros((n_out, ksize), np.int64)
    bounds = []
    for xx in range(n_out):
        center = (xx + 0.5) * scale
        ss = 1.0 / fs
        xmin = max(int(center - support + 0.5), 0)
        n = min(int(center + support + 0.5), n_in) - xmin
        w = [_bicubic((x + xmin - center + 0.5) * ss) for x in range(n)]
        ww = 0.0
        for v in w:
            ww += v
        w = [v / ww if ww != 0.0 else v for v in w]
        for x, v in enumerate(w):
            kk[xx, x] = int(-0.5 + v * (1 << PRECISION_BITS)) if v < 0 else int(0.5 + v * (1 << PRECISION_BITS))
        bounds.append((xmin, n))
    return kk, bounds


def _clip8(acc):
    return np.clip(acc >> PRECISION_BITS, 0, 255)


def pillow_resize_u8(img: np.ndarray, S: int) -> np.ndarray:
    """``np.asarray(Image.fromarray(img).resize((S, S)))`` for an RGB uint8 [H, W, 3] image, in int64 numpy: the
    horizontal pass over the source rows the vertical taps reach, a uint8 intermediate, then the vertical pass; a pass
    is skipped when its axis already has size S."""
    H, W = img.shape[:2]
    if (H, W) == (S, S):
        return img.copy()
    kx, bx = pillow_coeffs(W, S)
    ky, by = pillow_coeffs(H, S)
    y0, y1 = by[0][0], by[-1][0] + by[-1][1]
    src = img.astype(np.int64)
    if W != S:
        tmp = np.empty((y1 - y0, S, 3), np.int64)
        for xx, (xmin, n) in enumerate(bx):
            acc = (1 << (PRECISION_BITS - 1)) + np.einsum("yxc,x->yc", src[y0:y1, xmin:xmin + n], kx[xx, :n])
            tmp[:, xx] = _clip8(acc)
    else:
        y0, tmp = 0, src
    if H == S:
        return tmp.astype(np.uint8)
    out = np.empty((S, S, 3), np.int64)
    for yy, (ymin, n) in enumerate(by):
        acc = (1 << (PRECISION_BITS - 1)) + np.einsum("yxc,y->xc", tmp[ymin - y0:ymin - y0 + n], ky[yy, :n])
        out[yy] = _clip8(acc)
    return out.astype(np.uint8)


def normalized_frames(frames_u8: np.ndarray, S: int, float64_path: bool = False) -> torch.Tensor:
    """[N, H, W, 3] uint8 -> [N, 3, S, S] fp32 through ``pillow_resize_u8`` and upstream's normalisation: the
    synchronous loader's fp32 ``(v/255 - mean) / std`` or (``float64_path``) the async loader's float64 one, cast."""
    out = []
    for f in frames_u8:
        x = torch.from_numpy(pillow_resize_u8(f, S) / 255.0).permute(2, 0, 1)
        mean = torch.tensor(IMG_MEAN, dtype=torch.float32)[:, None, None]
        std = torch.tensor(IMG_STD, dtype=torch.float32)[:, None, None]
        out.append(((x - mean) / std).float() if float64_path else (x.float() - mean) / std)
    return torch.stack(out)


# ---- sam2/utils/misc.py ---------------------------------------------------------------------------------------------
def _load_img_as_tensor(img_path, image_size):
    img_pil = Image.open(img_path)
    img_np = np.array(img_pil.convert("RGB").resize((image_size, image_size)))
    if img_np.dtype == np.uint8:  # np.uint8 is expected for JPEG images
        img_np = img_np / 255.0
    else:
        raise RuntimeError(f"Unknown image dtype: {img_np.dtype} on {img_path}")
    img = torch.from_numpy(img_np).permute(2, 0, 1)
    video_width, video_height = img_pil.size  # the original video size
    return img, video_height, video_width


class AsyncVideoFrameLoader:
    """Loads frame 0 in the constructor and the rest in a daemon thread; frames are float64 [3, S, S]."""

    def __init__(self, img_paths, image_size, offload_video_to_cpu, img_mean, img_std, compute_device):
        self.img_paths = img_paths
        self.image_size = image_size
        self.offload_video_to_cpu = offload_video_to_cpu
        self.img_mean = img_mean
        self.img_std = img_std
        self.images = [None] * len(img_paths)
        self.exception = None
        self.video_height = None
        self.video_width = None
        self.compute_device = compute_device
        self.__getitem__(0)

        def _load_frames():
            try:
                for n in range(len(self.images)):
                    self.__getitem__(n)
            except Exception as e:
                self.exception = e

        self.thread = Thread(target=_load_frames, daemon=True)
        self.thread.start()

    def __getitem__(self, index):
        if self.exception is not None:
            raise RuntimeError("Failure in frame loading thread") from self.exception
        img = self.images[index]
        if img is not None:
            return img
        img, video_height, video_width = _load_img_as_tensor(self.img_paths[index], self.image_size)
        self.video_height = video_height
        self.video_width = video_width
        img -= self.img_mean
        img /= self.img_std
        if not self.offload_video_to_cpu:
            img = img.to(self.compute_device, non_blocking=True)
        self.images[index] = img
        return img

    def __len__(self):
        return len(self.images)


def load_video_frames_from_jpg_images(video_path, image_size, offload_video_to_cpu, img_mean=IMG_MEAN,
                                      img_std=IMG_STD, async_loading_frames=False, compute_device=torch.device("cuda")):
    if isinstance(video_path, str) and os.path.isdir(video_path):
        jpg_folder = video_path
    else:
        raise NotImplementedError("Only JPEG frames are supported at this moment.")
    frame_names = [p for p in os.listdir(jpg_folder) if os.path.splitext(p)[-1] in [".jpg", ".jpeg", ".JPG", ".JPEG"]]
    frame_names.sort(key=lambda p: int(os.path.splitext(p)[0]))
    num_frames = len(frame_names)
    if num_frames == 0:
        raise RuntimeError(f"no images found in {jpg_folder}")
    img_paths = [os.path.join(jpg_folder, frame_name) for frame_name in frame_names]
    img_mean = torch.tensor(img_mean, dtype=torch.float32)[:, None, None]
    img_std = torch.tensor(img_std, dtype=torch.float32)[:, None, None]
    if async_loading_frames:
        lazy_images = AsyncVideoFrameLoader(img_paths, image_size, offload_video_to_cpu, img_mean, img_std,
                                            compute_device)
        return lazy_images, lazy_images.video_height, lazy_images.video_width
    images = torch.zeros(num_frames, 3, image_size, image_size, dtype=torch.float32)
    for n, img_path in enumerate(img_paths):
        images[n], video_height, video_width = _load_img_as_tensor(img_path, image_size)
    if not offload_video_to_cpu:
        images = images.to(compute_device)
        img_mean = img_mean.to(compute_device)
        img_std = img_std.to(compute_device)
    images -= img_mean
    images /= img_std
    return images, video_height, video_width


def load_video_frames(video_path, image_size, offload_video_to_cpu, img_mean=IMG_MEAN, img_std=IMG_STD,
                      async_loading_frames=False, compute_device=torch.device("cuda")):
    is_bytes = isinstance(video_path, bytes)
    is_str = isinstance(video_path, str)
    is_mp4_path = is_str and os.path.splitext(video_path)[-1] in [".mp4", ".MP4"]
    if is_bytes or is_mp4_path:
        raise NotImplementedError("MP4 decoding (decord) is not restated in the oracle")
    elif is_str and os.path.isdir(video_path):
        return load_video_frames_from_jpg_images(video_path, image_size, offload_video_to_cpu, img_mean, img_std,
                                                 async_loading_frames, compute_device)
    raise NotImplementedError("Only MP4 video and JPEG folder are supported at this moment")


# ---- sam2/sam2_video_predictor.py: init_state ----------------------------------------------------------------------
class SAM2VideoPredictor(_OracleVideoPredictor):
    """The oracle video predictor with upstream's ``init_state``."""

    @torch.inference_mode()
    def init_state(self, video_path, offload_video_to_cpu=False, offload_state_to_cpu=False,
                   async_loading_frames=False):
        compute_device = self.device
        images, video_height, video_width = load_video_frames(
            video_path=video_path, image_size=self.image_size, offload_video_to_cpu=offload_video_to_cpu,
            async_loading_frames=async_loading_frames, compute_device=compute_device)
        inference_state = {}
        inference_state["images"] = images
        inference_state["num_frames"] = len(images)
        inference_state["offload_video_to_cpu"] = offload_video_to_cpu
        inference_state["offload_state_to_cpu"] = offload_state_to_cpu
        inference_state["video_height"] = video_height
        inference_state["video_width"] = video_width
        inference_state["device"] = compute_device
        if offload_state_to_cpu:
            inference_state["storage_device"] = torch.device("cpu")
        else:
            inference_state["storage_device"] = compute_device
        inference_state["point_inputs_per_obj"] = {}
        inference_state["mask_inputs_per_obj"] = {}
        inference_state["cached_features"] = {}
        inference_state["constants"] = {}
        inference_state["obj_id_to_idx"] = OrderedDict()
        inference_state["obj_idx_to_id"] = OrderedDict()
        inference_state["obj_ids"] = []
        inference_state["output_dict_per_obj"] = {}
        inference_state["temp_output_dict_per_obj"] = {}
        inference_state["frames_tracked_per_obj"] = {}
        self._get_image_feature(inference_state, frame_idx=0, batch_size=1)
        return inference_state


def build_sam2_video_predictor(config_file="large", ckpt_path=None, device="cpu", mode="eval", apply_postprocessing=True,
                               vos_optimized=False, state_dict=None, **kw):
    """``video_predictor.build_sam2_video_predictor`` returning the predictor with ``init_state``."""
    model = SAM2VideoPredictor(cfg=config_file, fill_hole_area=8, binarize_mask_from_pts_for_mem_enc=True,
                               dynamic_multimask_via_stability=bool(apply_postprocessing), **kw)
    _load(model, ckpt_path, state_dict)
    return model.to(device).eval()
