"""Drop-in for upstream's ``sam2.utils.misc.load_video_frames`` on a JPEG folder, with the resize and normalisation on
the device.

Frames are decoded on the host exactly as upstream decodes them (``Image.open(p).convert("RGB")``, in a thread pool),
cross PCIe as uint8 at their own size through pinned staging, and are resized and normalised by
``ops.resample_frames_u8``: Pillow's 8-bit bicubic ``resize((S, S))`` bit for bit, then a 3 x 256 lookup table built
here with upstream's own arithmetic. The frames therefore equal upstream's bit for bit.

Difference: upstream's ``async_loading_frames=True`` path returns float64 frames (its in-place normalisation promotes
them), which ``_get_image_feature`` casts with ``.float()``. ``AsyncVideoFrameLoader`` here returns fp32 frames equal to
that cast.
"""
from __future__ import annotations

import os
from concurrent.futures import ThreadPoolExecutor
from threading import Thread
from typing import List, Tuple

import numpy as np
import torch
from PIL import Image

from .. import ops

IMG_MEAN = (0.485, 0.456, 0.406)
IMG_STD = (0.229, 0.224, 0.225)
JPEG_EXTS = (".jpg", ".jpeg", ".JPG", ".JPEG")
CHUNK_FRAMES = 16  # frames decoded, staged and resized together; host memory holds at most two chunks


def normalize_lut(float64_path: bool = False) -> torch.Tensor:
    """[3, 256] fp32: the value upstream gives byte v of channel c. Synchronous path: ``v / 255.0`` in float64, stored
    as fp32, then ``(x - mean) / std`` in fp32. Async path (``float64_path``): the same in float64 against the fp32
    mean / std, rounded to fp32 (upstream's float64 frame after ``.float()``)."""
    v = torch.from_numpy(np.arange(256, dtype=np.uint8) / 255.0)  # float64
    mean = torch.tensor(IMG_MEAN, dtype=torch.float32)[:, None]
    std = torch.tensor(IMG_STD, dtype=torch.float32)[:, None]
    if float64_path:
        return ((v[None] - mean.double()) / std.double()).float().contiguous()
    return ((v.float()[None] - mean) / std).contiguous()


def jpeg_frame_paths(folder: str) -> List[str]:
    """Upstream's frame list: files with a JPEG extension, sorted by the integer value of their stem (a non-integer
    stem raises ValueError)."""
    names = [p for p in os.listdir(folder) if os.path.splitext(p)[-1] in JPEG_EXTS]
    names.sort(key=lambda p: int(os.path.splitext(p)[0]))
    if not names:
        raise RuntimeError(f"no images found in {folder}")
    return [os.path.join(folder, n) for n in names]


def _decode(path: str) -> Tuple[np.ndarray, int, int]:
    """-> (uint8 [H, W, 3], video_height, video_width), decoded as upstream's _load_img_as_tensor decodes."""
    with Image.open(path) as img:
        rgb = np.asarray(img.convert("RGB"))
        w, h = img.size
    return rgb, h, w


def _to_device_frames(rgbs: List[np.ndarray], S: int, lut: torch.Tensor, out: torch.Tensor) -> None:
    """Stage decoded frames through pinned memory and resize them into ``out`` [len(rgbs), 3, S, S] on the device: one
    kernel call per distinct frame size."""
    dev = out.device
    groups = {}
    for i, r in enumerate(rgbs):
        groups.setdefault(r.shape, []).append(i)
    for shape, idx in groups.items():
        stage = torch.empty((len(idx),) + shape, dtype=torch.uint8, pin_memory=True)
        host = stage.numpy()
        for j, i in enumerate(idx):
            host[j] = rgbs[i]
        frames = stage.to(dev, non_blocking=True)  # the pinned block is reused only after this copy completes
        if len(idx) == len(rgbs):
            ops.resample_frames_u8(frames, S, lut, out=out)
        else:
            out[torch.tensor(idx, device=dev)] = ops.resample_frames_u8(frames, S, lut)


def _load_jpg_frames(paths: List[str], S: int, offload_video_to_cpu: bool, device: torch.device):
    N = len(paths)
    lut = normalize_lut().to(device)
    images = torch.empty((N, 3, S, S), dtype=torch.float32, device="cpu" if offload_video_to_cpu else device)
    chunks = [paths[c:c + CHUNK_FRAMES] for c in range(0, N, CHUNK_FRAMES)]
    with ThreadPoolExecutor(max_workers=min(8, os.cpu_count() or 1)) as pool:
        pending = [pool.submit(_decode, p) for p in chunks[0]]
        c0 = 0
        for k in range(len(chunks)):
            decoded = [f.result() for f in pending]
            # decode the next chunk while this one is staged and resized
            pending = [pool.submit(_decode, p) for p in chunks[k + 1]] if k + 1 < len(chunks) else []
            n = len(decoded)
            dst = images[c0:c0 + n] if not offload_video_to_cpu else torch.empty((n, 3, S, S), dtype=torch.float32,
                                                                                   device=device)
            _to_device_frames([d[0] for d in decoded], S, lut, dst)
            if offload_video_to_cpu:
                images[c0:c0 + n].copy_(dst)
            c0 += n
            video_height, video_width = decoded[-1][1], decoded[-1][2]  # upstream's loop leaves the last frame's size
    return images, video_height, video_width


class AsyncVideoFrameLoader:
    """Upstream's lazy frame list: frame 0 is loaded before the constructor returns, a daemon thread (``.thread``)
    loads the rest in order. Frames are fp32 [3, S, S] (upstream: float64, see the module docstring); a frame made by
    the thread is complete before it is published and is returned ready to be read on the caller's stream. An error in
    the thread is raised from ``__getitem__``."""

    def __init__(self, img_paths, image_size, offload_video_to_cpu, compute_device):
        self.img_paths = img_paths
        self.image_size = image_size
        self.offload_video_to_cpu = offload_video_to_cpu
        self.compute_device = torch.device(compute_device)
        self.images = [None] * len(img_paths)
        self._side = [False] * len(img_paths)  # made on the loader thread's stream
        self.exception = None
        self._lut = normalize_lut(float64_path=True).to(self.compute_device)
        self._stream = torch.cuda.Stream(device=self.compute_device)
        self.video_height = None
        self.video_width = None
        self.__getitem__(0)  # fills video_height / video_width

        def _load_frames():
            try:
                with torch.cuda.device(self.compute_device), torch.cuda.stream(self._stream):
                    for n in range(len(self.images)):
                        self._load(n, side=True)
            except Exception as e:
                self.exception = e

        self.thread = Thread(target=_load_frames, daemon=True)
        self.thread.start()

    def _load(self, index, side=False):
        img = self.images[index]
        if img is not None:
            return img
        rgb, h, w = _decode(self.img_paths[index])
        if self.video_height is None:
            self.video_height, self.video_width = h, w
        stage = torch.empty((1,) + rgb.shape, dtype=torch.uint8, pin_memory=True)
        stage.numpy()[0] = rgb
        frames = stage.to(self.compute_device, non_blocking=True)
        img = ops.resample_frames_u8(frames, self.image_size, self._lut)[0]
        if self.offload_video_to_cpu:
            img = img.cpu()
        elif side:
            self._stream.synchronize()
        self._side[index] = side and not self.offload_video_to_cpu
        self.images[index] = img
        return img

    def __getitem__(self, index):
        if self.exception is not None:
            raise RuntimeError("Failure in frame loading thread") from self.exception
        img = self._load(index)
        if self._side[index]:
            # allocated on the loader's stream: keep its memory from being reused while the caller's stream reads it
            img.record_stream(torch.cuda.current_stream(self.compute_device))
        return img

    def __len__(self):
        return len(self.images)


def load_video_frames(video_path, image_size, offload_video_to_cpu, async_loading_frames=False,
                      compute_device=torch.device("cuda")):
    """upstream ``load_video_frames`` (default mean / std) -> (images, video_height, video_width). ``images`` is fp32
    [N, 3, S, S] on ``compute_device`` (on the host with ``offload_video_to_cpu``), or an ``AsyncVideoFrameLoader``."""
    is_bytes = isinstance(video_path, bytes)
    is_str = isinstance(video_path, str)
    if is_bytes or (is_str and os.path.splitext(video_path)[-1] in (".mp4", ".MP4")):
        raise NotImplementedError("MP4 video decoding is not built in saber_b200; extract the frames to a folder of "
                                  "JPEG files (e.g. with ffmpeg) and pass the folder")
    if not (is_str and os.path.isdir(video_path)):
        raise NotImplementedError("Only MP4 video and JPEG folder are supported at this moment")
    paths = jpeg_frame_paths(video_path)
    device = torch.device(compute_device)
    if device.type != "cuda":
        raise RuntimeError("saber_b200 resizes video frames on a CUDA device; there is no CPU path")
    with torch.cuda.device(device):
        if async_loading_frames:
            lazy = AsyncVideoFrameLoader(paths, image_size, offload_video_to_cpu, device)
            return lazy, lazy.video_height, lazy.video_width
        return _load_jpg_frames(paths, image_size, offload_video_to_cpu, device)
