"""Cost of loading a JPEG-folder video: the frame kernel and SAM2VideoPredictor.init_state.

Prints one JSON object with the card name and power limit read in the same run, and:
  * kernel: ops.resample_frames_u8 on 64 frames at 1080x1920 and 64 at 3000x4000 -> 1024^2 (uint8 in, fp32 out), median
    of CUDA-event times. The working sets (1.2 and 3.1 GB) are far larger than L2. The HBM floor counts the uint8 frames
    read once and the fp32 output written once, at 7.7 TB/s; the uint8 intermediate's write + read is reported apart;
  * init_state: wall time (host clock, ending in a device synchronise) of init_state on a folder of 200 JPEGs at
    1080x1920 (hiera-tiny, random init; frame 0 is encoded in both routes), alternating with the upstream route
    restated in the oracle (PIL decode + resize on the host, fp32 normalisation after the H2D copy) followed by the
    same state construction. The two image tensors are checked equal. The host JPEG decoding alone (the same thread
    pool) is timed too, and its share of init_state is reported.

    python tools/bench_video_frames.py [--out profiles/video_frames_bench.json]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

HBM_BYTES_PER_S = 7.7e12  # HGX B200 data sheet, one GPU
S = 1024


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else torch.cuda.get_device_name()


def kernel_rows(reps):
    from saber_b200 import ops
    from saber_b200.sam2 import video_io
    lut = video_io.normalize_lut().cuda()
    rows = []
    for (H, W) in ((1080, 1920), (3000, 4000)):
        N = 64
        g = torch.Generator(device="cuda").manual_seed(0)
        x = torch.randint(0, 256, (N, H, W, 3), dtype=torch.uint8, device="cuda", generator=g)
        out = torch.empty((N, 3, S, S), dtype=torch.float32, device="cuda")
        ops.resample_frames_u8(x, S, lut, out=out)
        times = []
        for _ in range(reps):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            ops.resample_frames_u8(x, S, lut, out=out)
            b.record()
            torch.cuda.synchronize()
            times.append(a.elapsed_time(b))
        _, _, _, y0, y1 = ops._frame_coeffs(H, S, x.device)
        floor_bytes = x.numel() + out.numel() * 4
        inter_bytes = 2 * N * (y1 - y0) * S * 3
        ms = float(np.median(times))
        rows.append({"frames": N, "in_hw": [H, W], "out": S, "ms": ms, "ms_per_frame": ms / N,
                     "floor_bytes": floor_bytes, "intermediate_bytes": inter_bytes,
                     "floor_ms": floor_bytes / HBM_BYTES_PER_S * 1e3,
                     "floor_with_intermediate_ms": (floor_bytes + inter_bytes) / HBM_BYTES_PER_S * 1e3,
                     "share_of_floor": floor_bytes / HBM_BYTES_PER_S * 1e3 / ms, "times_ms": times})
        print(json.dumps(rows[-1]), file=sys.stderr)
        del x, out
    return rows


def init_state_rows(reps, n_frames):
    from PIL import Image

    from oracle.sam2_ref import video_io as ovio
    from saber_b200.sam2 import video_io
    from saber_b200.sam2.sam2_video_predictor import build_sam2_video_predictor
    from saber_b200.sam2 import arch
    p = build_sam2_video_predictor("tiny", None, device="cuda:0", state_dict=arch.random_state_dict("tiny", seed=0))
    dev = p.device
    with tempfile.TemporaryDirectory() as folder:
        rng = np.random.default_rng(0)
        yy, xx = np.mgrid[0:1080, 0:1920].astype(np.float32)
        for i in range(n_frames):
            img = np.stack([128 + 90 * np.sin(xx / (150 + 7 * i) + c) * np.cos(yy / (110 + 3 * c)) for c in range(3)], -1)
            img = np.clip(img + rng.normal(0, 8, img.shape), 0, 255).astype(np.uint8)
            Image.fromarray(img).save(os.path.join(folder, f"{i:05d}.jpg"), quality=90)
        paths = video_io.jpeg_frame_paths(folder)

        def ours():
            st = p.init_state(folder)
            torch.cuda.synchronize()
            return st["images"]

        def upstream():
            images, vh, vw = ovio.load_video_frames(folder, S, False, compute_device=dev)
            p.new_inference_state(images, vh, vw, False, False, dev, dev)
            torch.cuda.synchronize()
            return images

        def decode_only():
            with ThreadPoolExecutor(max_workers=min(8, os.cpu_count() or 1)) as pool:
                list(pool.map(video_io._decode, paths))

        ours()
        upstream()
        t_ours, t_up, t_dec, equal = [], [], [], True
        for _ in range(reps):
            t = time.perf_counter()
            a = ours()
            t_ours.append(time.perf_counter() - t)
            t = time.perf_counter()
            b = upstream()
            t_up.append(time.perf_counter() - t)
            equal = equal and torch.equal(a, b)
            del a, b
            t = time.perf_counter()
            decode_only()
            t_dec.append(time.perf_counter() - t)
    row = {"frames": n_frames, "in_hw": [1080, 1920], "cpu_count": os.cpu_count(),
           "decode_threads": min(8, os.cpu_count() or 1), "init_state_s": float(np.median(t_ours)),
           "upstream_route_s": float(np.median(t_up)), "decode_only_s": float(np.median(t_dec)),
           "speedup": float(np.median(t_up) / np.median(t_ours)),
           "decode_share_of_init_state": float(np.median(t_dec) / np.median(t_ours)), "images_equal": bool(equal),
           "init_state_times_s": t_ours, "upstream_times_s": t_up, "decode_times_s": t_dec}
    print(json.dumps(row), file=sys.stderr)
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--init-reps", type=int, default=3)
    ap.add_argument("--frames", type=int, default=200)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_video_frames needs a CUDA device")
    res = {"card": card(), "kernel": kernel_rows(args.reps), "init_state": init_state_rows(args.init_reps, args.frames)}
    res["card_after"] = card()
    print(json.dumps(res))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
