"""Cost of the AMG's run-length encoded output modes ("uncompressed_rle", "coco_rle") against "binary_mask".

Prints one JSON object with the card name and power limit read in the same run, and:
  * kernels: the device RLE of 64 and 256 noise-like and blob-like 1024x1024 packed masks, per phase (sizing, counts,
    COCO sizing, COCO characters), median of CUDA-event times with L2 overwritten (a 256 MiB write) before every timed
    launch, against the HBM floor: the bytes the phase must move (packed masks read once; counts written; counts read
    and characters written) at 7.7 TB/s;
  * e2e: the wall time of generate() per slice (host clock around the call, which ends with the copies to the host) at
    config 1 — hiera-L random init, 1024^2 synthetic tomogram slices, SABER's AMG defaults with the thresholds opened as
    bench.py --thresholds open, min_mask_region_area 25 — for the three output modes, alternating mode order slice by
    slice, with the bytes each mode copies to the host.

    python tools/bench_rle.py [--slices 6] [--out profiles/rle_bench.json]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

HBM_BYTES_PER_S = 7.7e12  # HGX B200 data sheet, one GPU


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else torch.cuda.get_device_name()


def time_ms(fn, flush, reps=20, warm=3):
    for _ in range(warm):
        fn()
    ts = []
    for _ in range(reps):
        flush()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    return float(np.median(ts))


def masks(kind, m, H=1024, W=1024):
    g = torch.Generator(device="cuda").manual_seed(m + (0 if kind == "noise" else 1))
    if kind == "noise":
        return torch.randint(-2 ** 31, 2 ** 31 - 1, (m, H, W // 32), dtype=torch.int32, device="cuda", generator=g)
    # blob-like: one ellipse per mask, packed
    yy = torch.arange(H, device="cuda", dtype=torch.float32)[:, None]
    xx = torch.arange(W, device="cuda", dtype=torch.float32)[None, :]
    p = torch.rand((m, 4), device="cuda", generator=g)
    cy, cx = p[:, 0, None, None] * H, p[:, 1, None, None] * W
    ry, rx = 20 + p[:, 2, None, None] * H / 3, 20 + p[:, 3, None, None] * W / 3
    dense = ((yy - cy) / ry) ** 2 + ((xx - cx) / rx) ** 2 < 1  # [m, H, W]
    weights = (2 ** torch.arange(32, device="cuda", dtype=torch.int64))
    words = (dense.view(m, H, W // 32, 32).to(torch.int64) * weights).sum(-1)
    return words.to(torch.int64).where(words < 2 ** 31, words - 2 ** 32).to(torch.int32).contiguous()


def bench_kernels(kind, m, flush, H=1024, W=1024):
    from saber_b200 import lib, ops
    L = lib.load()
    bits = masks(kind, m, H, W)
    counts, off = ops.masks_to_rle(bits, None, m, W)
    chars, coff = ops.masks_to_rle(bits, None, m, W, coco=True)
    n_counts, n_chars = int(off[-1]), int(coff[-1])
    ws = torch.empty((2 * m * W,), dtype=torch.int32, device="cuda")
    off2, coff2 = torch.empty_like(off), torch.empty_like(coff)
    cnt2, chr2 = torch.empty_like(counts), torch.empty_like(chars)
    st = ops._stream

    def size():
        lib.check(L.sb_masks_rle_size(bits.data_ptr(), None, m, H, W, ws.data_ptr(), off2.data_ptr(), st()), "size")

    def emit():
        lib.check(L.sb_masks_rle_counts(bits.data_ptr(), None, m, H, W, ws.data_ptr(), off.data_ptr(),
                                        cnt2.data_ptr(), st()), "counts")

    def coco_size():
        lib.check(L.sb_masks_rle_coco_size(counts.data_ptr(), off.data_ptr(), m, coff2.data_ptr(), st()), "coco_size")

    def coco():
        lib.check(L.sb_masks_rle_coco(counts.data_ptr(), off.data_ptr(), m, coff.data_ptr(), chr2.data_ptr(), st()),
                  "coco")

    size()
    torch.cuda.synchronize()
    assert torch.equal(off2, off)
    in_bytes = m * H * (W // 32) * 4
    phases = {
        "size": (size, in_bytes + 2 * m * W * 4),               # masks read, column counts / last positions written
        "counts": (emit, in_bytes + 2 * m * W * 4 + 4 * n_counts),  # masks + column scans read, counts written
        "coco_size": (coco_size, 4 * n_counts),                  # counts read
        "coco_chars": (coco, 4 * n_counts + n_chars),            # counts read, characters written
    }
    out = {"kind": kind, "masks": m, "hw": [H, W], "counts": n_counts, "coco_chars": n_chars, "phases": {}}
    for name, (fn, nbytes) in phases.items():
        ms = time_ms(fn, flush)
        floor_ms = nbytes / HBM_BYTES_PER_S * 1e3
        out["phases"][name] = {"ms": ms, "bytes": nbytes, "hbm_floor_ms": floor_ms, "floor_share": floor_ms / ms}
    assert torch.equal(cnt2, counts) and torch.equal(chr2, chars)
    tot = sum(p["ms"] for p in out["phases"].values())
    out["uncompressed_ms"] = out["phases"]["size"]["ms"] + out["phases"]["counts"]["ms"]
    out["coco_ms"] = tot
    out["uncompressed_floor_share"] = (in_bytes + 4 * n_counts) / HBM_BYTES_PER_S * 1e3 / out["uncompressed_ms"]
    out["coco_floor_share"] = (in_bytes + n_chars) / HBM_BYTES_PER_S * 1e3 / out["coco_ms"]
    return out


def seg_bytes(recs):
    n = 0
    for r in recs:
        s = r["segmentation"]
        n += s.nbytes if isinstance(s, np.ndarray) else (4 * len(s["counts"]) if isinstance(s["counts"], list)
                                                          else len(s["counts"]))
    return n


def bench_e2e(n_slices):
    from saber_b200 import synth
    from saber_b200.adapters.base import cfgAMG
    from saber_b200.adapters.sam2 import build_amg
    from saber_b200.sam2.automatic_mask_generator import SAM2AutomaticMaskGenerator
    from saber_b200.utils import preprocessing as prep
    p = cfgAMG(sam2_cfg="large", pred_iou_thresh=0.3, stability_score_thresh=0.0).dict()
    model = build_amg(p, 100, allow_random_init=True).base_generator.predictor.model  # random-init hiera-L, as bench.py
    modes = ("binary_mask", "uncompressed_rle", "coco_rle")
    gens = {mode: SAM2AutomaticMaskGenerator(
        model, points_per_side=p["npoints"], points_per_batch=p["points_per_batch"],
        pred_iou_thresh=p["pred_iou_thresh"], stability_score_thresh=p["stability_score_thresh"],
        stability_score_offset=p["stability_score_offset"], crop_n_layers=p["crop_n_layers"],
        box_nms_thresh=p["box_nms_thresh"], crop_n_points_downscale_factor=p["crop_n_points_downscale_factor"],
        use_m2m=p["use_m2m"], multimask_output=p["multimask_output"], min_mask_region_area=25, output_mode=mode)
        for mode in modes}
    vol = synth.make_tomogram((n_slices + 2, 1024, 1024), seed=0)
    imgs = [torch.from_numpy(prep.prepare(vol[z].numpy(), to_rgb=True)).cuda() for z in range(n_slices + 2)]
    times = {mode: [] for mode in modes}
    counts = {mode: [] for mode in modes}
    host_bytes = {mode: [] for mode in modes}
    for z, img in enumerate(imgs):
        order = modes[z % 3:] + modes[:z % 3]
        for mode in order:
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            recs = gens[mode].generate(img)
            t1 = time.perf_counter()
            if z >= 2:  # the first two slices warm up every generator (graph capture, workspaces)
                times[mode].append((t1 - t0) * 1e3)
                counts[mode].append(len(recs))
                host_bytes[mode].append(seg_bytes(recs))
            del recs
    med = {mode: float(np.median(t)) for mode, t in times.items()}
    return {"ms_per_slice_median": med, "ms_per_slice_all": times, "masks_per_slice": counts,
            "segmentation_bytes_per_slice": host_bytes}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--slices", type=int, default=6)
    ap.add_argument("--out")
    args = ap.parse_args()
    from saber_b200 import ops
    ops.require_b200()
    scratch = torch.empty((256 << 20,), dtype=torch.uint8, device="cuda")
    flush = lambda: scratch.fill_(1)  # noqa: E731
    kernels = [bench_kernels(kind, m, flush) for kind in ("noise", "blob") for m in (64, 256)]
    del scratch
    res = {"card": card(), "kernels_1024": kernels, "e2e_config1_thresholds_open_A25": bench_e2e(args.slices)}
    print(json.dumps(res))
    if args.out:
        with open(args.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
