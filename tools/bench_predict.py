"""Cost of SAM2ImagePredictor's full-resolution output and of predict().

Prints one JSON object with the card name and power limit read in the same run, and:
  * kernel: ops.upsample_select (planes -> [P, 3, H, W] bool masks or fp32 logits in one launch) at 1024^2 and 4096^2
    with 1, 16 and 64 prompts x 3 masks, median of CUDA-event times with L2 overwritten (a 256 MiB write) before every
    timed launch, against the HBM floor: the output written once plus each candidate's 256 KB plane read once, at
    7.7 TB/s. In the same loop, alternating with it, the route it replaces: a gather copy of the planes,
    ops.upsample_bilinear to fp32, and (for masks) a torch compare; both outputs are checked equal;
  * predict: the wall time of predict() (host clock; the call ends with the copies to the host) at hiera-large, random
    init, on a 1024^2 image, for one point, one box, one box plus two points, and 64 boxes (multimask, bool masks).

    python tools/bench_predict.py [--out profiles/predict_bench.json]
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


def event_ms(fn, flush):
    flush()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    out = fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b), out


def kernel_rows(reps):
    from saber_b200 import ops
    scratch = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    flush = lambda: scratch.fill_(1)
    rows = []
    for hw in (1024, 4096):
        for P in (1, 16, 64):
            g = torch.Generator(device="cuda").manual_seed(P)
            planes = torch.randn(P, 4, 256, 256, device="cuda", generator=g) * 8.0
            for logits in (False, True):
                new = lambda: ops.upsample_select(planes, None, 3, hw, hw, 0.0, logits=logits)
                if logits:
                    old = lambda: ops.upsample_bilinear(planes[:, 1:4].contiguous(), hw, hw)
                else:
                    old = lambda: ops.upsample_bilinear(planes[:, 1:4].contiguous(), hw, hw) > 0.0
                equal = bool(torch.equal(new(), old()))
                for _ in range(2):  # warm both routes
                    new(), old()
                t_new, t_old = [], []
                for _ in range(reps):  # alternating
                    t, o = event_ms(new, flush)
                    t_new.append(t)
                    del o
                    t, o = event_ms(old, flush)
                    t_old.append(t)
                    del o
                nbytes = P * 3 * hw * hw * (4 if logits else 1) + P * 3 * 256 * 256 * 4
                floor_ms = nbytes / HBM_BYTES_PER_S * 1e3
                ms_new, ms_old = float(np.median(t_new)), float(np.median(t_old))
                rows.append(dict(hw=hw, prompts=P, candidates=3 * P, output="logits" if logits else "masks",
                                 bytes=nbytes, floor_ms=round(floor_ms, 4), kernel_ms=round(ms_new, 4),
                                 share_of_floor=round(floor_ms / ms_new, 3), old_route_ms=round(ms_old, 4),
                                 speedup=round(ms_old / ms_new, 2), outputs_equal=equal))
                print(json.dumps(rows[-1]), file=sys.stderr)
                torch.cuda.empty_cache()
    return rows


def predict_rows(reps):
    from saber_b200.sam2 import arch
    from saber_b200.sam2.build_sam import build_sam2
    from saber_b200.sam2.sam2_image_predictor import SAM2ImagePredictor
    model = build_sam2("large", None, device="cuda", state_dict=arch.random_state_dict("large", seed=0))
    pred = SAM2ImagePredictor(model)
    rng = np.random.default_rng(0)
    pred.set_image(rng.uniform(0, 1, (1024, 1024, 3)).astype(np.float32))
    xy = rng.uniform(0, 700, (64, 2))
    boxes = np.concatenate([xy, xy + rng.uniform(20, 300, (64, 2))], 1).astype(np.float32)
    cases = {
        "one_point": dict(point_coords=np.array([[500.0, 400.0]]), point_labels=np.array([1])),
        "one_box": dict(box=boxes[0]),
        "box_and_points": dict(box=boxes[0], point_coords=np.array([[120.0, 200.0], [300.0, 90.0]]),
                               point_labels=np.array([1, 0])),
        "64_boxes": dict(box=boxes),
    }
    rows = []
    for name, kw in cases.items():
        for _ in range(3):
            pred.predict(**kw)
        ts = []
        for _ in range(reps):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            pred.predict(**kw)
            ts.append((time.perf_counter() - t0) * 1e3)
        rows.append(dict(case=name, hw=1024, model="hiera-large", ms=round(float(np.median(ts)), 3),
                         ms_min=round(float(np.min(ts)), 3)))
        print(json.dumps(rows[-1]), file=sys.stderr)
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_predict needs a CUDA device")
    res = {"card": card(), "kernel": kernel_rows(args.reps), "predict": predict_rows(args.reps)}
    res["card_after"] = card()
    print(json.dumps(res))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
