#!/usr/bin/env python
"""bench.py — SABER slice-wise SAM2.1 hiera-large segmentation throughput (BASELINE.json configs[1]).

A *step* is one pass of the hot path over one batch of `--slices-per-step` z-slices of the synthetic
200x1024x1024 tomogram: per slice prepare (contrast / min-max) -> AMG at SABER's defaults (21 crops -> Hiera-L
encoder, 3 072 point prompts, multimask + m2m = 12 288 mask-decoder evaluations, stability / threshold / box /
NMS) -> area filter -> duplicate removal -> sort -> label stitch; then 26-connected 3-D components over the
batch's label slab (the `propagationSegmenter.slice_by_slice` body, REF saber/segmenters/propagation.py:164-189).

  value  : slices/s, whole job (all ranks), inputs resident in HBM, CUDA-event timed, max over ranks.
  e2e    : same metric through the reference-facing API `propagationSegmenter.slice_by_slice(numpy volume)`
           with HOST buffers (pinned H2D of the slab + D2H of the uint32 label volume inside the timed region).
  roofline: the tcgen05 GEMM kernel (dominant), algorithmic FLOPs / CUDA-event duration vs MEASURED_PEAKS.json.
  cpu_baseline: the oracle port (pure-torch fp32 restatement of upstream sam2 + SABER post-processing) timed on
           this box's host cores on a bounded sample, extrapolated to slices/s.

`--impl reference` times the CPU implementation only (rank 0) and prints the same JSON line shape.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SHAPE = (200, 1024, 1024)
METRIC = "tomogram slices/sec (SAM2.1 hiera-L, 1024^2 slice-wise AMG)"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--cfg", default="large")
    ap.add_argument("--slices-per-step", type=int, default=3,
                    help="slices per step; with 2 or more the slice workers overlap one slice's encoder with another's decoder")
    ap.add_argument("--thresholds", default="default", choices=["default", "open"],
                    help="'open' lowers pred_iou/stability thresholds so random-init weights exercise NMS/CC stages")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-roofline", action="store_true")
    ap.add_argument("--no-propagation", action="store_true",
                    help="skip the config-3 sub-record (3-D propagation of a 300x928x960 tomogram, z-slab relay over the ranks)")
    ap.add_argument("--prop-frames", type=int, default=300)
    ap.add_argument("--prop-objects", type=int, default=8)
    ap.add_argument("--no-extras", action="store_true",
                    help="skip thresholds_open / components_3d / bandwidth / gpu_eager_baseline (N = 1 only anyway)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed (rank 0) as DIR/<name>.npy: labels (3-D "
                         "components of the slab), slice_labels (stitched per-slice labels), masks_kept (per slice), "
                         "candidate_iou / candidate_stability (scores of every AMG candidate of the last slices)")
    args = ap.parse_args()
    if args.dump_outputs and args.steps < 1:
        ap.error("--dump-outputs needs --steps >= 1")
    return args


def workload_name(args):
    return (f"SAM2.1 hiera-{args.cfg} slice-wise zero-shot segmentation of a {SHAPE[0]}x{SHAPE[1]}x{SHAPE[2]} synthetic "
            f"tomogram (BASELINE configs[1]); AMG at SABER defaults (32 pts/side, 2 crop layers, multimask + m2m)"
            + ("" if args.thresholds == "default" else "; thresholds opened (pred_iou 0.3, stability filter off)"))


# ------------------------------------------------------------------------------------------------
# clocks sampling (nvidia-smi during the timed region)
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.gpu)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# CPU implementation (oracle port) — cpu_baseline leg and --impl reference
# ------------------------------------------------------------------------------------------------
def cpu_reference_sample(cfg: str, thresholds: str, n_points: int = 16):
    """One bounded sample of the CPU path (oracle port, fp32, all host threads): one crop encode + one batch of
    `n_points` prompts through both decoder passes and the post-processing, + prepare + per-slice integer
    stages; returns (seconds per slice extrapolated, description, cores)."""
    import numpy as np
    import torch
    from oracle import saber_ref
    from oracle.sam2_ref.amg import SAM2AutomaticMaskGenerator as OracleAMG
    from oracle.sam2_ref.sam2_base import SAM2Base
    from saber_b200 import synth
    from saber_b200.sam2 import arch

    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    st = cpu_reference_sample.__dict__
    if "model" not in st:
        sd = arch.random_state_dict(cfg, seed=0)
        m = SAM2Base(cfg, dynamic_multimask_via_stability=True)
        m.load_state_dict(sd, strict=True)
        st["model"] = m.eval()
        st["img"] = synth.make_tomogram(SHAPE, seed=0, z_range=(100, 101))[0].numpy()
    model, img = st["model"], st["img"]
    thr = dict(pred_iou_thresh=0.7, stability_score_thresh=0.92) if thresholds == "default" else \
        dict(pred_iou_thresh=0.3, stability_score_thresh=0.0)
    gen = OracleAMG(model, points_per_side=32, points_per_batch=64, stability_score_offset=0.7, crop_n_layers=2,
                    box_nms_thresh=0.7, crop_n_points_downscale_factor=2, use_m2m=True, multimask_output=True, **thr)
    t0 = time.perf_counter()
    rgb = saber_ref.prepare(img, to_rgb=True)
    t_prep = time.perf_counter() - t0
    t0 = time.perf_counter()
    with torch.no_grad():
        gen.predictor.set_image(rgb)  # one 1024^2 crop: resize + normalise + Hiera-L + FPN
    t_enc = time.perf_counter() - t0
    pts = gen.point_grids[0][:n_points] * np.array([[1024, 1024]])
    t0 = time.perf_counter()
    with torch.no_grad():
        gen._process_batch(pts, (1024, 1024), [0, 0, 1024, 1024], (1024, 1024), normalize=True)
    t_batch = time.perf_counter() - t0
    n_crops, n_pts = 21, 3072
    per_slice = t_prep + n_crops * t_enc + (n_pts / n_points) * t_batch
    desc = (f"1 slice prepare ({t_prep:.2f}s) + 1 of 21 crop encodes ({t_enc:.2f}s) + 1 batch of {n_points} of 3072 "
            f"prompts through decoder x(1+3 m2m) + post-processing ({t_batch:.2f}s); extrapolated "
            f"prep + 21*enc + {n_pts // n_points}*batch = {per_slice:.1f}s per slice (NMS/dedupe/CC not included)")
    return per_slice, desc, cores


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    for _ in range(args.warmup):
        cpu_reference_sample(args.cfg, args.thresholds, n_points=4)
    per, desc = [], ""
    t_all = time.perf_counter()
    for _ in range(args.steps):
        s, desc, cores = cpu_reference_sample(args.cfg, args.thresholds, n_points=8)
        per.append(s)
    wall = time.perf_counter() - t_all
    sec = sum(per) / len(per)
    val = 1.0 / sec
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": "slices/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * wall / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_name(args), "note": "each step is a bounded sample extrapolated to one slice"},
            "cpu_baseline": {"value": val, "unit": "slices/s", "cores": cores, "kind": "port", "sample": desc},
            "e2e": {"value": val, "unit": "slices/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    _emit(line)



# ------------------------------------------------------------------------------------------------
# Extra records of the one JSON line (rank 0, N = 1): the parts of the path the as-configured headline cannot show
# ------------------------------------------------------------------------------------------------
def _time_kernel(fn, flush, reps=5, warm=2):
    """Median CUDA-event time (ms) of fn() on the current stream, L2 flushed before every timed call."""
    import torch
    for _ in range(warm):
        fn()
    ts = []
    for _ in range(reps):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    ts.sort()
    return ts[len(ts) // 2]


def _hbm_peak():
    try:
        return float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (of measured)"
    except Exception:
        return 6650.0, "fallback 6.65 TB/s (of fallback)"


def measure_extras(args, seg, slab, labels, flush, dev):
    import numpy as np
    import torch

    from saber_b200 import ops, synth
    from saber_b200.segmenters import utils as sutils
    out = {}
    peak, peak_src = _hbm_peak()
    gen = seg.adapter._amg().base_generator
    S = slab.shape[0]

    # (i) thresholds opened: with random-init weights nothing passes pred_iou 0.7 / stability 0.92, so up-sampling,
    # stability, bit packing, NMS, duplicate removal, stitching and the slab CCL run on (almost) empty input in the
    # headline. Same workload with pred_iou 0.3 / stability filter off (SURVEY 8d's second reporting mode).
    saved = (gen.pred_iou_thresh, gen.stability_score_thresh)
    gen.pred_iou_thresh, gen.stability_score_thresh = 0.3, 0.0
    gen._graphs.clear()  # thresholds are baked into the captured launches
    try:
        n = max(2, min(args.steps, 5))
        for _ in range(2):
            seg.label_slices_device(slab, labels)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        kept = 0
        e0.record()
        for _ in range(n):
            flush.zero_()
            kept += sum(seg.label_slices_device(slab, labels))
            sutils.separate_masks_device(labels, min_mask_area=100)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / n
        host = slab.cpu().pin_memory()
        seg.slice_by_slice_host(host)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(n):
            flush.zero_()
            seg.slice_by_slice_host(host)
        torch.cuda.synchronize()
        out["thresholds_open"] = {"value": S / (ms / 1e3), "unit": "slices/s", "ms_per_step": ms, "steps": n,
                                  "masks_kept_per_slice": kept / (n * S),
                                  "e2e": {"value": n * S / (time.perf_counter() - t0), "unit": "slices/s"},
                                  "thresholds": {"pred_iou_thresh": 0.3, "stability_score_thresh": 0.0}}
    finally:
        gen.pred_iou_thresh, gen.stability_score_thresh = saved
        gen._graphs.clear()

    # (ii) 26-connected 3-D components (separate_masks) on the whole 200 x 1024 x 1024 label volume of configs[1]
    vol = synth.make_label_volume(SHAPE, seed=1, n_ellipsoids=300, device=dev, rmin=8.0, rmax=40.0, speckle=0.0005)
    ms = _time_kernel(lambda: sutils.separate_masks_device(vol, min_mask_area=100), flush, reps=3, warm=1)
    nvox = float(np.prod(SHAPE))
    gbs = 6.0 * nvox / (ms * 1e-3) / 1e9
    out["components_3d"] = {"workload": "separate_masks (26-connected CCL + size filter + compact relabel) on a 200x1024x1024 "
                                        "uint16 label volume, 300 ellipsoids + speckle", "ms": ms, "mvox_per_s": nvox / ms / 1e3,
                            "algorithmic_bytes_per_voxel": 6, "achieved_gbs": gbs, "peak_gbs": peak, "frac": gbs / peak,
                            "peak_source": peak_src}
    del vol

    # (iii) bandwidth kernels of subsystems (2) / (3): algorithmic bytes (SURVEY 8d) / CUDA-event time vs the HBM peak
    table = []

    def add(name, nbytes, fn, note=""):
        ms_ = _time_kernel(fn, flush)
        g = nbytes / (ms_ * 1e-3) / 1e9
        table.append({"kernel": name, "algorithmic_bytes": int(nbytes), "us": ms_ * 1e3, "gbs": g, "frac": g / peak, "note": note})

    v = synth.make_tomogram((64, 928, 960), seed=2, device=dev).contiguous()
    nv = v.numel()
    mm = ops.minmax(v)
    add("minmax (normalize_tomogram, pass 1)", 4 * nv, lambda: ops.minmax(v), "64x928x960 fp32: 4 B read / voxel")
    add("minmax_affine (normalize_tomogram, pass 2)", 8 * nv, lambda: ops.minmax_affine(v, mm, 0.0, 2.0, -1.0), "4 B + 4 B / voxel")
    from saber_b200.filters.gaussian import make_gaussian_kernel
    w15 = make_gaussian_kernel(5).to(dev, torch.float32).contiguous()
    add("gaussian_z (15 taps, zero padded)", 8 * nv, lambda: ops.gaussian_z(v, w15), "4 B + 4 B / voxel")
    add("zoom_linear_mirror (skimage resize 928x960 -> 1024^2, 2x-1)", 4 * nv + 4 * 64 * 1024 * 1024,
        lambda: ops.skimage_resize_stack(v, 1024, 2.0, -1.0), "4 B / input voxel + 4 B / output pixel")
    add("mean_z (slab projection, 20 slices)", 4 * 20 * 928 * 960 + 4 * 928 * 960, lambda: ops.mean_z(v, 22, 42))
    img = slab[0].contiguous()
    add("prepare_slice (box filter x4 + contrast + min-max)", 8 * img.numel(), lambda: ops.prepare_slice(img, 500, 3.0),
        "algorithmic 4 B in + 4 B out / pixel; executed: 6 launches, ~52 B / pixel of traffic (L2 resident at 1024^2)")
    del v
    # mask_post: bilinear up-sampling + IoU filter + stability + threshold + box + bit packing of 192 candidates of a
    # full-frame crop (every candidate kept: thresholds open)
    plan = gen._plan((SHAPE[1], SHAPE[2]))
    ws = gen._workspace(plan)
    crop = plan.crops[0]
    x0, y0, x1, y1 = crop.box
    planes = (torch.randn(192, 4, 256, 256, device=dev) * 4).contiguous()
    ious4 = torch.rand(192, 4, device=dev).contiguous()
    geom = ((y1 - y0, x1 - x0), (x0, y0), plan.hw, 1e-6, gen.mask_threshold, gen.stability_score_offset, 0.0, ws["keep"],
            ws["stab"], ws["iou"], ws["bbox"], ws["area"], ws["bits"])
    cap, gen.capture = gen.capture, None
    add("mask_post_kernel (192 candidates, 1024^2 crop, all kept)", 192 * (256 * 256 * 4 + SHAPE[1] * SHAPE[2] // 8),
        lambda: gen._post(0, planes, ious4, None, 1, 192, geom, 0), "256 KB logits read + 128 KB bits written per candidate")
    gen.capture = cap
    order = torch.arange(64, dtype=torch.int32, device=dev)
    lab1 = torch.empty((SHAPE[1], SHAPE[2]), dtype=torch.int16, device=dev)
    add("stitch_labels (64 masks -> uint16 slice)", 64 * SHAPE[1] * SHAPE[2] // 8 + 2 * SHAPE[1] * SHAPE[2],
        lambda: ops.stitch_labels(ws["bits"], order, 64, SHAPE[2], out=lab1), "128 KB bits per mask + 2 B / pixel")
    low = (torch.randn(64, 256, 256, device=dev)).contiguous()
    add("fill_holes (64 low-res masks, area <= 8)", 2 * low.numel() * 4, lambda: ops.fill_holes(low, 8), "4 B + 4 B / pixel")
    out["bandwidth"] = {"peak_gbs": peak, "peak_source": peak_src, "l2": "256 MiB flush before every timed launch",
                        "kernels": [t for t in table if t]}

    # (v) SURVEY 8f rows 2 / 3 (the import step before the path and the refinement step after it) at the BASELINE volume
    # size: FFT line passes against the HBM roofline, the whole rescale / band-pass calls, the membrane workflow
    try:
        from saber_b200.analysis.refine_membranes import FilteringConfig, OrganelleMembraneFilter
        from saber_b200.filters.downsample import FourierRescale3D
        from saber_b200.filters.tomograms import Filter3D
        shape3 = (200, 928, 960)
        v3 = synth.make_tomogram(shape3, seed=7, n_ellipsoids=30, device=dev).contiguous()
        n3 = v3.numel()
        spec = ops.fft_lines(v3, 2)
        fft_rows = []
        for name, fn, nbytes in [("fft x rows, real -> complex, n=960", lambda: ops.fft_lines(v3, 2), 12 * n3),
                                 ("fft y columns, complex, n=928 (2^5 x 29)", lambda: ops.fft_lines(spec, 1), 16 * n3),
                                 ("fft z columns, complex, n=200 (2^3 x 5^2)", lambda: ops.fft_lines(spec, 0), 16 * n3),
                                 ("ifft x rows, complex -> real, n=960", lambda: ops.fft_lines(spec, 2, inverse=True, out_mode="real"), 12 * n3)]:
            ms_ = _time_kernel(fn, flush, reps=3, warm=1)
            g = nbytes / (ms_ * 1e-3) / 1e9
            fft_rows.append({"kernel": name, "algorithmic_bytes": int(nbytes), "us": ms_ * 1e3, "gbs": g, "frac": g / peak})
        del spec
        rs = FourierRescale3D(10.0, 20.0)
        ms_rs = _time_kernel(lambda: rs.rescale_device(v3), flush, reps=3, warm=1)
        f3 = Filter3D(10.0, shape3, lp=60.0, lpd=6.0, hp=2000.0, hpd=2.0)
        ms_bp = _time_kernel(lambda: f3.apply(v3), flush, reps=3, warm=1)
        del v3
        org, mem = synth.make_organelle_membrane((200, 464, 480), 71, 12, blob=3.0)
        o_d, m_d = torch.from_numpy(org).to(dev), torch.from_numpy(mem).to(dev)
        filt = OrganelleMembraneFilter(FilteringConfig(ball_size=3, min_membrane_area=2000), gpu_id=dev.index or 0)
        filt.run_device(o_d, m_d)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        res = filt.run_device(o_d, m_d)
        torch.cuda.synchronize()
        ms_ref = (time.perf_counter() - t0) * 1e3
        out["next_rows"] = {
            "fft_passes": fft_rows, "peak_gbs": peak,
            "fourier_rescale_3d": {"workload": "200x928x960 fp32 -> 100x464x480 (voxel 10 -> 20 A)", "ms": ms_rs},
            "filter3d_bandpass": {"workload": "200x928x960 fp32, cosine low- + high-pass, 6 line passes", "ms": ms_bp,
                                  "gbs": 88.0 * n3 / (ms_bp * 1e-3) / 1e9, "frac": 88.0 * n3 / (ms_bp * 1e-3) / 1e9 / peak},
            "refine_membranes": {"workload": "200x464x480 int32 labels, 12 organelles + membrane shells, run_device (wall "
                                             "clock incl. the host reads of component counts)", "ms": ms_ref,
                                 "organelles_kept": int(torch.unique(res["organelles"]).numel()) - 1}}
    except Exception as e:  # the headline must not depend on the next-row probes
        out["next_rows"] = {"error": repr(e)}

    # (iv) same-box GPU bar: the oracle (plain PyTorch: cuBLASLt / cuDNN / SDPA) on this B200 for one crop encode + one
    # prompt batch (64 points + 192 m2m), extrapolated per slice like the CPU arm (SURVEY 8d)
    out["gpu_eager_baseline"] = gpu_eager_baseline(args, dev)
    return out


def measure_propagation(args, dev, world, rank):
    """BASELINE configs[2]: SAM2.1 hiera-large 3-D propagation (memory attention along z) of a synthetic 300x928x960
    tomogram, frames sharded by z-slab over the ranks (STRONG scaling: the volume is fixed). One step = set_volume
    (normalise + resize + encode this rank's slab; no feature exchange) + segment_volume (bidirectional tracking of
    `--prop-objects` seed masks from the middle slice as a relay: the memory-bank halo crosses each slab boundary
    point-to-point over NCCL, label slabs are all-gathered). Reported: slices/s over the whole step (max over ranks),
    bytes moved over NCCL per step and the CRC-32 of the label volume (identical for every N: compare the lines)."""
    import zlib

    import numpy as np
    import torch
    import torch.distributed as dist

    from saber_b200 import synth
    from saber_b200.adapters.base import SAM2AdapterConfig, cfgAMG
    from saber_b200.adapters.sam2 import SAM2Adapter

    Z, H, W = args.prop_frames, 928, 960
    sam_cfg = {"large": "large", "base_plus": "base", "small": "small", "tiny": "tiny"}[args.cfg]
    ad = SAM2Adapter(SAM2AdapterConfig(cfg=sam_cfg, amg_cfg=cfgAMG(sam2_cfg=sam_cfg), num_maskmem=2, seed=0,
                                       allow_random_init=True), device=str(dev))
    vol = synth.make_tomogram((Z, H, W), seed=3, n_ellipsoids=10, device=dev)
    rng = np.random.default_rng(0)
    yy, xx = np.mgrid[0:H, 0:W]
    seeds = []
    for _ in range(args.prop_objects):
        cy, cx, ry, rx = rng.uniform(200, 700), rng.uniform(200, 700), rng.uniform(30, 90), rng.uniform(30, 90)
        seeds.append(torch.from_numpy((((yy - cy) / ry) ** 2 + ((xx - cx) / rx) ** 2 <= 1).astype(np.float32)).to(dev))
    seeds = torch.stack(seeds)

    def sync():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def tmax(x):
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.item()

    ad._video()
    zw = min(Z, 16 * world)  # build + warm the kernels on a small volume (>= 15 frames per slab: the relay's minimum)
    ad.set_volume(vol[:zw].contiguous())
    ad.segment_volume_device(zw // 2, masks=seeds[:1], vol_shape=(zw, H, W), min_presence_score=-1e9)
    ad.reset_state()
    t_set, t_seg, out = [], [], None
    for rep in range(2):
        sync()
        t0 = time.perf_counter()
        ad.set_volume(vol)
        sync()
        t1 = time.perf_counter()
        out = ad.segment_volume_device(Z // 2, masks=seeds, vol_shape=(Z, H, W), min_presence_score=-1e9)
        sync()
        t2 = time.perf_counter()
        t_set.append(tmax(t1 - t0))
        t_seg.append(tmax(t2 - t1))
        ad.reset_state()
    sent = torch.tensor([float((ad.relay_stats or {}).get("bytes_sent", 0))], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(sent)
    label_bytes = (world - 1) * 2.0 * Z * H * W if world > 1 else 0.0  # all-gather of the uint16 slabs: received per rank x ranks / ... total
    rec = None
    if rank == 0:
        crc = zlib.crc32(out.cpu().numpy().tobytes())
        total = t_set[-1] + t_seg[-1]
        rec = {"workload": f"SAM2.1 hiera-{args.cfg} 3-D propagation of a {Z}x{H}x{W} synthetic tomogram, {args.prop_objects} objects "
                           f"seeded on slice {Z // 2} (BASELINE configs[2]), frames sharded by z-slab over {world} GPU(s)",
               "value": Z / total, "unit": "slices/s", "scaling": "strong", "n_gpus": world,
               "set_volume_ms": t_set[-1] * 1e3, "segment_volume_ms": t_seg[-1] * 1e3,
               "first_rep_ms": (t_set[0] + t_seg[0]) * 1e3,
               "nccl_bytes_per_step": {"memory_bank_halo": sent.item(), "label_slab_allgather_total": label_bytes,
                                       "frame_features": 0.0},
               "shard": ad.prop_shard, "label_volume_crc32": crc,
               "labels_present": int(torch.unique(out).numel() - 1),
               "timing": "wall clock around the public calls, device-synchronised + barrier on both sides, max over ranks; 2nd of 2 repetitions"}
    del ad, vol, out
    torch.cuda.empty_cache()
    return rec


def gpu_eager_baseline(args, dev):
    import numpy as np
    import torch

    from oracle.sam2_ref.amg import SAM2AutomaticMaskGenerator as OracleAMG
    from oracle.sam2_ref.sam2_base import SAM2Base
    from saber_b200 import synth
    from saber_b200.sam2 import arch
    res = {"what": "oracle restatement of upstream sam2 (PyTorch eager) on the same B200: 1 crop encode + 1 batch of 64 "
                   "points through decoder x(1+3 m2m) + upstream post-processing; per slice = 21 encodes + 48 batches",
           "modes": {}}
    sd = arch.random_state_dict(args.cfg, seed=0)
    m = SAM2Base(args.cfg, dynamic_multimask_via_stability=True)
    m.load_state_dict(sd, strict=True)
    m = m.to(dev).eval()
    img = synth.make_tomogram(SHAPE, seed=0, z_range=(100, 101))[0].numpy()
    rgb = np.repeat(((img - img.min()) / (img.max() - img.min() + 1e-8))[..., None], 3, axis=2).astype(np.float32)
    gen = OracleAMG(m, points_per_side=32, points_per_batch=64, stability_score_offset=0.7, crop_n_layers=2,
                    box_nms_thresh=0.7, crop_n_points_downscale_factor=2, use_m2m=True, multimask_output=True,
                    pred_iou_thresh=0.7, stability_score_thresh=0.92)
    pts = gen.point_grids[0][:64] * np.array([[1024, 1024]])
    old = (torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32)
    try:
        for mode in ("tf32", "bf16_autocast"):
            torch.backends.cuda.matmul.allow_tf32 = True   # REF saber/utils/io.py:127-130
            torch.backends.cudnn.allow_tf32 = True
            ctx = torch.autocast("cuda", dtype=torch.bfloat16) if mode == "bf16_autocast" else torch.autocast("cuda", enabled=False)

            def enc():
                with torch.no_grad(), ctx:
                    gen.predictor.set_image(rgb)

            def batch():
                with torch.no_grad(), ctx:
                    gen._process_batch(pts, (1024, 1024), [0, 0, 1024, 1024], (1024, 1024), normalize=True)

            for f in (enc, batch):
                f()
            torch.cuda.synchronize()
            t = {}
            for name, f, reps in (("encode", enc, 3), ("batch", batch, 3)):
                t0 = time.perf_counter()
                for _ in range(reps):
                    f()
                torch.cuda.synchronize()
                t[name] = (time.perf_counter() - t0) / reps
            per_slice = 21 * t["encode"] + 48 * t["batch"]
            res["modes"][mode] = {"encode_ms_per_crop": 1e3 * t["encode"], "batch_ms_per_64_points": 1e3 * t["batch"],
                                  "slices_per_s": 1.0 / per_slice}
    except Exception as e:  # the bar is informative; never let it take the bench line down
        res["error"] = f"{type(e).__name__}: {e}"
    finally:
        torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = old
    return res


# ------------------------------------------------------------------------------------------------
# B200 arm
# ------------------------------------------------------------------------------------------------
DUMP_BYTES = 60 << 20  # < 64 MB with the .npy headers


def dump_outputs(path, arrays):
    """Writes each array as path/<name>.npy, in float32 where that holds every value exactly, else float64, so that
    two builds can be compared output for output. Above DUMP_BYTES in all, each array keeps the same share of its
    flattened elements, picked by a fixed seed (identical positions from run to run for the same shapes)."""
    import numpy as np
    out = {}
    for name, a in arrays.items():
        f = a.astype(np.float32)
        out[name] = f if np.array_equal(f, a) else a.astype(np.float64)
    total = sum(f.nbytes for f in out.values())
    os.makedirs(path, exist_ok=True)
    for name, f in out.items():
        if total > DUMP_BYTES:
            k = f.size * DUMP_BYTES // total
            f = f.reshape(-1)[np.sort(np.random.default_rng(0).choice(f.size, k, replace=False))]
        np.save(os.path.join(path, name + ".npy"), f)


def candidate_scores(seg, S, hw):
    """Predicted IoU and stability score of every AMG candidate (all crops, prompts and multimask outputs) of the last
    step's slices, as their mask generators' workspaces hold them after the step: slice j of a step runs on slice
    worker j % nw, so the last nw slices are still there. With random-init weights at the default thresholds no
    candidate is kept, and these scores are the only non-zero results of the step."""
    import numpy as np
    nw = min(seg.slice_workers, S)
    rows = [seg._peers[j % nw].adapter._amg().base_generator._ws[tuple(hw)] for j in range(S - nw, S)]
    return {"candidate_iou": np.stack([ws["iou"].cpu().numpy() for ws in rows]),
            "candidate_stability": np.stack([ws["stab"].cpu().numpy() for ws in rows])}


def run_b200(args):
    import numpy as np
    import torch
    import torch.distributed as dist

    from saber_b200 import ops, synth
    from saber_b200.adapters.base import SAM2AdapterConfig, cfgAMG
    from saber_b200.segmenters import utils as sutils
    from saber_b200.segmenters.propagation import propagationSegmenter

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device(f"cuda:{local}")
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("TORCH_NCCL_SHOW_EAGER_INIT_P2P_SERIALIZATION_WARNING", "false")
        dist.init_process_group("nccl", device_id=dev)
    ops.require_b200()

    sam_cfg = {"large": "large", "base_plus": "base", "small": "small", "tiny": "tiny"}[args.cfg]
    amg_kw = dict(sam2_cfg=sam_cfg)
    if args.thresholds == "open":
        amg_kw.update(pred_iou_thresh=0.3, stability_score_thresh=0.0)
    seg = propagationSegmenter(deviceID=local, cfg=SAM2AdapterConfig(cfg=sam_cfg, amg_cfg=cfgAMG(**amg_kw),
                                                                    min_mask_area=100, allow_random_init=True),
                               min_mask_area=100)  # random-init weights of the named architecture (BASELINE: no checkpoints)
    if os.environ.get("SB_NO_GRAPH"):
        seg.adapter._amg().base_generator.use_cuda_graph = False
    S = args.slices_per_step
    Z = SHAPE[0]
    # z-slab sharding: rank r owns slices [r*Z/world, (r+1)*Z/world); each step takes the next S slices of the slab
    slab0 = rank * (Z // world)
    n_total = args.warmup + args.steps + 2
    zs = [slab0 + (i * S) % max(1, (Z // world) - S + 1) for i in range(n_total)]
    slabs = {}
    for z in sorted(set(zs)):
        slabs[z] = synth.make_tomogram(SHAPE, seed=0, device=dev, z_range=(z, z + S)).contiguous()
    labels = torch.empty((S,) + SHAPE[1:], dtype=torch.int16, device=dev)
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)  # 256 MiB > 126 MB L2

    def step(i):
        counts = seg.label_slices_device(slabs[zs[i]], labels)
        out = sutils.separate_masks_device(labels, min_mask_area=100)
        return counts, out

    def step_serial(i):
        # instrumented variant: one slice at a time with a device synchronisation in between, so that phase events and
        # per-launch GEMM timings of a slice are not stretched by the next slice's (asynchronously launched) kernels
        for z in range(S):
            seg.label_slices_device(slabs[zs[i]], labels, z, z + 1)
            torch.cuda.synchronize()
        return sutils.separate_masks_device(labels, min_mask_area=100)

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for i in range(args.warmup):
        step(i)
    sync_all()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    launches0 = ops.launch_count
    kept = 0
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sync_all()
    e0.record()
    for i in range(args.steps):
        flush.zero_()  # L2 flush between timed iterations (plus inputs/activations >> L2)
        counts, comps = step(args.warmup + i)
        kept += sum(counts)
    e1.record()
    sync_all()
    ms = e0.elapsed_time(e1)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"labels": comps.cpu().numpy().view(np.uint32),
                                         "slice_labels": labels.cpu().numpy().view(np.uint16),
                                         "masks_kept": np.array(counts),
                                         **candidate_scores(seg, S, labels.shape[1:])})
    launches = ops.launch_count - launches0
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = t.item()
    clocks = sampler.stop() if rank == 0 else None
    value = world * S * args.steps / (ms_max / 1e3)

    # ---- e2e through the reference-facing API with host buffers (pinned H2D + D2H inside the timed region)
    e2e = None
    if not args.no_e2e:
        # every one of the --steps slices goes host -> device -> host (pinned staging, wall clock around the public call)
        host = [slabs[zs[args.warmup + i]].cpu().pin_memory() for i in range(args.steps)]
        seg.slice_by_slice_host(host[0])  # warm the path
        sync_all()
        t0 = time.perf_counter()
        for h in host:
            flush.zero_()
            out = seg.slice_by_slice_host(h)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        tt = torch.tensor([dt], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        e2e = {"value": world * S * len(host) / tt.item(), "unit": "slices/s",
               "h2d_bytes_per_step": int(host[0].numel() * 4), "d2h_bytes_per_step": int(out.nbytes)}

    # ---- roofline of the dominant kernel: one extra instrumented step, CUDA events around every GEMM launch
    roofline = None
    phases = None
    if not args.no_roofline and rank == 0:
        gen = seg.adapter._amg().base_generator
        workers_was, seg.slice_workers = seg.slice_workers, 1  # instrumented steps run the slices one after the other
        step_serial(args.warmup + args.steps)  # un-instrumented pass first: the serial path runs on the caller's stream, whose
        torch.cuda.synchronize()               # allocator pool may not yet hold the encoder's transient buffers (cudaMalloc)
        gen.phase_ms = {}
        step_serial(args.warmup + args.steps)  # one more normal (graph-replay) step with phase events
        torch.cuda.synchronize()
        n_img = max(1, gen.phase_ms.get("images", 1))
        phases = {k: v / n_img for k, v in gen.phase_ms.items() if k != "images"}
        gen.phase_ms = None
        prof = ops.GemmProfiler()
        graph_was = gen.use_cuda_graph
        gen.use_cuda_graph = False  # eager launches: the decoder GEMMs inside the replayed graphs get their events too
        with prof:
            step_serial(args.warmup + args.steps)
        torch.cuda.synchronize()
        gen.use_cuda_graph = graph_was
        seg.slice_workers = workers_was
        r = prof.summary()
        if os.environ.get("SB_GEMM_SHAPES"):
            with open(os.environ["SB_GEMM_SHAPES"], "w") as fh:
                for tag, n, ms_, tf in prof.by_shape(40):
                    fh.write(f"{ms_:9.3f} ms  n={n:5d}  {tf:8.1f} TFLOP/s  {tag}\n")
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = peaks.get("bf16_tflops_sustained", 1400.0)
        traffic = None  # dram__bytes_read.sum + dram__bytes_write.sum of one representative launch (ncu --set full, profiles/)
        try:
            tj = json.load(open(os.path.join(ROOT, "profiles", "gemm_traffic.json")))
            traffic = tj["dram_bytes_per_launch"]
            traffic_detail = {"algorithmic_bytes": tj["algorithmic_bytes_per_launch"], "launch": tj["launch"],
                              "source": tj["source"]}
        except Exception:
            traffic_detail = None
        roofline = {"bound": "tensor", "kernel": "gemm_bf16_tcgen05_kernel + gemm2_bf16_tcgen05_kernel (single-CTA and CTA-pair tcgen05 GEMMs)", "achieved": r["tflops"], "peak": peak,
                    "unit": "TFLOP/s", "frac": r["tflops"] / peak, "traffic": traffic, "traffic_detail": traffic_detail,
                    "peak_source": "MEASURED_PEAKS.json bf16_tflops_sustained (of measured)" if peaks else "fallback 1.4 PFLOP/s (of fallback)",
                    "launches": r["launches"], "gemm_ms_per_step": r["ms"], "flops_per_step": r["flops"],
                    "share_of_step": r["ms"] / (ms_max / args.steps),  # GEMM ms of the serial instrumented step / concurrent step
                    "how": "1 extra instrumented step after the timed region, launched eagerly (no CUDA graph) so every tcgen05 GEMM launch of the step (encoder + both decoder passes: std / LN / up-scaling epilogues) is bracketed by CUDA events on the launch stream; achieved = sum(2MNK) / sum(duration)"}

        # north_star's encoder figure: algorithmic Hiera FLOPs of the slice's crops (SURVEY 8a U1, incl. window padding)
        # over the device-timed encode phase
        enc_gf = {"tiny": 292.0, "small": 360.0, "base_plus": 647.0, "base+": 647.0, "large": 1823.0}.get(args.cfg)
        if enc_gf and phases and phases.get("encode"):
            n_crops = sum(len(pl.crops) for pl in gen._plans.values()) // max(1, len(gen._plans))
            enc_tf = enc_gf * 1e9 * n_crops / (phases["encode"] * 1e-3) / 1e12
            roofline["encoder"] = {"crops_per_slice": n_crops, "gflop_per_crop": enc_gf, "ms_per_slice": phases["encode"],
                                   "achieved": enc_tf, "unit": "TFLOP/s", "frac": enc_tf / peak,
                                   "note": "all encoder kernels (GEMMs and the stage-3 window / global attention on tcgen05, the 8x8 / 4x4 / pooled windows on mma.sync, LayerNorm, pooling)"}
        roofline["not_counted"] = ("i2t_tc_kernel / t2i_tc_kernel (fused mask-decoder attention blocks on tcgen05) are not "
                                   "GEMM launches: HBM-bound, 4 MB resp. 2 MB of image stream per prompt; see DESIGN.md section 3")

    extras = {}
    if rank == 0 and world == 1 and not args.no_extras:
        extras = measure_extras(args, seg, slabs[zs[0]], labels, flush, dev)
    if not args.no_propagation:  # every rank takes part
        prop = measure_propagation(args, dev, world, rank)
        if prop is not None:
            extras["propagation"] = prop

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        sec, desc, cores = cpu_reference_sample(args.cfg, args.thresholds, n_points=16)
        cpu = {"value": 1.0 / sec, "unit": "slices/s", "cores": cores, "kind": "port", "sample": desc}

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": "slices/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms_max / args.steps, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
                "config": {"workload": workload_name(args), "slices_per_step": S, "sharding": f"z-slab x{world}",
                           "voxels_per_s": value * SHAPE[1] * SHAPE[2], "masks_kept_per_slice": kept / max(1, S * args.steps),
                           "l2": "256 MiB flush write between timed steps; per-step activations (>10 GB) exceed L2",
                           "weights": "random-init (seed 0) of the named architecture",
                           "phase_ms_per_slice": phases,
                           "slice_workers": getattr(seg, "slice_workers", 1),
                           "concurrency": "the slices of a step are dealt to slice_workers worker threads (own mask generator, workspaces, CUDA graphs and stream each; one shared model) so one slice's tensor-bound encoder overlaps another's HBM-bound decoder; phase_ms_per_slice and roofline are measured with the slices run one after the other",
                           "graph_lanes": int(os.environ.get("SB_GRAPH_LANES", "4")),
                           "encode_batch": int(os.environ.get("SB_ENCODE_BATCH", "24"))},
                "clocks": clocks, "e2e": e2e, "gpu_launches": launches, "roofline": roofline, "cpu_baseline": cpu}
        line.update(extras)
        _emit(line)
    if world > 1:
        dist.destroy_process_group()


_JSON_OUT = None


def _reserve_stdout():
    """The contract is ONE JSON line on stdout. Libraries (NCCL's version banner, torchrun children) write to file
    descriptor 1 directly, so keep a private duplicate of the real stdout for the JSON line and point fd 1 at stderr."""
    global _JSON_OUT
    sys.stdout.flush()
    _JSON_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)


def _emit(line: dict) -> None:
    out = _JSON_OUT if _JSON_OUT is not None else sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def main():
    args = parse_args()
    _reserve_stdout()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
