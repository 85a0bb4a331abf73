#!/usr/bin/env python
"""tools/boundary_iou_bench.py -- time of one ``dct_b200.boundary_iou`` call (Boundary IoU, default band width) against
one ``dct_confusion_labels_i64`` launch on the same int64 maps (the IoU meter's counting: it reads the same 16 B/pixel),
and against the host forms of the definition (cv2 and the scipy restatement, oracle/oracle_boundary_iou.py).

Shapes: an ACDC patient (10 x 256^2, C = 4), a Spleen batch (8 x 512^2, C = 2), a 16 x 512 x 1024 batch and a Cityscapes
batch (4 x 1024 x 2048), both C = 19; the last with ignore label 255 on a 2 % sprinkle plus blocks.  Maps: smooth random
blobs and salt-and-pepper (every pixel of another class than some neighbour), as tools/surface_dice_bench.py builds them.
GPU time: CUDA events around each call after warm-up, the two calls alternated in one loop, median and p10-p90 over
--reps pairs.  Per-launch device time: the mean over a torch.profiler trace of 8 calls, taken in a separate pass.
Algorithmic bytes: 16 B/pixel of int64 maps read + 2 B/pixel of records written and read back.  Host time: every class
of pred and gt of one image, single-threaded, times B (not a timed batch).  One JSON line per case, then a summary
table.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for _p in (ROOT, os.path.join(ROOT, "oracle")):
    sys.path.insert(0, _p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import oracle_boundary_iou as OB  # noqa: E402
import oracle_hausdorff as OH  # noqa: E402

CASES = [  # name, (B, H, W), C, ignore
    ("acdc", (10, 256, 256), 4, None),
    ("spleen", (8, 512, 512), 2, None),
    ("large", (16, 512, 1024), 19, None),
    ("cityscapes", (4, 1024, 2048), 19, 255),
]


def gpu_info():
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                            capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        pl = f"unavailable ({e})"
    return name, pl


def kernel_profile(fn, keys, calls=8):
    """(launches per call, {kernel: mean device us per call}) from a torch.profiler trace of `calls` calls (a trace of a
    single call can miss its longest kernels)."""
    from torch.profiler import ProfilerActivity, profile
    fn(); torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA], acc_events=True) as prof:
        for _ in range(calls):
            fn()
        torch.cuda.synchronize()
    per, n = {}, 0
    for e in prof.key_averages():
        if any(k in e.key for k in keys):
            name = e.key.split("(")[0].replace("void ", "").replace("dct::", "")
            per[name] = round(float(e.device_time_total) / calls, 1)
            n += e.count
    return n / calls, per


def stats(us):
    return float(np.median(us)), float(np.percentile(us, 10)), float(np.percentile(us, 90))


def host_time(p, g, C, d, band):
    t0 = time.perf_counter()
    for c in range(C):
        band(p == c, d); band(g == c, d)
    return time.perf_counter() - t0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--only", default=None, help="comma-separated case names")
    ap.add_argument("--no-host", action="store_true")
    args = ap.parse_args()
    assert args.reps >= 30
    assert torch.cuda.is_available(), "boundary_iou_bench measures the GPU call: no CUDA device found"
    import dct_b200
    try:
        import cv2
        cv2.setNumThreads(1)
    except ImportError:
        cv2 = None
    dev = torch.device("cuda:0")
    h = dct_b200._lib.lib()
    name, power = gpu_info()
    print(f"# GPU {name}, power limit {power}; host times single-threaded, one image times B", flush=True)
    rows = []
    for case, shape, C, ignore in CASES:
        if args.only and case not in args.only.split(","):
            continue
        B, H, W = shape
        d = OB.dilation_for(H, W)
        for kind in ("blobs", "saltpepper"):
            rng = np.random.default_rng(1)
            make = OH.blobs if kind == "blobs" else OH.salt_pepper
            p, g = make(rng, shape, C), make(rng, shape, C)
            if ignore is not None:
                g[rng.random(shape) < 0.02] = ignore
                for b in range(B):
                    for _ in range(6):
                        y, x = rng.integers(0, H - 128), rng.integers(0, W - 256)
                        g[b, y: y + 128, x: x + 256] = ignore
            pt, gt = torch.from_numpy(p).to(dev), torch.from_numpy(g).to(dev)
            conf = torch.zeros((C, C), dtype=torch.int64, device=dev)
            stream = torch.cuda.current_stream(dev).cuda_stream

            def biou():
                return dct_b200.boundary_iou(pt, gt, C=C, ignore_index=ignore)

            def confusion():
                h.dct_confusion_labels_i64(pt.data_ptr(), gt.data_ptr(), pt.numel(), C, conf.data_ptr(), None, stream)

            with dct_b200._runtime.check_mode("off"):
                for _ in range(args.warmup):
                    out = biou(); confusion()
                torch.cuda.synchronize()
                ev = [[torch.cuda.Event(enable_timing=True) for _ in range(4)] for _ in range(args.reps)]
                for e in ev:   # alternated: Boundary IoU, confusion counting
                    e[0].record(); biou(); e[1].record()
                    e[2].record(); confusion(); e[3].record()
                torch.cuda.synchronize()
                us_b = np.array([e[0].elapsed_time(e[1]) * 1e3 for e in ev])
                us_c = np.array([e[2].elapsed_time(e[3]) * 1e3 for e in ev])
                launches, per_kernel = kernel_profile(biou, ("biou_",))
                _, conf_kernel = kernel_profile(confusion, ("confusion",))
            want = OB.boundary_iou(p[:1], g[:1], C, d, ignore)["counts"]
            equal = bool(np.array_equal(out["counts"][:1].cpu().numpy(), want))
            host_cv2 = host_scipy = None
            if not args.no_host:
                host_scipy = host_time(p[0], g[0], C, d, OB.mask_to_boundary) * B
                if cv2 is not None:
                    host_cv2 = host_time(p[0], g[0], C, d, OB.mask_to_boundary_cv2) * B
            (b_m, b_10, b_90), (c_m, c_10, c_90) = stats(us_b), stats(us_c)
            npx = B * H * W
            r = {"case": case, "shape": list(shape), "C": C, "d": d, "ignore": ignore, "maps": kind,
                 "biou_us_median": b_m, "biou_us_p10": b_10, "biou_us_p90": b_90,
                 "confusion_us_median": c_m, "confusion_us_p10": c_10, "confusion_us_p90": c_90,
                 "ratio_vs_confusion": b_m / c_m, "reps": args.reps, "launches": launches,
                 "kernel_us": per_kernel, "confusion_kernel_us": conf_kernel,
                 "algorithmic_bytes": 20 * npx, "biou_GBps": 20 * npx / (b_m * 1e3),
                 "confusion_bytes": 16 * npx, "confusion_GBps": 16 * npx / (c_m * 1e3),
                 "host_cv2_s": host_cv2, "host_scipy_s": host_scipy,
                 "counts_equal_oracle_image0": equal, "gpu": name, "power_limit": power}
            rows.append(r)
            print(json.dumps(r), flush=True)
    print("\n| case | C | d | maps | boundary_iou us (median, p10-p90) | per launch us | confusion us | ratio | "
          "GB/s (20 B/px) | host cv2 s | host scipy s |")
    print("|---|---|---|---|---|---|---|---|---|---|---|")
    for r in rows:
        kern = " / ".join(f"{k.split('_')[1]} {v:.1f}" for k, v in r["kernel_us"].items())
        hc = "-" if r["host_cv2_s"] is None else f"{r['host_cv2_s']:.2f}"
        hs = "-" if r["host_scipy_s"] is None else f"{r['host_scipy_s']:.2f}"
        print(f"| {r['case']} {'x'.join(map(str, r['shape']))} | {r['C']} | {r['d']} | {r['maps']} | "
              f"{r['biou_us_median']:.1f} ({r['biou_us_p10']:.1f}-{r['biou_us_p90']:.1f}) | {kern} | "
              f"{r['confusion_us_median']:.1f} | {r['ratio_vs_confusion']:.2f} | {r['biou_GBps']:.0f} | {hc} | {hs} |")


if __name__ == "__main__":
    main()
