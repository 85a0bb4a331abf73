#!/usr/bin/env python
"""tools/hausdorff_bench.py -- time of one ``dct_b200.hausdorff`` call against the host scipy restatement of
medpy.metric.binary.hd (oracle/oracle_hausdorff.py) on the same class maps.

Shapes are the ones a user evaluates: an ACDC patient (10 x 256^2, C = 4, '2d' and '3d', spacing (10, 1.5625, 1.5625)), a
Spleen batch (8 x 512^2, C = 2) and a Cityscapes-sized batch (16 x 512 x 1024, C = 19).  Class maps are smooth random blobs
and salt-and-pepper noise (almost every pixel a border pixel: the most features and queries per line).  GPU time: CUDA
events around each call after warm-up, median and spread over --reps calls (inputs and scratch stay in L2 where they fit:
this is the time of a call in an evaluation loop).  Launches per call: kernels in a torch.profiler trace of one call,
taken in a separate pass.  One JSON line per case, then a summary table.
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

import oracle_hausdorff as OH  # noqa: E402

ACDC_SPACING = (10.0, 1.5625, 1.5625)
CASES = [  # name, (B, H, W), C, method
    ("acdc", (10, 256, 256), 4, "2d"),
    ("acdc", (10, 256, 256), 4, "3d"),
    ("spleen", (8, 512, 512), 2, "2d"),
    ("spleen", (8, 512, 512), 2, "3d"),
    ("large", (16, 512, 1024), 19, "2d"),
]


def gpu_info():
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                            capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        pl = f"unavailable ({e})"
    return name, pl


def launches_per_call(fn):
    from torch.profiler import ProfilerActivity, profile
    fn(); torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA], acc_events=True) as prof:
        fn(); torch.cuda.synchronize()
    counts = {e.key.split("(")[0].replace("void ", ""): e.count for e in prof.key_averages()
              if "hd_" in e.key and "kernel" in e.key}
    return sum(counts.values()), sorted(counts)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--host-reps", type=int, default=1)
    ap.add_argument("--only", default=None, help="comma-separated case names")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "hausdorff_bench measures the GPU call: no CUDA device found"
    import dct_b200
    dev = torch.device("cuda:0")
    name, power = gpu_info()
    cores = len(os.sched_getaffinity(0))
    print(f"# GPU {name}, power limit {power}; host: {cores} cores available to this process "
          f"(scipy's EDT is single-threaded)", flush=True)
    rows = []
    for case, shape, C, method in CASES:
        if args.only and case not in args.only.split(","):
            continue
        sp = ACDC_SPACING if method == "3d" else ACDC_SPACING[1:]
        for kind in ("blobs", "saltpepper"):
            rng = np.random.default_rng(1)
            make = OH.blobs if kind == "blobs" else OH.salt_pepper
            p, g = make(rng, shape, C), make(rng, shape, C)
            pt, gt = torch.from_numpy(p).to(dev), torch.from_numpy(g).to(dev)

            def call():
                return dct_b200.hausdorff(pt, gt, C=C, method=method, voxelspacing=sp)

            with dct_b200._runtime.check_mode("off"):
                for _ in range(args.warmup):
                    out = call()
                torch.cuda.synchronize()
                ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.reps)]
                for a, b in ev:
                    a.record(); call(); b.record()
                torch.cuda.synchronize()
                us = np.array([a.elapsed_time(b) * 1e3 for a, b in ev])
                nl, knames = launches_per_call(call)
            gpu = out.cpu().numpy()
            host = []
            for _ in range(args.host_reps):
                t0 = time.perf_counter()
                ref = OH.hausdorff(p, g, C, method, sp)
                host.append(time.perf_counter() - t0)
            nan = np.isnan(ref)
            err = float(np.max(np.abs(gpu[~nan] - ref[~nan]) / ref[~nan].clip(min=1e-30))) if (~nan).any() else 0.0
            r = {"case": case, "shape": list(shape), "C": C, "method": method, "maps": kind, "spacing": list(sp),
                 "gpu_us_median": float(np.median(us)), "gpu_us_p10": float(np.percentile(us, 10)),
                 "gpu_us_p90": float(np.percentile(us, 90)), "gpu_us_min": float(us.min()), "reps": args.reps,
                 "launches_per_call": nl, "kernels": knames,
                 "host_scipy_s": float(np.median(host)), "host_reps": args.host_reps, "host_cores": cores,
                 "speedup": float(np.median(host)) / (float(np.median(us)) * 1e-6),
                 "max_rel_err_vs_oracle": err, "nan_match": bool(np.array_equal(np.isnan(gpu), nan)),
                 "gpu": name, "power_limit": power}
            rows.append(r)
            print(json.dumps(r), flush=True)
    print(f"\n| case | C | method | maps | GPU us (median, p10-p90) | launches | host scipy s ({cores} cores) | speedup |")
    print("|---|---|---|---|---|---|---|---|")
    for r in rows:
        print(f"| {r['case']} {'x'.join(map(str, r['shape']))} | {r['C']} | {r['method']} | {r['maps']} | "
              f"{r['gpu_us_median']:.1f} ({r['gpu_us_p10']:.1f}-{r['gpu_us_p90']:.1f}) | {r['launches_per_call']} | "
              f"{r['host_scipy_s']:.3f} | {r['speedup']:.0f}x |")


if __name__ == "__main__":
    main()
