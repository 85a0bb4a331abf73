#!/usr/bin/env python
"""tools/surface_distance_bench.py -- time of one ``dct_b200.surface_distances`` call (HD, HD95, ASD, ASSD) against one
``dct_b200.hausdorff`` call on the same class maps, and against the host scipy restatement of medpy hd95 / asd / assd
(oracle/oracle_surface.py).

Shapes are those of tools/hausdorff_bench.py (DESIGN.md §3.9): an ACDC patient (10 x 256^2, C = 4, '2d' and '3d', spacing
(10, 1.5625, 1.5625)), a Spleen batch (8 x 512^2, C = 2) and a Cityscapes-sized batch (16 x 512 x 1024, C = 19), with
smooth random blobs and salt-and-pepper maps (almost every pixel a border pixel: the most queries and the fullest
histogram bins).  GPU time: CUDA events around each call after warm-up, the two calls alternated in one loop, median and
spread over --reps pairs (inputs and scratch stay in L2 where they fit: the time of a call in an evaluation loop).
Launches per call and the device time per kernel: a torch.profiler trace of one call, taken in a separate pass.  One JSON
line per case, then a summary table.
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
import oracle_surface as OS  # noqa: E402

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


def kernel_profile(fn):
    """(launches, {kernel: device us}) of one call from a torch.profiler trace."""
    from torch.profiler import ProfilerActivity, profile
    fn(); torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA], acc_events=True) as prof:
        fn(); torch.cuda.synchronize()
    per = {}
    n = 0
    for e in prof.key_averages():
        if ("hd_" in e.key or "sd_" in e.key) and "kernel" in e.key:
            name = e.key.split("(")[0].replace("void ", "").replace("dct::", "")
            per[name] = round(float(e.device_time_total), 1)
            n += e.count
    return n, per


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--host-reps", type=int, default=1)
    ap.add_argument("--only", default=None, help="comma-separated case names")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "surface_distance_bench measures the GPU call: no CUDA device found"
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

            def surf():
                return dct_b200.surface_distances(pt, gt, C=C, method=method, voxelspacing=sp)

            def hd():
                return dct_b200.hausdorff(pt, gt, C=C, method=method, voxelspacing=sp)

            with dct_b200._runtime.check_mode("off"):
                for _ in range(args.warmup):
                    out = surf(); hd_out = hd()
                torch.cuda.synchronize()
                ev = [[torch.cuda.Event(enable_timing=True) for _ in range(4)] for _ in range(args.reps)]
                for e in ev:   # alternated: surface, then hausdorff
                    e[0].record(); surf(); e[1].record()
                    e[2].record(); hd(); e[3].record()
                torch.cuda.synchronize()
                us_s = np.array([e[0].elapsed_time(e[1]) * 1e3 for e in ev])
                us_h = np.array([e[2].elapsed_time(e[3]) * 1e3 for e in ev])
                nl_s, k_s = kernel_profile(surf)
                nl_h, _ = kernel_profile(hd)
            got = {k: v.cpu().numpy() for k, v in out.items()}
            hd_same = bool(np.array_equal(got["hd"].view(np.uint32), hd_out.cpu().numpy().view(np.uint32)))
            host = []
            for _ in range(args.host_reps):
                t0 = time.perf_counter()
                ref = OS.surface(p, g, C, method, sp)
                host.append(time.perf_counter() - t0)
            err = {}
            for k in OS.KEYS:
                nan = np.isnan(ref[k])
                ok = ~nan & (ref[k] > 0)
                err[k] = float(np.max(np.abs(got[k][ok] - ref[k][ok]) / ref[k][ok])) if ok.any() else 0.0
                err[k + "_nan_match"] = bool(np.array_equal(np.isnan(got[k]), nan))
            r = {"case": case, "shape": list(shape), "C": C, "method": method, "maps": kind, "spacing": list(sp),
                 "surface_us_median": float(np.median(us_s)), "surface_us_p10": float(np.percentile(us_s, 10)),
                 "surface_us_p90": float(np.percentile(us_s, 90)),
                 "hausdorff_us_median": float(np.median(us_h)), "hausdorff_us_p10": float(np.percentile(us_h, 10)),
                 "hausdorff_us_p90": float(np.percentile(us_h, 90)),
                 "ratio": float(np.median(us_s) / np.median(us_h)), "reps": args.reps,
                 "launches_surface": nl_s, "launches_hausdorff": nl_h, "surface_kernel_us": k_s,
                 "host_scipy_s": float(np.median(host)), "host_reps": args.host_reps, "host_cores": cores,
                 "speedup": float(np.median(host)) / (float(np.median(us_s)) * 1e-6),
                 "hd_bitwise_equal_hausdorff": hd_same, "max_rel_err_vs_oracle": err,
                 "gpu": name, "power_limit": power}
            rows.append(r)
            print(json.dumps(r), flush=True)
    print(f"\n| case | C | method | maps | surface us (median, p10-p90) | hausdorff us (median, p10-p90) | ratio | "
          f"launches | host scipy s ({cores} cores) | speedup |")
    print("|---|---|---|---|---|---|---|---|---|---|")
    for r in rows:
        print(f"| {r['case']} {'x'.join(map(str, r['shape']))} | {r['C']} | {r['method']} | {r['maps']} | "
              f"{r['surface_us_median']:.1f} ({r['surface_us_p10']:.1f}-{r['surface_us_p90']:.1f}) | "
              f"{r['hausdorff_us_median']:.1f} ({r['hausdorff_us_p10']:.1f}-{r['hausdorff_us_p90']:.1f}) | "
              f"{r['ratio']:.2f} | {r['launches_surface']} / {r['launches_hausdorff']} | {r['host_scipy_s']:.3f} | "
              f"{r['speedup']:.0f}x |")


if __name__ == "__main__":
    main()
