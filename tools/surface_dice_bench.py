#!/usr/bin/env python
"""tools/surface_dice_bench.py -- time of one ``dct_b200.surface_dice`` call (normalized surface Dice) against one
``dct_b200.hausdorff`` and one ``dct_b200.surface_distances`` call on the same class maps, and against the host scipy
restatement (oracle/oracle_surface_dice.py).

Shapes and maps are those of tools/surface_distance_bench.py (DESIGN.md §3.9 / §3.11): an ACDC patient (10 x 256^2, C = 4,
'2d' and '3d', spacing (10, 1.5625, 1.5625)), a Spleen batch (8 x 512^2, C = 2) and a Cityscapes-sized batch
(16 x 512 x 1024, C = 19), with smooth random blobs and salt-and-pepper maps (almost every pixel a border pixel).
Tolerance: 2 spacing units (3.125 at this spacing) for every class.  GPU time: CUDA events around each call after
warm-up, the three calls alternated in one loop, median and p10-p90 over --reps triples.  Launches per call and the
device time per kernel: a torch.profiler trace of one call, taken in a separate pass.  One JSON line per case, then a
summary table.
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
import oracle_surface_dice as OD  # noqa: E402

ACDC_SPACING = (10.0, 1.5625, 1.5625)
TOLERANCE = 3.125
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
        if ("hd_" in e.key or "sd_" in e.key or "nsd_" in e.key) and "kernel" in e.key:
            name = e.key.split("(")[0].replace("void ", "").replace("dct::", "")
            per[name] = round(float(e.device_time_total), 1)
            n += e.count
    return n, per


def stats(us):
    return float(np.median(us)), float(np.percentile(us, 10)), float(np.percentile(us, 90))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--host-reps", type=int, default=1)
    ap.add_argument("--only", default=None, help="comma-separated case names")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "surface_dice_bench measures the GPU call: no CUDA device found"
    import dct_b200
    dev = torch.device("cuda:0")
    name, power = gpu_info()
    cores = len(os.sched_getaffinity(0))
    print(f"# GPU {name}, power limit {power}; host: {cores} cores available to this process "
          f"(scipy's EDT is single-threaded); tolerance {TOLERANCE}", flush=True)
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

            def nsd():
                return dct_b200.surface_dice(pt, gt, TOLERANCE, C=C, method=method, voxelspacing=sp)

            def hd():
                return dct_b200.hausdorff(pt, gt, C=C, method=method, voxelspacing=sp)

            def surf():
                return dct_b200.surface_distances(pt, gt, C=C, method=method, voxelspacing=sp)

            fns = (nsd, hd, surf)
            with dct_b200._runtime.check_mode("off"):
                for _ in range(args.warmup):
                    out = nsd(); hd(); surf()
                torch.cuda.synchronize()
                ev = [[torch.cuda.Event(enable_timing=True) for _ in range(6)] for _ in range(args.reps)]
                for e in ev:   # alternated: surface Dice, hausdorff, surface distances
                    for i, f in enumerate(fns):
                        e[2 * i].record(); f(); e[2 * i + 1].record()
                torch.cuda.synchronize()
                us = [np.array([e[2 * i].elapsed_time(e[2 * i + 1]) * 1e3 for e in ev]) for i in range(3)]
                launches = [kernel_profile(f) for f in fns]
            got = out["counts"].cpu().numpy()
            host = []
            for _ in range(args.host_reps):
                t0 = time.perf_counter()
                ref = OD.surface_dice(p, g, C, TOLERANCE, method, sp)
                host.append(time.perf_counter() - t0)
            diff = np.abs(got - ref["counts"])
            (n_m, n_10, n_90), (h_m, h_10, h_90), (s_m, s_10, s_90) = (stats(u) for u in us)
            r = {"case": case, "shape": list(shape), "C": C, "method": method, "maps": kind, "spacing": list(sp),
                 "tolerance": TOLERANCE,
                 "nsd_us_median": n_m, "nsd_us_p10": n_10, "nsd_us_p90": n_90,
                 "hausdorff_us_median": h_m, "hausdorff_us_p10": h_10, "hausdorff_us_p90": h_90,
                 "surface_us_median": s_m, "surface_us_p10": s_10, "surface_us_p90": s_90,
                 "ratio_vs_hausdorff": n_m / h_m, "ratio_vs_surface": n_m / s_m, "reps": args.reps,
                 "launches_nsd": launches[0][0], "launches_hausdorff": launches[1][0],
                 "launches_surface": launches[2][0], "nsd_kernel_us": launches[0][1],
                 "host_scipy_s": float(np.median(host)), "host_reps": args.host_reps, "host_cores": cores,
                 "speedup": float(np.median(host)) / (n_m * 1e-6),
                 "counts_equal_oracle": bool(not diff.any()), "max_count_diff": int(diff.max()),
                 "gpu": name, "power_limit": power}
            rows.append(r)
            print(json.dumps(r), flush=True)
    print(f"\n| case | C | method | maps | surface_dice us (median, p10-p90) | hausdorff us | surface_distances us | "
          f"launches | host scipy s ({cores} cores) | speedup |")
    print("|---|---|---|---|---|---|---|---|---|---|")
    for r in rows:
        print(f"| {r['case']} {'x'.join(map(str, r['shape']))} | {r['C']} | {r['method']} | {r['maps']} | "
              f"{r['nsd_us_median']:.1f} ({r['nsd_us_p10']:.1f}-{r['nsd_us_p90']:.1f}) | "
              f"{r['hausdorff_us_median']:.1f} ({r['hausdorff_us_p10']:.1f}-{r['hausdorff_us_p90']:.1f}) | "
              f"{r['surface_us_median']:.1f} ({r['surface_us_p10']:.1f}-{r['surface_us_p90']:.1f}) | "
              f"{r['launches_nsd']} / {r['launches_hausdorff']} / {r['launches_surface']} | {r['host_scipy_s']:.3f} | "
              f"{r['speedup']:.0f}x |")


if __name__ == "__main__":
    main()
