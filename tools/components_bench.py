#!/usr/bin/env python
"""tools/components_bench.py -- time of one ``dct_b200.largest_component`` and one ``dct_b200.connected_components`` call
against the host scipy restatement (oracle/oracle_components.py: ``scipy.ndimage.label`` per class and grid), and next
to one ``dct_b200.surface_distances`` call on the same prediction, which is what the post-processing sits in front of.

Shapes: an ACDC patient (10 x 256^2, C = 4, '2d' and '3d'), a Spleen volume (64 x 512^2, C = 2, '3d') and a
Cityscapes-sized batch (16 x 512 x 1024, C = 19, '2d').  Maps: smooth random blobs (the usual case), salt-and-pepper
(about one component per few pixels: the most roots, sizes and counts) and a one-pixel-wide serpentine through every
tile (one component with long merge chains and one hot root).  Connectivity 1 (scipy's and nnU-Net's default) and the
full one (skimage's default).  GPU time: CUDA events around each call after warm-up, the three calls alternated in one
loop, median and spread over --reps rounds (inputs and scratch stay in L2 where they fit: the time of a call in an
evaluation loop).  Launches per call and device time per kernel: a torch.profiler trace of one call, in a separate pass.
One JSON line per case, then a summary table.
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

import oracle_components as OC  # noqa: E402
import oracle_hausdorff as OH  # noqa: E402

CASES = [  # name, (B, H, W), C, method
    ("acdc", (10, 256, 256), 4, "2d"),
    ("acdc", (10, 256, 256), 4, "3d"),
    ("spleen", (64, 512, 512), 2, "3d"),
    ("large", (16, 512, 1024), 19, "2d"),
]


def serpentine(shape):
    """Class 1 on a one-pixel-wide path through every row pair of every even slice, odd slices joining the paths' ends."""
    B, H, W = shape
    m = np.zeros(shape, np.int64)
    for b in range(0, B, 2):
        m[b, 0::2, :] = 1
        for y in range(1, H, 2):
            m[b, y, W - 1 if y % 4 == 1 else 0] = 1
        if b + 1 < B:
            m[b + 1, H - 1 if (H - 1) % 2 == 0 else H - 2, 0] = 1
    return m


def gpu_info():
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                            capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        pl = f"unavailable ({e})"
    return name, pl


def kernel_profile(fn, prefixes):
    """(launches, {kernel: device us}) of one call from a torch.profiler trace."""
    from torch.profiler import ProfilerActivity, profile
    fn(); torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA], acc_events=True) as prof:
        fn(); torch.cuda.synchronize()
    per, n = {}, 0
    for e in prof.key_averages():
        if any(p in e.key for p in prefixes) and "kernel" in e.key:
            name = e.key.split("(")[0].replace("void ", "").replace("dct::", "")
            per[name] = round(float(e.device_time_total), 1)
            n += e.count
    return n, per


def stats_us(a):
    return float(np.median(a)), float(np.percentile(a, 10)), float(np.percentile(a, 90))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--only", default=None, help="comma-separated case names")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "components_bench measures the GPU call: no CUDA device found"
    import dct_b200
    dev = torch.device("cuda:0")
    name, power = gpu_info()
    cores = len(os.sched_getaffinity(0))
    print(f"# GPU {name}, power limit {power}; host: {cores} cores available to this process "
          f"(scipy.ndimage.label is single-threaded)", flush=True)
    rows = []
    for case, shape, C, method in CASES:
        if args.only and case not in args.only.split(","):
            continue
        sp = (10.0, 1.5625, 1.5625) if method == "3d" else (1.5625, 1.5625)
        for kind in ("blobs", "saltpepper", "serpentine"):
            rng = np.random.default_rng(1)
            if kind == "serpentine":
                p = serpentine(shape)
                g = OH.blobs(rng, shape, C)
            else:
                make = OH.blobs if kind == "blobs" else OH.salt_pepper
                p, g = make(rng, shape, C), make(rng, shape, C)
            pt, gt = torch.from_numpy(p).to(dev), torch.from_numpy(g).to(dev)
            for conn in (1, 3 if method == "3d" else 2):
                def largest():
                    return dct_b200.largest_component(pt, C=C, method=method, connectivity=conn)

                def labels():
                    return dct_b200.connected_components(pt, C=C, method=method, connectivity=conn)

                def surf():
                    return dct_b200.surface_distances(pt, gt, C=C, method=method, voxelspacing=sp)

                with dct_b200._runtime.check_mode("off"):
                    for _ in range(args.warmup):
                        big = largest(); cc = labels(); surf()
                    torch.cuda.synchronize()
                    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(6)] for _ in range(args.reps)]
                    for e in ev:   # alternated: largest_component, connected_components, surface_distances
                        e[0].record(); largest(); e[1].record()
                        e[2].record(); labels(); e[3].record()
                        e[4].record(); surf(); e[5].record()
                    torch.cuda.synchronize()
                    us = [np.array([e[2 * i].elapsed_time(e[2 * i + 1]) * 1e3 for e in ev]) for i in range(3)]
                    nl_big, k_big = kernel_profile(largest, ("cc_",))
                    nl_cc, _ = kernel_profile(labels, ("cc_",))
                t0 = time.perf_counter()
                want = OC.components(p, C, method, conn)
                host_s = time.perf_counter() - t0
                stats = torch.stack((cc["count"], cc["largest"]), -1).cpu().numpy()
                equal = bool(np.array_equal(cc["labels"].cpu().numpy(), want[0]) and np.array_equal(stats, want[1])
                             and np.array_equal(big.cpu().numpy(), want[2]))
                (lm, l10, l90), (cm, c10, c90), (sm, s10, s90) = (stats_us(u) for u in us)
                r = {"case": case, "shape": list(shape), "C": C, "method": method, "maps": kind, "connectivity": conn,
                     "largest_us_median": lm, "largest_us_p10": l10, "largest_us_p90": l90,
                     "components_us_median": cm, "components_us_p10": c10, "components_us_p90": c90,
                     "surface_us_median": sm, "surface_us_p10": s10, "surface_us_p90": s90,
                     "largest_over_surface": lm / sm, "reps": args.reps,
                     "launches_largest": nl_big, "launches_components": nl_cc, "largest_kernel_us": k_big,
                     "host_scipy_s": host_s, "host_cores": cores, "speedup_largest": host_s / (lm * 1e-6),
                     "equal_to_oracle": equal, "gpu": name, "power_limit": power}
                rows.append(r)
                print(json.dumps(r), flush=True)
    print(f"\n| case | C | method | maps | conn | largest_component us (median, p10-p90) | connected_components us | "
          f"surface_distances us | largest / surface | launches | host scipy s | speedup | equal |")
    print("|---|---|---|---|---|---|---|---|---|---|---|---|---|")
    for r in rows:
        print(f"| {r['case']} {'x'.join(map(str, r['shape']))} | {r['C']} | {r['method']} | {r['maps']} | "
              f"{r['connectivity']} | {r['largest_us_median']:.1f} ({r['largest_us_p10']:.1f}-{r['largest_us_p90']:.1f}) | "
              f"{r['components_us_median']:.1f} | {r['surface_us_median']:.1f} | {r['largest_over_surface']:.3f} | "
              f"{r['launches_largest']} / {r['launches_components']} | {r['host_scipy_s']:.3f} | "
              f"{r['speedup_largest']:.0f}x | {r['equal_to_oracle']} |")


if __name__ == "__main__":
    main()
