#!/usr/bin/env python
"""tools/distance_bench.py -- time of one ``dct_b200.signed_distance_map`` call (signed map of every class) and one
``dct_b200.distance_transform_edt`` call (inside distances of the foreground, scipy's function), against the host scipy
restatement (oracle/oracle_distance.py) on the same maps.

Shapes and maps are those of tools/surface_distance_bench.py (DESIGN.md §3.9): an ACDC patient (10 x 256^2, C = 4, '2d'
and '3d', spacing (10, 1.5625, 1.5625)), a Spleen batch (8 x 512^2, C = 2) and a Cityscapes-sized batch (16 x 512 x 1024,
C = 19), with smooth random blobs and salt-and-pepper maps.  The EDT call takes the mask ``map != 0``.  GPU time: CUDA
events around each call after warm-up, the two calls alternated in one loop, median and p10-p90 over --reps pairs.
Launches per call and the device time per kernel: a torch.profiler trace of one call, taken in a separate pass.  Host
time: the oracle's signed maps of every class (one scipy EDT per mask and complement, per grid and class) and scipy's
``distance_transform_edt`` of the mask per grid.  One JSON line per case, then a summary table.
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
from scipy.ndimage import distance_transform_edt  # noqa: E402

import oracle_distance as ODM  # noqa: E402
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


def kernel_profile(fn):
    """(launches, {kernel: device us}) of one call from a torch.profiler trace."""
    from torch.profiler import ProfilerActivity, profile
    fn(); torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA], acc_events=True) as prof:
        fn(); torch.cuda.synchronize()
    per = {}
    n = 0
    for e in prof.key_averages():
        if ("hd_" in e.key or "dm_" in e.key) and "kernel" in e.key:
            name = e.key.split("(")[0].replace("void ", "").replace("dct::", "")
            per[name] = round(float(e.device_time_total), 1)
            n += e.count
    return n, per


def stats(us):
    return float(np.median(us)), float(np.percentile(us, 10)), float(np.percentile(us, 90))


def host_time(fn, reps):
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        out = fn()
        ts.append(time.perf_counter() - t0)
    return float(np.median(ts)), out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--host-reps", type=int, default=1)
    ap.add_argument("--only", default=None, help="comma-separated case names")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "distance_bench measures the GPU call: no CUDA device found"
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
            m = (OH.blobs if kind == "blobs" else OH.salt_pepper)(rng, shape, C)
            mt = torch.from_numpy(m).to(dev)

            def sdm():
                return dct_b200.signed_distance_map(mt, C=C, method=method, voxelspacing=sp)

            def edt():
                return dct_b200.distance_transform_edt(mt, sampling=sp, method=method)

            fns = (sdm, edt)
            with dct_b200._runtime.check_mode("off"):
                for _ in range(args.warmup):
                    phi = sdm(); d = edt()
                torch.cuda.synchronize()
                ev = [[torch.cuda.Event(enable_timing=True) for _ in range(4)] for _ in range(args.reps)]
                for e in ev:   # alternated: signed maps, EDT
                    for i, f in enumerate(fns):
                        e[2 * i].record(); f(); e[2 * i + 1].record()
                torch.cuda.synchronize()
                us = [np.array([e[2 * i].elapsed_time(e[2 * i + 1]) * 1e3 for e in ev]) for i in range(2)]
                launches = [kernel_profile(f) for f in fns]
            grids = [m != 0] if method == "3d" else list(m != 0)
            h_sdm, ref = host_time(lambda: ODM.distance_map(m, C, 0, method, sp), args.host_reps)
            h_edt, ref_edt = host_time(lambda: [distance_transform_edt(g, sampling=sp) for g in grids], args.host_reps)
            ref_edt = np.stack(ref_edt).reshape(m.shape)
            rel = lambda g, w: float(np.max(np.abs(g.cpu().numpy() - w) / np.maximum(np.abs(w), 1e-30)))  # noqa: E731
            (s_m, s_10, s_90), (e_m, e_10, e_90) = (stats(u) for u in us)
            r = {"case": case, "shape": list(shape), "C": C, "method": method, "maps": kind, "spacing": list(sp),
                 "sdm_us_median": s_m, "sdm_us_p10": s_10, "sdm_us_p90": s_90,
                 "edt_us_median": e_m, "edt_us_p10": e_10, "edt_us_p90": e_90, "reps": args.reps,
                 "launches_sdm": launches[0][0], "launches_edt": launches[1][0],
                 "sdm_kernel_us": launches[0][1], "edt_kernel_us": launches[1][1],
                 "host_sdm_s": h_sdm, "host_edt_s": h_edt, "host_reps": args.host_reps, "host_cores": cores,
                 "speedup_sdm": h_sdm / (s_m * 1e-6), "speedup_edt": h_edt / (e_m * 1e-6),
                 "max_rel_err_sdm": rel(phi, ref), "max_rel_err_edt": rel(d, ref_edt),
                 "gpu": name, "power_limit": power}
            rows.append(r)
            print(json.dumps(r), flush=True)
    print(f"\n| case | C | method | maps | signed_distance_map us (median, p10-p90) | distance_transform_edt us | "
          f"launches | host scipy s, maps / EDT ({cores} cores) | speedup maps / EDT |")
    print("|---|---|---|---|---|---|---|---|---|")
    for r in rows:
        print(f"| {r['case']} {'x'.join(map(str, r['shape']))} | {r['C']} | {r['method']} | {r['maps']} | "
              f"{r['sdm_us_median']:.1f} ({r['sdm_us_p10']:.1f}-{r['sdm_us_p90']:.1f}) | "
              f"{r['edt_us_median']:.1f} ({r['edt_us_p10']:.1f}-{r['edt_us_p90']:.1f}) | "
              f"{r['launches_sdm']} / {r['launches_edt']} | {r['host_sdm_s']:.3f} / {r['host_edt_s']:.3f} | "
              f"{r['speedup_sdm']:.0f}x / {r['speedup_edt']:.0f}x |")


if __name__ == "__main__":
    main()
