#!/usr/bin/env python
"""Developer tool: in-kernel timeline of one consistency step (GPU box).

Every CTA of every launch stamps %globaltimer (dct_dev_trace_begin / _end, include/dct_b200.h): after its
programmatic-dependency wait, at a kernel-specific mid point, and at its end.  Printed per launch, relative to the first
stamp of the chain: when the first / last CTA started, when the first data landed, when the first / last CTA ended --
i.e. where a step's microseconds go BETWEEN the kernels (launch-to-launch gaps, ramps, tails), which event timing of
whole launches cannot show.

Then each launch's end segments, the chain a CTA runs after its last tile or store: tile pipeline "tiles done" ->
"stores read out" -> "ticket drawn" -> end, cluster normalisation "stores issued" -> end; the median and the maximum
over the launch's CTAs, and "tail": the last CTA's "tiles done" / "stores issued" -> the last CTA end.

    python tools/step_trace.py [--workload c2] [--steps 6] [--graph 1]
"""
import argparse
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import dct_b200  # noqa: E402
from bench import WORKLOADS  # noqa: E402
from dct_b200.engine import ConsistencyStep, StepBuffers  # noqa: E402

SLOTS = 8   # kTraceSlots (csrc/dct_common.cuh)
END_POINTS = [(4, "done"), (5, "read"), (6, "ticket"), (3, "end")]   # end-segment stamps in chain order


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="c2")
    ap.add_argument("--steps", type=int, default=6)
    ap.add_argument("--parts", default="", help="comma list: trace a chain of these parts instead of whole steps")
    args = ap.parse_args()
    K, C, B, H, W, cin, _ = WORKLOADS[args.workload]
    dev = torch.device("cuda", 0)
    h = dct_b200._lib.lib()
    with_vat, with_dice = args.workload != "c1", args.workload != "c4"
    step = ConsistencyStep(K, C, B, H, W, cin=cin, with_vat=with_vat, with_dice=with_dice)
    gen = torch.Generator(device=dev).manual_seed(1)
    R = 4
    sets = [StepBuffers.allocate(K, C, B, H, W, cin, dev, gen) for _ in range(R)]
    dct_b200.set_check_mode("deferred")
    parts = [p for p in args.parts.split(",") if p] or list(step.parts())
    for s in sets:   # warm-up (workspace allocation, module load, function attributes)
        for p in parts:
            step.run_part(s, p)
    torch.cuda.synchronize()
    max_ctas, nl = 1024, args.steps * len(parts)
    buf = torch.zeros(nl * max_ctas * SLOTS, dtype=torch.int64, device=dev)
    # the chain is captured into ONE CUDA graph while tracing is on (every captured launch gets its slice of the trace
    # buffer baked in), then replayed: no host launch latency between the kernels, as in bench.py
    side = torch.cuda.Stream(device=dev)
    side.wait_stream(torch.cuda.current_stream(dev))
    with torch.cuda.stream(side):
        for p in parts:
            step.run_part(sets[0], p)
    torch.cuda.current_stream(dev).wait_stream(side)
    torch.cuda.synchronize()
    assert h.dct_dev_trace_begin(buf.data_ptr(), max_ctas, nl) == 0
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=side):
        for i in range(args.steps):
            for p in parts:
                step.run_part(sets[i % R], p)
    g.replay()
    torch.cuda.synchronize()
    buf.zero_()
    torch.cuda.synchronize()
    g.replay()
    torch.cuda.synchronize()
    n = h.dct_dev_trace_end()
    t = buf.view(nl, max_ctas, SLOTS).cpu().numpy().astype("int64")
    names = [parts[i % len(parts)] for i in range(n)]
    t0 = None
    prev_end = None
    print(f"{args.workload}: {n} traced launches; times in us relative to the first start; one CUDA graph, launches chained with PDL")
    print(f"{'launch':<14}{'ctas':>5} {'start0':>8} {'startN':>8} {'mid1_0':>8} {'mid1_N':>8} {'mid2_N':>8} {'end0':>8} {'endN':>8}"
          f" {'window':>8} {'gap':>6} {'life':>7}")
    rows = []
    segs = []   # per launch: (name, {segment: (median, max)}, tail)
    for i in range(n):
        a = t[i]
        live = a[:, 0] > 0
        if not live.any():
            continue
        s, e = a[live, 0], a[live, 3]
        m1 = a[live, 1][a[live, 1] > 0]
        m2 = a[live, 2][a[live, 2] > 0]
        if t0 is None:
            t0 = s.min()
        us = lambda v: (v - t0) / 1e3  # noqa: E731
        gap = (s.min() - prev_end) / 1e3 if prev_end is not None else float("nan")
        prev_end = e.max()
        rows.append((names[i], int(live.sum()), us(s.min()), us(s.max()), us(m1.min()) if m1.size else float("nan"),
                     us(m1.max()) if m1.size else float("nan"), us(m2.max()) if m2.size else float("nan"), us(e.min()),
                     us(e.max()), (e.max() - s.min()) / 1e3, gap, float((e - s).mean()) / 1e3))
        pts = [(k, nm) for k, nm in END_POINTS if (a[live, k] > 0).all()]
        seg = {}
        for (k0, n0), (k1, n1) in zip(pts, pts[1:]):
            d = (a[live, k1] - a[live, k0]) / 1e3
            seg[f"{n0}->{n1}"] = (float(np.median(d)), float(d.max()))
        tail = (e.max() - a[live, pts[0][0]].max()) / 1e3 if len(pts) > 1 else float("nan")
        segs.append((names[i], seg, tail))
    for r in rows[len(parts):]:   # skip the first step (cold instruction caches)
        print(f"{r[0]:<14}{r[1]:>5} " + " ".join(f"{v:8.2f}" for v in r[2:9]) + f" {r[9]:8.2f} {r[10]:6.2f} {r[11]:7.2f}")
    # per-part means over the traced steps (first step skipped)
    print("\nmeans per part: window = first start -> last end; gap = previous launch's last end -> this launch's first start")
    for p in parts:
        rr = [r for r in rows[len(parts):] if r[0] == p]
        if rr:
            print(f"  {p:<14} window {sum(r[9] for r in rr) / len(rr):7.2f}  gap {sum(r[10] for r in rr) / len(rr):5.2f}  "
                  f"start spread {sum(r[3] - r[2] for r in rr) / len(rr):5.2f}  first data {sum(r[4] - r[2] for r in rr) / len(rr):5.2f}  "
                  f"end spread {sum(r[8] - r[7] for r in rr) / len(rr):5.2f}  mean CTA life {sum(r[11] for r in rr) / len(rr):6.2f}")
    print("\nend segments per part (us; median / max over a launch's CTAs, mean over the traced steps); tail = last "
          "'done' -> last end")
    for p in parts:
        ss = [x for x in segs[len(parts):] if x[0] == p and x[1]]
        if ss:
            keys = list(ss[0][1])
            cols = "  ".join(f"{k} {np.mean([x[1][k][0] for x in ss]):5.2f} / {np.mean([x[1][k][1] for x in ss]):5.2f}" for k in keys)
            print(f"  {p:<14} {cols}  tail {np.mean([x[2] for x in ss]):5.2f}")
    per_step = (rows[-1][8] - rows[len(parts) - 1][8]) / max(args.steps - 1, 1)
    print(f"  chain period: {per_step:.2f} us per step of {len(parts)} launches")


if __name__ == "__main__":
    main()
