#!/usr/bin/env python
"""bench.py -- consistency-loss pixels/s (fwd+bwd) of the Deep Co-Training unlabeled-branch hot path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload c2] [--dump-outputs DIR]

One "step" = one pass of the hot path over one synthetic unlabeled batch (BASELINE.json configs[1]:
ACDC co-training, K=3 views, C=4 classes, 256x256, batch 32 per GPU, JSD + VAT adversarial):
fused K-view JSD forward+backward from logits + the K Dice-count reductions, the three VAT
L2-normalisations, kl_div_with_logit forward+backward, and the adversarial KL forward+backward.
The networks between those points are out of scope (stock cuDNN); their outputs are seeded synthetic
tensors.  Prints ONE JSON line (rank 0).  See DESIGN.md "Measurement" for every field.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for _p in (ROOT, os.path.join(ROOT, "oracle")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

WORKLOADS = {  # name: (K, C, B per GPU, H, W, Cin, description)
    "c1": (2, 4, 4, 256, 256, 1, "ACDC 2 views C=4 256x256 B=4 (JSD only)"),
    "c2": (3, 4, 32, 256, 256, 1, "ACDC 3 views C=4 256x256 B=32/GPU, JSD + VAT adversarial + Dice meters"),
    "c3": (2, 2, 4, 512, 512, 1, "Spleen 2 views C=2 512x512 B=4/GPU"),
    "c4": (2, 19, 16, 512, 1024, 3, "Cityscapes 2 views C=19 512x1024 B=16/GPU, JSD + VAT adversarial (no meters on the "
                                    "unlabeled branch: trainer/cotraining_city.py:250-257)"),
}
METRIC = "consistency-loss pixels/sec (fwd+bwd)"
UNIT = "pixels/s"


def csrc_sha16():
    """Hash of the kernel sources the loaded library was built from (tools/ncu_traffic.py stamps captures with it).
    Comments and white space are stripped first: only a change that can alter the generated code invalidates a capture."""
    import hashlib
    import re
    d = os.path.join(ROOT, "deep-co-training-for-semi-supervised-image-segmentation_b200", "csrc")
    h = hashlib.sha256()
    for f in sorted(os.listdir(d)):
        if f.endswith((".cu", ".cuh")):
            src = open(os.path.join(d, f), "r", encoding="utf-8", errors="replace").read()
            src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
            src = re.sub(r"//[^\n]*", "", src)
            h.update(f.encode())
            h.update("".join(src.split()).encode())
    return h.hexdigest()[:16]


def load_traffic(workload):
    """DRAM bytes per launch of the dominant kernel from the committed ncu --set full capture (profiles/traffic.json) --
    only if that capture was taken from the kernel sources this build was made of; else None (traffic is never guessed)."""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))[workload]
        if t.get("csrc_sha16") != csrc_sha16():
            return {"bytes": None, "stale": f"capture {t.get('source')} was taken from other kernel sources "
                                            f"({t.get('csrc_sha16')} != {csrc_sha16()})"}
        return t
    except Exception:
        return None


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed regions run."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
                for n, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                continue
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        top = sorted(sm)[len(sm) // 2:]  # under load = upper half of the samples
        return {"sm_mhz": statistics.median(top), "sm_max_mhz": max(mx), "reasons": sorted(reasons),
                "samples": len(sm)}


# ---------------------------------------------------------------------------------------------------
# CPU arm: the oracle port (the reference is pure Python and cannot travel to the GPU box)
# ---------------------------------------------------------------------------------------------------
def cpu_step_inputs(K, C, B, H, W, cin, seed=1234):
    import numpy as np
    rng = np.random.default_rng(seed)
    f = lambda *s: rng.standard_normal(s, dtype=np.float32)  # noqa: E731
    z = [3 * f(B, C, H, W) for _ in range(K)]
    gt = rng.integers(0, C, (B, 1, H, W), dtype=np.int64)
    d, dg = f(B, cin, H, W), f(B, cin, H, W)
    img = rng.random((B, cin, H, W), dtype=np.float32)
    yhat, adv = 3 * f(B, C, H, W), 3 * f(B, C, H, W)
    return z, gt, d, dg, img, yhat, adv


def cpu_step(O, inp, K, C, with_vat=True):
    """The same step as ConsistencyStep.run, on the CPU oracle (all OpenMP threads)."""
    import numpy as np
    z, gt, d, dg, img, yhat, adv = inp
    n = z[0].shape[0] * z[0].shape[2] * z[0].shape[3]
    mean, _, gz = O.jsd_logits_fwdbwd(z, 1.0, want_map=False, want_grad=True)
    for k in range(K):
        O.dice_counts(z[k], gt)
    if with_vat:
        d1 = O.l2_normalize(d)
        d2 = O.l2_normalize(d1) * np.float32(1e-6)
        gout = np.full((z[0].shape[0],) + z[0].shape[2:], 1.0 / n, np.float32)
        O.kl_logit(z[0], yhat, gout)
        r = O.l2_normalize(dg)
        O.vat_apply(img, r, 10.0)
        real = O.softmax(z[1])
        p = O.softmax(adv)
        O.kl_fwd(p, real)
        gp, _ = O.kl_bwd(p, real, gout)
        O.softmax_bwd(p, gp)
    return mean


def time_cpu(K, C, B, H, W, cin, steps, warmup, with_vat=True, budget_s=None):
    """Times `steps` CPU steps on a bounded sample.  If budget_s is given the sample batch (and, below one
    image, the image height) is shrunk so that steps+warmup fit the budget; pixels/s is size-independent
    beyond the caches.  Returns (pixels/s, s/step, threads, sample description)."""
    import oracle as O
    O.build()
    O.set_num_threads(os.cpu_count() or 1)
    Bs, Hs = min(B, 8), H
    if budget_s is not None:
        probe = cpu_step_inputs(K, C, 1, H, W, cin)
        cpu_step(O, probe, K, C, with_vat)
        t0 = time.perf_counter()
        cpu_step(O, probe, K, C, with_vat)
        t_img = max(time.perf_counter() - t0, 1e-6)
        per_step = budget_s / max(steps + warmup, 1)
        Bs = int(max(1, min(B, per_step / t_img)))
        if per_step < t_img:
            Hs = int(max(8, (H * per_step / t_img) // 8 * 8))
    inp = cpu_step_inputs(K, C, Bs, Hs, W, cin)
    for _ in range(warmup):
        cpu_step(O, inp, K, C, with_vat)
    t0 = time.perf_counter()
    for _ in range(steps):
        cpu_step(O, inp, K, C, with_vat)
    dt = time.perf_counter() - t0
    sample = (f"same step on {Bs} image(s) of {Hs}x{W} (workload: {B} of {H}x{W}), {steps} steps, "
              f"C/OpenMP oracle port on all {O.num_threads()} host threads")
    return Bs * Hs * W * steps / dt, dt / steps, O.num_threads(), sample


def reference_staged():
    """The unmodified reference ($DCT_REFERENCE_ROOT, or baseline/_ref staged by tools/stage_reference.sh), if present."""
    try:
        import ref_trainer
        return ref_trainer if ref_trainer.available() else None
    except Exception:
        return None


def time_cpu_reference(rt, K, C, B, H, W, cin, steps, warmup, with_vat, with_dice, budget_s):
    """The reference's OWN modules (generalframework.loss / .metrics / .utils.AEGenerator through oracle/ref_trainer.py) on
    the host cores, torch intra-op threads = all of them, on a bounded sample of the workload's batch."""
    import torch
    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    dev = torch.device("cpu")
    _, t_img, _ = rt.time_reference_step(dev, K, C, 1, H, W, cin, steps=1, warmup=1, with_vat=with_vat, with_dice=with_dice)
    per_step = budget_s / max(steps + warmup, 1)
    Bs = int(max(1, min(B, per_step / max(t_img, 1e-6))))
    v, sec, losses = rt.time_reference_step(dev, K, C, Bs, H, W, cin, steps=steps, warmup=warmup, with_vat=with_vat,
                                            with_dice=with_dice)
    sample = (f"same step on {Bs} image(s) of {H}x{W} (workload: {B}), {steps} steps, the unmodified reference's modules "
              f"(JSD_2D, DiceMeter, VATGenerator statics, KL_Divergence_2D) on torch CPU, {threads} intra-op threads")
    return v, sec, threads, sample


def run_reference(args, wl):
    """--impl reference: the path's CPU implementation on the host cores.  The reference is pure Python on PyTorch: when
    it is staged (baseline/_ref) its own modules run, unmodified (kind "reference"); otherwise the C/OpenMP oracle port
    (kind "port" -- a FASTER baseline than the real one).  Bounded sample of the same workload."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    K, C, B, H, W, cin, desc = wl
    with_vat, with_dice = args.workload != "c1", args.workload != "c4"
    rt = reference_staged()
    if rt is not None:
        val, sec, cores, sample = time_cpu_reference(rt, K, C, B, H, W, cin, args.steps, max(min(args.warmup, 2), 1), with_vat,
                                                     with_dice, budget_s=150.0)
        kind = "reference"
    else:
        val, sec, cores, sample = time_cpu(K, C, B, H, W, cin, args.steps, max(args.warmup, 1), with_vat=with_vat, budget_s=150.0)
        kind = "port"
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"{args.workload}: {desc}", "K": K, "C": C, "H": H, "W": W, "batch_per_gpu": B},
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


# ---------------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------------
DUMP_BYTES = 48 << 20   # per-pixel outputs are sampled down to this many bytes in all (the rest is a few KB)


def dump_outputs(path, step, bufs):
    """Write what one step left in ``bufs`` -- the arrays a caller of the step receives -- as ``path/<name>.npy``.

    Losses, raw loss sums and Dice counts are written whole.  The per-pixel outputs (gradients, the VAT direction,
    r_adv, img_adv) are written whole as [B, C, H, W] when they fit DUMP_BYTES together, else as [P, C] rows at P pixels
    drawn once with a fixed seed (same pixels for every output; ``pixel_index.npy`` holds their flat b*H*W + h*W + w).
    Integer outputs are stored as float64 (exact)."""
    import numpy as np
    import torch
    os.makedirs(path, exist_ok=True)
    small = {"losses": torch.stack(step.losses(bufs)), "loss_sums": bufs.sums}
    pix = {f"grad_logits{k}": g for k, g in enumerate(bufs.grad_logits)}
    if step.with_dice:
        small["dice_counts"] = bufs.dice_counts.double()
    if step.with_vat:
        pix.update(vat_direction=bufs.d, r_adv=bufs.r_adv, img_adv=bufs.img_adv, grad_yhat=bufs.grad_yhat,
                   grad_adv=bufs.grad_adv)
    B, _, H, W = bufs.logits[0].shape
    n = B * H * W
    per_pixel = sum(t.shape[1] * t.element_size() for t in pix.values())
    P = min(n, DUMP_BYTES // per_pixel)
    if P < n:
        idx = np.sort(np.random.default_rng(20240).choice(n, size=P, replace=False))
        small["pixel_index"] = torch.from_numpy(idx.astype(np.float64))
        di = torch.from_numpy(idx).to(bufs.logits[0].device)
        pix = {k: t.permute(0, 2, 3, 1).reshape(n, t.shape[1]).index_select(0, di) for k, t in pix.items()}
    for name, t in {**small, **pix}.items():
        np.save(os.path.join(path, name + ".npy"), t.detach().cpu().numpy())


def use_nccl_later(world, px):
    return world > 1 and px is None


def run_ours(args, wl):
    import torch
    import torch.distributed as dist

    import dct_b200
    from dct_b200.engine import ConsistencyStep, StepBuffers

    K, C, B, H, W, cin, desc = wl
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py --impl ours needs a GPU (there is no CPU fallback)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    assert dct_b200._lib.lib().dct_device_check(local) == 0, "not an sm_100 device"
    with_vat = args.workload != "c1"
    # CoTrainer_City keeps its IoU meters on the labeled branch only (trainer/cotraining_city.py:236-241 vs :250-257)
    with_dice = args.workload != "c4"
    n_local = B * H * W
    # The path's only exchange (SURVEY 8e): the loss sums of every step.  They are stored into every rank's mailbox over
    # NVLink peer memory (distributed.PeerExchange) -- no collective launch.  "p2p-early" (default at N > 1): by the first
    # CTA to finish the NEXT step's first kernel (the sums are final by then; the ~2 us of the publication sit in that
    # launch's own tail); "p2p": by a one-CTA kernel chained to the step's last kernel (+2.3 us per step); "p2p-fused":
    # by that last kernel's last CTA (+2.2 us); "p2p-deferred": one step late on a forked graph branch (+6.8 us) --
    # profiles/r45, r46, DESIGN.md 5;
    # "nccl": one all-reduce per step on a side stream (the baseline this replaces, kept for A/B).
    px, exchange = None, "none"
    if world > 1 or args.exchange in ("p2p", "p2p-fused", "p2p-deferred", "p2p-early"):   # (at N = 1: loopback on the own mailbox, for A/B)
        exchange = args.exchange
        if exchange in ("p2p", "p2p-fused", "p2p-deferred", "p2p-early", "auto"):
            try:
                from dct_b200.distributed import PeerExchange
                px = PeerExchange(dev, n=4, nslots=64)
                ok = torch.ones(1, device=dev)
            except Exception as e:  # IPC / peer mapping refused on this box
                if args.exchange != "auto":
                    raise
                print(f"[bench rank {rank}] peer exchange unavailable ({e}); using NCCL", file=sys.stderr)
                ok = torch.zeros(1, device=dev)
            if world > 1:
                dist.all_reduce(ok, op=dist.ReduceOp.MIN)
            if ok.item() == 0:
                px = None
            exchange = (args.exchange if args.exchange in ("p2p", "p2p-fused", "p2p-deferred") else "p2p-early") if px is not None else "nccl"
    step = ConsistencyStep(K, C, B, H, W, cin=cin, jsd_weight=1.0, adv_weight=1.0, n_global=n_local * world,
                           with_vat=with_vat, with_dice=with_dice, exchange=px,
                           exchange_mode={"p2p-fused": "fused", "p2p-deferred": "deferred", "p2p-early": "early"}.get(exchange, "chained"))
    gen = torch.Generator(device=dev).manual_seed(1234 + rank)
    # R independent buffer sets, rotated every step so that no step finds its inputs in the 126 MB L2
    per_set = sum(t.numel() * t.element_size() for t in StepBuffers.allocate(K, C, 1, H, W, cin, dev).input_tensors()) * B
    R = max(2, min(8, int(1.5e9 // max(per_set, 1)) or 2))
    sets = [StepBuffers.allocate(K, C, B, H, W, cin, dev, gen) for _ in range(R)]
    dct_b200.set_check_mode("deferred")  # no host sync inside the path; flags are read once at the end
    deferred = px is not None and step.exchange_mode in ("deferred", "early")
    prev_of = (lambda j: sets[(j - 1) % R]) if deferred else (lambda j: None)   # step i publishes step i-1's sums
    graphs = [step.capture(s, publish_prev=prev_of(j)) for j, s in enumerate(sets)] if args.graph else None
    # One graph holding R consecutive steps (one per buffer set): inside a graph consecutive launches chain by programmatic
    # dependent launch (0.5 us from one kernel's last CTA to the next one's first), between two graph launches they do not
    # (~2.5 us, profiles/r26): the timed loop replays this graph for every full round of R steps and the single-step graphs
    # for the remainder.  Every step still is the full 5 launches on its own buffer set.
    round_graph = None
    early = px is not None and step.exchange_mode == "early"
    if args.graph and (not deferred or early) and not use_nccl_later(world, px):
        round_graph = step.capture_many(sets, publish_chain=early)
    # the path's only exchange (SURVEY 8e): the loss scalars of every step, all-reduced over NCCL on a side stream
    # so that the collective of step i overlaps the kernels of step i+1 (the gradients never depend on it: the
    # global 1/N is folded into the kernels through n_global)
    use_nccl = world > 1 and px is None
    comm = torch.cuda.Stream(device=dev) if use_nccl else None
    reds = [torch.zeros(4, dtype=torch.float64, device=dev) for _ in range(R)]
    copied = [None] * R
    pending = []

    def one(i):
        j = i % R
        s = sets[j]
        main = torch.cuda.current_stream(dev)
        if use_nccl and copied[j] is not None:
            main.wait_event(copied[j])  # step i-R's sums have been staged before this step overwrites them
        if graphs is not None:
            graphs[j].replay()
        else:
            step.run(s, publish_prev=prev_of(j))
        if use_nccl:
            done = torch.cuda.Event()
            done.record(main)
            with torch.cuda.stream(comm):
                comm.wait_event(done)
                reds[j].copy_(s.sums)
                ev = torch.cuda.Event()
                ev.record(comm)
                copied[j] = ev
                pending.append(dist.all_reduce(reds[j], async_op=True))
                if len(pending) > R:
                    pending.pop(0).wait()

    def drain():
        if use_nccl:
            with torch.cuda.stream(comm):
                while pending:
                    pending.pop(0).wait()
            torch.cuda.current_stream(dev).wait_stream(comm)

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    for i in range(args.warmup):
        one(i)
    if round_graph is not None:
        for _ in range(max(1, args.warmup // R)):
            round_graph.replay()
    drain()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    if round_graph is not None:
        full = args.steps // R
        for _ in range(full):
            round_graph.replay()
        for i in range(full * R, args.steps):
            one(i)
    else:
        for i in range(args.steps):
            one(i)
    if deferred:
        px.publish(sets[(args.steps - 1) % R].sums)   # the last step's sums (every earlier step was published by its successor)
    drain()   # the timed region ends when the last step's exchange has completed
    e1.record()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    if args.dump_outputs and rank == 0:   # before anything below runs the step again on these buffers
        dump_outputs(args.dump_outputs, step, sets[(args.steps - 1) % R])
    ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_total = float(ms.item())
    value = n_local * world * args.steps / (ms_total * 1e-3)
    exchange_check = None
    if px is not None:
        # every rank has finished (barrier above): the last publication of every rank must sit in this rank's mailbox,
        # and its rank-ordered sum must equal an NCCL all-reduce of the same sums
        q = px.published()
        got = px.read(q)
        last = sets[(args.steps - 1) % R].sums.clone()
        if world > 1:
            dist.all_reduce(last)
        err = float((got - last[:4]).abs().max().item()) / max(float(last[:4].abs().max().item()), 1e-30)
        assert err <= 1e-12, f"peer exchange disagrees with the NCCL all-reduce of the same sums (rel {err:.2e})"
        exchange_check = {"publications": q, "rel_err_vs_nccl_allreduce": err}

    # ---- roofline of the dominant kernel (fused JSD fwd+bwd, + the K Dice count sets when C <= 4): its average
    # launch duration over a timed region of back-to-back launches on the launching stream, CUDA events on that
    # stream, rotating over the R buffer sets (R x inputs+grads >> the 126 MB L2, so no launch finds its inputs cached)
    fused_dice = with_dice and C <= 4 and K * C <= 16
    side = torch.cuda.Stream(device=dev)

    def time_part(part, reps):
        """Average duration of ONE launch sequence of `part` (a graph of R back-to-back runs rotating over the buffer
        sets, replayed `reps` times), CUDA events on the launching stream."""
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            for i in range(2 * R):
                step.run_part(sets[i % R], part)
        torch.cuda.current_stream(dev).wait_stream(side)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=side):
            for j in range(R):
                step.run_part(sets[j], part)
        for _ in range(3):
            g.replay()
        torch.cuda.synchronize()
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        for _ in range(reps):
            g.replay()
        t1.record()
        torch.cuda.synchronize()
        return t0.elapsed_time(t1) / (reps * R)

    rounds = max(3, min(args.steps, 400) // R)
    part_ms = {p: time_part(p, rounds) for p in step.parts()}
    k_ms = part_ms["jsd"]
    jsd_only = step
    alg = jsd_only.part_bytes()["jsd"]
    peak, peak_src = load_peaks()
    achieved = alg / (k_ms * 1e-3) / 1e9
    roofline = {"bound": "hbm", "kernel": "tile_kernel<JsdOp<K,logits,fwd+bwd,%s>> via dct_jsd_fwdbwd_f32 "
                                          "(K-view JSD forward+backward%s, one launch)"
                                          % (("dice", " + K Dice count sets") if fused_dice else ("nodice", "")),
                "launches_timed": rounds * R,
                "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "frac_of_8TBps_nominal": achieved / 8000.0, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": alg, "kernel_ms": k_ms,
                "traffic": (load_traffic(args.workload) or {}).get("bytes"), "traffic_detail": load_traffic(args.workload),
                "step_algorithmic_bytes": step.algorithmic_bytes(),
                # every launch of the step timed on its own the same way (back to back with itself, cold inputs)
                "step_kernels": [{"part": p, "us": part_ms[p] * 1e3, "algorithmic_bytes": step.part_bytes()[p],
                                  "GBps": step.part_bytes()[p] / (part_ms[p] * 1e-3) / 1e9,
                                  "frac": step.part_bytes()[p] / (part_ms[p] * 1e-3) / 1e9 / peak} for p in step.parts()],
                "step_achieved_GBps": sum(step.algorithmic_bytes().values()) / (ms_total * 1e-3 / args.steps) / 1e9}

    # ---- e2e: host buffers in pinned memory -> H2D -> the public autograd API -> D2H of losses + Dice rows
    e2e = run_e2e(args, dct_b200, step, sets[0], dev, world, n_local, K, C, B, H, W, with_vat, with_dice)
    dct_b200.raise_if_flagged()
    clocks = sampler.stop() if rank == 0 else None
    steps_per_graph = R if round_graph is not None else (1 if args.graph else 0)
    del graphs, round_graph, sets
    torch.cuda.empty_cache()
    extras = {}
    if not args.no_extras:
        extras = run_extras(args, dct_b200, dev, rank, world, local, peak)

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        v, sec, cores, sample = time_cpu(K, C, B, H, W, cin, steps=10, warmup=1, with_vat=with_vat, budget_s=10.0)
        cpu = {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample}
        rt = reference_staged()
        if rt is not None:   # the reference itself is staged: ITS modules are the baseline, the C port is kept beside it
            try:
                rv, rsec, rcores, rsample = time_cpu_reference(rt, K, C, B, H, W, cin, 3, 1, with_vat, with_dice, budget_s=20.0)
                cpu = {"value": rv, "unit": UNIT, "cores": rcores, "kind": "reference", "sample": rsample,
                       "oracle_port": {"value": v, "cores": cores, "sample": sample}}
            except Exception as e:
                cpu["reference_error"] = f"{type(e).__name__}: {e}"
    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms_total / args.steps, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": {"workload": f"{args.workload}: {desc}", "K": K, "C": C, "H": H, "W": W, "batch_per_gpu": B,
                           "global_batch": B * world, "parallelism": f"dp{world}", "cuda_graph": bool(args.graph),
                           "steps_per_graph": steps_per_graph,
                           "exchange": {"none": "none (1 GPU)", "nccl": "NCCL all-reduce of the loss sums per step (side stream)",
                                        "p2p": "a one-CTA kernel chained to the step's last kernel by programmatic dependent "
                                               "launch stores the loss sums into every rank's mailbox over NVLink peer memory "
                                               "(no collective, no NCCL kernel)",
                                        "p2p-early": "the first CTA to finish the NEXT step's first kernel stores the step's loss sums into "
                                                     "every rank's mailbox over NVLink peer memory (no collective, no extra launch; "
                                                     "the last step's sums by a one-CTA kernel)",
                                        "p2p-deferred": "a one-CTA kernel on a forked graph branch stores step i-1's loss sums into "
                                                        "every rank's mailbox next to step i's first kernel",
                                        "p2p-fused": "the step's last kernel itself stores the loss sums into every rank's "
                                                     "mailbox over NVLink peer memory"}[exchange],
                           "exchange_check": exchange_check,
                           "l2": f"inputs larger than L2: {R} rotating buffer sets of {per_set / 2**20:.0f} MiB inputs"},
                "clocks": clocks, "e2e": e2e, "gpu_launches": step.launches_per_step * args.steps,
                "roofline": roofline, "cpu_baseline": cpu, **extras}
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def bench_workload(dct, name, dev, world, steps, peak):
    """ms/step and the dominant kernel's roofline fraction of another BASELINE workload (c1 / c3 / c4), same method as the
    headline: R rotating buffer sets larger than L2, R steps per CUDA graph, CUDA events."""
    import torch
    from dct_b200.engine import ConsistencyStep, StepBuffers
    K, C, B, H, W, cin, desc = WORKLOADS[name]
    with_vat, with_dice = name != "c1", name != "c4"
    step = ConsistencyStep(K, C, B, H, W, cin=cin, n_global=B * H * W * world, with_vat=with_vat, with_dice=with_dice)
    gen = torch.Generator(device=dev).manual_seed(4321)
    per_set = sum(t.numel() * t.element_size() for t in StepBuffers.allocate(K, C, 1, H, W, cin, dev).input_tensors()) * B
    R = max(2, min(8, int(1.5e9 // max(per_set, 1)) or 2))
    sets = [StepBuffers.allocate(K, C, B, H, W, cin, dev, gen) for _ in range(R)]
    g = step.capture_many(sets)
    rounds = max(2, steps // R)
    for _ in range(2):
        g.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(rounds):
        g.replay()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / (rounds * R)
    # the dominant (JSD) launch on its own
    side = torch.cuda.Stream(device=dev)
    side.wait_stream(torch.cuda.current_stream(dev))
    kg = torch.cuda.CUDAGraph()
    with torch.cuda.graph(kg, stream=side):
        for s in sets:
            step.run_part(s, "jsd")
    kg.replay()
    torch.cuda.synchronize()
    e0.record()
    for _ in range(rounds):
        kg.replay()
    e1.record()
    torch.cuda.synchronize()
    k_ms = e0.elapsed_time(e1) / (rounds * R)
    pb = step.part_bytes()
    out = {"workload": f"{name}: {desc}", "value": B * H * W * 1e3 / ms, "unit": UNIT, "ms_per_step": ms, "steps": rounds * R,
           "step_achieved_GBps": sum(pb.values()) / (ms * 1e-3) / 1e9, "step_frac": sum(pb.values()) / (ms * 1e-3) / 1e9 / peak,
           "dominant_kernel_ms": k_ms, "dominant_kernel_frac": pb["jsd"] / (k_ms * 1e-3) / 1e9 / peak,
           "n_gpus": world, "per_gpu": True}
    del g, kg, sets
    torch.cuda.empty_cache()
    return out


def run_extras(args, dct, dev, rank, world, local, peak):
    """The rest of BASELINE.json's metric in the same JSON line: the reference's stock ATen composition of the step on this
    GPU (SURVEY 8d: the meaningful speed-up denominator), co-training iterations/s (the reference's own trainer stock vs
    with the drop-ins installed at N = 1; the DDP engine and the networks-alone floor at every N), and the other workloads."""
    import torch
    import torch.distributed as dist
    K, C, B, H, W, cin, desc = WORKLOADS[args.workload]
    with_vat, with_dice = args.workload != "c1", args.workload != "c4"
    out = {}
    rt = reference_staged()
    # ---- the step through the reference's own modules on this GPU (N = 1 only, like cpu_baseline)
    if rank == 0 and world == 1:
        if rt is not None:
            try:
                v, sec, losses = rt.time_reference_step(dev, K, C, B, H, W, cin, steps=3, warmup=1, with_vat=with_vat,
                                                        with_dice=with_dice)
                out["aten_gpu_baseline"] = {"value": v, "unit": UNIT, "ms_per_step": sec * 1e3, "steps": 3, "kind": "reference",
                                            "what": "the same step through the unmodified reference's modules (DiceMeter.add x K, "
                                                    "JSD_2D, VATGenerator statics, KL_Divergence_2D, autograd backward) in stock "
                                                    "ATen on this GPU, inputs resident in HBM, losses + Dice rows read back",
                                            "last_losses": losses}
            except Exception as e:
                out["aten_gpu_baseline"] = {"unavailable": f"{type(e).__name__}: {e}"}
        else:
            out["aten_gpu_baseline"] = {"unavailable": "reference not staged (tools/stage_reference.sh -> baseline/_ref)"}
    torch.cuda.empty_cache()
    if world > 1:
        dist.barrier()
    # ---- co-training iterations/s
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import cotrain_bench as cb
    cot = {}
    for cfg_name, iters, warm in (("c1", 20, 3), (args.workload if args.workload != "c1" else "c3", 4 if args.workload == "c2" else 8, 1)):
        entry = {}
        try:
            lines = cb.measure(cfg_name, ["ours", "nets"], iters, warm, dev, rank, world, local)
            for ln in lines:
                entry["engine_ddp" if ln["arm"] == "ours" else "networks_alone"] = {"it_per_s": ln["value"], "ms_per_iter": ln["ms_per_iter"]}
            entry["config"] = lines[0]["config"]
            entry["images_per_iter_per_gpu"] = lines[0]["images_per_iter_per_gpu"]
        except Exception as e:
            entry["engine_error"] = f"{type(e).__name__}: {e}"
        if world == 1 and rt is not None:
            Kc, Cc, cinc, Hc, Wc, BL, BU = cb.CONFIGS[cfg_name]
            if cinc == 1 and Cc == 4:   # the reference trainer's validation loop hard-codes C = 4 and its datasets are grey-scale
                try:
                    kw = dict(iters=iters if cfg_name == "c1" else 3, K=Kc, arch=cb.REF_ARCH[cfg_name], C=Cc, B=BL, H=Hc, W=Wc,
                              train_jsd=True, train_adv=True, deterministic=False, warmup_iters=1, tf32=None)
                    stock = rt.run_train_loop(dev, False, **kw)
                    drop = rt.run_train_loop(dev, True, **kw)
                    entry["reference_trainer_stock"] = {"it_per_s": stock["it_per_s"], "iters": stock["iters"]}
                    entry["reference_trainer_with_dropins"] = {"it_per_s": drop["it_per_s"], "iters": drop["iters"],
                                                               "first_total_loss_rel_diff": float(abs(drop["total_loss"][0] - stock["total_loss"][0]) / abs(stock["total_loss"][0]))}
                except Exception as e:
                    entry["reference_trainer_error"] = f"{type(e).__name__}: {e}"
        cot[cfg_name] = entry
        torch.cuda.empty_cache()
    out["cotrain_it_s"] = cot
    # ---- the other workloads of BASELINE.json (per-GPU numbers; at N > 1 every rank runs them, rank 0 reports)
    others = {}
    for name in ("c1", "c3", "c4"):
        if name == args.workload:
            continue
        try:
            others[name] = bench_workload(dct, name, dev, world, 240 if name != "c4" else 60, peak)
        except Exception as e:
            others[name] = {"error": f"{type(e).__name__}: {e}"}
        if world > 1:
            v = torch.tensor([others[name].get("ms_per_step", 0.0)], dtype=torch.float64, device=dev)
            dist.all_reduce(v, op=dist.ReduceOp.MAX)
            if "ms_per_step" in others[name]:
                Kx, Cx, Bx, Hx, Wx, _, _ = WORKLOADS[name]
                others[name]["ms_per_step_max_over_ranks"] = float(v.item())
                others[name]["value_all_gpus"] = Bx * Hx * Wx * world * 1e3 / float(v.item())
    out["other_workloads"] = others
    return out


def run_e2e(args, dct, step, dev_set, dev, world, n_local, K, C, B, H, W, with_vat, with_dice=True):
    """Same step through the PUBLIC API (autograd Functions / meters / generators) with host buffers:
    every step copies its inputs from pinned host memory (copy stream, double-buffered against the
    compute of the previous step) and reads the losses and Dice rows back to the host."""
    import torch
    import torch.distributed as dist
    host = [t.cpu().pin_memory() for t in dev_set.input_tensors()]
    h2d = sum(t.numel() * t.element_size() for t in host)
    nbuf = 2
    slots = [[torch.empty_like(t, device=dev) for t in host] for _ in range(nbuf)]
    copy_stream = torch.cuda.Stream(device=dev)
    ready = [torch.cuda.Event() for _ in range(nbuf)]
    freed = [torch.cuda.Event() for _ in range(nbuf)]
    out_host = torch.empty(3 + K * B * C, dtype=torch.float32).pin_memory()
    meters = [dct.DiceMeter(method="2d", C=C) for _ in range(K)]
    n_glob = n_local * world
    d2h = out_host.numel() * 4

    def upload(i):
        j = i % nbuf
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(freed[j])
            for dst, src in zip(slots[j], host):
                dst.copy_(src, non_blocking=True)
            ready[j].record(copy_stream)

    def compute(i):
        j = i % nbuf
        cur = torch.cuda.current_stream(dev)
        cur.wait_event(ready[j])
        t = slots[j]
        logits = [x.requires_grad_() for x in t[:K]]
        labels, d, d_grad, img, yhat, adv, real = t[K:K + 7]
        counts = torch.empty(K, B, C, 3, dtype=torch.int64, device=dev)
        if with_dice:
            loss = dct.jsd_consistency_from_logits(logits, weight=1.0, labels=labels, dice_counts=counts, n_global=n_glob,
                                                   accumulate=False)
        else:
            loss = dct.jsd_consistency_from_logits(logits, weight=1.0, n_global=n_glob)
        total = loss
        outs = [loss.detach()]
        if with_vat:
            dct.l2_normalize(d, scale=1e-6, passes=2)
            yh = yhat.requires_grad_()
            vkl = dct.kl_div_with_logit(logits[0].detach(), yh).mean()
            vkl.backward()
            r_adv, img_adv = dct.l2_normalize(d_grad, scale=10.0, out=torch.empty_like(d_grad), img=img)
            advl = dct.kl_consistency_from_logits(adv.requires_grad_(), real, weight=1.0, n_global=n_glob)
            total = total + advl
            outs += [vkl.detach(), advl.detach()]
        else:
            outs += [loss.detach() * 0, loss.detach() * 0]
        total.backward()
        rows = []
        for k in range(K):
            meters[k].reset()
            meters[k].add_counts(counts[k])
            rows.append(meters[k].log.reshape(-1))
        res = torch.cat([torch.stack(outs)] + rows)
        if world > 1:
            dist.all_reduce(res[:3])
        out_host.copy_(res, non_blocking=True)
        for x in t:
            x.requires_grad_(False) if x.is_floating_point() else None
            x.grad = None
        freed[j].record(cur)

    steps = max(3, min(args.steps, args.e2e_steps))

    def timed(fn_upload, fn_compute):
        for j in range(nbuf):
            freed[j].record(torch.cuda.current_stream(dev))
        for i in range(3):  # warm-up
            fn_upload(i); fn_compute(i)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        fn_upload(0)
        for i in range(steps):
            if i + 1 < steps:
                fn_upload(i + 1)
            fn_compute(i)
        torch.cuda.synchronize()
        dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        return float(dt.item())

    dt = timed(upload, compute)

    # The same uploads with NO compute behind them: what the host link alone sustains with N ranks copying at once.  When
    # the end-to-end step time equals this, the limiter is the host side (PCIe / host DRAM shared by the N GPUs), not a kernel.
    def no_compute(i):
        j = i % nbuf
        cur = torch.cuda.current_stream(dev)
        cur.wait_event(ready[j])
        freed[j].record(cur)

    dt_copy = timed(upload, no_compute)
    res = {"value": n_glob * steps / dt, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
           "steps": steps, "ms_per_step": dt / steps * 1e3, "h2d_GBps_per_gpu": h2d * steps / dt / 1e9,
           "copy_only": {"ms_per_step": dt_copy / steps * 1e3, "h2d_GBps_per_gpu": h2d * steps / dt_copy / 1e9,
                         "what": "the same pinned-memory uploads with no kernels behind them, all ranks at once (max over ranks)"},
           "api": "jsd_consistency_from_logits + DiceMeter.add_counts + l2_normalize + kl_div_with_logit + "
                  "kl_consistency_from_logits (autograd), pinned host inputs, double-buffered H2D",
           "last_losses": [float(v) for v in out_host[:3]]}

    # bf16 variant (networks under autocast hand the path bf16 logits): the [B,C,H,W] tensors travel as 2-byte elements
    # (images, the VAT direction and the int64 labels as they are), fp32 math in the kernels, bf16 gradients.
    try:
        is_big = [t.is_floating_point() and t.dim() == 4 and t.shape[1] == C and C > 1 for t in host]
        host16 = [t.to(torch.bfloat16).pin_memory() if big else t for t, big in zip(host, is_big)]
        # the detached target must stay a simplex to 1e-5 after rounding (the reference's own assert): a one-hot target does
        host16[K + 6] = torch.nn.functional.one_hot(host[K + 6].argmax(1), C).permute(0, 3, 1, 2).contiguous().to(torch.bfloat16).pin_memory()
        slots16 = [[torch.empty_like(t, device=dev) for t in host16] for _ in range(nbuf)]
        h2d16 = sum(t.numel() * t.element_size() for t in host16)

        def upload16(i):
            j = i % nbuf
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(freed[j])
                for dst, src in zip(slots16[j], host16):
                    dst.copy_(src, non_blocking=True)
                ready[j].record(copy_stream)

        def compute16(i):
            nonlocal slots
            keep, slots = slots, slots16
            try:
                compute(i)
            finally:
                slots = keep

        dt16 = timed(upload16, compute16)
        res["bf16"] = {"value": n_glob * steps / dt16, "unit": UNIT, "h2d_bytes_per_step": h2d16, "ms_per_step": dt16 / steps * 1e3,
                       "h2d_GBps_per_gpu": h2d16 * steps / dt16 / 1e9, "last_losses": [float(v) for v in out_host[:3]],
                       "what": "same step, logits / probabilities as bfloat16 in host memory and on the device"}
    except Exception as e:
        res["bf16"] = {"error": f"{type(e).__name__}: {e}"}
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS))
    ap.add_argument("--graph", type=int, default=1, help="replay the step as a CUDA graph (1) or launch eagerly (0)")
    ap.add_argument("--e2e-steps", type=int, default=50)
    ap.add_argument("--exchange", default="auto", choices=["auto", "p2p", "p2p-early", "p2p-deferred", "p2p-fused", "nccl"],
                    help="N > 1: how the loss sums cross ranks (auto = p2p, NCCL if peer mapping is refused)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true",
                    help="skip aten_gpu_baseline / cotrain_it_s / other_workloads (developer A/B runs)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the outputs of the last timed step (rank 0) as DIR/<name>.npy; "
                         "the same arguments give the same inputs, so two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    wl = WORKLOADS[args.workload]
    if args.impl == "reference":
        run_reference(args, wl)
    else:
        run_ours(args, wl)


if __name__ == "__main__":
    main()
