"""Allocation-free execution of one unlabeled-branch consistency step.

The autograd drop-ins in :mod:`loss` / :mod:`metrics` allocate their outputs per call, which is
what a drop-in must do.  A training loop that owns its buffers can instead bind them once and
replay the whole per-pixel path -- K-view JSD forward+backward with the K Dice counts, the VAT
power-iteration arithmetic and the adversarial KL -- as a fixed sequence of C-ABI launches on
one stream, optionally captured in a CUDA graph (the inner loop is launch-bound at ACDC sizes:
~10 kernels of 5-40 us each).

Where the step sits in the reference iteration (generalframework/trainer/cotraining_totalloss.py):
  :223-226  unlab_preds -> unlabdiceMeters.add x K -> JSD_2D -> .mean()        [jsd + dice]
  AEGenerator.py:93-119 (VAT): normalise(d) -> xi*normalise(d) -> net -> kl_div_with_logit.mean().backward()
                               -> eps*normalise(d.grad) -> clamp(img + r)       [l2 x3, kl_logit]
  :391-392  KL_Divergence_2D(reduce=True)(softmax(adv_logits), real.detach())   [kl_from_logits]
Both the JSD and kl_div_with_logit read the first view's logits (pred = views[0]).  The JSD's outputs are only consumed
at totalLoss.backward() and by the meters, so the JSD can wait for the VAT forward yhat = net(img + xi*d): where the shape
allows (see ConsistencyStep.fused_vat) one launch does both, and the step is l2_direction, jsd (+ VAT KL), l2_radv, kl_adv.
The network forward/backward passes between those points stay in PyTorch/cuDNN; here their
outputs are whatever tensors the caller binds (synthetic ones in bench.py).
"""
import ctypes
from dataclasses import dataclass
from typing import List, Optional

import torch

from . import _lib, _runtime


@dataclass
class StepBuffers:
    """Device tensors of one consistency step (all float32 NCHW unless noted)."""
    logits: List[torch.Tensor]          # K x [B,C,H,W]  unlabeled-branch logits of the K views   (in)
    labels: torch.Tensor                # [B,1,H,W] int64 unlabeled ground truth for the meters    (in)
    grad_logits: List[torch.Tensor]     # K x [B,C,H,W]  d(w_jsd * mean JSD)/d logits              (out)
    dice_counts: torch.Tensor           # [K,B,C,3] int64 (I,G,P)                                   (out)
    d: torch.Tensor                     # [B,Cin,H,W] VAT direction, N(0,1) on entry                (in/out)
    d_grad: torch.Tensor                # [B,Cin,H,W] dKL/dd coming back from the net               (in)
    img: torch.Tensor                   # [B,Cin,H,W] unlabeled images in [0,1]                     (in)
    r_adv: torch.Tensor                 # [B,Cin,H,W]                                               (out)
    img_adv: torch.Tensor               # [B,Cin,H,W]                                               (out)
    yhat_logits: torch.Tensor           # [B,C,H,W] net(img + d)                                    (in)
    grad_yhat: torch.Tensor             # [B,C,H,W] d mean KL_logit / d yhat                        (out)
    adv_logits: torch.Tensor            # [B,C,H,W] other view on img_adv                           (in)
    real_probs: torch.Tensor            # [B,C,H,W] detached clean prediction (probabilities)       (in)
    grad_adv: torch.Tensor              # [B,C,H,W] d(w_adv * KL mean)/d adv_logits                 (out)
    sums: torch.Tensor                  # [4] float64: sum JSD map, sum VAT KL map, sum adv KL map, -  (out)

    @staticmethod
    def allocate(K, C, B, H, W, cin, device, generator: Optional[torch.Generator] = None) -> "StepBuffers":
        """Synthetic, seeded contents (SURVEY.md 8d): logits 3*randn, labels randint, images rand, d randn."""
        def rn(*s):
            return torch.randn(*s, device=device, dtype=torch.float32, generator=generator)
        logits = [3 * rn(B, C, H, W) for _ in range(K)]
        e = lambda: torch.empty(B, C, H, W, device=device, dtype=torch.float32)  # noqa: E731
        ei = lambda: torch.empty(B, cin, H, W, device=device, dtype=torch.float32)  # noqa: E731
        return StepBuffers(
            logits=logits,
            labels=torch.randint(0, C, (B, 1, H, W), device=device, dtype=torch.int64, generator=generator),
            grad_logits=[e() for _ in range(K)],
            dice_counts=torch.zeros(K, B, C, 3, dtype=torch.int64, device=device),
            d=rn(B, cin, H, W), d_grad=rn(B, cin, H, W),
            img=torch.rand(B, cin, H, W, device=device, dtype=torch.float32, generator=generator),
            r_adv=ei(), img_adv=ei(),
            yhat_logits=3 * rn(B, C, H, W), grad_yhat=e(),
            adv_logits=3 * rn(B, C, H, W), real_probs=torch.softmax(3 * rn(B, C, H, W), 1), grad_adv=e(),
            sums=torch.zeros(4, dtype=torch.float64, device=device))

    def input_tensors(self):
        return list(self.logits) + [self.labels, self.d, self.d_grad, self.img, self.yhat_logits, self.adv_logits,
                                    self.real_probs]

    def result_tensors(self):
        return [self.sums, self.dice_counts]


class ConsistencyStep:
    """Binds shapes and hyper-parameters; ``run(buffers)`` enqueues the step on the current stream.

    ``jsd_weight`` / ``adv_weight`` are the ramp values the trainer multiplies the two consistency
    losses with (cotraining_totalloss.py:246); ``n_global`` the pixel count over all ranks.
    """

    def __init__(self, K, C, B, H, W, cin=1, jsd_weight=1.0, adv_weight=1.0, xi=1e-6, eps=10.0, kl_eps=1e-10,
                 n_global: Optional[int] = None, with_vat=True, with_dice=True, exchange=None, exchange_mode="chained"):
        self.K, self.C, self.B, self.HW, self.M = K, C, B, H * W, cin * H * W
        self.n = B * H * W if n_global is None else int(n_global)
        self.jsd_weight, self.adv_weight, self.xi, self.eps, self.kl_eps = jsd_weight, adv_weight, xi, eps, kl_eps
        self.with_vat, self.with_dice = with_vat, with_dice
        # distributed.PeerExchange or None: the kernel that writes the step's last sum also pushes the sums into every
        # data-parallel rank's mailbox over NVLink (no collective launch; SURVEY.md 8e)
        self.exchange = exchange
        # "chained" (default): the plain kernel, then the one-CTA publication kernel chained by programmatic dependent
        #            launch (+2.4 us per step, measured);
        # "fused":   the adversarial-KL kernel's own last CTA publishes (dct_kl_from_logits_fwdbwd_pub_f32) -- no extra
        #            launch, but ptxas generates a slower tile loop for that kernel (+3.7 us at c2, +82 us at c4)
        # "deferred": like "chained", but the publication of step i-1's sums runs on a forked branch next to step i's
        #            first kernel (run(bufs, publish_prev=previous buffers)): nothing is added to the step's critical path;
        #            the caller publishes the last step's sums itself (exchange.publish) when the loop ends
        # "early":   like "deferred", without a launch: the step's FIRST kernel (dct_jsd_fwdbwd_pub_f32) carries the previous
        #            step's sums and its first finishing CTA publishes them inside the launch's own tail (CTAs end 3-4 us apart)
        assert exchange_mode in ("fused", "chained", "deferred", "early")
        self.exchange_mode = exchange_mode
        self._pub_stream = None
        self._h = _lib.lib()
        # the VAT KL rides the JSD launch (dct_jsd_vat_kl_fwdbwd_f32) where that launch's stage holds the K views and yhat in
        # 5..16 rows of 256-pixel tensor-map tiles; other shapes (C = 19) keep the two launches
        self.fused_vat = with_vat and K >= 2 and C <= 4 and (K + 1) * C <= 16 and self.HW % 4 == 0
        # kernels launched per run(): the JSD kernel (Dice fused for C <= 4, else K counting launches), the two KL kernels,
        # the two normalisations (one launch each up to 16 x 256 x 64 floats per sample, else a sum-of-squares launch + a
        # scale launch each), the publication kernel of a chained / deferred exchange
        big = (self.M > 16 * 256 * 64) or (self.M % 4 != 0)   # (a cluster of 16 CTAs serves samples up to 1 MB)
        self.launches_per_step = 1 + (0 if (not with_dice or (C <= 4 and K * C <= 16)) else K) + \
            ((2 + (2 + 2 if big else 2) - (1 if self.fused_vat else 0)) if with_vat else 0) + \
            (1 if (exchange is not None and exchange_mode != "early" and (not with_vat or exchange_mode != "fused")) else 0)

    # bytes that MUST move per step (algorithmic, fp32): see DESIGN.md "Algorithmic bytes"
    def algorithmic_bytes(self):
        return self.part_bytes()

    def _publish_forked(self, prev: StepBuffers, dev) -> "torch.cuda.Event":
        """Publication of ``prev.sums`` on a side branch of the current stream (a fork/join that CUDA-graph capture records
        as such): it runs next to the kernels enqueued between this call and the join."""
        cur = torch.cuda.current_stream(dev)
        if self._pub_stream is None:
            self._pub_stream = torch.cuda.Stream(device=dev)
        fork = torch.cuda.Event()
        fork.record(cur)
        self._pub_stream.wait_event(fork)
        with torch.cuda.stream(self._pub_stream):
            self.exchange.publish(prev.sums)
            done = torch.cuda.Event()
            done.record(self._pub_stream)
        return done

    def run(self, bufs: StepBuffers, zero_counts: bool = True, publish_prev: Optional[StepBuffers] = None) -> None:
        h, K, C, B, HW = self._h, self.K, self.C, self.B, self.HW
        dev = bufs.logits[0].device
        joined = None
        if self.exchange is not None and self.exchange_mode == "deferred" and publish_prev is not None:
            joined = self._publish_forked(publish_prev, dev)
        try:
            self._run(bufs, zero_counts, publish_prev if self.exchange_mode == "early" else None)
        finally:
            if joined is not None:
                torch.cuda.current_stream(dev).wait_event(joined)

    # the step's launches by name, in stream order (bench.py times each one on its own as well)
    PARTS = ("jsd", "l2_direction", "kl_logit", "l2_radv", "kl_adv")
    FUSED_VAT_PARTS = ("l2_direction", "jsd", "l2_radv", "kl_adv")   # "jsd" also runs the VAT KL (fused_vat)

    def parts(self):
        if not self.with_vat:
            return self.PARTS[:1]
        return self.FUSED_VAT_PARTS if self.fused_vat else self.PARTS

    def part_bytes(self):
        """Algorithmic bytes of every launch of :meth:`parts` (what MUST cross HBM; DESIGN.md 3)."""
        K, C, n = self.K, self.C, self.B * self.HW
        cin = self.M // self.HW
        fused = self.with_dice and C <= 4 and K * C <= 16   # Dice counted inside the JSD kernel: + labels only
        kv = K + 1 if self.fused_vat else K                 # fused VAT KL: yhat read, grad_yhat written as well
        b = {"jsd": n * (2 * kv * C * 4) + (n * 8 if fused else 0) +
                    ((n * K * (C * 4 + 8)) if (self.with_dice and not fused) else 0)}
        if self.with_vat:
            b.update({"l2_direction": n * cin * 4 * 2,      # d read, xi * normalise(normalise(d)) written (one launch)
                      "kl_logit": n * 3 * C * 4,            # two logits tensors read, one gradient written
                      "l2_radv": n * cin * 4 * 4,           # d.grad + img read, r_adv + img_adv written
                      "kl_adv": n * 3 * C * 4})
            if self.fused_vat:
                del b["kl_logit"]
        return b

    def run_part(self, bufs: StepBuffers, part: str, zero_counts: bool = True, publish_prev: Optional[StepBuffers] = None) -> None:
        h, K, C, B, HW = self._h, self.K, self.C, self.B, self.HW
        dev = bufs.logits[0].device
        st = _runtime.state(dev)
        ws, s = st.workspace.data_ptr(), _runtime.stream_ptr(dev)
        fl = _runtime.flags_ptr(st)
        sums = bufs.sums.data_ptr()
        if part == "jsd" and self.fused_vat:
            # JSD fwd+bwd + Dice and kl_div_with_logit(pred.detach(), y_hat) + backward to y_hat in one launch; it also
            # publishes the previous step's sums when asked (as dct_jsd_fwdbwd_pub_f32 below)
            pub = None
            if self.exchange is not None and publish_prev is not None:
                pub = ctypes.byref(self.exchange.descriptor(publish_prev.sums))
            _lib.check(h.dct_jsd_vat_kl_fwdbwd_f32(_lib.ptr_array(bufs.logits), K, C, B, HW, self.jsd_weight / self.n, sums,
                                                   _lib.ptr_array(bufs.grad_logits),
                                                   bufs.labels.data_ptr() if self.with_dice else None,
                                                   bufs.dice_counts.data_ptr() if self.with_dice else None,
                                                   _lib.COUNTS_OVERWRITE if zero_counts else _lib.COUNTS_ACCUMULATE,
                                                   bufs.yhat_logits.data_ptr(), 1.0 / self.n, sums + 8,
                                                   bufs.grad_yhat.data_ptr(), fl, ws, pub, s),
                       "dct_jsd_vat_kl_fwdbwd_f32")
        elif part == "jsd" and self.exchange is not None and publish_prev is not None:
            # the step's first kernel also publishes the PREVIOUS step's sums (final since that step's last kernel completed)
            _lib.check(h.dct_jsd_fwdbwd_pub_f32(_lib.ptr_array(bufs.logits), K, C, B, HW, _lib.IN_LOGITS,
                                                self.jsd_weight / self.n, None, sums, _lib.ptr_array(bufs.grad_logits),
                                                bufs.labels.data_ptr() if self.with_dice else None,
                                                bufs.dice_counts.data_ptr() if self.with_dice else None,
                                                _lib.COUNTS_OVERWRITE if zero_counts else _lib.COUNTS_ACCUMULATE, fl, ws,
                                                ctypes.byref(self.exchange.descriptor(publish_prev.sums)), s),
                       "dct_jsd_fwdbwd_pub_f32")
        elif part == "jsd":
            # counts_mode 1: the launch overwrites the counters (zeroed by its own first CTA) -- no fill launch per step
            _lib.check(h.dct_jsd_fwdbwd_f32(_lib.ptr_array(bufs.logits), K, C, B, HW, _lib.IN_LOGITS,
                                            self.jsd_weight / self.n, None, sums, _lib.ptr_array(bufs.grad_logits),
                                            bufs.labels.data_ptr() if self.with_dice else None,
                                            bufs.dice_counts.data_ptr() if self.with_dice else None,
                                            _lib.COUNTS_OVERWRITE if zero_counts else _lib.COUNTS_ACCUMULATE, fl, ws, s),
                       "dct_jsd_fwdbwd_f32")
        elif part == "l2_direction":
            # d <- normalise(N(0,1));  d <- xi * normalise(d)                       (AEGenerator.py:97-98,103)
            d = bufs.d.data_ptr()
            _lib.check(h.dct_l2_normalize_f32(d, d, B, self.M, 2, self.xi, None, None, ws, s), "dct_l2_normalize_f32")
        elif part == "kl_logit":
            # delta_kl = kl_div_with_logit(pred.detach(), y_hat); delta_kl.mean().backward()       (:107-108)
            _lib.check(h.dct_kl_logit_f32(bufs.logits[0].data_ptr(), bufs.yhat_logits.data_ptr(), C, B, HW, None, sums + 8,
                                          1, None, None, 1.0 / self.n, bufs.grad_yhat.data_ptr(), None, ws, s),
                       "dct_kl_logit_f32")
        elif part == "l2_radv":
            # r_adv = eps * normalise(d.grad); img_adv = clamp(img + r_adv, 0, 1)                  (:113-117)
            _lib.check(h.dct_l2_normalize_f32(bufs.d_grad.data_ptr(), bufs.r_adv.data_ptr(), B, self.M, 1, self.eps,
                                              bufs.img.data_ptr(), bufs.img_adv.data_ptr(), ws, s), "dct_l2_normalize_f32")
        elif part == "kl_adv":
            # adv loss: KL_Divergence_2D(reduce=True)(softmax(adv_logits), real.detach()) + backward (cotraining :391-392)
            if self.exchange is not None and self.exchange_mode == "fused":
                # the step's last kernel also stores the three sums into every data-parallel rank's mailbox (NVLink)
                _lib.check(h.dct_kl_from_logits_fwdbwd_pub_f32(bufs.adv_logits.data_ptr(), bufs.real_probs.data_ptr(), C, B, HW,
                                                               self.kl_eps, self.adv_weight / self.n, None, sums + 16,
                                                               bufs.grad_adv.data_ptr(), fl, ws,
                                                               ctypes.byref(self.exchange.descriptor(bufs.sums)), s),
                           "dct_kl_from_logits_fwdbwd_pub_f32")
            else:
                _lib.check(h.dct_kl_from_logits_fwdbwd_f32(bufs.adv_logits.data_ptr(), bufs.real_probs.data_ptr(), C, B, HW,
                                                           self.kl_eps, self.adv_weight / self.n, None, sums + 16,
                                                           bufs.grad_adv.data_ptr(), fl, ws, s), "dct_kl_from_logits_fwdbwd_f32")
        else:
            raise ValueError(part)

    def _run(self, bufs: StepBuffers, zero_counts: bool, publish_prev: Optional[StepBuffers] = None) -> None:
        for part in self.parts():
            self.run_part(bufs, part, zero_counts, publish_prev if part == "jsd" else None)
        if self.exchange is not None and self.exchange_mode == "chained":
            self.exchange.publish(bufs.sums)   # the one-CTA publication kernel behind the step's last kernel
        elif self.exchange is not None and self.exchange_mode == "fused" and not self.with_vat:
            self.exchange.publish(bufs.sums)   # JSD-only step: no fused variant of its last kernel

    def capture(self, bufs: StepBuffers, publish_prev: Optional[StepBuffers] = None) -> "torch.cuda.CUDAGraph":
        """Capture ``run(bufs, publish_prev=...)`` into a CUDA graph (replay with ``graph.replay()``)."""
        dev = bufs.logits[0].device
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            self.run(bufs, publish_prev=publish_prev)  # warm-up on the side stream (allocates the per-stream workspace)
        torch.cuda.current_stream(dev).wait_stream(side)
        torch.cuda.synchronize(dev)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=side):
            self.run(bufs, publish_prev=publish_prev)
        return g

    def capture_many(self, sets, publish_chain: bool = False) -> "torch.cuda.CUDAGraph":
        """One CUDA graph holding ``run(s)`` for every buffer set of ``sets`` in order (a round of consecutive steps: the
        launches of neighbouring steps chain by programmatic dependent launch, which two separate graph launches do not).
        ``publish_chain`` ("early" exchange): every step publishes the sums of the set before it, the first one those of the
        last set (the previous round's last step)."""
        dev = sets[0].logits[0].device
        prev = (lambda j: sets[(j - 1) % len(sets)]) if publish_chain else (lambda j: None)
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            self.run(sets[0], publish_prev=prev(0))
        torch.cuda.current_stream(dev).wait_stream(side)
        torch.cuda.synchronize(dev)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=side):
            for j, s in enumerate(sets):
                self.run(s, publish_prev=prev(j))
        return g

    def losses(self, bufs: StepBuffers):
        """(jsd_loss, vat_kl_mean, adv_loss) as 0-d float32 tensors on the device (no sync)."""
        s = bufs.sums
        return ((s[0] * (self.jsd_weight / self.n)).float(), (s[1] / self.n).float(),
                (s[2] * (self.adv_weight / self.n)).float())
