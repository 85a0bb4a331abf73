"""Drive the UNMODIFIED reference trainer on synthetic data (TEST / BENCH INFRASTRUCTURE, not product code).

``CoTrainer._train_loop`` (generalframework/trainer/cotraining_totalloss.py:158-271) is the north star's contract: its
loss / meter call sites must work unchanged once ``dct_b200.install()`` has rebound the names.  This module builds that
trainer exactly as ``train_ACDC_cotraining.py:38-63`` does -- ``Segmentator``s from the config dicts, criterions from the
``get_loss_fn`` registry, ``CoTrainer(...)`` -- over synthetic loaders of the dataset API the loop expects
(``([img, gt], meta, name)`` items, ``set_mode``, a writable ``training``; SURVEY.md Appendix A), truncates the
hard-coded 300 iterations through the module-global ``tqdm_`` and records, without touching the reference:

  * every ``totalLoss`` (the tensor ``.backward()`` is called on at cotraining_totalloss.py:247),
  * every Dice row any ``DiceMeter.add`` appends (labeled and unlabeled meters),
  * the tensors ``_train_loop`` returns,
  * wall time per iteration (device-synchronised).

The reference is found through ``oracle/ref_shim.py``: ``$DCT_REFERENCE_ROOT``, else ``baseline/_ref`` (staged by
``tools/stage_reference.sh``).
"""
import os
import sys
import tempfile
import time
import warnings

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
if HERE not in sys.path:
    sys.path.insert(0, HERE)
import ref_shim  # noqa: E402


def available() -> bool:
    return ref_shim.reference_available()


class _Trunc:
    """Stand-in for ``tqdm_(range(300))``: the first ``n`` items, with the progress-bar methods the loop calls."""

    def __init__(self, it, n):
        self.it, self.n = it, n

    def __iter__(self):
        for i, x in enumerate(self.it):
            if i >= self.n:
                return
            yield x

    def set_postfix(self, *a, **k):
        pass

    def set_description(self, *a, **k):
        pass


class SynthSet(torch.utils.data.Dataset):
    """Seeded images in [0,1] and labels in [0,C) with the reference datasets' item structure and mode switches
    (dataset/medicalDataLoader.py:22-162)."""

    def __init__(self, n, C, H, W, seed, cin=1):
        g = torch.Generator().manual_seed(seed)
        self.img = torch.rand(n, cin, H, W, generator=g)
        # blocky labels (8 x 8 patches) so that the classes form regions, as segmentation masks do
        small = torch.randint(0, C, (n, 1, (H + 7) // 8, (W + 7) // 8), generator=g)
        self.gt = small.repeat_interleave(8, 2).repeat_interleave(8, 3)[:, :, :H, :W].contiguous()
        self.training = None

    def set_mode(self, mode):
        self.training = mode

    def __len__(self):
        return self.img.shape[0]

    def __getitem__(self, i):
        return [self.img[i], self.gt[i]], i, f"synth_{i:04d}"


def run_train_loop(device, use_dropins, iters=3, K=2, arch="enet", C=4, B=4, H=256, W=256, seed=1234, train_jsd=True,
                   train_adv=True, cot_weight=0.5, adv_weight=0.05, eps=0.03, deterministic=True, warmup_iters=0,
                   keep_inputs=0, tf32=False, check_mode=None):
    """One truncated epoch of the reference's co-training loop, stock (``use_dropins=False``) or after
    ``dct_b200.install()``.  Returns a dict of recorded values (numpy) and timings."""
    ref_shim.install()
    warnings.filterwarnings("ignore")
    import generalframework.trainer.cotraining_totalloss as ct
    from generalframework import ModelMode
    from generalframework.loss import get_loss_fn
    from generalframework.models import Segmentator

    old_check = None
    if use_dropins:
        import dct_b200
        dct_b200.install()
        if check_mode is not None:   # 'deferred': the drop-ins' contract flags are read once, after the loop, not after every call
            old_check = dct_b200.set_check_mode(check_mode)
    # process-wide torch switches: saved here, restored in the `finally` below.  ``tf32=False`` (parity runs): exact fp32
    # convolutions, so that both arms see the same network outputs; ``tf32=None`` (timing runs): PyTorch's defaults untouched
    saved_flags = (torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark, torch.backends.cudnn.allow_tf32,
                   torch.backends.cuda.matmul.allow_tf32)
    if deterministic:
        torch.backends.cudnn.deterministic = True
        torch.backends.cudnn.benchmark = False
    if tf32 is not None:
        torch.backends.cudnn.allow_tf32 = bool(tf32)
        torch.backends.cuda.matmul.allow_tf32 = bool(tf32)
    torch.manual_seed(seed)
    np.random.seed(seed)
    import random
    random.seed(seed)

    arch_dict = {"name": arch, "num_classes": C}
    optim_dict = {"name": "Adam", "lr": 0.001, "weight_decay": 0.0001}          # config/ACDC_config_cotraing.yaml:5-8
    sched_dict = {"name": "StepLR", "step_size": 90, "gamma": 0.1}
    segs = [Segmentator(arch_dict=dict(arch_dict), optim_dict=dict(optim_dict), scheduler_dict=dict(sched_dict))
            for _ in range(K)]
    mk = lambda s: torch.utils.data.DataLoader(SynthSet(B * max(iters + warmup_iters, 2), C, H, W, s), batch_size=B,  # noqa: E731
                                               shuffle=False, drop_last=True, num_workers=0)
    labeled = [mk(seed + 10 + k) for k in range(K)]
    unlabeled = mk(seed + 99)
    val = mk(seed + 77)
    criterions = {"sup": get_loss_fn("cross_entropy"), "jsd": get_loss_fn("jsd"), "adv": get_loss_fn("jsd")}
    save_dir = tempfile.mkdtemp(prefix="dct_ref_trainer_")
    const = lambda v: {"name": "ConstantScheduler", "begin_epoch": 0, "max_value": v}  # noqa: E731
    trainer = ct.CoTrainer(segmentators=segs, labeled_dataloaders=labeled, unlabeled_dataloader=unlabeled,
                           val_dataloader=val, criterions=criterions, max_epoch=1, save_dir=save_dir, device=str(device),
                           axises=list(range(1, C)), adv_scheduler_dict=const(adv_weight),
                           cot_scheduler_dict=const(cot_weight), adv_training_dict={"eplision": eps}, use_tqdm=True)

    # ---- recorders (monkey-patches of module globals / torch; restored below; the reference files are not touched)
    losses, rows, meter_inputs = [], [], []
    orig_backward = torch.Tensor.backward
    orig_tqdm = ct.tqdm_
    Meter = ct.DiceMeter

    class RecMeter(Meter):
        def add(self, pred_logit, gt):
            super().add(pred_logit, gt)
            rows.append(self.diceLog[-1].detach().clone())
            if len(meter_inputs) < keep_inputs:   # the first adds' inputs, for the near-tie analysis of the GPU test
                meter_inputs.append((pred_logit.detach().clone(), gt.detach().clone()))

    def rec_backward(self, *a, **k):
        losses.append(self.detach().clone())
        return orig_backward(self, *a, **k)

    def run(n):
        ct.tqdm_ = lambda it, **k: _Trunc(it, n)
        return trainer._train_loop(labeled_dataloaders=labeled, unlabeled_dataloader=unlabeled, epoch=0,
                                   mode=ModelMode.TRAIN, save=False, train_jsd=train_jsd, train_adv=train_adv,
                                   augment_labeled_data=False, augment_unlabeled_data=False)

    try:
        if warmup_iters:
            run(warmup_iters)       # cuDNN autotuning, module load; re-seeds at its start like every epoch
        ct.DiceMeter = RecMeter
        torch.Tensor.backward = rec_backward
        if device.type == "cuda":
            torch.cuda.synchronize(device)
        t0 = time.perf_counter()
        lab_dice, unlab_dice = run(iters)
        if device.type == "cuda":
            torch.cuda.synchronize(device)
        dt = time.perf_counter() - t0
    finally:
        torch.Tensor.backward = orig_backward
        ct.tqdm_ = orig_tqdm
        ct.DiceMeter = Meter
        if use_dropins:
            import dct_b200
            if old_check is not None:
                try:
                    dct_b200.raise_if_flagged()
                finally:
                    dct_b200.set_check_mode(old_check)
            dct_b200.uninstall()
        (torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark, torch.backends.cudnn.allow_tf32,
         torch.backends.cuda.matmul.allow_tf32) = saved_flags
    per_iter = 2 if train_adv else 1      # FSGMGenerator back-propagates its own CE loss before the total loss
    total = [float(v) for v in losses[per_iter - 1::per_iter]]
    return {"total_loss": np.asarray(total, dtype=np.float64),
            "all_backward_losses": np.asarray([float(v) for v in losses], dtype=np.float64),
            "dice_rows": [r.float().cpu().numpy() for r in rows], "meter_inputs": meter_inputs,
            "lab_dice": lab_dice.detach().cpu().numpy(), "unlab_dice": unlab_dice.detach().cpu().numpy(),
            "seconds": dt, "iters": iters, "it_per_s": iters / dt,
            "meter_class": f"{Meter.__module__}.{Meter.__name__}",
            "jsd_class": f"{type(criterions['jsd']).__module__}.{type(criterions['jsd']).__name__}"}


# ----------------------------------------------------------------------------------------------------
# The consistency STEP of bench.py through the reference's own modules (stock ATen composition), on any device
# ----------------------------------------------------------------------------------------------------
def reference_step_inputs(device, K, C, B, H, W, cin, seed=1234):
    """The synthetic tensors of one step (SURVEY.md 8d), same distributions as engine.StepBuffers.allocate."""
    g = torch.Generator(device="cpu").manual_seed(seed)
    rn = lambda *s: torch.randn(*s, generator=g)  # noqa: E731
    t = {"logits": [3 * rn(B, C, H, W) for _ in range(K)],
         "labels": torch.randint(0, C, (B, 1, H, W), generator=g),
         "d": rn(B, cin, H, W), "d_grad": rn(B, cin, H, W), "img": torch.rand(B, cin, H, W, generator=g),
         "yhat": 3 * rn(B, C, H, W), "adv": 3 * rn(B, C, H, W), "real": torch.softmax(3 * rn(B, C, H, W), 1)}
    mv = lambda x: [v.to(device) for v in x] if isinstance(x, list) else x.to(device)  # noqa: E731
    return {k: mv(v) for k, v in t.items()}


def reference_step(inp, with_vat=True, with_dice=True, xi=1e-6, eps=10.0):
    """One pass of the hot path exactly as the reference composes it, with the reference's own classes:
    ``unlabdiceMeters[k].add(prob_k, gt)`` x K -> ``JSD_2D(probs).mean()`` (cotraining_totalloss.py:223-226); the VAT
    arithmetic (AEGenerator.py:97-117: ``_l2_normalize`` x 3, ``kl_div_with_logit(...).mean().backward()``); the
    adversarial ``KL_Divergence_2D(reduce=True)`` (:391-392); backward; losses and Dice rows read back to the host.
    The network passes between those points are not part of the path (their outputs are the synthetic tensors)."""
    ref_shim.install()
    import torch.nn.functional as F
    from generalframework.loss import JSD_2D, KL_Divergence_2D
    from generalframework.metrics import DiceMeter
    from generalframework.utils.AEGenerator import VATGenerator
    K, C = len(inp["logits"]), inp["logits"][0].shape[1]
    z = [x.detach().requires_grad_() for x in inp["logits"]]
    probs = [F.softmax(x, 1) for x in z]
    rows = []
    if with_dice:
        for k in range(K):
            m = DiceMeter(method="2d", C=C)
            m.add(probs[k], inp["labels"])
            rows.append(m.log)
    jsd = JSD_2D()(probs).mean()
    total = jsd
    outs = [jsd.detach()]
    if with_vat:
        d = VATGenerator._l2_normalize(inp["d"].clone())
        d = xi * VATGenerator._l2_normalize(d)
        yh = inp["yhat"].detach().requires_grad_()
        vkl = VATGenerator.kl_div_with_logit(z[0].detach(), yh).mean()
        vkl.backward()
        r_adv = eps * VATGenerator._l2_normalize(inp["d_grad"].clone())
        img_adv = torch.clamp(inp["img"] + r_adv.detach(), 0, 1)  # noqa: F841
        adv = KL_Divergence_2D(reduce=True)(F.softmax(inp["adv"].detach().requires_grad_(), 1), inp["real"].detach())
        total = total + adv
        outs += [vkl.detach(), adv.detach()]
    total.backward()
    res = torch.stack(outs).cpu()
    rows = [r.cpu() for r in rows]
    return res, rows


def time_reference_step(device, K, C, B, H, W, cin, steps, warmup, with_vat=True, with_dice=True, threads=None):
    """(pixels/s, s/step, last losses) of ``reference_step`` on ``device`` over ``steps`` timed steps."""
    if threads:
        torch.set_num_threads(threads)
    inp = reference_step_inputs(device, K, C, B, H, W, cin)
    for _ in range(warmup):
        res, _ = reference_step(inp, with_vat, with_dice)
    if device.type == "cuda":
        torch.cuda.synchronize(device)
    t0 = time.perf_counter()
    for _ in range(steps):
        res, _ = reference_step(inp, with_vat, with_dice)
    if device.type == "cuda":
        torch.cuda.synchronize(device)
    dt = time.perf_counter() - t0
    return B * H * W * steps / dt, dt / steps, [float(v) for v in res]
