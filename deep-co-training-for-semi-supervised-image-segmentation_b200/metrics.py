"""Drop-in meters of the consistency path, backed by the integer kernels.

Mirrors ``generalframework/metrics`` of the reference:

  DiceMeter        metrics/dice_meter.py:36-83   (``add`` is one counting launch + one tiny divide launch)
  ConfusionMatrix  metrics/confusionmatrix.py:7-98
  IoU              metrics/iou.py:8-113

plus ``hausdorff`` / ``HausdorffMeter``: the Hausdorff distance Summary.py:25 takes from the external ``deepclustering``
package, with the definition of ``medpy.metric.binary.hd`` (exact distance transforms on the device), and
``surface_distances`` / ``SurfaceDistanceMeter``: HD95, ASD and ASSD (``medpy.metric.binary`` hd95 / asd / assd) from the
same distance transforms.

``add`` never leaves the device (no one-hot tensors, no ``torch.unique(a.cpu())``, no numpy
``bincount``); ``value()`` / ``summary()`` keep the reference's return structures.  Counts are exact
int64; ``conf`` is exposed as the reference's ``np.int32`` view.
"""
import ctypes

import numpy as np
import torch

from . import _lib, _runtime


class Metric(object):
    """Base class (metrics/metric.py:9-29)."""

    def reset(self):
        pass

    def add(self, **kwargs):
        pass

    def value(self, **kwargs):
        pass

    def summary(self) -> dict:
        raise NotImplementedError

    def detailed_summary(self) -> dict:
        raise NotImplementedError


def _scores_and_labels(pred, gt, what):
    _runtime.require_cuda(pred, what)
    _runtime.require_cuda(gt, what)
    if pred.dtype != torch.float32:
        raise TypeError(f"{what}: float32 scores expected, got {pred.dtype}")
    assert pred.dim() >= 2
    b, c = pred.shape[0], pred.shape[1]
    hw = pred.numel() // max(b * c, 1)
    if gt.dtype != torch.int64:
        gt = gt.to(torch.int64)
    assert gt.numel() == b * hw, f"label shape {tuple(gt.shape)} does not match scores {tuple(pred.shape)}"
    return pred.detach().contiguous(), gt.contiguous(), b, c, hw


def dice_counts(pred_logit: torch.Tensor, gt: torch.Tensor, out: torch.Tensor = None, accumulate=False) -> torch.Tensor:
    """int64 ``[B,C,3]`` = (intersection, |gt|, |pred|) per image and class, pred = argmax softmax(pred_logit)."""
    x, g, b, c, hw = _scores_and_labels(pred_logit, gt, "dice_counts")
    st = _runtime.state(x.device)
    if out is None:
        out = torch.empty((b, c, 3), dtype=torch.int64, device=x.device)
        accumulate = False
    _lib.check(_lib.lib().dct_dice_counts_f32(x.data_ptr(), g.data_ptr(), c, b, hw, out.data_ptr(), int(accumulate),
                                              _runtime.flags_ptr(st), _runtime.stream_ptr(x.device)),
               "dct_dice_counts_f32")
    _runtime.after_call(st)
    return out


def dice_from_counts(counts: torch.Tensor, batch_sum: bool = False) -> torch.Tensor:
    """``(2*I + 1e-8) / (G + P + 1e-8)`` in float32: ``[B,C]`` rows, or one ``[1,C]`` row summed over the batch."""
    _runtime.require_cuda(counts, "dice_from_counts")
    assert counts.dtype == torch.int64 and counts.dim() == 3 and counts.shape[2] == 3
    counts = counts.contiguous()
    b, c = counts.shape[0], counts.shape[1]
    out = torch.empty((1 if batch_sum else b, c), dtype=torch.float32, device=counts.device)
    _lib.check(_lib.lib().dct_dice_from_counts_f32(counts.data_ptr(), b, c, int(batch_sum), out.data_ptr(),
                                                   _runtime.stream_ptr(counts.device)), "dct_dice_from_counts_f32")
    return out


class DiceMeter(Metric):
    """Drop-in for ``DiceMeter`` (metrics/dice_meter.py:36-83; ``metrics2`` twin has the same ``add``)."""

    def __init__(self, method='2d', report_axises='all', C=4) -> None:
        super().__init__()
        assert method in ('2d', '3d')
        assert report_axises == 'all' or isinstance(report_axises, list)
        self.method = method
        self.report_axis = report_axises
        self.diceLog = []
        self.C = C
        self._cat = None
        self._value = None       # value() of the current log (trainers ask for it ~8 times per meter and iteration)
        self._axis_index = None  # report axes as a device index tensor (a Python-list index costs a blocking H2D copy per use)

    def reset(self):
        self.diceLog = []
        self._cat = None
        self._value = None

    def add(self, pred_logit, gt):
        counts = dice_counts(pred_logit, gt)
        self.add_counts(counts)

    def add_counts(self, counts: torch.Tensor):
        """Append rows from precomputed counts ``[B,C,3]`` (e.g. the fused consistency kernel's)."""
        dice_value = dice_from_counts(counts, batch_sum=(self.method == '3d'))
        assert dice_value.shape.__len__() == 2
        self.diceLog.append(dice_value)
        self._cat = None
        self._value = None

    def value(self, **kwargs):
        """Same statistics, same tensor ops as the reference (dice_meter.py:57-64).  The result is kept until the log
        changes: the reference trainer evaluates ``value()`` once per (model, axis) per iteration for its progress bar
        (cotraining_totalloss.py:252-258) -- eight times per meter on an unchanged log; the tensors returned are the same
        objects then (the reference builds new ones each time: do not modify them in place)."""
        key = self._log_key()
        if self._value is not None and self._value[0] == key:
            return self._value[1]
        log = self.log
        means = log.mean(0)
        stds = log.std(0)
        if self.report_axis == 'all':
            report_means = log.mean(1)
        elif log.is_cuda:
            if self._axis_index is None or self._axis_index.device != log.device:
                self._axis_index = torch.tensor(self.report_axis, dtype=torch.long, device=log.device)
            report_means = log.index_select(1, self._axis_index).mean(1)   # == log[:, self.report_axis].mean(1)
        else:
            report_means = log[:, self.report_axis].mean(1)
        report_std = report_means.std()
        report_mean = report_means.mean()
        self._value = (key, ((report_mean, report_std), (means, stds)))   # keyed on the log's identity: ``diceLog`` is a public list
        return self._value[1]

    def _log_key(self):
        # identity of the log's content as far as a list of immutable-by-convention rows goes: ``diceLog`` is a public
        # attribute of the reference's meter (callers read it, tests append to it), so the caches below cannot rely on
        # add() / reset() alone
        return (len(self.diceLog), id(self.diceLog[-1]) if self.diceLog else 0)

    @property
    def log(self):
        key = self._log_key()
        if self._cat is None or self._cat[0] != key:
            if len(self.diceLog) > 0:
                log = torch.cat(self.diceLog)
            else:
                log = torch.Tensor([0 for _ in range(self.C)])
            if len(log.shape) == 1:
                log = log.unsqueeze(0)
            assert len(log.shape) == 2
            self._cat = (key, log)
        return self._cat[1]

    def detailed_summary(self) -> dict:
        _, (means, _) = self.value()
        return {f'DSC{i}': means[i].item() for i in range(len(means))}

    def summary(self) -> dict:
        (means, var), (_, _) = self.value()
        return {f'mDSC': means.item(), 'mVars': var.item()}


class DiceMeter2(DiceMeter):
    """Drop-in for the ``metrics2`` flavour of ``DiceMeter`` (generalframework/metrics2/dice_meter.py:36-84; user:
    trainer/mean_teacher_trainer.py:18).  Same ``add`` (same counting kernel); the host side differs in two places:
    ``report_axises='all'`` becomes ``list(range(C))`` (:43) and ``summary()`` reports one ``DSC{i}`` per report axis
    (:82-84) instead of ``mDSC`` / ``mVars``."""

    def __init__(self, method='2d', report_axises='all', C=4) -> None:
        super().__init__(method=method, report_axises=report_axises, C=C)
        if isinstance(report_axises, str) and report_axises == 'all':
            self.report_axis = list(range(C))

    def summary(self) -> dict:
        _, (means, _) = self.value()
        return {f'DSC{i}': means[i].item() for i in self.report_axis}


def _class_map(t, C, what):
    """int64 ``[B,H,W]`` class map from an integer ``[B,H,W]`` / ``[B,1,H,W]`` tensor."""
    _runtime.require_cuda(t, what)
    if t.is_floating_point():
        raise TypeError(f"{what}: integer class map expected, got {t.dtype}")
    if t.dim() == 4 and t.shape[1] == 1:
        t = t[:, 0]
    assert t.dim() == 3, f"{what}: class map [B,H,W] or [B,1,H,W] expected, got {tuple(t.shape)}"
    return t.to(torch.int64).contiguous()


def _distance_args(pred, gt, C, method, voxelspacing, what):
    """Arguments of ``hausdorff`` / ``surface_distances``: int64 class maps ``p``, ``g`` ``[B,H,W]``, ``C``, whether the
    batch is one volume, and the spacing as a ctypes double array (``None`` = ones)."""
    assert method in ('2d', '3d')
    if pred.is_floating_point():
        from .utils import _classmap
        assert pred.dim() == 4, f"{what}: scores [B,C,H,W] expected, got {tuple(pred.shape)}"
        if pred.dtype != torch.float32:
            raise TypeError(f"{what}: float32 scores expected, got {pred.dtype}")
        assert C is None or C == pred.shape[1], f"C={C} does not match scores {tuple(pred.shape)}"
        C = pred.shape[1]
        p = _classmap(pred.detach(), 1, want_cls=True)[0]
    else:
        assert C is not None, f"{what}: C is required for an integer class map"
        p = _class_map(pred, C, what)
    g = _class_map(gt, C, what)
    assert g.shape == p.shape, f"label shape {tuple(gt.shape)} does not match prediction {tuple(pred.shape)}"
    volume = method == '3d'
    sp = None
    if voxelspacing is not None:
        vals = [float(v) for v in voxelspacing]
        assert len(vals) == (3 if volume else 2), f"voxelspacing for '{method}' has {3 if volume else 2} values, got {vals}"
        sp = (ctypes.c_double * len(vals))(*vals)
    return p, g, C, volume, sp


def hausdorff(pred, gt, C=None, method='2d', voxelspacing=None) -> torch.Tensor:
    """Hausdorff distance per class, float32 ``[rows, C]`` on the input's device (``rows`` = B for ``'2d'``, 1 for ``'3d'``).

    Definition of ``medpy.metric.binary.hd`` (the ACDC challenge's evaluation code; the reference's Summary.py:25 gets the
    metric from the external ``deepclustering`` package): the largest distance from a border pixel of ``{pred == c}`` to the
    border of ``{gt == c}`` and back, borders taken with the cross structuring element and the grid's outside as
    background, distances scaled by ``voxelspacing``.  ``'2d'`` measures every slice ``[H,W]`` on its own; ``'3d'`` measures
    the batch as one ``[B,H,W]`` volume (under ``PatientSampler`` one batch is one patient).  A class absent from ``pred``
    or ``gt`` gives NaN (medpy raises there).

    ``pred``: float32 scores ``[B,C,H,W]`` -- reduced to a class map with the arg-max ``DiceMeter.add`` uses, so the Dice and
    the HD of one batch describe the same segmentation -- or an integer class map ``[B,H,W]`` / ``[B,1,H,W]`` (e.g.
    ``ensemble.vote_class(...)``; then ``C`` is required).  ``gt``: integer ``[B,H,W]`` / ``[B,1,H,W]``.
    ``voxelspacing``: ``(sy, sx)`` for ``'2d'``, ``(sz, sy, sx)`` for ``'3d'``, ``None`` = ones.  Values outside ``[0, C)``
    belong to no class and raise the label / prediction range checks under the current check mode.
    """
    p, g, C, volume, sp = _distance_args(pred, gt, C, method, voxelspacing, "hausdorff")
    B, H, W = p.shape
    h = _lib.lib()
    nbytes = h.dct_hausdorff_scratch_bytes(C, B, H, W, int(volume))
    if nbytes == 0:
        _lib.check(_lib.ERR_UNSUPPORTED, f"dct_hausdorff_scratch_bytes (C={C}, shape {(B, H, W)})")
    scratch = torch.empty(nbytes, dtype=torch.uint8, device=p.device)
    out = torch.empty((1 if volume else B, C), dtype=torch.float32, device=p.device)
    st = _runtime.state(p.device)
    _lib.check(h.dct_hausdorff_i64(p.data_ptr(), g.data_ptr(), C, B, H, W, int(volume), sp, out.data_ptr(),
                                   _runtime.flags_ptr(st), scratch.data_ptr(), _runtime.stream_ptr(p.device)),
               "dct_hausdorff_i64")
    _runtime.after_call(st)
    return out


_SURFACE_KEYS = ('hd', 'hd95', 'asd', 'assd')


def surface_distances(pred, gt, C=None, method='2d', voxelspacing=None) -> dict:
    """Surface distances per class: ``{'hd', 'hd95', 'asd', 'assd'}``, each float32 ``[rows, C]`` on the input's device,
    from one device call.  Arguments, borders, grids, spacing and NaN are those of ``hausdorff``.

    With ``S_pg`` the distances from each border pixel of ``{pred == c}`` to the border of ``{gt == c}`` and ``S_gp`` the
    other direction (``medpy.metric.binary``, connectivity 1): ``hd`` = ``hausdorff(...)`` bit for bit; ``hd95`` =
    ``np.percentile(np.hstack((S_pg, S_gp)), 95)`` (medpy ``hd95``); ``asd`` = ``mean(S_pg)`` (medpy ``asd(pred, gt)``,
    directional); ``assd`` = ``(mean(S_pg) + mean(S_gp)) / 2`` (medpy ``assd``).
    """
    p, g, C, volume, sp = _distance_args(pred, gt, C, method, voxelspacing, "surface_distances")
    B, H, W = p.shape
    h = _lib.lib()
    nbytes = h.dct_surface_distance_scratch_bytes(C, B, H, W, int(volume))
    if nbytes == 0:
        _lib.check(_lib.ERR_UNSUPPORTED, f"dct_surface_distance_scratch_bytes (C={C}, shape {(B, H, W)})")
    scratch = torch.empty(nbytes, dtype=torch.uint8, device=p.device)
    out = torch.empty((4, 1 if volume else B, C), dtype=torch.float32, device=p.device)
    st = _runtime.state(p.device)
    _lib.check(h.dct_surface_distances_i64(p.data_ptr(), g.data_ptr(), C, B, H, W, int(volume), sp, out.data_ptr(),
                                           _runtime.flags_ptr(st), scratch.data_ptr(), _runtime.stream_ptr(p.device)),
               "dct_surface_distances_i64")
    _runtime.after_call(st)
    return dict(zip(_SURFACE_KEYS, out.unbind(0)))


def _nan_mean_std(x: torch.Tensor, dim: int):
    """Mean and unbiased standard deviation along ``dim`` over the non-NaN entries (NaN where fewer than 1 / 2 remain)."""
    valid = ~torch.isnan(x)
    n = valid.sum(dim)
    mean = torch.nanmean(x, dim)
    dev = torch.where(valid, x - mean.unsqueeze(dim), torch.zeros_like(x))
    var = (dev * dev).sum(dim) / (n - 1)
    return mean, torch.where(n > 1, var.sqrt(), torch.full_like(var, float('nan')))


def _nan_statistics(log: torch.Tensor, report_axis):
    """``HausdorffMeter.value`` of a ``[rows, C]`` log."""
    means, stds = _nan_mean_std(log, 0)
    axes = log if report_axis == 'all' else log[:, report_axis]
    report_mean, report_std = _nan_mean_std(torch.nanmean(axes, 1), 0)
    return (report_mean, report_std), (means, stds)


class HausdorffMeter(Metric):
    """Hausdorff distance per class next to ``DiceMeter`` (same ``method`` / ``report_axises`` / ``C``; definition of
    ``medpy.metric.binary.hd``, see ``hausdorff``).  ``add`` appends one row per image (``'2d'``) or per batch
    (``'3d'``); the statistics skip the NaN of classes absent from a prediction or a label."""

    def __init__(self, method='2d', report_axises='all', C=4) -> None:
        super().__init__()
        assert method in ('2d', '3d')
        assert report_axises == 'all' or isinstance(report_axises, list)
        self.method = method
        self.report_axis = report_axises
        self.C = C
        self.hdLog = []

    def reset(self):
        self.hdLog = []

    def add(self, pred, gt, voxelspacing=None):
        self.hdLog.append(hausdorff(pred, gt, C=self.C, method=self.method, voxelspacing=voxelspacing))

    @property
    def log(self):
        if len(self.hdLog) == 0:
            return torch.full((1, self.C), float('nan'))
        return torch.cat(self.hdLog)

    def value(self, **kwargs):
        """``((mean, std), (means[C], stds[C]))``: per class over the rows, and of the per-row mean over the report
        axes; NaN entries skipped, unbiased standard deviations."""
        return _nan_statistics(self.log, self.report_axis)

    def detailed_summary(self) -> dict:
        _, (means, _) = self.value()
        return {f'HD{i}': means[i].item() for i in range(len(means))}

    def summary(self) -> dict:
        (mean, var), _ = self.value()
        return {'mHD': mean.item(), 'mHDVars': var.item()}


class SurfaceDistanceMeter(Metric):
    """HD, HD95, ASD and ASSD per class next to ``DiceMeter`` (same ``method`` / ``report_axises`` / ``C``; definitions of
    ``surface_distances``).  ``add`` makes one device call and appends one row per image (``'2d'``) or per batch
    (``'3d'``) to each metric's log; the statistics are ``HausdorffMeter``'s and skip the NaN of absent classes."""

    _NAMES = (('hd', 'HD', 'HD'), ('hd95', 'HD95', 'HD95_'), ('asd', 'ASD', 'ASD'), ('assd', 'ASSD', 'ASSD'))   # key, summary, detailed

    def __init__(self, method='2d', report_axises='all', C=4) -> None:
        super().__init__()
        assert method in ('2d', '3d')
        assert report_axises == 'all' or isinstance(report_axises, list)
        self.method = method
        self.report_axis = report_axises
        self.C = C
        self.reset()

    def reset(self):
        self.logs = {k: [] for k in _SURFACE_KEYS}

    def add(self, pred, gt, voxelspacing=None):
        r = surface_distances(pred, gt, C=self.C, method=self.method, voxelspacing=voxelspacing)
        for k in _SURFACE_KEYS:
            self.logs[k].append(r[k])

    def log(self, metric='hd95') -> torch.Tensor:
        rows = self.logs[metric]
        if len(rows) == 0:
            return torch.full((1, self.C), float('nan'))
        return torch.cat(rows)

    def value(self, metric='hd95'):
        """``((mean, std), (means[C], stds[C]))`` of one metric's log, as ``HausdorffMeter.value``."""
        return _nan_statistics(self.log(metric), self.report_axis)

    def detailed_summary(self) -> dict:
        out = {}
        for k, _, prefix in self._NAMES:
            _, (means, _) = self.value(k)
            out.update({f'{prefix}{i}': means[i].item() for i in range(len(means))})
        return out

    def summary(self) -> dict:
        out = {}
        for k, name, _ in self._NAMES:
            (mean, var), _ = self.value(k)
            out.update({f'm{name}': mean.item(), f'm{name}Vars': var.item()})
        return out


class ConfusionMatrix(Metric):
    """Drop-in for ``ConfusionMatrix`` (metrics/confusionmatrix.py:7-98).

    The matrix accumulates on the device as int64 ``[C,C]`` (rows = ground truth); ``conf`` /
    ``value()`` copy it to the host as the reference's ``np.int32`` array.
    """

    def __init__(self, num_classes, ignore_index=255, normalized=False):
        super().__init__()
        self.normalized = normalized
        self.num_classes = num_classes
        self.ignore_index = ignore_index
        self._dev = None
        self._host = np.zeros((num_classes, num_classes), dtype=np.int64)

    def reset(self):
        self._host.fill(0)
        if self._dev is not None:
            self._dev.zero_()

    def _device_conf(self, device):
        if self._dev is None or self._dev.device != device:
            self._flush()
            self._dev = torch.zeros((self.num_classes, self.num_classes), dtype=torch.int64, device=device)
        return self._dev

    def _flush(self):
        if self._dev is not None:
            self._host += self._dev.cpu().numpy()
            self._dev.zero_()

    def add_scores(self, scores, target):
        """scores ``[N,C,H,W]`` float32: arg-max over dim 1 fused into the counting kernel."""
        x, g, b, c, hw = _scores_and_labels(scores, target, "ConfusionMatrix.add_scores")
        assert c == self.num_classes, 'number of predictions does not match size of confusion matrix'
        conf = self._device_conf(x.device)
        _lib.check(_lib.lib().dct_confusion_f32(x.data_ptr(), g.data_ptr(), c, b, hw, conf.data_ptr(),
                                                _runtime.stream_ptr(x.device)), "dct_confusion_f32")

    def device_counts(self, device) -> torch.Tensor:
        """The int64 ``[C,C]`` device accumulator itself: pass it as ``confusion=`` to ``supervised_from_logits`` and the
        loss kernel counts straight into this meter (no second pass over the logits)."""
        return self._device_conf(torch.device(device))

    def add(self, predicted, target):
        """predicted / target: integer class maps of equal shape (tensors or numpy arrays)."""
        if not torch.is_tensor(predicted):
            predicted = torch.as_tensor(np.asarray(predicted))
        if not torch.is_tensor(target):
            target = torch.as_tensor(np.asarray(target))
        if not predicted.is_cuda and target.is_cuda:
            predicted = predicted.to(target.device)
        if not target.is_cuda and predicted.is_cuda:
            target = target.to(predicted.device)
        _runtime.require_cuda(predicted, "ConfusionMatrix.add")
        assert predicted.shape == target.shape
        p = predicted.to(torch.int64).contiguous().view(-1)
        t = target.to(torch.int64).contiguous().view(-1)
        st = _runtime.state(p.device)
        conf = self._device_conf(p.device)
        _lib.check(_lib.lib().dct_confusion_labels_i64(p.data_ptr(), t.data_ptr(), p.numel(), self.num_classes,
                                                       conf.data_ptr(), _runtime.flags_ptr(st),
                                                       _runtime.stream_ptr(p.device)), "dct_confusion_labels_i64")
        _runtime.after_call(st)

    @property
    def conf64(self) -> np.ndarray:
        self._flush()
        return self._host.copy()

    @property
    def conf(self) -> np.ndarray:
        return self.conf64.astype(np.int32)

    def value(self):
        conf = self.conf
        if self.normalized:
            conf = conf.astype(np.float32)
            return conf / conf.sum(1).clip(min=1e-12)[:, None]
        return conf


class IoU(Metric):
    """Drop-in for ``IoU`` (metrics/iou.py:8-113)."""

    def __init__(self, num_classes, normalized=False, ignore_index=255):
        super().__init__()
        self.conf_metric = ConfusionMatrix(num_classes, ignore_index=ignore_index, normalized=normalized)
        if ignore_index is None:
            self.ignore_index = None
        elif isinstance(ignore_index, int):
            self.ignore_index = (ignore_index,)
        else:
            try:
                self.ignore_index = tuple(ignore_index)
            except TypeError:
                raise ValueError("'ignore_index' must be an int or iterable")

    def reset(self):
        self.conf_metric.reset()

    def device_counts(self, device) -> torch.Tensor:
        """int64 ``[C,C]`` accumulator on ``device`` for the fused loss + meter launch (``supervised_from_logits(...,
        confusion=meter.device_counts(dev))`` replaces ``meter.add(predicted=pred, target=gt)``)."""
        return self.conf_metric.device_counts(device)

    def add(self, predicted, target):
        assert predicted.size(0) == target.size(0), 'number of targets and predicted outputs do not match'
        assert predicted.dim() == 3 or predicted.dim() == 4, \
            "predictions must be of dimension (N, H, W) or (N, K, H, W)"
        assert target.dim() == 3 or target.dim() == 4, "targets must be of dimension (N, H, W) or (N, K, H, W)"
        if predicted.dim() == 4:
            self.conf_metric.add_scores(predicted, target)
        else:
            self.conf_metric.add(predicted.reshape(-1), target.reshape(-1))

    def value(self):
        hist = self.conf_metric.value()
        with np.errstate(divide='ignore', invalid='ignore'):
            acc = np.diag(hist).sum() / hist.sum()
            acc_cls = np.nanmean(np.diag(hist) / hist.sum(axis=1))
            iu = np.diag(hist) / (hist.sum(axis=1) + hist.sum(axis=0) - np.diag(hist))
            valid = hist.sum(axis=1) > 0
            mean_iu = np.nanmean(iu[valid])
            freq = hist.sum(axis=1) / hist.sum()
            fwavacc = (freq[freq > 0] * iu[freq > 0]).sum()
            mean_all = np.nanmean(iu)
        return {
            "Overall_Acc": acc,
            "Mean_Acc": acc_cls,
            "FreqW_Acc": fwavacc,
            "Validated_Mean_IoU": mean_iu,
            "Mean_IoU": mean_all,
            "Class_IoU": torch.from_numpy(iu).float(),
        }
