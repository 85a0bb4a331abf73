"""Drop-in losses of the consistency path, backed by the sm_100a kernels.

Mirrors ``generalframework/loss/loss.py`` of the reference (class names, ctor
arguments, call signatures, return shapes/dtypes, AssertionError behaviour):

  JSD_2D, JSD            loss.py:183-196, 165-180
  Entropy_2D, Entropy    loss.py:70-84, 53-67
  KL_Divergence_2D       loss.py:110-134
  KL_Divergence_2D_Logit loss.py:137-162
  KL_div                 loss.py:87-107
  CrossEntropyLoss2d     loss.py:12-25           (supervised branch, SURVEY.md 8f.1)
  get_loss_fn / LOSS     loss/__init__.py:6-16   (the hot-path entries)

plus the fast path the north star asks for -- one pass over the K views' LOGITS
producing the weighted mean JSD, its gradient and (optionally) the K Dice count
tensors: :func:`jsd_consistency_from_logits` / :class:`FusedJSDConsistency`, and
:func:`kl_consistency_from_logits` for the adversarial KL.

Every forward/backward is a ``torch.autograd.Function`` whose body is one call
into the C ABI (``include/dct_b200.h``); inputs must be CUDA float32 tensors.  The one-pass-over-logits
forms (:func:`jsd_consistency_from_logits`, :func:`kl_consistency_from_logits`, :func:`kl_div_with_logit`,
:func:`supervised_from_logits` / ``CrossEntropyLoss2d``) also take bfloat16 logits (autocast networks): bf16 rows
through the same tile pipeline, fp32 math and loss, bf16 gradients.
"""
from typing import List, Optional, Sequence

import torch
import torch.nn as nn

from . import _lib, _runtime


def _prep(t: torch.Tensor, what: str) -> torch.Tensor:
    _runtime.require_cuda(t, what)
    if t.dtype != torch.float32:
        raise TypeError(f"{what}: float32 expected, got {t.dtype}")
    return t.contiguous()


def _prep_lp(t: torch.Tensor, what: str) -> torch.Tensor:
    """float32 or bfloat16 (the one-pass-over-logits ops also take the bf16 logits of an autocast network)."""
    _runtime.require_cuda(t, what)
    if t.dtype not in (torch.float32, torch.bfloat16):
        raise TypeError(f"{what}: float32 or bfloat16 expected, got {t.dtype}")
    return t.contiguous()


def _promote(t: torch.Tensor) -> torch.Tensor:
    return t.float() if t.dtype == torch.bfloat16 else t


def _all_bf16(ts) -> bool:
    """bf16 kernels run only when every tensor is bf16; mixed inputs are promoted to float32 (as torch would)."""
    return all(t.dtype == torch.bfloat16 for t in ts)


def _bchw(t: torch.Tensor):
    b, c = t.shape[0], t.shape[1]
    hw = 1
    for s in t.shape[2:]:
        hw *= s
    return b, c, hw


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else t.data_ptr()


def _views_args(views: Sequence[torch.Tensor], what: str):
    assert len(views) >= 1
    vs = [_prep(v, what) for v in views]
    for v in vs[1:]:
        assert v.shape == vs[0].shape, "all views must have the same shape"
    if len(vs) > _lib.MAX_VIEWS or vs[0].shape[1] > _lib.MAX_CLASSES:
        raise ValueError(f"{what}: at most {_lib.MAX_VIEWS} views and {_lib.MAX_CLASSES} classes are supported")
    return vs


# ------------------------------------------------------------------------------------------------
# JSD
# ------------------------------------------------------------------------------------------------
class _JSDFn(torch.autograd.Function):
    """map = JSD(views) with views given as probs or logits; backward recomputes from the inputs."""

    @staticmethod
    def forward(ctx, in_kind: int, reduce: bool, *views):
        vs = _views_args(views, "JSD")
        b, c, hw = _bchw(vs[0])
        dev = vs[0].device
        st = _runtime.state(dev)
        h = _lib.lib()
        out_map = None if reduce else torch.empty((b,) + tuple(vs[0].shape[2:]), dtype=torch.float32, device=dev)
        total = torch.empty(1, dtype=torch.float64, device=dev) if reduce else None
        _lib.check(h.dct_jsd_fwd_f32(_lib.ptr_array(vs), len(vs), c, b, hw, in_kind, _ptr(out_map), _ptr(total),
                                     _runtime.flags_ptr(st) if in_kind == _lib.IN_PROBS else None,
                                     st.workspace.data_ptr(), _runtime.stream_ptr(dev)), "dct_jsd_fwd_f32")
        if in_kind == _lib.IN_PROBS:
            _runtime.after_call(st)
        ctx.save_for_backward(*vs)
        ctx.in_kind, ctx.reduce, ctx.n = in_kind, reduce, b * hw
        if reduce:
            return (total / float(b * hw)).to(torch.float32).reshape(())
        return out_map

    @staticmethod
    def backward(ctx, g):
        vs = ctx.saved_tensors
        b, c, hw = _bchw(vs[0])
        dev = vs[0].device
        g = g.contiguous().to(torch.float32)
        grads = [torch.empty_like(v) for v in vs]
        if ctx.reduce:
            gmap, gscalar, gconst = None, g, 1.0 / ctx.n
        else:
            gmap, gscalar, gconst = g, None, 1.0
        _lib.check(_lib.lib().dct_jsd_bwd_f32(_lib.ptr_array(vs), len(vs), c, b, hw, ctx.in_kind, _ptr(gmap),
                                              _ptr(gscalar), gconst, _lib.ptr_array(grads),
                                              _runtime.stream_ptr(dev)), "dct_jsd_bwd_f32")
        return (None, None) + tuple(grads)


class JSD_2D(nn.Module):
    """K-view Jensen-Shannon divergence map; drop-in for ``JSD_2D`` (loss.py:183-196).

    ``forward(List[Tensor[B,C,H,W]] of probabilities) -> Tensor[B,H,W]``, differentiable w.r.t.
    every list element; AssertionError on non-4-D or non-simplex input (unless ``python -O``).
    """

    def __init__(self):
        super().__init__()

    def forward(self, input: List[torch.Tensor]):
        for inprob in input:
            assert inprob.shape.__len__() == 4
        return _JSDFn.apply(_lib.IN_PROBS, False, *input)


class JSD(nn.Module):
    """N-d variant with optional mean; drop-in for ``JSD`` (loss.py:165-180)."""

    def __init__(self):
        super().__init__()

    def forward(self, input: List[torch.Tensor], reduce=True):
        for inprob in input:
            assert inprob.shape.__len__() >= 2
        return _JSDFn.apply(_lib.IN_PROBS, bool(reduce), *input)


def jsd_map_from_logits(logits: Sequence[torch.Tensor]) -> torch.Tensor:
    """``JSD_2D([softmax(z, 1) for z in logits])`` without materialising the probabilities."""
    return _JSDFn.apply(_lib.IN_LOGITS, False, *logits)


def _finish_grads(grads, g, dtypes):
    """Upstream scaling of gradients that were produced in the forward pass (a zero-traffic launch for the usual
    upstream of exactly 1) and the cast back to each input's dtype (no-op unless an input was promoted).  bf16
    gradients are scaled by the fp32 upstream with one fp32 multiply and one rounding, not by a bf16-rounded upstream."""
    h = _lib.lib()
    out = []
    for gr, dt in zip(grads, dtypes):
        if gr.dtype == torch.float32:
            _lib.check(h.dct_scale_if_not_one_f32(gr.data_ptr(), gr.numel(), g.data_ptr(),
                                                  _runtime.stream_ptr(gr.device)), "dct_scale_if_not_one_f32")
        else:
            _lib.check(h.dct_scale_if_not_one_bf16(gr.data_ptr(), gr.numel(), g.data_ptr(),
                                                   _runtime.stream_ptr(gr.device)), "dct_scale_if_not_one_bf16")
        out.append(gr if gr.dtype == dt else gr.to(dt))
    return out


class _FusedJSDFn(torch.autograd.Function):
    """weight * mean(JSD(softmax(logits))) and its gradient in ONE pass (dct_jsd_fwdbwd_f32)."""

    @staticmethod
    def forward(ctx, weight: float, n_global: Optional[int], labels, counts, in_kind: int, accumulate: bool, *views):
        in_dtypes = [v.dtype for v in views]
        cmode = _lib.COUNTS_ACCUMULATE if accumulate else _lib.COUNTS_OVERWRITE
        lp = in_kind == _lib.IN_LOGITS and _all_bf16(views)
        if in_kind == _lib.IN_LOGITS and not lp and any(d == torch.bfloat16 for d in in_dtypes):
            views = [_promote(v) for v in views]   # mixed precisions: promote
        vs = [_prep_lp(v, "jsd_consistency") for v in views] if lp else _views_args(views, "jsd_consistency")
        b, c, hw = _bchw(vs[0])
        dev = vs[0].device
        st = _runtime.state(dev)
        n = b * hw if n_global is None else int(n_global)
        need_grad = any(ctx.needs_input_grad[6:])
        ctx.in_dtypes = in_dtypes
        total = torch.empty(1, dtype=torch.float64, device=dev)
        h = _lib.lib()
        lab = None
        if labels is not None:
            _runtime.require_cuda(labels, "labels")
            assert labels.dtype == torch.int64 and labels.numel() == b * hw
            assert counts is not None and counts.dtype == torch.int64 and counts.numel() == len(vs) * b * c * 3
            lab = labels.contiguous()
        fl = _runtime.flags_ptr(st)
        if lp:
            # bf16 logits: one launch of the bf16 tile pipeline (fp32 math); shapes it does not take are promoted
            for v in vs[1:]:
                assert v.shape == vs[0].shape, "all views must have the same shape"
            grads = [torch.empty_like(v) for v in vs] if need_grad else None
            fuse_dice = lab is not None and need_grad and c <= 4
            rc = h.dct_jsd_fwdbwd_bf16(_lib.ptr_array(vs), len(vs), c, b, hw, float(weight) / n, None, _ptr(total),
                                       _lib.ptr_array(grads) if need_grad else None, _ptr(lab) if fuse_dice else None,
                                       _ptr(counts) if fuse_dice else None, cmode, fl, st.workspace.data_ptr(),
                                       _runtime.stream_ptr(dev))
            if rc == _lib.ERR_UNSUPPORTED:
                lp = False
                vs = [v.float() for v in vs]
            else:
                _lib.check(rc, "dct_jsd_fwdbwd_bf16")
                if lab is not None and not fuse_dice:  # C > 4 / evaluation: the meters count on their own
                    for k, v in enumerate(vs):
                        vf = v.float()
                        _lib.check(h.dct_dice_counts_f32(vf.data_ptr(), lab.data_ptr(), c, b, hw,
                                                         counts.data_ptr() + k * b * c * 3 * 8, int(accumulate), fl,
                                                         _runtime.stream_ptr(dev)), "dct_dice_counts_f32")
                ctx.grads = grads
        if lp:
            pass
        elif need_grad:
            grads = [torch.empty_like(v) for v in vs]
            _lib.check(h.dct_jsd_fwdbwd_f32(_lib.ptr_array(vs), len(vs), c, b, hw, in_kind, float(weight) / n, None,
                                            _ptr(total), _lib.ptr_array(grads), _ptr(lab), _ptr(counts), cmode, fl,
                                            st.workspace.data_ptr(), _runtime.stream_ptr(dev)), "dct_jsd_fwdbwd_f32")
            ctx.grads = grads
        else:
            _lib.check(h.dct_jsd_fwd_f32(_lib.ptr_array(vs), len(vs), c, b, hw, in_kind, None, _ptr(total), fl,
                                         st.workspace.data_ptr(), _runtime.stream_ptr(dev)), "dct_jsd_fwd_f32")
            if lab is not None:
                for k, v in enumerate(vs):
                    _lib.check(h.dct_dice_counts_f32(v.data_ptr(), lab.data_ptr(), c, b, hw,
                                                     counts.data_ptr() + k * b * c * 3 * 8, int(accumulate), fl,
                                                     _runtime.stream_ptr(dev)), "dct_dice_counts_f32")
            ctx.grads = None
        if lab is not None or in_kind == _lib.IN_PROBS:
            _runtime.after_call(st)
        return (total * (float(weight) / n)).to(torch.float32).reshape(())

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, g):
        grads = ctx.grads
        ctx.grads = None
        if grads is None:
            raise RuntimeError("jsd_consistency: backward called twice or without grad-requiring inputs")
        g = g.contiguous().to(torch.float32)
        h = _lib.lib()
        dev = grads[0].device
        grads = _finish_grads(grads, g, ctx.in_dtypes)
        return (None, None, None, None, None, None) + tuple(grads)


def jsd_consistency_from_logits(logits: Sequence[torch.Tensor], weight: float = 1.0,
                                labels: Optional[torch.Tensor] = None, dice_counts: Optional[torch.Tensor] = None,
                                n_global: Optional[int] = None, accumulate: bool = True) -> torch.Tensor:
    """``weight * JSD_2D([softmax(z,1) for z in logits]).mean()`` in one pass over the logits.

    The gradient w.r.t. every logits tensor is produced by the same kernel launch (upstream
    ``weight / N`` folded in), so ``loss.backward()`` costs no further pass.  If ``labels``
    ([B,1,H,W] / [B,H,W] int64) and ``dice_counts`` (int64 ``[K,B,C,3]``, accumulated into) are
    given, the K views' Dice counts (I, G, P) against ``labels`` are produced as well
    (what ``unlabdiceMeters[k].add`` computes, cotraining_totalloss.py:224).
    ``n_global``: total pixel count over all data-parallel ranks (defaults to the local B*H*W).
    ``accumulate=False``: the launch clears ``dice_counts`` itself (hand it ``torch.empty``: no fill launch per step).
    """
    return _FusedJSDFn.apply(float(weight), n_global, labels, dice_counts, _lib.IN_LOGITS, bool(accumulate), *logits)


class FusedJSDConsistency(nn.Module):
    """Module form of :func:`jsd_consistency_from_logits` (logits in, weighted scalar loss out)."""

    def __init__(self, weight: float = 1.0):
        super().__init__()
        self.weight = weight

    def forward(self, logits: List[torch.Tensor], labels=None, dice_counts=None, n_global=None, accumulate=True):
        return jsd_consistency_from_logits(logits, self.weight, labels, dice_counts, n_global, accumulate)


# ------------------------------------------------------------------------------------------------
# Entropy
# ------------------------------------------------------------------------------------------------
class _EntropyFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, p):
        p = _prep(p, "Entropy")
        b, c, hw = _bchw(p)
        st = _runtime.state(p.device)
        out = torch.empty((b,) + tuple(p.shape[2:]), dtype=torch.float32, device=p.device)
        _lib.check(_lib.lib().dct_entropy_fwd_f32(p.data_ptr(), c, b, hw, out.data_ptr(), None, _runtime.flags_ptr(st),
                                                  st.workspace.data_ptr(), _runtime.stream_ptr(p.device)),
                   "dct_entropy_fwd_f32")
        _runtime.after_call(st)
        ctx.save_for_backward(p)
        return out

    @staticmethod
    def backward(ctx, g):
        (p,) = ctx.saved_tensors
        b, c, hw = _bchw(p)
        gp = torch.empty_like(p)
        g = g.contiguous().to(torch.float32)
        _lib.check(_lib.lib().dct_entropy_bwd_f32(p.data_ptr(), c, b, hw, g.data_ptr(), None, 1.0, gp.data_ptr(),
                                                  _runtime.stream_ptr(p.device)), "dct_entropy_bwd_f32")
        return gp


class Entropy(nn.Module):
    """``-sum_c p log(p + 1e-16)`` over dim 1; drop-in for ``Entropy`` (loss.py:53-67)."""

    def __init__(self):
        super().__init__()

    def forward(self, input: torch.Tensor):
        assert input.shape.__len__() >= 2
        return _EntropyFn.apply(input)


class Entropy_2D(nn.Module):
    """Drop-in for ``Entropy_2D`` (loss.py:70-84): 4-D input -> [B,H,W]."""

    def __init__(self):
        super().__init__()

    def forward(self, input: torch.Tensor):
        assert input.shape.__len__() == 4
        return _EntropyFn.apply(input)


# ------------------------------------------------------------------------------------------------
# KL family
# ------------------------------------------------------------------------------------------------
class _KLProbFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, p, y, reduce: bool, eps: float):
        p = _prep(p, "KL_Divergence_2D"); y = _prep(y, "KL_Divergence_2D")
        assert p.shape == y.shape
        b, c, hw = _bchw(p)
        dev = p.device
        st = _runtime.state(dev)
        out_map = None if reduce else torch.empty((b,) + tuple(p.shape[2:]), dtype=torch.float32, device=dev)
        total = torch.empty(1, dtype=torch.float64, device=dev) if reduce else None
        _lib.check(_lib.lib().dct_kl_fwd_f32(p.data_ptr(), y.data_ptr(), c, b, hw, float(eps), _ptr(out_map),
                                             _ptr(total), _runtime.flags_ptr(st), st.workspace.data_ptr(),
                                             _runtime.stream_ptr(dev)), "dct_kl_fwd_f32")
        _runtime.after_call(st)
        ctx.save_for_backward(p, y)
        ctx.reduce, ctx.eps, ctx.n = reduce, float(eps), b * hw
        if reduce:
            return (total / float(b * hw)).to(torch.float32).reshape(())
        return out_map

    @staticmethod
    def backward(ctx, g):
        p, y = ctx.saved_tensors
        b, c, hw = _bchw(p)
        g = g.contiguous().to(torch.float32)
        gp = torch.empty_like(p) if ctx.needs_input_grad[0] else None
        gy = torch.empty_like(y) if ctx.needs_input_grad[1] else None
        if gp is None and gy is None:
            return None, None, None, None
        if ctx.reduce:
            gmap, gscalar, gconst = None, g, 1.0 / ctx.n
        else:
            gmap, gscalar, gconst = g, None, 1.0
        _lib.check(_lib.lib().dct_kl_bwd_f32(p.data_ptr(), y.data_ptr(), c, b, hw, ctx.eps, _ptr(gmap), _ptr(gscalar),
                                             gconst, _ptr(gp), _ptr(gy), _runtime.stream_ptr(p.device)),
                   "dct_kl_bwd_f32")
        return gp, gy, None, None


class KL_Divergence_2D(nn.Module):
    """Drop-in for ``KL_Divergence_2D`` (loss.py:110-134): ``sum_c y log(y+eps) - y log(p+eps)``."""

    def __init__(self, reduce=False, eps=1e-10):
        super().__init__()
        self.reduce = reduce
        self.eps = eps

    def forward(self, p_prob: torch.Tensor, y_prob: torch.Tensor):
        return _KLProbFn.apply(p_prob, y_prob, bool(self.reduce), self.eps)


class _KLLogitFn(torch.autograd.Function):
    """kl_div_with_logit(q_logit, p_logit): map and both gradients from one launch each way."""

    @staticmethod
    def forward(ctx, q_logit, p_logit, reduce: bool):
        ctx.in_dtypes = (q_logit.dtype, p_logit.dtype)
        lp = _all_bf16((q_logit, p_logit))
        if not lp:
            q_logit, p_logit = _prep(_promote(q_logit), "kl_div_with_logit"), _prep(_promote(p_logit), "kl_div_with_logit")
        ql = _prep_lp(q_logit, "kl_div_with_logit"); pl = _prep_lp(p_logit, "kl_div_with_logit")
        assert ql.shape == pl.shape
        b, c, hw = _bchw(ql)
        dev = ql.device
        st = _runtime.state(dev)
        out_map = None if reduce else torch.empty((b,) + tuple(ql.shape[2:]), dtype=torch.float32, device=dev)
        total = torch.empty(1, dtype=torch.float64, device=dev) if reduce else None
        if lp:  # bf16 logits (fp32 map): the bf16 tile pipeline, or promotion for shapes it does not take
            rc = _lib.lib().dct_kl_logit_bf16(ql.data_ptr(), pl.data_ptr(), c, b, hw, _ptr(out_map), _ptr(total), 0,
                                              None, None, 1.0, None, None, st.workspace.data_ptr(),
                                              _runtime.stream_ptr(dev))
            if rc == _lib.ERR_UNSUPPORTED:
                lp, ql, pl = False, ql.float(), pl.float()
            else:
                _lib.check(rc, "dct_kl_logit_bf16")
        if not lp:
            _lib.check(_lib.lib().dct_kl_logit_f32(ql.data_ptr(), pl.data_ptr(), c, b, hw, _ptr(out_map), _ptr(total), 0,
                                                   None, None, 1.0, None, None, st.workspace.data_ptr(),
                                                   _runtime.stream_ptr(dev)), "dct_kl_logit_f32")
        ctx.save_for_backward(ql, pl)
        ctx.reduce, ctx.n = reduce, b * hw
        if reduce:
            return (total / float(b * hw)).to(torch.float32).reshape(())
        return out_map

    @staticmethod
    def backward(ctx, g):
        ql, pl = ctx.saved_tensors
        b, c, hw = _bchw(ql)
        dev = ql.device
        g = g.contiguous().to(torch.float32)
        gq = torch.empty_like(ql) if ctx.needs_input_grad[0] else None
        gp = torch.empty_like(pl) if ctx.needs_input_grad[1] else None
        if gq is None and gp is None:
            return None, None, None
        if ctx.reduce:
            gmap, gscalar, gconst = None, g, 1.0 / ctx.n
        else:
            gmap, gscalar, gconst = g, None, 1.0
            if ql.dtype == torch.bfloat16 and g.data_ptr() % 16 != 0:
                # the bf16 tile pipeline reads the upstream map in 16-byte rows; autograd may hand over a slice at any
                # 4-byte offset (e.g. of a torch.cat of the map with a tensor whose size is not a multiple of 4)
                gmap = g.clone()
        st = _runtime.state(dev)
        fn = _lib.lib().dct_kl_logit_bf16 if ql.dtype == torch.bfloat16 else _lib.lib().dct_kl_logit_f32
        _lib.check(fn(ql.data_ptr(), pl.data_ptr(), c, b, hw, None, None, 1, _ptr(gmap), _ptr(gscalar), gconst,
                      _ptr(gp), _ptr(gq), st.workspace.data_ptr(), _runtime.stream_ptr(dev)), "dct_kl_logit")
        if gq is not None and gq.dtype != ctx.in_dtypes[0]:
            gq = gq.to(ctx.in_dtypes[0])
        if gp is not None and gp.dtype != ctx.in_dtypes[1]:
            gp = gp.to(ctx.in_dtypes[1])
        return gq, gp, None


def kl_div_with_logit(q_logit: torch.Tensor, p_logit: torch.Tensor) -> torch.Tensor:
    """Drop-in for ``VATGenerator.kl_div_with_logit`` (utils/AEGenerator.py:78-91) -> [B,H,W]."""
    return _KLLogitFn.apply(q_logit, p_logit, False)


class KL_Divergence_2D_Logit(nn.Module):
    """Drop-in for ``KL_Divergence_2D_Logit`` (loss.py:137-162); ``y_logit`` plays the role of q."""

    def __init__(self, reduce=False, eps=1e-10):
        super().__init__()
        self.reduce = reduce
        self.eps = eps

    def forward(self, p_logit: torch.Tensor, y_logit: torch.Tensor):
        return _KLLogitFn.apply(y_logit, p_logit, bool(self.reduce))


class _KLDivFn(torch.autograd.Function):
    """KL_div's map / mean and, like the reference's autograd graph, its gradients w.r.t. both arguments."""

    @staticmethod
    def forward(ctx, p, q, reduce: bool, eps: float):
        p = _prep(p, "KL_div"); q = _prep(q, "KL_div")
        assert p.shape == q.shape
        b, c, hw = _bchw(p)
        dev = p.device
        st = _runtime.state(dev)
        out_map = None if reduce else torch.empty((b,) + tuple(p.shape[2:]), dtype=torch.float32, device=dev)
        total = torch.empty(1, dtype=torch.float64, device=dev) if reduce else None
        _lib.check(_lib.lib().dct_kl_div_fwd_f32(p.data_ptr(), q.data_ptr(), c, b, hw, float(eps), _ptr(out_map),
                                                 _ptr(total), _runtime.flags_ptr(st), st.workspace.data_ptr(),
                                                 _runtime.stream_ptr(dev)), "dct_kl_div_fwd_f32")
        _runtime.after_call(st)
        ctx.save_for_backward(p, q)
        ctx.reduce, ctx.eps, ctx.n = reduce, float(eps), b * hw
        if reduce:
            return (total / float(b * hw)).to(torch.float32).reshape(())
        return out_map

    @staticmethod
    def backward(ctx, g):
        p, q = ctx.saved_tensors
        b, c, hw = _bchw(p)
        if not (ctx.needs_input_grad[0] or ctx.needs_input_grad[1]):
            return None, None, None, None
        g = g.contiguous().to(torch.float32)
        gp = torch.empty_like(p)
        gq = torch.empty_like(q) if ctx.needs_input_grad[1] else None
        if ctx.reduce:
            gmap, gscalar, gconst = None, g, 1.0 / ctx.n
        else:
            gmap, gscalar, gconst = g, None, 1.0
        _lib.check(_lib.lib().dct_kl_div_bwd_f32(p.data_ptr(), q.data_ptr(), c, b, hw, ctx.eps, _ptr(gmap), _ptr(gscalar),
                                                 gconst, gp.data_ptr(), _ptr(gq), _runtime.stream_ptr(p.device)),
                   "dct_kl_div_bwd_f32")
        return (gp if ctx.needs_input_grad[0] else None), gq, None, None


class KL_div(nn.Module):
    """Drop-in for ``KL_div`` (loss.py:87-107): ``sum_c -p log(q/p + eps)``, map or mean (``reduce`` is the ctor's, the
    call-time argument is ignored exactly as the reference ignores it), differentiable w.r.t. ``p`` and ``q``."""

    def __init__(self, reduce=True, eps=1e-10):
        super().__init__()
        self.eps = eps
        self.reduce = reduce

    def forward(self, p, q, reduce=False):
        return _KLDivFn.apply(p, q, bool(self.reduce), self.eps)


class _KLFromLogitsFn(torch.autograd.Function):
    """weight * KL_Divergence_2D(reduce=True)(softmax(p_logit), y_prob.detach()) + grad in one pass."""

    @staticmethod
    def forward(ctx, p_logit, y_prob, weight: float, eps: float, n_global: Optional[int]):
        ctx.in_dtype = p_logit.dtype
        lp = _all_bf16((p_logit, y_prob))
        if not lp:
            p_logit, y_prob = _prep(_promote(p_logit), "kl_consistency"), _prep(_promote(y_prob), "kl_consistency")
        pl = _prep_lp(p_logit, "kl_consistency"); y = _prep_lp(y_prob, "kl_consistency")
        assert pl.shape == y.shape
        b, c, hw = _bchw(pl)
        dev = pl.device
        st = _runtime.state(dev)
        n = b * hw if n_global is None else int(n_global)
        total = torch.empty(1, dtype=torch.float64, device=dev)
        grad = torch.empty_like(pl) if ctx.needs_input_grad[0] else None
        if lp:
            rc = _lib.lib().dct_kl_from_logits_fwdbwd_bf16(pl.data_ptr(), y.data_ptr(), c, b, hw, float(eps),
                                                           float(weight) / n, None, total.data_ptr(), _ptr(grad),
                                                           _runtime.flags_ptr(st), st.workspace.data_ptr(),
                                                           _runtime.stream_ptr(dev))
            if rc == _lib.ERR_UNSUPPORTED:  # shape outside the bf16 tile pipeline: promote
                lp, pl, y = False, pl.float(), y.float()
                grad = torch.empty_like(pl) if grad is not None else None
            else:
                _lib.check(rc, "dct_kl_from_logits_fwdbwd_bf16")
        if not lp:
                _lib.check(_lib.lib().dct_kl_from_logits_fwdbwd_f32(pl.data_ptr(), y.data_ptr(), c, b, hw, float(eps),
                                                                float(weight) / n, None, total.data_ptr(), _ptr(grad),
                                                                _runtime.flags_ptr(st), st.workspace.data_ptr(),
                                                                _runtime.stream_ptr(dev)), "dct_kl_from_logits_fwdbwd_f32")
        _runtime.after_call(st)
        ctx.grad = grad
        return (total * (float(weight) / n)).to(torch.float32).reshape(())

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, g):
        grad = ctx.grad
        ctx.grad = None
        if grad is None:
            return None, None, None, None, None
        g = g.contiguous().to(torch.float32)
        return _finish_grads([grad], g, [ctx.in_dtype])[0], None, None, None, None


def kl_consistency_from_logits(adv_logit: torch.Tensor, real_prob: torch.Tensor, weight: float = 1.0,
                               eps: float = 1e-10, n_global: Optional[int] = None) -> torch.Tensor:
    """``weight * KL_Divergence_2D(reduce=True)(softmax(adv_logit,1), real_prob.detach())`` in one pass.

    The adversarial loss of ``CoTrainer._FSGM_adv_training`` (cotraining_totalloss.py:391-392) /
    ``VatTrainer`` (vattrainer.py:152-154) with the softmax, the mean and the backward fused.
    """
    return _KLFromLogitsFn.apply(adv_logit, real_prob.detach(), float(weight), float(eps), n_global)


# ------------------------------------------------------------------------------------------------
# softmax as a standalone op (Segmentator.predict(logit=False), models/segmentators.py:46-50)
# ------------------------------------------------------------------------------------------------
class _SoftmaxFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x):
        x = _prep(x, "softmax")
        b, c, hw = _bchw(x)
        p = torch.empty_like(x)
        _lib.check(_lib.lib().dct_softmax_fwd_f32(x.data_ptr(), c, b, hw, p.data_ptr(), _runtime.stream_ptr(x.device)),
                   "dct_softmax_fwd_f32")
        ctx.save_for_backward(p)
        return p

    @staticmethod
    def backward(ctx, gp):
        (p,) = ctx.saved_tensors
        b, c, hw = _bchw(p)
        gp = gp.contiguous().to(torch.float32)
        gx = torch.empty_like(p)
        _lib.check(_lib.lib().dct_softmax_bwd_f32(p.data_ptr(), gp.data_ptr(), c, b, hw, gx.data_ptr(),
                                                  _runtime.stream_ptr(p.device)), "dct_softmax_bwd_f32")
        return gx


def softmax_dim1(x: torch.Tensor) -> torch.Tensor:
    """``F.softmax(x, 1)`` for [B,C,*] CUDA float32 tensors."""
    return _SoftmaxFn.apply(x)


# ------------------------------------------------------------------------------------------------
# supervised branch: CrossEntropyLoss2d (+ the Dice counting of the same logits / labels), SURVEY.md 8f.1
# ------------------------------------------------------------------------------------------------
def _ce_labels(targets: torch.Tensor, b: int, hw: int) -> torch.Tensor:
    _runtime.require_cuda(targets, "CrossEntropyLoss2d targets")
    if targets.dtype != torch.int64:
        raise TypeError(f"CrossEntropyLoss2d: int64 targets expected, got {targets.dtype}")
    assert targets.numel() == b * hw, "targets must be [B,H,W] (or [B,1,H,W]) matching the logits"
    return targets.contiguous()


def _ce_weight_sum(lab, c, ignore_index, weight, st, dev):
    """W = sum_i w[t_i] over the kept pixels as a float64 device scalar (dct_label_hist_i64 + a C-element dot)."""
    hist = torch.empty(c + 2, dtype=torch.int64, device=dev)
    _lib.check(_lib.lib().dct_label_hist_i64(lab.data_ptr(), lab.numel(), c, int(ignore_index), hist.data_ptr(),
                                             _runtime.stream_ptr(dev)), "dct_label_hist_i64")
    kept = hist[:c].to(torch.float64)
    return kept.sum() if weight is None else (kept * weight.to(torch.float64)).sum()


class _CEFn(torch.autograd.Function):
    """nn.NLLLoss(weight, ignore_index, reduction)(log_softmax(logits, 1), targets) -- one pass for mean / sum
    (loss AND gradient from dct_ce_fwdbwd_f32, optionally with the Dice counts of the same tensors), map forward +
    map backward for reduction 'none'."""

    @staticmethod
    def forward(ctx, logits, targets, weight, ignore_index: int, reduction: str, n_global, dice_counts, confusion=None):
        ctx.in_dtype = logits.dtype
        lp = logits.dtype == torch.bfloat16 and reduction != "none" and ctx.needs_input_grad[0] and confusion is None
        x = _prep_lp(logits, "CrossEntropyLoss2d") if lp else _prep(_promote(logits), "CrossEntropyLoss2d")
        assert x.dim() >= 2
        b, c, hw = _bchw(x)
        if c > _lib.MAX_CLASSES:
            raise ValueError(f"CrossEntropyLoss2d: at most {_lib.MAX_CLASSES} classes are supported")
        dev = x.device
        lab = _ce_labels(targets, b, hw)
        st = _runtime.state(dev)
        h = _lib.lib()
        w = None
        if weight is not None:
            w = weight.to(device=dev, dtype=torch.float32).contiguous()
            assert w.numel() == c, "weight must have one entry per class"
        if dice_counts is not None:
            assert dice_counts.dtype == torch.int64 and dice_counts.is_cuda and dice_counts.numel() == b * c * 3
        if confusion is not None:
            assert confusion.dtype == torch.int64 and confusion.is_cuda and confusion.is_contiguous() and \
                confusion.numel() == c * c, "confusion must be a contiguous int64 [C,C] CUDA tensor"
            assert dice_counts is None and reduction != "none", "confusion counting fuses with the mean / sum loss only"
        fl, ws, s = _runtime.flags_ptr(st), st.workspace.data_ptr(), _runtime.stream_ptr(dev)
        ctx.reduction, ctx.ignore_index = reduction, int(ignore_index)
        if reduction == "none":
            out = torch.empty((b,) + tuple(x.shape[2:]), dtype=torch.float32, device=dev)
            _lib.check(h.dct_ce_fwd_f32(x.data_ptr(), lab.data_ptr(), c, b, hw, _ptr(w), int(ignore_index),
                                        out.data_ptr(), None, fl, ws, s), "dct_ce_fwd_f32")
            if dice_counts is not None:
                _lib.check(h.dct_dice_counts_f32(x.data_ptr(), lab.data_ptr(), c, b, hw, dice_counts.data_ptr(), 1, fl, s),
                           "dct_dice_counts_f32")
            _runtime.after_call(st)
            ctx.save_for_backward(x, lab, *([w] if w is not None else []))
            ctx.grad = None
            return out
        total = torch.empty(1, dtype=torch.float64, device=dev)
        inv = None        # float32 device scalar 1/W ('mean' with a data-dependent denominator)
        gconst = 1.0
        if reduction == "mean":
            if n_global is not None:
                gconst = 1.0 / float(n_global)
            elif w is None and dice_counts is not None and confusion is None and _runtime.get_check_mode() != "off":
                # the fused meter asserts every label in [0,C) (class2one_hot, utils/utils.py:190; raised through
                # the label flag in 'eager' / 'deferred' mode), so no pixel is ignored and W is the pixel count: no
                # histogram pass.  In mode 'off' nothing would ever report an ignored / bad label, and NLLLoss' mean
                # is sum / #kept: the histogram branch below counts the kept pixels instead.
                gconst = 1.0 / float(b * hw)
            else:
                inv64 = 1.0 / _ce_weight_sum(lab, c, ignore_index, w, st, dev)
                inv = inv64.to(torch.float32).reshape(1)
        if lp:  # bf16 logits: one launch of the bf16 tile pipeline, or promotion for shapes it does not take
            grad = torch.empty_like(x)
            rc = h.dct_ce_fwdbwd_bf16(x.data_ptr(), lab.data_ptr(), c, b, hw, _ptr(w), int(ignore_index), _ptr(inv),
                                      gconst, None, total.data_ptr(), grad.data_ptr(), _ptr(dice_counts), fl, ws, s)
            if rc == _lib.ERR_UNSUPPORTED:
                lp, x = False, x.float()
            else:
                _lib.check(rc, "dct_ce_fwdbwd_bf16")
                ctx.grad = grad
        if lp:
            pass
        elif ctx.needs_input_grad[0] and confusion is not None:
            grad = torch.empty_like(x)
            _lib.check(h.dct_ce_fwdbwd_conf_f32(x.data_ptr(), lab.data_ptr(), c, b, hw, _ptr(w), int(ignore_index),
                                                _ptr(inv), gconst, None, total.data_ptr(), grad.data_ptr(),
                                                confusion.data_ptr(), fl, ws, s), "dct_ce_fwdbwd_conf_f32")
            ctx.grad = grad
        elif ctx.needs_input_grad[0]:
            grad = torch.empty_like(x)
            _lib.check(h.dct_ce_fwdbwd_f32(x.data_ptr(), lab.data_ptr(), c, b, hw, _ptr(w), int(ignore_index),
                                           _ptr(inv), gconst, None, total.data_ptr(), grad.data_ptr(),
                                           _ptr(dice_counts), fl, ws, s), "dct_ce_fwdbwd_f32")
            ctx.grad = grad
        else:
            _lib.check(h.dct_ce_fwd_f32(x.data_ptr(), lab.data_ptr(), c, b, hw, _ptr(w), int(ignore_index), None,
                                        total.data_ptr(), fl, ws, s), "dct_ce_fwd_f32")
            if dice_counts is not None:
                _lib.check(h.dct_dice_counts_f32(x.data_ptr(), lab.data_ptr(), c, b, hw, dice_counts.data_ptr(), 1, fl, s),
                           "dct_dice_counts_f32")
            if confusion is not None:
                _lib.check(h.dct_confusion_f32(x.data_ptr(), lab.data_ptr(), c, b, hw, confusion.data_ptr(), s),
                           "dct_confusion_f32")
            ctx.grad = None
        _runtime.after_call(st)
        if inv is not None:
            return (total * inv.to(torch.float64)).to(torch.float32).reshape(())
        return (total * gconst).to(torch.float32).reshape(())

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, g):
        g = g.contiguous().to(torch.float32)
        h = _lib.lib()
        if ctx.reduction == "none":
            x, lab = ctx.saved_tensors[:2]
            w = ctx.saved_tensors[2] if len(ctx.saved_tensors) > 2 else None
            b, c, hw = _bchw(x)
            grad = torch.empty_like(x)
            _lib.check(h.dct_ce_bwd_f32(x.data_ptr(), lab.data_ptr(), c, b, hw, _ptr(w), ctx.ignore_index, g.data_ptr(),
                                        None, 1.0, grad.data_ptr(), None, _runtime.stream_ptr(x.device)),
                       "dct_ce_bwd_f32")
            return grad.to(ctx.in_dtype), None, None, None, None, None, None, None
        grad = ctx.grad
        ctx.grad = None
        if grad is None:
            raise RuntimeError("CrossEntropyLoss2d: backward called twice or without grad-requiring logits")
        return _finish_grads([grad], g, [ctx.in_dtype])[0], None, None, None, None, None, None, None


class CrossEntropyLoss2d(nn.Module):
    """Drop-in for ``CrossEntropyLoss2d`` (loss.py:12-25): ``NLLLoss(weight, ignore_index)(log_softmax(x,1), t)``.

    Same ctor (``weight=None, reduce=True, size_average=True, ignore_index=255``) and call
    (``forward(outputs[B,C,H,W], targets[B,H,W] int64)``).  The loss and its gradient come from one
    pass over the logits; ``loss.backward()`` costs no further pass for the default reductions."""

    def __init__(self, weight=None, reduce=True, size_average=True, ignore_index=255):
        super().__init__()
        self.ignore_index = ignore_index
        self.reduction = "none" if not reduce else ("mean" if size_average else "sum")
        if weight is not None:
            self.register_buffer("weight", torch.as_tensor(weight, dtype=torch.float32).clone())
        else:
            self.weight = None

    def forward(self, outputs: torch.Tensor, targets: torch.Tensor):
        return _CEFn.apply(outputs, targets, self.weight, int(self.ignore_index), self.reduction, None, None, None)


def supervised_from_logits(logits: torch.Tensor, gt: torch.Tensor, weight: Optional[torch.Tensor] = None,
                           ignore_index: int = 255, dice_counts: Optional[torch.Tensor] = None,
                           n_global: Optional[int] = None, confusion: Optional[torch.Tensor] = None) -> torch.Tensor:
    """``CrossEntropyLoss2d(weight)(logits, gt.squeeze(1))`` and ``DiceMeter.add(logits, gt)`` in ONE pass.

    The two consecutive lines of the labeled loop (cotraining_totalloss.py:211-212) read the same
    logits and labels; here one kernel launch produces the mean cross-entropy, its gradient
    (upstream 1/W folded in) and, if ``dice_counts`` (int64 ``[B,C,3]``, accumulated into) is given,
    the (I, G, P) counts of ``argmax softmax(logits)`` against ``gt`` (feed them to
    ``DiceMeter.add_counts``).  ``n_global``: pixel count over all data-parallel ranks for the
    unweighted global mean (defaults to the local denominator) -- valid ONLY without class weights and without
    ignored pixels (it replaces NLLLoss' data-dependent denominator ``sum_i w[t_i]`` by a constant); with either,
    leave it None and all-reduce the per-rank losses weighted by their kept weight instead.

    ``confusion`` (int64 ``[C,C]``, accumulated into; instead of ``dice_counts``): the Cityscapes trainers keep an
    ``IoU`` meter on the same line pair (cotraining_city.py:236-241: ``metrics[k].add(predicted=pred, target=gt)``);
    the same launch then counts ``conf[gt][argmax logits]`` over the pixels with ``0 <= gt < C`` -- hand the tensor
    to ``IoU.add_confusion`` / read it back at ``value()`` time."""
    w = None if weight is None else torch.as_tensor(weight, dtype=torch.float32)
    return _CEFn.apply(logits, gt, w, int(ignore_index), "mean", n_global, dice_counts, confusion)


# ------------------------------------------------------------------------------------------------
# registry (loss/__init__.py:6-16); the entries that live on the hot path
# ------------------------------------------------------------------------------------------------
LOSS = {"jsd": JSD_2D, "cross_entropy": CrossEntropyLoss2d}


def get_loss_fn(name: str, **kwargs):
    try:
        return LOSS.get(name)(**kwargs)
    except Exception as e:
        raise ValueError("name error when inputting the loss name, with %s" % str(e))
