"""Import shim for the upstream reference (TEST INFRASTRUCTURE ONLY).

Makes ``import generalframework`` work from a read-only copy of the original
project's source tree, where several of its eager imports (skimage,
tensorboardX, visdom, matplotlib) may be absent.  Nothing in that tree is
modified.  This file is only used by ``oracle/make_golden*.py``, by
``oracle/ref_trainer.py`` and by tests that are skipped when the tree is not
found (the repository does not contain it).

Why each stub is needed (reference file:line):
  generalframework/utils/__init__.py:1-2  -> utils/utils.py:16 (skimage.io.imsave)
  generalframework/utils/visualize.py:2,4,6,9 (tensorboardX, visdom, matplotlib, skimage)
  generalframework/trainer/cotraining_totalloss.py:6 (tensorboardX)
  generalframework/utils/utils.py:318,342 + dataset/augment.py:141 (collections.Mapping...)
  generalframework/trainer/mean_teacher_trainer.py:10 (easydict; only when the package is absent)

Where the reference is looked for: $DCT_REFERENCE_ROOT, else <repo>/baseline/_ref (a staged copy;
tools/stage_reference.sh).
"""
import collections
import collections.abc
import os
import sys
import types

_REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _find_root() -> str:
    cands = [os.environ.get("DCT_REFERENCE_ROOT"), os.path.join(_REPO, "baseline", "_ref")]
    for c in cands:
        if c and os.path.isdir(os.path.join(c, "generalframework")):
            return c
    return cands[0] or cands[1]


REFERENCE_ROOT = _find_root()


def reference_available() -> bool:
    return os.path.isdir(os.path.join(REFERENCE_ROOT, "generalframework"))


def _stub(name, **attrs):
    m = types.ModuleType(name)
    m.__dict__.update(attrs)
    sys.modules.setdefault(name, m)
    return sys.modules[name]


class _EasyDict(dict):
    """Stand-in for easydict.EasyDict (attribute access to dict keys, nested dicts converted)."""

    def __init__(self, d=None, **kw):
        super().__init__()
        for k, v in dict(d or {}, **kw).items():
            self[k] = v

    def __setitem__(self, k, v):
        super().__setitem__(k, _EasyDict(v) if isinstance(v, dict) and not isinstance(v, _EasyDict) else v)

    __setattr__ = __setitem__

    def __getattr__(self, k):
        try:
            return self[k]
        except KeyError:
            raise AttributeError(k)


class _SummaryWriter:
    def __init__(self, *a, **k):
        pass

    def add_scalars(self, *a, **k):
        pass


def install():
    """Idempotently make ``generalframework`` importable. Returns the package."""
    if not reference_available():
        raise RuntimeError(f"reference tree not found at {REFERENCE_ROOT}")
    sk = _stub("skimage")
    sk.io = _stub("skimage.io", imsave=lambda *a, **k: None)
    sk.transform = _stub("skimage.transform", resize=None)
    sk.data = None
    _stub("tensorboardX", SummaryWriter=_SummaryWriter)
    _stub("visdom", Visdom=object)
    try:
        import easydict  # noqa: F401
    except ImportError:
        _stub("easydict", EasyDict=_EasyDict)
    mpl = _stub("matplotlib")
    mpl.pyplot = _stub("matplotlib.pyplot")
    for n in ("Mapping", "MutableMapping", "Iterable"):
        if not hasattr(collections, n):
            setattr(collections, n, getattr(collections.abc, n))
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)
    import generalframework  # noqa: F401
    return generalframework
