"""Connected components of a predicted class map on the device: labels, per-class statistics, and the largest component
per class (the ``getLargestCC`` post-processing of the UA-MT / DTC / MC-Net test scripts; nnU-Net's "remove all but the
largest component").  Backed by ``dct_components_i64`` (``csrc/dct_components.cu``); DESIGN.md §3.12.
"""
import torch

from . import _lib, _runtime
from .metrics import _prediction_map


def _components(pred, C, method, connectivity, what, want_labels, want_stats, want_largest):
    assert method in ('2d', '3d')
    p, C = _prediction_map(pred, C, what)
    B, H, W = p.shape
    volume = method == '3d'
    h = _lib.lib()
    nbytes = h.dct_components_scratch_bytes(C, B, H, W, int(volume))
    if nbytes == 0:
        _lib.check(_lib.ERR_UNSUPPORTED, f"dct_components_scratch_bytes (C={C}, shape {(B, H, W)})")
    scratch = torch.empty(nbytes, dtype=torch.uint8, device=p.device)
    labels = torch.empty((B, H, W), dtype=torch.int32, device=p.device) if want_labels else None
    stats = torch.empty((1 if volume else B, C, 2), dtype=torch.int64, device=p.device) if want_stats else None
    largest = torch.empty_like(p) if want_largest else None
    st = _runtime.state(p.device)
    _lib.check(h.dct_components_i64(p.data_ptr(), C, B, H, W, int(volume), int(connectivity),
                                    None if labels is None else labels.data_ptr(),
                                    None if stats is None else stats.data_ptr(),
                                    None if largest is None else largest.data_ptr(),
                                    _runtime.flags_ptr(st), scratch.data_ptr(), _runtime.stream_ptr(p.device)),
               "dct_components_i64")
    _runtime.after_call(st)
    return labels, stats, largest


def connected_components(pred, C=None, method='2d', connectivity=1) -> dict:
    """Connected components of every class: ``{'labels', 'count', 'largest'}`` on the input's device.

    ``pred``: float32 scores ``[B,C,H,W]`` (reduced with the arg-max ``DiceMeter.add`` uses) or an integer class map
    ``[B,H,W]`` / ``[B,1,H,W]`` (then ``C`` is required), as for ``hausdorff``.  ``'2d'`` labels every ``[H,W]`` slice on
    its own (adjacency never crosses slices); ``'3d'`` labels the batch as one ``[B,H,W]`` volume.  ``connectivity`` is
    that of ``scipy.ndimage.generate_binary_structure``: for ``'2d'`` 1 = 4 neighbours, 2 = 8; for ``'3d'`` 1 = 6, 2 = 18,
    3 = 26.  The default, 1, is ``scipy.ndimage.label``'s and nnU-Net's; ``skimage.measure.label`` (which ``getLargestCC``
    uses) defaults to full connectivity: 2 for ``'2d'``, 3 for ``'3d'``.

    Two pixels are in one component when they hold the same class and are joined through neighbours of that class;
    every class, 0 included, is labelled.
      ``labels``  int32 ``[B,H,W]``: the linear index in the ``[B,H,W]`` tensor of the component's first pixel in raster
                  order (its smallest index; scipy numbers components in the same order), -1 for a value outside
                  ``[0, C)``.
      ``count``   int64 ``[rows, C]``: number of components per class (``rows`` = B for ``'2d'``, 1 for ``'3d'``).
      ``largest`` int64 ``[rows, C]``: size in pixels of the largest component, 0 for an absent class.
    Values outside ``[0, C)`` belong to no component and raise the prediction range check under the current check mode.
    Every output is an exact integer, the same from call to call.
    """
    labels, stats, _ = _components(pred, C, method, connectivity, "connected_components", True, True, False)
    return {'labels': labels, 'count': stats[..., 0], 'largest': stats[..., 1]}


def largest_component(pred, C=None, method='2d', connectivity=1) -> torch.Tensor:
    """The class map with every class c >= 1 cut down to its largest connected component on each grid: int64
    ``[B,H,W]``, pixels of c outside that component set to 0.  Class 0 is never filtered; ties go to the component whose
    first pixel comes first in raster order (``np.argmax(np.bincount(labels.flat)[1:])`` on scipy's labels); values
    outside ``[0, C)`` are copied unchanged.  Arguments, grids and connectivity as for ``connected_components``.

    The usual post-processing before the surface distances, in one line::

        sd = surface_distances(largest_component(logits, method='3d'), gt, C=4, method='3d', voxelspacing=sp)
    """
    return _components(pred, C, method, connectivity, "largest_component", False, False, True)[2]
