"""Exact Euclidean distance maps on the device: ``distance_transform_edt`` (scipy's function for a batch of binary
masks) and ``signed_distance_map`` (one signed map per class of a class map).  Backed by ``dct_distance_map_i64``
(``csrc/dct_hausdorff.cu``, the separable distance passes of the Hausdorff metrics); DESIGN.md §3.14.
"""
import ctypes

import torch

from . import _lib, _runtime
from .metrics import _prediction_map


def _spacing(values, method, what):
    """The spacing as a ctypes double array (``None`` = ones): a scalar for every axis, or one value per grid axis."""
    if values is None:
        return None
    n = 3 if method == '3d' else 2
    vals = [float(values)] * n if isinstance(values, (int, float)) else [float(v) for v in values]
    assert len(vals) == n, f"{what}: spacing for '{method}' has {n} values, got {vals}"
    return (ctypes.c_double * n)(*vals)


def _distance_map(m, C, first_class, method, sp, signed_map, what):
    assert method in ('2d', '3d')
    assert 0 <= first_class < C, f"{what}: no class to compute (C={C}, first_class={first_class})"
    B, H, W = m.shape
    volume = int(method == '3d')
    h = _lib.lib()
    nbytes = h.dct_distance_map_scratch_bytes(C, first_class, B, H, W, volume, int(signed_map))
    if nbytes == 0:
        _lib.check(_lib.ERR_UNSUPPORTED, f"{what}: dct_distance_map_scratch_bytes (C={C}, shape {(B, H, W)})")
    scratch = torch.empty(nbytes, dtype=torch.uint8, device=m.device)
    out = torch.empty((B, C - first_class, H, W), dtype=torch.float32, device=m.device)
    st = _runtime.state(m.device)
    _lib.check(h.dct_distance_map_i64(m.data_ptr(), C, first_class, B, H, W, volume, sp, int(signed_map),
                                      out.data_ptr(), _runtime.flags_ptr(st), scratch.data_ptr(),
                                      _runtime.stream_ptr(m.device)), "dct_distance_map_i64")
    _runtime.after_call(st)
    return out


def distance_transform_edt(input, sampling=None, method='2d') -> torch.Tensor:
    """``scipy.ndimage.distance_transform_edt`` of a batch of masks on the device: float32 ``[B,H,W]``.

    ``input``: a CUDA tensor ``[B,H,W]`` or ``[B,1,H,W]`` of any dtype; nonzero is foreground.  Each foreground pixel gets
    its distance to the nearest background pixel of its grid, ``min ||(x - y) * sampling||_2``; background pixels get 0.
    ``'2d'`` takes every ``[H,W]`` slice as its own grid, ``'3d'`` the batch as one ``[B,H,W]`` volume.  ``sampling``:
    ``None`` (ones), a scalar, or ``(sy, sx)`` / ``(sz, sy, sx)``, as scipy's argument of that name.  Cells off the grid are
    not background, as in scipy.

    Where scipy differs: a grid with no background pixel has no defined distance; here its pixels are +inf, while scipy
    returns an artifact of its feature transform (``[[1, 1.414, 2.236, 3.162]]`` for an all-true 1 x 4 array).  At unit
    spacing every value is scipy's float64 value rounded to float32, bit for bit; otherwise within 1e-6 relative.
    ``return_distances`` / ``return_indices`` are not offered: this returns the distances only.
    """
    _runtime.require_cuda(input, "distance_transform_edt")
    if input.dim() == 4 and input.shape[1] == 1:
        input = input[:, 0]
    assert input.dim() == 3, f"distance_transform_edt: [B,H,W] or [B,1,H,W] expected, got {tuple(input.shape)}"
    m = (input != 0).to(torch.int64).contiguous()
    sp = _spacing(sampling, method, "distance_transform_edt")
    return _distance_map(m, 2, 1, method, sp, False, "distance_transform_edt")[:, 0]


def signed_distance_map(pred, C=None, method='2d', voxelspacing=None, include_background=True) -> torch.Tensor:
    """Signed Euclidean distance map of every class: float32 ``[B, C, H, W]`` (``[B, C - 1, H, W]`` without class 0).

    ``pred``: float32 scores ``[B,C,H,W]`` (reduced with the arg-max ``DiceMeter.add`` uses) or an integer class map
    ``[B,H,W]`` / ``[B,1,H,W]`` (then ``C`` is required), as for ``hausdorff``.  ``'2d'`` takes every ``[H,W]`` slice as its
    own grid, ``'3d'`` the batch as one ``[B,H,W]`` volume; ``voxelspacing``: ``(sy, sx)`` / ``(sz, sy, sx)``, ``None`` =
    ones.  With ``in_c = {map == c}``, ``out_c`` its complement on the grid and ``d(x, S)`` the smallest scaled distance
    to a pixel of ``S`` on the grid (scipy's EDT semantics)::

        phi_c(x) = d(x, in_c) for x in out_c,   -d(x, out_c) for x in in_c

    positive outside, negative inside, no offset or normalisation.  A grid on which ``in_c`` or ``out_c`` is empty (the
    class is absent, or fills it) has no boundary: ``phi_c`` is 0 there.  Values outside ``[0, C)`` belong to no class
    (``out_c`` for every c) and raise the prediction range check under the current check mode.  At unit spacing every
    value is the float32 of ``scipy.ndimage.distance_transform_edt`` on the corresponding mask, bit for bit; otherwise
    within 1e-6 relative.

    The usual training targets are plain torch over ``phi``, for example the boundary loss's map (distance outside,
    offset by one inside) and a DTC-style target normalised per (image, class) to ``[-1, 1]``::

        bl = torch.where(phi < 0, phi + 1, phi)
        dtc = torch.where(phi < 0, phi / -phi.amin((2, 3), keepdim=True), phi / phi.amax((2, 3), keepdim=True)).nan_to_num(0)

    (written from the papers' definitions, not checked against those repositories).
    """
    assert method in ('2d', '3d')
    m, C = _prediction_map(pred, C, "signed_distance_map")
    sp = _spacing(voxelspacing, method, "signed_distance_map")
    return _distance_map(m, C, 0 if include_background else 1, method, sp, True, "signed_distance_map")
