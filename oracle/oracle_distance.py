"""Distance map oracle (test infrastructure): the signed and inside Euclidean distance maps of a class map restated with
scipy's ``distance_transform_edt``, and a brute-force form it is checked against.

Per grid (every ``[H,W]`` slice for '2d', the ``[B,H,W]`` batch for '3d') and class c, with ``in_c = {map == c}``,
``out_c`` its complement on the grid and ``d(x, S)`` the smallest distance ``||(x - y) * spacing||_2`` to a pixel y of S
on the grid (cells off the grid are not features: scipy's EDT semantics):
  inside  ``d_in(x) = d(x, out_c)`` on ``in_c``, 0 elsewhere; +inf where ``out_c`` is empty (scipy returns an artifact of
          its feature transform there, so that case is written out);
  signed  ``phi(x) = d(x, in_c)`` on ``out_c``, ``-d(x, out_c)`` on ``in_c``; all 0 where ``in_c`` or ``out_c`` is empty.
Values outside ``[0, C)`` belong to no class (they are in ``out_c`` for every c).
"""
import numpy as np
from scipy.ndimage import distance_transform_edt
from scipy.spatial.distance import cdist


def _edt(mask: np.ndarray, spacing) -> np.ndarray:
    """d(x, ~mask) for x in mask, 0 elsewhere; +inf on mask where ~mask is empty."""
    if mask.all():
        return np.full(mask.shape, np.inf)
    return distance_transform_edt(mask, sampling=None if spacing is None else np.asarray(spacing, np.float64))


def _edt_brute(mask: np.ndarray, spacing) -> np.ndarray:
    sp = np.ones(mask.ndim) if spacing is None else np.asarray(spacing, dtype=np.float64)
    out = np.zeros(mask.shape)
    inside, feats = np.argwhere(mask), np.argwhere(~mask)
    if len(inside):
        out[mask] = cdist(inside * sp, feats * sp).min(1) if len(feats) else np.inf
    return out


def inside_binary(inside: np.ndarray, spacing=None, brute: bool = False) -> np.ndarray:
    """float64 d_in of one grid."""
    return (_edt_brute if brute else _edt)(inside.astype(bool), spacing)


def signed_binary(inside: np.ndarray, spacing=None, brute: bool = False) -> np.ndarray:
    """float64 phi of one grid."""
    inside = inside.astype(bool)
    if inside.all() or not inside.any():
        return np.zeros(inside.shape)
    f = _edt_brute if brute else _edt
    return f(~inside, spacing) - f(inside, spacing)


def distance_map(m: np.ndarray, C: int, first_class: int = 0, method: str = "2d", spacing=None, signed: bool = True,
                 brute: bool = False) -> np.ndarray:
    """float64 ``[B, C - first_class, H, W]`` for an integer map ``[B,H,W]``: phi (signed) or d_in per computed class."""
    assert method in ("2d", "3d") and m.ndim == 3 and 0 <= first_class < C
    f = signed_binary if signed else inside_binary
    out = np.zeros((m.shape[0], C - first_class) + m.shape[1:])
    for c in range(first_class, C):
        if method == "3d":
            out[:, c - first_class] = f(m == c, spacing, brute)
        else:
            for b in range(m.shape[0]):
                out[b, c - first_class] = f(m[b] == c, spacing, brute)
    return out
