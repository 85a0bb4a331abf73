"""Hausdorff distance oracle (test infrastructure): the definition of ``medpy.metric.binary.hd`` restated with scipy, and a
brute-force form it is checked against.

medpy (``medpy/metric/binary.py``): ``hd(result, reference, voxelspacing, connectivity=1)`` is
``max(__surface_distances(result, reference).max(), __surface_distances(reference, result).max())``, where
``__surface_distances`` takes the border of each mask as ``mask ^ binary_erosion(mask, structure=generate_binary_structure(
ndim, 1), iterations=1)`` (scipy's default ``border_value=0``: the outside of the grid is background) and reads
``distance_transform_edt(~reference_border, sampling=voxelspacing)`` at the result's border pixels.  medpy raises
``RuntimeError`` when either mask is empty; here the value is NaN.

Per class c of integer maps: ``'2d'`` applies it to every slice ``[H,W]`` of a ``[B,H,W]`` batch (rows = B), ``'3d'`` to
the batch as one volume (one row).  Values outside ``[0,C)`` belong to no class.
"""
import numpy as np
from scipy.ndimage import binary_erosion, distance_transform_edt, generate_binary_structure
from scipy.spatial.distance import cdist


def border(mask: np.ndarray) -> np.ndarray:
    return mask ^ binary_erosion(mask, structure=generate_binary_structure(mask.ndim, 1), iterations=1)


def hd_binary(a: np.ndarray, g: np.ndarray, spacing=None) -> float:
    """medpy.metric.binary.hd(a, g, voxelspacing=spacing), NaN for an empty mask."""
    a, g = a.astype(bool), g.astype(bool)
    if not a.any() or not g.any():
        return float("nan")
    sp = None if spacing is None else np.asarray(spacing, dtype=np.float64)
    ba, bg = border(a), border(g)
    d_to_g = distance_transform_edt(~bg, sampling=sp)
    d_to_a = distance_transform_edt(~ba, sampling=sp)
    return float(max(d_to_g[ba].max(), d_to_a[bg].max()))


def hd_binary_brute(a: np.ndarray, g: np.ndarray, spacing=None) -> float:
    """The same from the border coordinates: all pairwise distances (argwhere + cdist)."""
    a, g = a.astype(bool), g.astype(bool)
    if not a.any() or not g.any():
        return float("nan")
    sp = np.ones(a.ndim) if spacing is None else np.asarray(spacing, dtype=np.float64)
    pa, pg = np.argwhere(border(a)) * sp, np.argwhere(border(g)) * sp
    d = cdist(pa, pg)
    return float(max(d.min(1).max(), d.min(0).max()))


def hausdorff(pred: np.ndarray, gt: np.ndarray, C: int, method: str = "2d", spacing=None, brute: bool = False) -> np.ndarray:
    """float64 ``[rows, C]`` for integer maps ``[B,H,W]`` (rows = B for '2d', 1 for '3d')."""
    assert method in ("2d", "3d") and pred.shape == gt.shape and pred.ndim == 3
    f = hd_binary_brute if brute else hd_binary
    grids = [(pred, gt)] if method == "3d" else [(pred[b], gt[b]) for b in range(pred.shape[0])]
    return np.array([[f(p == c, g == c, spacing) for c in range(C)] for p, g in grids], dtype=np.float64)


def blobs(rng: np.random.Generator, shape, C: int, smooth: float = 4.0) -> np.ndarray:
    """Smooth random class map: arg-max over C low-pass-filtered noise fields (per slice for a [B,H,W] shape)."""
    from scipy.ndimage import gaussian_filter
    noise = rng.standard_normal((C,) + tuple(shape))
    sig = (0,) + (0,) * (len(shape) - 2) + (smooth, smooth)
    return gaussian_filter(noise, sigma=sig).argmax(0).astype(np.int64)


def salt_pepper(rng: np.random.Generator, shape, C: int) -> np.ndarray:
    """Independent uniform classes per pixel: almost every pixel is a border pixel."""
    return rng.integers(0, C, size=shape, dtype=np.int64)
