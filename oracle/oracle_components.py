"""Connected-component oracle (test infrastructure): ``dct_components_i64`` restated with ``scipy.ndimage.label``, and an
independent breadth-first flood fill it is checked against.

Per class c of an integer map ``[B,H,W]`` and per grid (every slice for ``'2d'``, the batch as one volume for ``'3d'``):
``scipy.ndimage.label(grid == c, structure=generate_binary_structure(rank, connectivity))``.  scipy numbers components in
the raster order of their first pixels, so label k's first pixel is the first pixel of the mask holding k.  Outputs:
  labels  int32 ``[B,H,W]``: linear index in the batch tensor of the component's first pixel, -1 outside ``[0, C)``;
  stats   int64 ``[rows, C, 2]``: (number of components, size of the largest), (0, 0) for an absent class;
  largest int64 ``[B,H,W]``: pixels of c >= 1 outside the component ``np.argmax(np.bincount(lab.flat)[1:]) + 1`` set to 0
          (the first of equal sizes), class 0 and values outside ``[0, C)`` unchanged.
"""
from collections import deque
from itertools import product

import numpy as np
from scipy.ndimage import generate_binary_structure, label


def _grids(shape, method):
    """(index into the batch, rank) of every grid: one per slice for '2d', the whole batch for '3d'."""
    if method == "3d":
        return [(np.s_[:, :, :], 3)]
    return [(np.s_[b:b + 1, :, :], 2) for b in range(shape[0])]


def components(m: np.ndarray, C: int, method: str = "2d", connectivity: int = 1):
    """(labels, stats, largest) of an integer class map ``[B,H,W]``."""
    assert method in ("2d", "3d") and m.ndim == 3
    assert 1 <= connectivity <= (3 if method == "3d" else 2)
    m = np.asarray(m, dtype=np.int64)
    grids = _grids(m.shape, method)
    labels = np.full(m.shape, -1, dtype=np.int32)
    stats = np.zeros((len(grids), C, 2), dtype=np.int64)
    largest = m.copy()
    index = np.arange(m.size, dtype=np.int64).reshape(m.shape)
    for row, (sl, rank) in enumerate(grids):
        grid, idx = m[sl], index[sl]
        if rank == 2:
            grid, idx = grid[0], idx[0]
        structure = generate_binary_structure(rank, connectivity)
        for c in range(C):
            mask = grid == c
            lab, n = label(mask, structure=structure)
            if n == 0:
                continue
            flat = lab[mask]                                   # raster order
            _, first = np.unique(flat, return_index=True)      # first occurrence of labels 1..n
            first_index = idx[mask][first]                     # ascending, as scipy numbers in raster order
            assert np.all(np.diff(first_index) > 0)
            out = labels[sl][0] if rank == 2 else labels[sl]
            out[mask] = first_index[flat - 1].astype(np.int32)
            sizes = np.bincount(lab.ravel())[1:]
            stats[row, c] = (n, sizes.max())
            if c >= 1:
                keep = np.argmax(sizes) + 1
                big = largest[sl][0] if rank == 2 else largest[sl]
                big[mask & (lab != keep)] = 0
    return labels, stats, largest


def _neighbours(rank: int, connectivity: int):
    """Offsets of the neighbourhood: not all zero, at most ``connectivity`` non-zero entries."""
    return [d for d in product((-1, 0, 1), repeat=rank) if 0 < sum(map(abs, d)) <= connectivity]


def components_bfs(m: np.ndarray, C: int, method: str = "2d", connectivity: int = 1):
    """The same outputs from a breadth-first flood fill, scanning pixels in raster order (slow; small grids only)."""
    m = np.asarray(m, dtype=np.int64)
    B, H, W = m.shape
    volume = method == "3d"
    offs = [(0,) + d for d in _neighbours(2, connectivity)] if not volume else _neighbours(3, connectivity)
    labels = np.full(m.shape, -1, dtype=np.int32)
    rows = 1 if volume else B
    comps = [[[] for _ in range(C)] for _ in range(rows)]   # per (row, class): (first index, size) in discovery order
    for start in range(m.size):
        z, y, x = np.unravel_index(start, m.shape)
        c = m[z, y, x]
        if not (0 <= c < C) or labels[z, y, x] >= 0:
            continue
        labels[z, y, x] = start
        todo, size = deque([(z, y, x)]), 0
        while todo:
            pz, py, px = todo.popleft()
            size += 1
            for dz, dy, dx in offs:
                q = (pz + dz, py + dy, px + dx)
                if 0 <= q[0] < B and 0 <= q[1] < H and 0 <= q[2] < W and m[q] == c and labels[q] < 0:
                    labels[q] = start
                    todo.append(q)
        comps[0 if volume else z][c].append((start, size))
    stats = np.zeros((rows, C, 2), dtype=np.int64)
    largest = m.copy()
    for r in range(rows):
        for c in range(C):
            found = comps[r][c]
            if not found:
                continue
            best = max(found, key=lambda fs: (fs[1], -fs[0]))   # largest, then first in raster order
            stats[r, c] = (len(found), best[1])
            if c >= 1:
                sl = np.s_[:] if volume else np.s_[r]
                largest[sl][(m[sl] == c) & (labels[sl] != best[0])] = 0
    return labels, stats, largest
