"""GPU: the evaluation-path distance and component kernels at the limits their ABI accepts.

* Unit spacing past 2^24.  A squared distance of 4096 pixels or more is no longer exact in float, so the distance passes
  carry d^2 as an exact integer at unit spacing.  Single-pixel masks at offsets where rounding d^2 (or the volume's
  intermediate d^2 after the row pass) to float would change hd, hd95, asd or the surface-Dice counts; the offsets are
  chosen here by emulating the float arithmetic, and the reference is the exact integer d^2, square-rooted in double and
  rounded once to float32.
* Long and thin grids against the scipy oracles (all four entry points, unit and anisotropic spacing): lines longer than
  12288 positions, which launch_envelope runs as one line per CTA with more than 48 KiB of shared memory, axes of 32768
  (the largest that 16-bit stack entries and column distances hold), and a column distance of 32767.
* Connected components on N x 1 x 1 and 1 x 1 x N grids (tiles grown along the long axis) and on 2^31 - 43707 pixels,
  where every index is close to the int32 limit."""
import math

import numpy as np
import pytest
import torch

import oracle_components as OC
import oracle_surface as OS
import oracle_surface_dice as OD
from test_gpu_components import assert_equal_to_oracle, run as run_components
from test_gpu_surface_dice import assert_matches as assert_nsd_matches, assert_ratios, counts_of, near_counts
from test_gpu_surface_distance import assert_matches as assert_surface_matches

pytestmark = pytest.mark.gpu

SPACING = {"2d": (1.5625, 1.25), "3d": (10.0, 1.5625, 1.25)}
METHOD_CONN = {"2d": (1, 2), "3d": (1, 2, 3)}


@pytest.fixture(scope="module")
def dct():
    import dct_b200
    assert torch.cuda.is_available()
    return dct_b200


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda:0")


def T(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def bits(t):
    return t.detach().cpu().numpy().view(np.uint32)


# ---- exactness at unit spacing past 2^24 --------------------------------------------------------------------------------

def f32(x):
    """Round to float32 (elementwise), as a float64 value."""
    return np.asarray(x, dtype=np.float64).astype(np.float32).astype(np.float64)


def float_path(d2, f=None):
    """d^2 as float arithmetic would leave it: rounded once, or (a volume's depth pass) the row-pass intermediate `f`
    rounded first and the sum rounded again."""
    return f32(d2) if f is None else f32(f32(f) + (np.asarray(d2) - np.asarray(f)))


def exact_hd(d2):
    """float32 of the exact distance (what hd, hd95, asd and assd of one pixel pair must be)."""
    return np.sqrt(np.asarray(d2, dtype=np.float64)).astype(np.float32)


def float_hd(d2f):
    return np.sqrt(np.asarray(d2f).astype(np.float32))   # correctly rounded float square root of the float d^2


def within_floor(d2, d2f):
    """(exact, float-path) verdicts of `distance <= floor(distance)`, the NSD test at tolerance floor(sqrt(d^2))."""
    k = np.floor(np.sqrt(np.asarray(d2, dtype=np.float64)))
    return np.asarray(d2) <= k * k, np.sqrt(d2f) <= k


def first_offset(short, long, wrong):
    """First (s, l) in raster order over short x long for which `wrong(d2, d2f)` holds, d2 = s^2 + l^2 rounded once."""
    s, l = np.meshgrid(np.asarray(short, np.int64), np.asarray(long, np.int64), indexing="ij")
    d2 = s * s + l * l
    bad = wrong(d2, float_path(d2))
    i, j = np.argwhere(bad)[0]
    return int(s[i, j]), int(l[i, j])


def hd_wrong(d2, d2f):
    return exact_hd(d2) != float_hd(d2f)


def nsd_wrong(d2, d2f):
    a, b = within_floor(d2, d2f)
    return a != b


def _offset_cases():
    """(name, metric, method, grid shape, label pixel, prediction pixel); the label pixel is the grid's origin."""
    w_nsd, w_hd = (1, 4100), (3, 5462)   # (dy, dx) on a slice
    assert nsd_wrong(np.int64(w_nsd[0] ** 2 + w_nsd[1] ** 2), float_path(w_nsd[0] ** 2 + w_nsd[1] ** 2))
    assert hd_wrong(np.int64(w_hd[0] ** 2 + w_hd[1] ** 2), float_path(w_hd[0] ** 2 + w_hd[1] ** 2))
    # an attained integer distance k whose float k^2 rounds above k^2 (the tolerance k then excludes it)
    k_att = first_offset([0], range(4096, 32768), nsd_wrong)[1]
    # split across W and the depth: the row pass leaves dx^2 > 2^24 in the intermediate, the depth pass adds dz^2; chosen
    # so that rounding the intermediate alone breaks the metric, while rounding only the final d^2 would not
    split = {}
    for metric, base in (("hd", hd_wrong), ("nsd", nsd_wrong)):
        dz, dx = np.meshgrid(np.arange(1, 64, dtype=np.int64), np.arange(4097, 8192, dtype=np.int64), indexing="ij")
        d2, f = dz * dz + dx * dx, dx * dx
        teeth = (base(d2, float_path(d2, f)) & base(d2, np.round(f32(f)) + dz * dz)   # the float intermediate breaks it
                 & ~base(d2, f32(d2)))                                                # one rounding of d^2 would not
        i, j = np.argwhere(teeth)[0]
        split[metric] = (int(dz[i, j]), int(dx[i, j]))
    out = []
    for metric, (s, l) in (("nsd", w_nsd), ("hd", w_hd), ("nsd_attained", (0, k_att))):
        out.append((f"W_{metric}_{s}_{l}", metric, "2d", (1, s + 1, l + 1), (0, s, l)))
        out.append((f"H_{metric}_{l}_{s}", metric, "2d", (1, l + 1, s + 1), (0, l, s)))
        out.append((f"depth_{metric}_{l}_{s}", metric, "3d", (l + 1, s + 1, 1), (l, s, 0)))
    for metric, (dz, dx) in split.items():
        out.append((f"split_{metric}_{dz}_{dx}", metric, "3d", (dz + 1, 1, dx + 1), (dz, 0, dx)))
    return out


OFFSET_CASES = _offset_cases()


@pytest.mark.parametrize("case", OFFSET_CASES, ids=lambda c: c[0])
def test_unit_spacing_exact_past_2_24(case, dct, dev):
    name, metric, method, shape, pix = case
    d2 = sum(v * v for v in pix)
    assert d2 > 2 ** 24
    # the case has teeth: float arithmetic would get this metric wrong
    d2f = float_path(d2, pix[2] ** 2 if name.startswith("split") else None)
    if metric == "hd":
        assert exact_hd(d2) != float_hd(d2f)
    else:
        assert nsd_wrong(np.int64(d2), d2f)
    C = 2
    g = np.zeros(shape, np.int64); g[0, 0, 0] = 1
    p = np.zeros(shape, np.int64); p[pix] = 1
    pt, gt = T(p, dev), T(g, dev)
    want_d = exact_hd(d2)
    want = OS.surface(p, g, C, method)
    assert want["hd"][0, 1].astype(np.float32) == want_d   # scipy's EDT is exact here too
    hd = dct.hausdorff(pt, gt, C=C, method=method)
    sd = dct.surface_distances(pt, gt, C=C, method=method)
    assert np.array_equal(bits(hd), bits(sd["hd"]))
    for k in OS.KEYS:   # one border pixel per side: every statistic is the distance itself
        assert bits(sd[k][0, 1]) == np.float32(want_d).view(np.uint32), k
    assert_surface_matches(sd, want, True)
    k = math.isqrt(d2)
    dists = OD.distances(p, g, C, method)
    for tol in (k, math.sqrt(d2), k - 1, k + 1):
        got = dct.surface_dice(pt, gt, float(tol), C=C, method=method)
        within = int(d2 <= tol * tol) if tol != math.sqrt(d2) else 1
        assert got["counts"][0, 1].tolist() == [within, 1, within, 1], tol
        assert_nsd_matches(got, dists, [float(tol)] * C)
    # explicit unit spacing takes the same exact path
    for sp in ((1.0,) * (3 if method == "3d" else 2),):
        assert np.array_equal(bits(dct.hausdorff(pt, gt, C=C, method=method, voxelspacing=sp)), bits(hd))
        got = dct.surface_dice(pt, gt, float(k), C=C, method=method, voxelspacing=sp)
        assert got["counts"][0, 1].tolist() == [int(d2 == k * k), 1, int(d2 == k * k), 1]


# ---- long and thin grids ------------------------------------------------------------------------------------------------

# launch_envelope gives a pass over lines of n positions R = clamp(48 KiB / 4n, 1, 64) lines per CTA
LONG_GRIDS = [
    ((2, 48, 16384), "2d"),    # row pass n = 16384 > 12288: R = 1, 64 KiB of shared memory (opt-in)
    ((1, 24, 32768), "2d"),    # row pass n = 32768, the largest axis: R = 1, 128 KiB
    ((1, 32768, 24), "2d"),    # column pass over 32768 rows (distances up to 32767 in uint16); row pass n = 24, R = 64
    ((16384, 6, 5), "3d"),     # depth pass n = 16384: R = 1, 64 KiB; row pass n = 5, R = 64
    ((32768, 2, 3), "3d"),     # depth pass n = 32768: R = 1, 128 KiB
]
LONG_C = 4
LONG_TOLS = [0.0, 1.0, math.sqrt(2), 4096.0, 10000.0, 32767.0]
ANISO_TOLS = [0.0, 1.25, 4096.0, 20000.0]


def long_axis(shape, method):
    return 0 if method == "3d" else 1 + int(np.argmax(shape[1:]))


def long_maps(shape, method, seed):
    """Sparse classes on background 0: islands of classes 1 and 2 of up to 3 pixels a side, a third of them near either
    end of the long axis, so that distances pass 4096; class 3 is one pixel at each end of the long axis in the first
    grid, the label's at the start and the prediction's at the end (for H = 32768 its column holds nothing else: the
    column distance reaches 32767)."""
    rng = np.random.default_rng(seed)
    ax = long_axis(shape, method)
    L = shape[ax]
    out = []
    for side in range(2):
        m = np.zeros(shape, np.int64)
        for c in (1, 2):
            for _ in range(12):
                lo = [int(rng.integers(0, n)) for n in shape]
                r = rng.random()
                if r < 1 / 3:
                    lo[ax] = int(rng.integers(0, 16))
                elif r < 2 / 3:
                    lo[ax] = L - 1 - int(rng.integers(0, 16))
                if method == "2d":
                    lo[0] = int(rng.integers(0, shape[0]))
                ext = [1 if (method == "2d" and i == 0) else int(rng.integers(1, 4)) for i in range(3)]
                m[tuple(slice(a, a + e) for a, e in zip(lo, ext))] = c
        at = [0, shape[1] // 3, shape[2] // 3]
        at[ax] = L - 1 if side == 0 else 0
        m[tuple(at)] = 3
        out.append(m)
    return out[0], out[1]   # prediction, label


@pytest.mark.parametrize("unit", [True, False], ids=["unit", "aniso"])
@pytest.mark.parametrize("shape,method", LONG_GRIDS, ids=lambda v: "x".join(map(str, v)) if isinstance(v, tuple) else v)
def test_long_grids_vs_oracle(shape, method, unit, dct, dev):
    C = LONG_C
    p, g = long_maps(shape, method, seed=sum(shape))
    sp = None if unit else SPACING[method]
    pt, gt = T(p, dev), T(g, dev)
    want = OS.surface(p, g, C, method, sp)
    ax = long_axis(shape, method)
    assert np.nanmax(want["hd"]) > 4096   # the distances pass 4096 pixels
    assert want["hd"][0, 3] == pytest.approx((shape[ax] - 1) * (1.0 if unit else SPACING[method][ax - (method == "2d")]))
    sd = dct.surface_distances(pt, gt, C=C, method=method, voxelspacing=sp)
    assert np.array_equal(bits(sd["hd"]), bits(dct.hausdorff(pt, gt, C=C, method=method, voxelspacing=sp)))
    assert_surface_matches(sd, want, unit)
    dists = OD.distances(p, g, C, method, sp)
    for tau in (LONG_TOLS if unit else ANISO_TOLS):
        got = dct.surface_dice(pt, gt, tau, C=C, method=method, voxelspacing=sp)
        if unit:
            assert_nsd_matches(got, dists, [tau] * C)
            continue
        c = got["counts"].cpu().numpy()
        want_c = counts_of(dists, [tau] * C)
        np.testing.assert_array_equal(c[..., 1::2], want_c[..., 1::2])
        assert np.all(np.abs(c[..., 0::2] - want_c[..., 0::2]) <= near_counts(dists, [tau] * C)), tau
        assert_ratios(got, c)
    if unit:
        for m in (p, g):
            for conn in METHOD_CONN[method]:
                assert_equal_to_oracle(run_components(dct, m, C, method, conn, dev), m, C, method, conn)


# ---- components on thin grids and near 2^31 - 1 pixels ------------------------------------------------------------------

def runs_map(n, C, seed):
    """Runs of 1 to 8 pixels of random classes along a line of n pixels."""
    rng = np.random.default_rng(seed)
    return np.repeat(rng.integers(0, C, size=n), rng.integers(1, 9, size=n))[:n].astype(np.int64)


@pytest.mark.parametrize("shape,method", [((1, 1, 1 << 20), "2d"), ((1, 1 << 20, 1), "2d"), ((1 << 20, 1, 1), "3d"),
                                          ((3, 1, 1 << 18), "2d")])
def test_components_thin_grids(shape, method, dct, dev):
    C = 3
    m = runs_map(int(np.prod(shape)), C, seed=len(shape) + shape[0]).reshape(shape)
    for conn in METHOD_CONN[method]:
        got = run_components(dct, m, C, method, conn, dev)
        assert_equal_to_oracle(got, m, C, method, conn)


def test_components_near_int32_limit(dct, dev):
    """1 x 46340 x 46341 = 2^31 - 43707 pixels of width-1 vertical stripes (class x % 2): at connectivity 1 and 2 every
    column is one component of H pixels whose label is its column index x, so the class-1 winner is column 1.  Checked
    on the device, row block by row block."""
    h = dct._lib.lib()
    C, B, H, W = 2, 1, 46340, 46341
    N = B * H * W
    assert N <= 2 ** 31 - 1 and N + W > 2 ** 31 - 1
    nbytes = h.dct_components_scratch_bytes(C, B, H, W, 0)
    assert nbytes > 0
    free, _ = torch.cuda.mem_get_info(dev)
    margin = 1 << 30
    need_small = 8 * N + 4 * N + nbytes + margin            # map, labels, scratch
    with_largest = free >= need_small + 8 * N
    if free < need_small:
        pytest.skip(f"needs {need_small / 2 ** 30:.1f} GiB of free device memory, {free / 2 ** 30:.1f} GiB free")
    print(f"\ncomponents at {N} pixels: {free / 2 ** 30:.1f} GiB free, largest_map {'checked' if with_largest else 'skipped'}")
    xs = torch.arange(W, device=dev)
    m = (xs % 2).expand(H, W).contiguous()
    labels = torch.empty((H, W), dtype=torch.int32, device=dev)
    stats = torch.empty((1, C, 2), dtype=torch.int64, device=dev)
    largest = torch.empty((H, W), dtype=torch.int64, device=dev) if with_largest else None
    scratch = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    stream = torch.cuda.current_stream(dev).cuda_stream
    want_labels = xs.to(torch.int32)
    want_largest = (xs == 1).to(torch.int64)
    try:
        for conn in (1, 2):
            labels.fill_(-7); stats.fill_(-7)
            if largest is not None:
                largest.fill_(-7)
            rc = h.dct_components_i64(m.data_ptr(), C, B, H, W, 0, conn, labels.data_ptr(), stats.data_ptr(),
                                      None if largest is None else largest.data_ptr(), None, scratch.data_ptr(), stream)
            assert rc == 0
            torch.cuda.synchronize(dev)
            assert stats[0].tolist() == [[(W + 1) // 2, H], [W // 2, H]], conn
            for y0 in range(0, H, 2048):
                y1 = min(y0 + 2048, H)
                assert torch.equal(labels[y0:y1], want_labels.expand(y1 - y0, W)), (conn, y0)
                if largest is not None:
                    assert torch.equal(largest[y0:y1], want_largest.expand(y1 - y0, W)), (conn, y0)
    finally:
        del m, labels, stats, largest, scratch
        torch.cuda.empty_cache()
