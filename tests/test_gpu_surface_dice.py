"""GPU parity of the normalized surface Dice (dct_surface_dice_i64 through ``dct_b200.surface_dice`` /
``SurfaceDiceMeter``) against the scipy restatement (oracle/oracle_surface_dice.py).

At unit spacing the kernels carry every d^2 as the exact integer, so ``sqrt((double)d2) <= tol`` compares the same doubles
scipy's EDT gives: the counts equal the oracle's exactly, tolerances equal to attained distances included, and nsd and the overlaps are the
oracle's double ratios rounded to float32.  At anisotropic spacing d^2 is rounded to float, so a count may differ only by
the number of distances within 1e-6 relative of the tolerance; away from every attained distance the counts are exact."""
import ctypes
import math

import numpy as np
import pytest
import torch

import oracle_components as OC
import oracle_hausdorff as OH
import oracle_surface_dice as OD

pytestmark = pytest.mark.gpu

KEYS = OD.KEYS
SPACING = {"2d": (1.5625, 1.25), "3d": (10.0, 1.5625, 1.25)}
UNIT_TOLS = [0.0, 1.0, math.sqrt(2), 2.0, 3.5, math.sqrt(5)]
ANISO_TOLS = [0.0, 1.25, 1.5625, 2.0, 3.5, 10.0]
CASES = [((3, 17, 23), 2), ((3, 17, 23), 4), ((3, 17, 23), 19), ((5, 33, 47), 19),
         ((10, 256, 256), 4),      # ACDC patient
         ((8, 512, 512), 2),       # Spleen
         ((1, 512, 1024), 19)]     # one large image


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


def maps(shape, C, kind, seed):
    rng = np.random.default_rng(seed)
    make = OH.blobs if kind == "blobs" else OH.salt_pepper
    return make(rng, shape, C), make(rng, shape, C)


def counts_of(dists, tols):
    """int64 [rows, C, 4] from the oracle's distances (OD.distances) at per-class tolerances."""
    return np.array([[[int((s_pg <= tols[c]).sum()), s_pg.size, int((s_gp <= tols[c]).sum()), s_gp.size]
                      for c, (s_pg, s_gp) in enumerate(row)] for row in dists], dtype=np.int64)


def near_counts(dists, tols, rel=1e-6):
    """int64 [rows, C, 2]: distances within `rel` relative of the tolerance, per direction (pg, gp)."""
    return np.array([[[int((np.abs(s_pg - tols[c]) <= rel * tols[c]).sum()),
                       int((np.abs(s_gp - tols[c]) <= rel * tols[c]).sum())]
                      for c, (s_pg, s_gp) in enumerate(row)] for row in dists], dtype=np.int64)


def assert_ratios(got, counts):
    """nsd and the overlaps equal the double ratios of `counts`, rounded to float32, NaN where they are NaN."""
    want = np.array([[OD.ratios(cc) for cc in row] for row in counts], dtype=np.float64).reshape(counts.shape[:2] + (3,))
    for i, k in enumerate(KEYS):
        g = got[k].detach().cpu().numpy()
        assert g.dtype == np.float32 and g.shape == counts.shape[:2], k
        w = want[..., i].astype(np.float32)
        assert np.array_equal(g, w, equal_nan=True), (k, np.argwhere(~((g == w) | (np.isnan(g) & np.isnan(w))))[:4])


def assert_matches(got, dists, tols):
    c = got["counts"].cpu().numpy()
    want = counts_of(dists, tols)
    assert c.dtype == np.int64 and c.shape == want.shape
    np.testing.assert_array_equal(c, want)
    assert_ratios(got, c)


def away_tolerance(dists, near):
    """A tolerance near `near` with no attained distance within 1e-4 relative (midpoint of a gap of the distances)."""
    d = np.unique(np.hstack([np.hstack(p) for row in dists for p in row] + [np.zeros(1)]))
    d = d[np.isfinite(d)]
    gaps = [(abs((a + b) / 2 - near), (a + b) / 2) for a, b in zip(d[:-1], d[1:]) if b - a > 2e-4 * b]
    return min(gaps)[1] if gaps else near


@pytest.mark.parametrize("unit", [True, False], ids=["unit", "aniso"])
@pytest.mark.parametrize("method", ["2d", "3d"])
@pytest.mark.parametrize("kind", ["blobs", "saltpepper"])
@pytest.mark.parametrize("shape,C", CASES)
def test_surface_dice_vs_oracle(shape, C, kind, method, unit, dct, dev):
    p, g = maps(shape, C, kind, seed=C * 1000 + shape[1])
    sp = None if unit else SPACING[method]
    pt, gt = T(p, dev), T(g, dev)
    dists = OD.distances(p, g, C, method, sp)
    rows = 1 if method == "3d" else shape[0]
    for tau in (UNIT_TOLS if unit else ANISO_TOLS):
        tols = [tau] * C
        got = dct.surface_dice(pt, gt, tau, C=C, method=method, voxelspacing=sp)
        assert set(got) == set(KEYS) | {"counts"}
        assert all(got[k].shape == (rows, C) and got[k].device == dev for k in KEYS)
        assert got["counts"].shape == (rows, C, 4) and got["counts"].dtype == torch.int64
        if unit:
            assert_matches(got, dists, tols)
            continue
        c = got["counts"].cpu().numpy()
        want = counts_of(dists, tols)
        np.testing.assert_array_equal(c[..., 1::2], want[..., 1::2])     # |S_pg|, |S_gp|: no rounding involved
        assert np.all(np.abs(c[..., 0::2] - want[..., 0::2]) <= near_counts(dists, tols)), tau
        assert_ratios(got, c)
    if not unit:
        tau = away_tolerance(dists, 3.0)
        assert_matches(dct.surface_dice(pt, gt, tau, C=C, method=method, voxelspacing=sp), dists, [tau] * C)


def _edge_cases():
    out = []
    p = np.zeros((2, 6, 7), np.int64); g = np.zeros((2, 6, 7), np.int64)
    g[:, 2:4, 3] = 1; p[:, 1, 1] = 2
    out.append(("empty_pred_gt_both", p, g, 4))
    p = np.zeros((1, 9, 9), np.int64); g = np.zeros((1, 9, 9), np.int64)
    p[0, 3, 3] = 1; g[0, 4, 5] = 1
    out.append(("sqrt5_apart", p, g, 2))
    full = np.ones((2, 8, 10), np.int64); g = full.copy(); g[:, 3:5, 4:6] = 0; g[1, 0, :] = 0
    out.append(("whole_grid", full, g, 2))
    rng = np.random.default_rng(11)
    for shape in [(2, 1, 31), (3, 29, 1), (1, 1, 1), (2, 1, 1)]:
        out.append((f"line_{shape}", OH.salt_pepper(rng, shape, 3), OH.salt_pepper(rng, shape, 3), 3))
    m = OH.blobs(rng, (3, 40, 24), 4, smooth=2.0)
    out.append(("identical", m, m.copy(), 4))
    return out


@pytest.mark.parametrize("method", ["2d", "3d"])
@pytest.mark.parametrize("case", _edge_cases(), ids=lambda c: c[0])
def test_surface_dice_edge_cases(case, method, dct, dev):
    name, p, g, C = case
    pt, gt = T(p, dev), T(g, dev)
    dists = OD.distances(p, g, C, method)
    for tau in UNIT_TOLS:
        assert_matches(dct.surface_dice(pt, gt, tau, C=C, method=method), dists, [tau] * C)
    if name == "identical":
        got = dct.surface_dice(pt, gt, 0.0, C=C, method=method)
        present = got["counts"][..., 1] > 0
        assert bool(present.any()) and bool((got["nsd"][present] == 1.0).all())


def test_per_class_tolerances(dct, dev):
    C = 4
    p, g = maps((6, 80, 72), C, "blobs", seed=41)
    pt, gt = T(p, dev), T(g, dev)
    tols = [0.0, 1.0, math.sqrt(2), 3.5]
    for method in ("2d", "3d"):
        got = dct.surface_dice(pt, gt, tols, C=C, method=method)
        assert_matches(got, OD.distances(p, g, C, method), tols)
        for c, t in enumerate(tols):
            one = dct.surface_dice(pt, gt, t, C=C, method=method)
            assert torch.equal(got["counts"][:, c], one["counts"][:, c])
        as_tensor = dct.surface_dice(pt, gt, torch.tensor(tols, dtype=torch.float64), C=C, method=method)
        assert torch.equal(got["counts"], as_tensor["counts"])


@pytest.mark.parametrize("C", [2, 4, 19])
def test_scores_path_equals_class_map_path(C, dct, dev):
    gen = torch.Generator().manual_seed(C)
    x = (3 * torch.randn(3, C, 45, 38, generator=gen)).to(dev)
    x[0, :, 0, 0] = 0.0   # ties resolve as DiceMeter's arg-max does
    g = torch.randint(0, C, (3, 1, 45, 38), generator=gen).to(dev)
    cls = dct.utils._classmap(x, 1, want_cls=True)[0]
    for method in ("2d", "3d"):
        a = dct.surface_dice(x, g, 2.0, method=method)
        b = dct.surface_dice(cls, g, 2.0, C=C, method=method)
        assert torch.equal(a["counts"], b["counts"])
        for k in KEYS:
            assert np.array_equal(bits(a[k]), bits(b[k])), k


@pytest.mark.parametrize("method", ["2d", "3d"])
def test_out_of_range_values_flag_and_keep_other_classes(method, dct, dev):
    C = 4
    p, g = maps((4, 37, 29), C, "blobs", seed=5)
    p[0, 3, 4] = C; p[2, 10, 0] = -1; g[1, 36, 28] = C + 7
    dists = OD.distances(np.where(p < C, p, -1), np.where(g < C, g, -1), C, method)   # no class for those pixels
    st = dct._runtime.state(dev)
    with dct._runtime.check_mode("deferred"):
        st.flags.zero_()
        got = dct.surface_dice(T(p, dev), T(g, dev), 2.0, C=C, method=method)
        flags = st.flags.cpu().numpy()
        st.flags.zero_()
    assert flags[dct._lib.FLAG_PRED] == 2 and flags[dct._lib.FLAG_LABEL] == 1
    assert flags[dct._lib.FLAG_SIMPLEX] == 0 and flags[dct._lib.FLAG_ONEHOT] == 0
    assert_matches(got, dists, [2.0] * C)
    if dct.get_check_mode() == "eager":
        with pytest.raises(AssertionError):
            dct.surface_dice(T(p, dev), T(g, dev), 2.0, C=C, method=method)


def test_two_calls_are_bit_identical(dct, dev):
    for kind in ("blobs", "saltpepper"):
        p, g = maps((4, 256, 384), 19, kind, seed=2)
        pt, gt = T(p, dev), T(g, dev)
        for method in ("2d", "3d"):
            a = dct.surface_dice(pt, gt, 3.0, C=19, method=method, voxelspacing=SPACING[method])
            b = dct.surface_dice(pt, gt, 3.0, C=19, method=method, voxelspacing=SPACING[method])
            assert torch.equal(a["counts"], b["counts"]), (kind, method)
            for k in KEYS:
                assert np.array_equal(bits(a[k]), bits(b[k])), (kind, method, k)


@pytest.mark.parametrize("method", ["2d", "3d"])
def test_cuda_graph_capture_and_replay(method, dct, dev):
    C = 4
    p0, g0 = maps((6, 64, 80), C, "blobs", seed=9)
    p1, g1 = maps((6, 64, 80), C, "saltpepper", seed=10)
    tols = [0.0, 1.0, math.sqrt(2), 2.0]
    pt, gt = T(p0, dev), T(g0, dev)
    s = torch.cuda.Stream(dev)
    with dct._runtime.check_mode("deferred"):
        s.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(s):
            dct.surface_dice(pt, gt, tols, C=C, method=method)   # warm-up on the capture stream
        torch.cuda.current_stream(dev).wait_stream(s)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=s):
            out = dct.surface_dice(pt, gt, tols, C=C, method=method)
        for p, g in ((p0, g0), (p1, g1)):
            pt.copy_(T(p, dev)); gt.copy_(T(g, dev))
            graph.replay()
            torch.cuda.synchronize(dev)
            assert_matches(out, OD.distances(p, g, C, method), tols)
            eager = dct.surface_dice(pt, gt, tols, C=C, method=method)
            assert torch.equal(out["counts"], eager["counts"])
            for k in KEYS:
                assert np.array_equal(bits(out[k]), bits(eager[k])), k


def _abi_call(h, pt, gt, C, B, H, W, volume, sp, tol, out, counts, buf, stream):
    return h.dct_surface_dice_i64(pt.data_ptr(), gt.data_ptr(), C, B, H, W, volume, sp, tol, out.data_ptr(),
                                  None if counts is None else counts.data_ptr(), None, buf.data_ptr(), stream)


@pytest.mark.parametrize("method", ["2d", "3d"])
def test_scratch_query_is_sufficient(method, dct, dev):
    """The call stays inside the queried scratch (a canary behind it survives) and needs no initial state in it: the
    scratch starts as 0xAB bytes and is reused as the previous call left it."""
    C, (B, H, W) = 19, (3, 70, 90)
    p, g = maps((B, H, W), C, "saltpepper", seed=4)
    h = dct._lib.lib()
    volume = int(method == "3d")
    nbytes = h.dct_surface_dice_scratch_bytes(C, B, H, W, volume)
    assert nbytes > h.dct_hausdorff_scratch_bytes(C, B, H, W, volume)
    buf = torch.full((nbytes + 4096,), 0xAB, dtype=torch.uint8, device=dev)
    pt, gt = T(p, dev), T(g, dev)
    rows = 1 if volume else B
    out = torch.empty((3, rows, C), dtype=torch.float32, device=dev)
    counts = torch.empty((rows, C, 4), dtype=torch.int64, device=dev)
    stream = torch.cuda.current_stream(dev).cuda_stream
    tols = [0.5 * c for c in range(C)]
    tol = (ctypes.c_double * C)(*tols)
    dists = OD.distances(p, g, C, method)
    for with_counts in (True, False, True):
        out.fill_(-1.0); counts.fill_(-7)
        assert _abi_call(h, pt, gt, C, B, H, W, volume, None, tol, out, counts if with_counts else None, buf,
                         stream) == 0
        torch.cuda.synchronize(dev)
        want = counts_of(dists, tols)
        assert_ratios(dict(zip(KEYS, out.unbind(0))), want)
        if with_counts:
            np.testing.assert_array_equal(counts.cpu().numpy(), want)
        else:
            assert bool((counts == -7).all())
        assert bool((buf[nbytes:] == 0xAB).all())
    sp = (ctypes.c_double * len(SPACING[method]))(*SPACING[method])
    assert _abi_call(h, pt, gt, C, B, H, W, volume, sp, tol, out, counts, buf, stream) == 0
    torch.cuda.synchronize(dev)
    c = counts.cpu().numpy()
    dists = OD.distances(p, g, C, method, SPACING[method])
    want = counts_of(dists, tols)
    assert np.all(np.abs(c - want)[..., 0::2] <= near_counts(dists, tols))
    np.testing.assert_array_equal(c[..., 1::2], want[..., 1::2])
    assert bool((buf[nbytes:] == 0xAB).all())


def test_argument_errors_leave_outputs_untouched(dct, dev):
    C, (B, H, W) = 4, (2, 16, 16)
    p, g = maps((B, H, W), C, "blobs", seed=6)
    h = dct._lib.lib()
    pt, gt = T(p, dev), T(g, dev)
    buf = torch.zeros(h.dct_surface_dice_scratch_bytes(C, B, H, W, 1), dtype=torch.uint8, device=dev)
    out = torch.full((3, B, C), -1.0, dtype=torch.float32, device=dev)
    counts = torch.full((B, C, 4), -7, dtype=torch.int64, device=dev)
    stream = torch.cuda.current_stream(dev).cuda_stream

    def tol(*v):
        return (ctypes.c_double * len(v))(*v)

    for bad in (None, tol(1.0, -1.0, 1.0, 1.0), tol(1.0, float("nan"), 1.0, 1.0), tol(1.0, 1.0, 1.0, float("inf"))):
        for volume in (0, 1):
            assert _abi_call(h, pt, gt, C, B, H, W, volume, None, bad, out, counts, buf, stream) == -1
    assert _abi_call(h, pt, gt, C, B, H, W, 1, tol(1.0, 0.0, 1.0), tol(1, 1, 1, 1), out, counts, buf, stream) == -1
    assert _abi_call(h, pt, gt, 65, B, H, W, 0, None, tol(*[1.0] * 65), out, counts, buf, stream) == -2
    torch.cuda.synchronize(dev)
    assert bool((out == -1.0).all()) and bool((counts == -7).all())
    for bad in (-1.0, float("nan"), float("inf"), [1.0, 1.0, -2.0, 1.0]):
        with pytest.raises(ValueError):
            dct.surface_dice(pt, gt, bad, C=C)
    with pytest.raises(AssertionError):
        dct.surface_dice(pt, gt, [1.0, 2.0], C=C)


@pytest.mark.parametrize("method,axes", [("2d", "all"), ("3d", "all"), ("2d", [1, 2, 3])])
def test_meter_matches_nan_statistics_of_oracle_rows(method, axes, dct, dev):
    import warnings
    C = 4
    tols = [1.0, 2.0, math.sqrt(2), 3.0]
    meter = dct.SurfaceDiceMeter(tols, method=method, report_axises=axes, C=C)
    rows = []
    for i in range(3):
        p, g = maps((4, 48, 40), C, "blobs", seed=20 + i)
        if i == 1:
            p[p == 3] = 0; g[g == 3] = 0   # class 3 absent from both: NaN rows skipped by the statistics
        meter.add(T(p, dev), T(g, dev)[:, None])   # unit spacing: the rows equal the oracle's exactly
        rows.append(OD.surface_dice(p, g, C, tols, method)["nsd"])
    log = np.concatenate(rows)
    assert np.isnan(log).any()
    got = meter.log.cpu().numpy()
    assert np.array_equal(np.isnan(got), np.isnan(log))
    assert np.array_equal(got, log.astype(np.float32), equal_nan=True)
    with np.errstate(all="ignore"), warnings.catch_warnings():
        warnings.simplefilter("ignore", RuntimeWarning)
        (mean, std), (means, stds) = meter.value()
        rep = np.nanmean(log if axes == "all" else log[:, axes], 1)
        np.testing.assert_allclose(means.cpu().numpy(), np.nanmean(log, 0), rtol=1e-5)
        np.testing.assert_allclose(stds.cpu().numpy(), np.nanstd(log, 0, ddof=1), rtol=1e-5, equal_nan=True)
        np.testing.assert_allclose(mean.item(), np.nanmean(rep), rtol=1e-5)
        np.testing.assert_allclose(std.item(), np.nanstd(rep, ddof=1), rtol=1e-5, equal_nan=True)
    s = meter.summary()
    assert set(s) == {"mNSD", "mNSDVars"} and s["mNSD"] == pytest.approx(mean.item())
    assert list(meter.detailed_summary()) == [f"NSD{i}" for i in range(C)]
    meter.reset()
    assert meter.nsdLog == []


@pytest.mark.parametrize("method", ["2d", "3d"])
def test_surface_dice_of_the_largest_component(method, dct, dev):
    C = 4
    rng = np.random.default_rng(12)
    g = OH.blobs(rng, (10, 96, 96), C)
    p = g.copy()
    noise = rng.random(p.shape) < 0.002    # stray islands far from the organs
    p[noise] = rng.integers(1, C, size=int(noise.sum()))
    conn = 3 if method == "3d" else 2
    x = torch.nn.functional.one_hot(T(p, dev), C).permute(0, 3, 1, 2).float() * 4.0   # scores whose arg-max is p
    want_big = OC.components(p, C, method, conn)[2]
    tols = [1.0, 2.0, math.sqrt(2), math.sqrt(5)]
    got = dct.surface_dice(dct.largest_component(x, method=method, connectivity=conn), T(g, dev), tols, C=C,
                           method=method)
    assert_matches(got, OD.distances(want_big, g, C, method), tols)
    assert_matches(dct.surface_dice(x, T(g, dev), tols, method=method), OD.distances(p, g, C, method), tols)
