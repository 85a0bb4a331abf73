"""GPU parity of the surface distances (dct_surface_distances_i64 through ``dct_b200.surface_distances`` /
``SurfaceDistanceMeter``) against the scipy restatement of medpy hd95 / asd / assd (oracle/oracle_surface.py).

``hd`` equals ``hausdorff()`` bit for bit.  At unit spacing every d^2 is an integer below 2^24, so both sides interpolate
the same doubles and ``hd95`` equals the oracle rounded to float32 bit for bit; ``asd`` / ``assd`` sum in another order
(within 1e-6 relative).  At anisotropic spacing everything is within 1e-6 relative.  NaN where a class is absent from one
side."""
import ctypes

import numpy as np
import pytest
import torch

import oracle_hausdorff as OH
import oracle_surface as OS

pytestmark = pytest.mark.gpu

KEYS = OS.KEYS
SPACING = {"2d": (1.5625, 1.25), "3d": (10.0, 1.5625, 1.25)}
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


def assert_matches(got: dict, want: dict, unit: bool):
    assert set(got) == set(KEYS)
    for k in KEYS:
        g = got[k].detach().cpu().numpy()
        w = want[k]
        assert g.dtype == np.float32 and g.shape == w.shape, k
        nan = np.isnan(w)
        assert np.array_equal(np.isnan(g), nan), k
        if unit and k in ("hd", "hd95"):
            assert np.array_equal(g[~nan], w[~nan].astype(np.float32)), k
        else:
            np.testing.assert_allclose(g[~nan], w[~nan], rtol=1e-6, atol=0, err_msg=k)


def maps(shape, C, kind, seed):
    rng = np.random.default_rng(seed)
    make = OH.blobs if kind == "blobs" else OH.salt_pepper
    return make(rng, shape, C), make(rng, shape, C)


@pytest.mark.parametrize("unit", [True, False], ids=["unit", "aniso"])
@pytest.mark.parametrize("method", ["2d", "3d"])
@pytest.mark.parametrize("kind", ["blobs", "saltpepper"])
@pytest.mark.parametrize("shape,C", CASES)
def test_surface_distances_vs_oracle(shape, C, kind, method, unit, dct, dev):
    p, g = maps(shape, C, kind, seed=C * 1000 + shape[1])
    sp = None if unit else SPACING[method]
    pt, gt = T(p, dev), T(g, dev)
    got = dct.surface_distances(pt, gt, C=C, method=method, voxelspacing=sp)
    rows = 1 if method == "3d" else shape[0]
    assert all(got[k].shape == (rows, C) and got[k].device == dev for k in KEYS)
    assert np.array_equal(bits(got["hd"]), bits(dct.hausdorff(pt, gt, C=C, method=method, voxelspacing=sp)))
    assert_matches(got, OS.surface(p, g, C, method, sp), unit)


def _edge_cases():
    out = []
    p = np.zeros((2, 6, 7), np.int64); g = np.zeros((2, 6, 7), np.int64)
    g[:, 2:4, 3] = 1; p[:, 1, 1] = 2
    out.append(("empty_pred_gt_both", p, g, 4))
    p = np.zeros((1, 9, 9), np.int64); g = np.zeros((1, 9, 9), np.int64)
    p[0, 1, 2] = 1; g[0, 7, 5] = 1
    out.append(("single_pixels", p, g, 2))
    full = np.ones((2, 8, 10), np.int64); g = full.copy(); g[:, 3:5, 4:6] = 0; g[1, 0, :] = 0
    out.append(("whole_grid", full, g, 2))
    rng = np.random.default_rng(11)
    for shape in [(2, 1, 31), (3, 29, 1), (1, 1, 1), (2, 1, 1)]:
        out.append((f"line_{shape}", OH.salt_pepper(rng, shape, 3), OH.salt_pepper(rng, shape, 3), 3))
    m = OH.blobs(rng, (3, 40, 24), 4, smooth=2.0)
    out.append(("identical", m, m.copy(), 4))
    # one pixel against a 6x6 square (20 border pixels): n = 21, (n - 1) * 0.95 = 19 exactly, t = 0
    p = np.zeros((1, 12, 12), np.int64); g = np.zeros((1, 12, 12), np.int64)
    p[0, 1, 1] = 1; g[0, 4:10, 4:10] = 1
    out.append(("rank_integral", p, g, 2))
    return out


@pytest.mark.parametrize("method", ["2d", "3d"])
@pytest.mark.parametrize("case", _edge_cases(), ids=lambda c: c[0])
def test_surface_distances_edge_cases(case, method, dct, dev):
    name, p, g, C = case
    pt, gt = T(p, dev), T(g, dev)
    for sp in (None, SPACING[method]):
        got = dct.surface_distances(pt, gt, C=C, method=method, voxelspacing=sp)
        assert_matches(got, OS.surface(p, g, C, method, sp), sp is None)
        assert np.array_equal(bits(got["hd"]), bits(dct.hausdorff(pt, gt, C=C, method=method, voxelspacing=sp)))
    if name == "identical":
        got = dct.surface_distances(pt, gt, C=C, method=method)
        assert all(np.all(got[k].cpu().numpy() == 0) for k in KEYS)


@pytest.mark.parametrize("unit", [True, False], ids=["unit", "aniso"])
@pytest.mark.parametrize("method", ["2d", "3d"])
def test_swapping_pred_and_gt(method, unit, dct, dev):
    C = 4
    p, g = maps((4, 60, 52), C, "blobs", seed=31)
    p[2][p[2] == 1] = 0   # class 1 absent from one prediction slice
    sp = None if unit else SPACING[method]
    a = dct.surface_distances(T(p, dev), T(g, dev), C=C, method=method, voxelspacing=sp)
    b = dct.surface_distances(T(g, dev), T(p, dev), C=C, method=method, voxelspacing=sp)
    for k in ("hd", "hd95", "assd"):
        assert np.array_equal(bits(a[k]), bits(b[k])), k
    want = OS.surface(g, p, C, method, sp)["asd"]   # asd(gt, pred): label border to prediction border
    nan = np.isnan(want)
    got = b["asd"].cpu().numpy()
    assert np.array_equal(np.isnan(got), nan)
    np.testing.assert_allclose(got[~nan], want[~nan], rtol=1e-6, atol=0)


@pytest.mark.parametrize("C", [2, 4, 19])
def test_scores_path_equals_class_map_path(C, dct, dev):
    gen = torch.Generator().manual_seed(C)
    x = (3 * torch.randn(3, C, 45, 38, generator=gen)).to(dev)
    x[0, :, 0, 0] = 0.0   # ties resolve as DiceMeter's arg-max does
    g = torch.randint(0, C, (3, 1, 45, 38), generator=gen).to(dev)
    cls = dct.utils._classmap(x, 1, want_cls=True)[0]
    for method in ("2d", "3d"):
        a = dct.surface_distances(x, g, method=method)
        b = dct.surface_distances(cls, g, C=C, method=method)
        for k in KEYS:
            assert np.array_equal(a[k].cpu().numpy(), b[k].cpu().numpy(), equal_nan=True), k


@pytest.mark.parametrize("method", ["2d", "3d"])
def test_out_of_range_values_flag_and_keep_other_classes(method, dct, dev):
    C = 4
    p, g = maps((4, 37, 29), C, "blobs", seed=5)
    p[0, 3, 4] = C; p[2, 10, 0] = -1; g[1, 36, 28] = C + 7
    sp = SPACING[method]
    want = OS.surface(np.where(p < C, p, -1), np.where(g < C, g, -1), C, method, sp)   # no class for those pixels
    st = dct._runtime.state(dev)
    with dct._runtime.check_mode("deferred"):
        st.flags.zero_()
        got = dct.surface_distances(T(p, dev), T(g, dev), C=C, method=method, voxelspacing=sp)
        flags = st.flags.cpu().numpy()
        st.flags.zero_()
    assert flags[dct._lib.FLAG_PRED] == 2 and flags[dct._lib.FLAG_LABEL] == 1
    assert flags[dct._lib.FLAG_SIMPLEX] == 0 and flags[dct._lib.FLAG_ONEHOT] == 0
    assert_matches(got, want, False)
    if dct.get_check_mode() == "eager":
        with pytest.raises(AssertionError):
            dct.surface_distances(T(p, dev), T(g, dev), C=C, method=method)


def test_two_calls_are_bit_identical(dct, dev):
    for kind in ("blobs", "saltpepper"):
        p, g = maps((4, 256, 384), 19, kind, seed=2)
        pt, gt = T(p, dev), T(g, dev)
        for method in ("2d", "3d"):
            a = dct.surface_distances(pt, gt, C=19, method=method, voxelspacing=SPACING[method])
            b = dct.surface_distances(pt, gt, C=19, method=method, voxelspacing=SPACING[method])
            for k in KEYS:
                assert np.array_equal(bits(a[k]), bits(b[k])), (kind, method, k)


@pytest.mark.parametrize("method", ["2d", "3d"])
def test_cuda_graph_capture_and_replay(method, dct, dev):
    C = 4
    p0, g0 = maps((6, 64, 80), C, "blobs", seed=9)
    p1, g1 = maps((6, 64, 80), C, "saltpepper", seed=10)
    sp = SPACING[method]
    pt, gt = T(p0, dev), T(g0, dev)
    s = torch.cuda.Stream(dev)
    with dct._runtime.check_mode("deferred"):
        s.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(s):
            dct.surface_distances(pt, gt, C=C, method=method, voxelspacing=sp)   # warm-up on the capture stream
        torch.cuda.current_stream(dev).wait_stream(s)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=s):
            out = dct.surface_distances(pt, gt, C=C, method=method, voxelspacing=sp)
        for p, g in ((p0, g0), (p1, g1)):
            pt.copy_(T(p, dev)); gt.copy_(T(g, dev))
            graph.replay()
            torch.cuda.synchronize(dev)
            assert_matches(out, OS.surface(p, g, C, method, sp), False)
            eager = dct.surface_distances(pt, gt, C=C, method=method, voxelspacing=sp)
            for k in KEYS:
                assert np.array_equal(bits(out[k]), bits(eager[k])), k


@pytest.mark.parametrize("method", ["2d", "3d"])
def test_scratch_query_is_sufficient(method, dct, dev):
    """The call stays inside the queried scratch (a canary behind it survives) and needs no initial state in it: the
    scratch starts as 0xAB bytes and is reused as the previous call left it."""
    C, (B, H, W) = 19, (3, 70, 90)
    p, g = maps((B, H, W), C, "saltpepper", seed=4)
    h = dct._lib.lib()
    volume = int(method == "3d")
    nbytes = h.dct_surface_distance_scratch_bytes(C, B, H, W, volume)
    assert nbytes > h.dct_hausdorff_scratch_bytes(C, B, H, W, volume)
    buf = torch.full((nbytes + 4096,), 0xAB, dtype=torch.uint8, device=dev)
    pt, gt = T(p, dev), T(g, dev)
    rows = 1 if volume else B
    out = torch.empty((4, rows, C), dtype=torch.float32, device=dev)
    stream = torch.cuda.current_stream(dev).cuda_stream
    want = OS.surface(p, g, C, method)
    for _ in range(2):
        out.fill_(-1.0)
        assert h.dct_surface_distances_i64(pt.data_ptr(), gt.data_ptr(), C, B, H, W, volume, None, out.data_ptr(), None,
                                           buf.data_ptr(), stream) == 0
        torch.cuda.synchronize(dev)
        assert_matches(dict(zip(KEYS, out.unbind(0))), want, True)
        assert bool((buf[nbytes:] == 0xAB).all())
    sp = (ctypes.c_double * len(SPACING[method]))(*SPACING[method])
    assert h.dct_surface_distances_i64(pt.data_ptr(), gt.data_ptr(), C, B, H, W, volume, sp, out.data_ptr(), None,
                                       buf.data_ptr(), stream) == 0
    torch.cuda.synchronize(dev)
    assert_matches(dict(zip(KEYS, out.unbind(0))), OS.surface(p, g, C, method, SPACING[method]), False)
    assert bool((buf[nbytes:] == 0xAB).all())


@pytest.mark.parametrize("method,axes", [("2d", "all"), ("3d", "all"), ("2d", [1, 2, 3])])
def test_meter_matches_nan_statistics_of_oracle_rows(method, axes, dct, dev):
    import warnings
    C = 4
    meter = dct.SurfaceDistanceMeter(method=method, report_axises=axes, C=C)
    rows = {k: [] for k in KEYS}
    for i in range(3):
        p, g = maps((4, 48, 40), C, "blobs", seed=20 + i)
        if i == 1:
            p[p == 3] = 0   # class 3 absent from this prediction: NaN rows skipped by the statistics
        sp = SPACING[method]
        meter.add(T(p, dev), T(g, dev)[:, None], voxelspacing=sp)
        want = OS.surface(p, g, C, method, sp)
        for k in KEYS:
            rows[k].append(want[k])
    with np.errstate(all="ignore"), warnings.catch_warnings():
        warnings.simplefilter("ignore", RuntimeWarning)
        for k in KEYS:
            log = np.concatenate(rows[k])
            assert np.array_equal(np.isnan(meter.log(k).cpu().numpy()), np.isnan(log))
            (mean, std), (means, stds) = meter.value(k)
            rep = np.nanmean(log if axes == "all" else log[:, axes], 1)
            np.testing.assert_allclose(means.cpu().numpy(), np.nanmean(log, 0), rtol=1e-5)
            np.testing.assert_allclose(stds.cpu().numpy(), np.nanstd(log, 0, ddof=1), rtol=1e-5, equal_nan=True)
            np.testing.assert_allclose(mean.item(), np.nanmean(rep), rtol=1e-5)
            np.testing.assert_allclose(std.item(), np.nanstd(rep, ddof=1), rtol=1e-5, equal_nan=True)
    (m95, _), _ = meter.value()
    assert m95.item() == meter.value("hd95")[0][0].item()
    s = meter.summary()
    assert set(s) == {f"m{n}{v}" for n in ("HD", "HD95", "ASD", "ASSD") for v in ("", "Vars")}
    assert s["mHD95"] == pytest.approx(m95.item())
    d = meter.detailed_summary()
    assert list(d) == ([f"HD{i}" for i in range(C)] + [f"HD95_{i}" for i in range(C)] + [f"ASD{i}" for i in range(C)]
                       + [f"ASSD{i}" for i in range(C)])
    meter.reset()
    assert all(v == [] for v in meter.logs.values())
