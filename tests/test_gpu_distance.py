"""GPU parity of the distance maps (dct_distance_map_i64 through ``dct_b200.signed_distance_map`` /
``distance_transform_edt``) against the scipy restatement (oracle/oracle_distance.py) and scipy itself.

At unit spacing the kernels carry every d^2 as the exact integer and take one square root in double, so every value is
the float32 of scipy's float64 value, bit for bit.  At anisotropic spacing the volume's row pass rounds d^2 to float, so
values agree within 1e-6 relative."""
import ctypes
from functools import lru_cache

import numpy as np
import pytest
import torch
from scipy.ndimage import distance_transform_edt

import oracle_distance as ODM
import oracle_hausdorff as OH

pytestmark = pytest.mark.gpu

SPACING = {"2d": (1.5625, 1.5625), "3d": (10.0, 1.5625, 1.5625)}
CASES = [((10, 256, 256), 4),      # ACDC patient
         ((8, 512, 512), 2),       # Spleen
         ((5, 33, 47), 19),        # a C = 19 batch
         ((64, 512, 512), 2)]      # a volume of 64 slices


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


@lru_cache(maxsize=4)
def make_map(shape, C, kind, seed):
    rng = np.random.default_rng(seed)
    return (OH.blobs if kind == "blobs" else OH.salt_pepper)(rng, shape, C)


def assert_exact(got, want):
    g = got.detach().cpu().numpy()
    w = np.asarray(want).astype(np.float32)
    assert g.dtype == np.float32 and g.shape == w.shape
    bad = g.view(np.uint32) != w.view(np.uint32)
    assert not bad.any(), (int(bad.sum()), np.argwhere(bad)[:4], g[bad][:4], w[bad][:4])


def assert_close(got, want, rel=1e-6):
    g = got.detach().cpu().numpy().astype(np.float64)
    w = np.asarray(want, dtype=np.float64)
    assert g.shape == w.shape
    ok = (g == w) | (np.abs(g - w) <= rel * np.abs(w))
    assert ok.all(), (int((~ok).sum()), np.argwhere(~ok)[:4], g[~ok][:4], w[~ok][:4])


def check(got, want, unit):
    (assert_exact if unit else assert_close)(got, want)


@pytest.mark.parametrize("unit", [True, False], ids=["unit", "aniso"])
@pytest.mark.parametrize("signed", [True, False], ids=["signed", "inside"])
@pytest.mark.parametrize("method", ["2d", "3d"])
@pytest.mark.parametrize("kind", ["blobs", "saltpepper"])
@pytest.mark.parametrize("shape,C", CASES)
def test_distance_map_vs_oracle(shape, C, kind, method, signed, unit, dct, dev):
    if shape[0] == 64 and method == "2d" and kind == "saltpepper":
        pytest.skip("covered by the smaller slice batches")
    m = make_map(shape, C, kind, seed=C * 1000 + shape[1])
    sp = None if unit else SPACING[method]
    want = ODM.distance_map(m, C, 0, method, sp, signed)
    mt = T(m, dev)
    if signed:
        got = dct.signed_distance_map(mt, C=C, method=method, voxelspacing=sp)
    else:
        h = dct._lib.lib()
        B, H, W = shape
        vol = int(method == "3d")
        out = torch.empty((B, C, H, W), dtype=torch.float32, device=dev)
        buf = torch.empty(h.dct_distance_map_scratch_bytes(C, 0, B, H, W, vol, 0), dtype=torch.uint8, device=dev)
        spa = None if sp is None else (ctypes.c_double * len(sp))(*sp)
        assert h.dct_distance_map_i64(mt.data_ptr(), C, 0, B, H, W, vol, spa, 0, out.data_ptr(), None,
                                      buf.data_ptr(), torch.cuda.current_stream(dev).cuda_stream) == 0
        got = out
    assert got.shape == (shape[0], C) + shape[1:] and got.device == dev
    check(got, want, unit)
    if signed and C > 2:   # without the background: the same planes 1 .. C-1
        check(dct.signed_distance_map(mt, C=C, method=method, voxelspacing=sp, include_background=False),
              want[:, 1:], unit)


@pytest.mark.parametrize("method", ["2d", "3d"])
def test_scores_path_and_background(method, dct, dev):
    C = 4
    gen = torch.Generator().manual_seed(3)
    x = (3 * torch.randn(3, C, 45, 38, generator=gen)).to(dev)
    x[0, :, 0, 0] = 0.0   # ties resolve as DiceMeter's arg-max does
    cls = dct.utils._classmap(x, 1, want_cls=True)[0]
    a = dct.signed_distance_map(x, method=method)
    assert torch.equal(a, dct.signed_distance_map(cls, C=C, method=method))
    assert_exact(a, ODM.distance_map(cls.cpu().numpy(), C, 0, method))
    b = dct.signed_distance_map(x, method=method, include_background=False, voxelspacing=SPACING[method])
    assert b.shape == (3, C - 1, 45, 38)
    assert_close(b, ODM.distance_map(cls.cpu().numpy(), C, 1, method, SPACING[method]))


@pytest.mark.parametrize("method", ["2d", "3d"])
def test_distance_transform_edt_is_scipy(method, dct, dev):
    rng = np.random.default_rng(8)
    m = OH.blobs(rng, (6, 96, 80), 2) != 0
    m[2] = False            # no foreground: all 0
    sp3 = (2.5, 0.75, 1.25)
    for inp in (T(m, dev), T(m.astype(np.float32) * 0.5, dev), T(m.astype(np.uint8), dev)[:, None]):
        for sampling in (None, 1.75, sp3[3 - (2 if method == "2d" else 3):]):
            got = dct.distance_transform_edt(inp, sampling=sampling, method=method)
            assert got.shape == m.shape and got.dtype == torch.float32
            grids = [m] if method == "3d" else list(m)
            want = np.stack([distance_transform_edt(g, sampling=sampling) for g in grids]).reshape(m.shape)
            check(got, want, sampling is None)
    full = torch.ones((2, 3, 4), dtype=torch.bool, device=dev)   # no background: +inf, not scipy's artifact
    assert bool(torch.isinf(dct.distance_transform_edt(full)).all())


@pytest.mark.parametrize("method", ["2d", "3d"])
@pytest.mark.parametrize("signed", [True, False], ids=["signed", "inside"])
def test_long_axes(method, signed, dct, dev):
    """32768-long W (one line per CTA with 128 KiB of stack) and H = 32768 with a column distance of 32767, and for a
    volume a 32768-long B axis."""
    rng = np.random.default_rng(4)
    maps = []
    m = np.zeros((2, 3, 32768), np.int64); m[0, 1, 5] = 1; m[1, :, 32000:] = 1; m[1, 2, 100:140] = 2
    maps.append(m)
    m = np.zeros((1, 32768, 2), np.int64); m[0, 0, 0] = 1
    maps.append(m)
    maps.append(rng.integers(0, 3, size=(2, 32768, 3)) * (rng.random((2, 32768, 3)) < 0.001))
    if method == "3d":
        m = np.zeros((32768, 1, 2), np.int64); m[0, 0, 1] = 1; m[20000:, 0, 0] = 2
        maps.append(m)
    for m in maps:
        m = m.astype(np.int64)
        want = ODM.distance_map(m, 3, 0, method, None, signed)
        got = dct.signed_distance_map(T(m, dev), C=3, method=method) if signed else \
            _inside(dct, T(m, dev), 3, method, None)
        assert_exact(got, want)
        sp = SPACING[method]
        got = dct.signed_distance_map(T(m, dev), C=3, method=method, voxelspacing=sp) if signed else \
            _inside(dct, T(m, dev), 3, method, sp)
        assert_close(got, ODM.distance_map(m, 3, 0, method, sp, signed))
    if not signed and method == "2d":
        d = dct.distance_transform_edt(T(maps[1] == 0, dev))
        assert d[0, 32767, 0].item() == 32767.0 and d[0, 32767, 1].item() == np.float32(np.sqrt(32767.0 ** 2 + 1))


def _inside(dct, mt, C, method, sp):
    """Inside distances of every class: one unsigned call per class through distance_transform_edt of its mask."""
    return torch.stack([dct.distance_transform_edt(mt == c, sampling=sp, method=method) for c in range(C)], 1)


@pytest.mark.parametrize("method", ["2d", "3d"])
def test_out_of_range_values_flag(method, dct, dev):
    C = 4
    m = make_map((4, 37, 29), C, "blobs", seed=5).copy()
    m[0, 3, 4] = C; m[2, 10, 0] = -1; m[3, 36, 28] = C + 7
    st = dct._runtime.state(dev)
    with dct._runtime.check_mode("deferred"):
        st.flags.zero_()
        got = dct.signed_distance_map(T(m, dev), C=C, method=method)
        flags = st.flags.cpu().numpy()
        st.flags.zero_()
    assert flags[dct._lib.FLAG_PRED] == 3 and flags[dct._lib.FLAG_LABEL] == 0
    assert flags[dct._lib.FLAG_SIMPLEX] == 0 and flags[dct._lib.FLAG_ONEHOT] == 0
    assert_exact(got, ODM.distance_map(m, C, 0, method))
    if dct.get_check_mode() == "eager":
        with pytest.raises(AssertionError):
            dct.signed_distance_map(T(m, dev), C=C, method=method)


def test_two_calls_are_bit_identical(dct, dev):
    for kind in ("blobs", "saltpepper"):
        mt = T(make_map((4, 256, 384), 19, kind, seed=2), dev)
        for method in ("2d", "3d"):
            a = dct.signed_distance_map(mt, C=19, method=method, voxelspacing=SPACING[method])
            b = dct.signed_distance_map(mt, C=19, method=method, voxelspacing=SPACING[method])
            assert torch.equal(a.view(torch.int32), b.view(torch.int32)), (kind, method)


@pytest.mark.parametrize("method", ["2d", "3d"])
def test_cuda_graph_capture_and_replay(method, dct, dev):
    C = 4
    m0 = make_map((6, 64, 80), C, "blobs", seed=9)
    m1 = make_map((6, 64, 80), C, "saltpepper", seed=10)
    mt = T(m0, dev)
    s = torch.cuda.Stream(dev)
    with dct._runtime.check_mode("deferred"):
        s.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(s):
            dct.signed_distance_map(mt, C=C, method=method)   # warm-up on the capture stream
            dct.distance_transform_edt(mt, method=method)
        torch.cuda.current_stream(dev).wait_stream(s)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=s):
            phi = dct.signed_distance_map(mt, C=C, method=method)
            edt = dct.distance_transform_edt(mt, method=method)
        for m in (m0, m1):
            mt.copy_(T(m, dev))
            graph.replay()
            torch.cuda.synchronize(dev)
            assert_exact(phi, ODM.distance_map(m, C, 0, method))
            assert_exact(edt, ODM.distance_map((m != 0).astype(np.int64), 2, 1, method, signed=False)[:, 0])


@pytest.mark.parametrize("signed", [1, 0])
@pytest.mark.parametrize("method", ["2d", "3d"])
def test_scratch_query_is_sufficient(method, signed, dct, dev):
    """The call stays inside the queried scratch (a canary behind it survives) and needs no initial state in it: the
    scratch starts as 0xAB bytes and is reused as the previous call left it."""
    C, first, (B, H, W) = 19, 2, (3, 70, 90)
    m = make_map((B, H, W), C, "saltpepper", seed=4)
    h = dct._lib.lib()
    volume = int(method == "3d")
    nbytes = h.dct_distance_map_scratch_bytes(C, first, B, H, W, volume, signed)
    buf = torch.full((nbytes + 4096,), 0xAB, dtype=torch.uint8, device=dev)
    mt = T(m, dev)
    out = torch.empty((B, C - first, H, W), dtype=torch.float32, device=dev)
    stream = torch.cuda.current_stream(dev).cuda_stream
    want = ODM.distance_map(m, C, first, method, None, bool(signed))
    for _ in range(2):
        out.fill_(-7.0)
        assert h.dct_distance_map_i64(mt.data_ptr(), C, first, B, H, W, volume, None, signed, out.data_ptr(), None,
                                      buf.data_ptr(), stream) == 0
        torch.cuda.synchronize(dev)
        assert_exact(out, want)
        assert bool((buf[nbytes:] == 0xAB).all())


def test_argument_errors_leave_outputs_untouched(dct, dev):
    C, (B, H, W) = 4, (2, 16, 16)
    mt = T(make_map((B, H, W), C, "blobs", seed=6), dev)
    h = dct._lib.lib()
    buf = torch.zeros(h.dct_distance_map_scratch_bytes(C, 0, B, H, W, 1, 1), dtype=torch.uint8, device=dev)
    out = torch.full((B, C, H, W), -1.0, dtype=torch.float32, device=dev)
    stream = torch.cuda.current_stream(dev).cuda_stream

    def call(C=C, first=0, volume=0, sp=None, signed=1):
        spa = None if sp is None else (ctypes.c_double * len(sp))(*sp)
        return h.dct_distance_map_i64(mt.data_ptr(), C, first, B, H, W, volume, spa, signed, out.data_ptr(), None,
                                      buf.data_ptr(), stream)

    assert call(first=4) == -1 and call(first=-1) == -1 and call(signed=2) == -1
    assert call(sp=(1.0, 0.0)) == -1 and call(volume=1, sp=(1.0, float("nan"), 1.0)) == -1
    assert call(C=65) == -2
    torch.cuda.synchronize(dev)
    assert bool((out == -1.0).all())
    with pytest.raises(AssertionError):
        dct.signed_distance_map(mt, C=1, include_background=False)
    with pytest.raises(AssertionError):
        dct.signed_distance_map(mt, C=C, method="3d", voxelspacing=(1.0, 1.0))
    with pytest.raises(dct.DctError):
        dct.signed_distance_map(mt, C=65)
    with pytest.raises(RuntimeError):
        dct.distance_transform_edt(mt.cpu())


@pytest.mark.parametrize("method", ["2d", "3d"])
def test_signed_map_is_the_border_distance_outside(method, dct, dev):
    """At a pixel outside b, phi_b is its distance to b, and the nearest pixel of b is a border pixel of b: so on the
    border pixels of a that lie outside b, phi_b equals the distance to border(b) that hausdorff(a, b) folds, and the
    largest of them is at most hausdorff(a, b)."""
    C = 3
    a = make_map((4, 64, 72), C, "blobs", seed=31)
    b = make_map((4, 64, 72), C, "blobs", seed=32)
    phi_b = dct.signed_distance_map(T(b, dev), C=C, method=method).cpu().numpy()
    hd = dct.hausdorff(T(a, dev), T(b, dev), C=C, method=method).cpu().numpy()
    grids = [(0, slice(None))] if method == "3d" else [(i, i) for i in range(4)]
    checked = 0
    for c in range(C):
        for row, sl in grids:
            outside = OH.border(a[sl] == c) & (b[sl] != c)
            if not outside.any() or not (b[sl] == c).any():
                continue
            want = distance_transform_edt(~OH.border(b[sl] == c))[outside]
            got = (phi_b[sl, c] if method == "2d" else phi_b[:, c])[outside]
            np.testing.assert_array_equal(got, want.astype(np.float32))
            assert got.max() <= hd[row, c]
            checked += 1
    assert checked > 0
