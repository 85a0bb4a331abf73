"""GPU parity of Boundary IoU (dct_boundary_iou_i64 through ``dct_b200.boundary_iou`` / ``BoundaryIoUMeter``) against the
scipy restatement of ``mask_to_boundary`` (oracle/oracle_boundary_iou.py).

The counts are integers, so they must equal the oracle's exactly, and ``biou`` must be the float32 of the oracle's float64
quotient bit for bit (NaN where the union is empty)."""
import ctypes

import numpy as np
import pytest
import torch

import oracle_boundary_iou as OB
import oracle_hausdorff as OH

pytestmark = pytest.mark.gpu

CASES = [((3, 17, 23), 2), ((3, 17, 23), 4), ((3, 17, 23), 19), ((5, 33, 47), 19),
         ((10, 256, 256), 4),      # ACDC patient
         ((8, 512, 512), 2),       # Spleen
         ((2, 1024, 2048), 19)]    # Cityscapes


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


def assert_matches(got, want):
    c = got["counts"].cpu().numpy()
    assert c.dtype == np.int64 and c.shape == want["counts"].shape
    np.testing.assert_array_equal(c, want["counts"])
    b = got["biou"].cpu().numpy()
    w = want["biou"].astype(np.float32)
    assert b.dtype == np.float32 and b.shape == w.shape
    assert np.array_equal(b.view(np.uint32)[~np.isnan(w)], w.view(np.uint32)[~np.isnan(w)])
    assert np.array_equal(np.isnan(b), np.isnan(w))


def check(dct, dev, p, g, C, d, ignore_index=None):
    got = dct.boundary_iou(T(p, dev), T(g, dev), C=C, dilation=d, ignore_index=ignore_index)
    assert_matches(got, OB.boundary_iou(p, g, C, d, ignore_index))
    return got


@pytest.mark.parametrize("kind", ["blobs", "saltpepper"])
@pytest.mark.parametrize("shape,C", CASES)
def test_boundary_iou_vs_oracle(shape, C, kind, dct, dev):
    p, g = maps(shape, C, kind, seed=C * 1000 + shape[1])
    B, H, W = shape
    big = (min(H, W) + 1) // 2   # 2d+1 > min(H, W): every class pixel is band along that axis
    for d in (1, OB.dilation_for(H, W), big):
        check(dct, dev, p, g, C, d)
    got = dct.boundary_iou(T(p, dev), T(g, dev), C=C)   # default ratio
    assert_matches(got, OB.boundary_iou(p, g, C, OB.dilation_for(H, W)))


@pytest.mark.parametrize("shape", [(1, 1, 1), (2, 1, 37), (2, 41, 1), (1, 1, 700), (1, 900, 1), (3, 2, 2)])
def test_lines_and_tiny_images(shape, dct, dev):
    rng = np.random.default_rng(sum(shape))
    for C in (2, 3):
        for p, g in ((OH.salt_pepper(rng, shape, C), OH.salt_pepper(rng, shape, C)),
                     (np.zeros(shape, np.int64), np.zeros(shape, np.int64))):
            for d in (1, 2, 5, 400):
                check(dct, dev, p, g, C, d)


def _runs(rng, shape, C, mean_run):
    """Maps of long runs along both axes: few breaks, so the halo searches run many steps before finding one."""
    B, H, W = shape
    out = np.zeros(shape, np.int64)
    for b in range(B):
        ys = np.sort(rng.choice(np.arange(1, H), size=max(1, H // mean_run), replace=False))
        xs = np.sort(rng.choice(np.arange(1, W), size=max(1, W // mean_run), replace=False))
        out[b] = (np.searchsorted(ys, np.arange(H), side="right")[:, None] * 7 +
                  np.searchsorted(xs, np.arange(W), side="right")[None, :] * 3) % C
    return out


@pytest.mark.parametrize("shape,d", [((1, 3000, 700), 150), ((2, 1500, 2600), 400), ((1, 4097, 300), 1000),
                                     ((1, 700, 5000), 60), ((1, 2500, 40), 1100), ((1, 40, 2500), 1100)])
def test_long_lines_and_large_dilation(shape, d, dct, dev):
    """Halos longer than one search step (64 rows along H, 128 pixels along W), uniform stretches longer than a segment
    (256 along either axis), segments whose halo reaches past the line's other end, and 2d+1 > H with 2d+1 <= W (and the
    transpose)."""
    rng = np.random.default_rng(d)
    C = 3
    p, g = _runs(rng, shape, C, mean_run=3 * d), _runs(rng, shape, C, mean_run=2 * d)
    g[:, :, : shape[2] // 3] = p[:, :, : shape[2] // 3]
    for dd in (d, d // 2 + 1, 7):
        check(dct, dev, p, g, C, dd)
    check(dct, dev, np.full(shape, 1, np.int64), g, C, d)   # one class fills the prediction


@pytest.mark.parametrize("layout", ["sprinkle", "blocks"])
def test_ignore_index(layout, dct, dev):
    C, shape = 19, (3, 160, 272)
    p, g = maps(shape, C, "blobs", seed=31)
    rng = np.random.default_rng(32)
    if layout == "sprinkle":
        g[rng.random(shape) < 0.02] = 255
    else:
        for b in range(shape[0]):
            y, x = rng.integers(0, 120), rng.integers(0, 220)
            g[b, y: y + 40, x: x + 50] = 255
        g[:, :, -7:] = 255
    for d in (1, 3, OB.dilation_for(*shape[1:])):
        got = check(dct, dev, p, g, C, d, ignore_index=255)
        plain = OB.boundary_iou(p, g, C, d)   # ignored pixels then still leave the band pixels of P in P
        assert (got["counts"].cpu().numpy()[..., 2] <= plain["counts"][..., 2]).all()
    with pytest.raises(ValueError):
        dct.boundary_iou(T(p, dev), T(g, dev), C=C, ignore_index=3)


def test_out_of_range_values_flag_and_keep_other_classes(dct, dev):
    C = 4
    p, g = maps((4, 37, 29), C, "blobs", seed=5)
    p[0, 3, 4] = C; p[2, 10, 0] = -1; g[1, 36, 28] = C + 7; g[3, 5, 5] = 255
    want = OB.boundary_iou(p, g, C, 2, ignore_index=255)
    st = dct._runtime.state(dev)
    with dct._runtime.check_mode("deferred"):
        st.flags.zero_()
        got = dct.boundary_iou(T(p, dev), T(g, dev), C=C, dilation=2, ignore_index=255)
        flags = st.flags.cpu().numpy()
        st.flags.zero_()
    assert flags[dct._lib.FLAG_PRED] == 2 and flags[dct._lib.FLAG_LABEL] == 1
    assert flags[dct._lib.FLAG_SIMPLEX] == 0 and flags[dct._lib.FLAG_ONEHOT] == 0
    assert_matches(got, want)
    if dct.get_check_mode() == "eager":
        with pytest.raises(AssertionError):
            dct.boundary_iou(T(p, dev), T(g, dev), C=C, dilation=2)


@pytest.mark.parametrize("C", [2, 4, 19])
def test_scores_path_equals_class_map_path(C, dct, dev):
    gen = torch.Generator().manual_seed(C)
    x = (3 * torch.randn(3, C, 45, 38, generator=gen)).to(dev)
    x[0, :, 0:4, 0:6] = 0.0          # ties: the first index, as torch.max
    x[1, 1, 5:9, 3:8] = float("nan")  # NaN is maximal, as torch.max
    g = torch.randint(0, C, (3, 1, 45, 38), generator=gen).to(dev)
    cls = dct.utils._classmap(x, 0, want_cls=True)[0]
    assert torch.equal(cls, torch.max(x, 1)[1])
    for d in (1, 3):
        a = dct.boundary_iou(x, g, dilation=d)
        b = dct.boundary_iou(cls, g, C=C, dilation=d)
        assert torch.equal(a["counts"], b["counts"])
        assert np.array_equal(bits(a["biou"]), bits(b["biou"]))


def _abi_call(h, pt, gt, C, B, H, W, d, ignore, biou, counts, buf, stream, flags=None):
    return h.dct_boundary_iou_i64(pt.data_ptr(), gt.data_ptr(), C, B, H, W, d, ignore, biou.data_ptr(),
                                  None if counts is None else counts.data_ptr(),
                                  None if flags is None else flags.data_ptr(), buf.data_ptr(), stream)


def test_scratch_query_is_sufficient_and_counts_nullable(dct, dev):
    """The call stays inside the queried scratch (a canary behind it survives) and needs no initial state in it: the
    scratch starts as 0xAB bytes and is reused as the previous call left it."""
    C, (B, H, W) = 19, (3, 300, 290)
    p, g = maps((B, H, W), C, "saltpepper", seed=4)
    p2, g2 = maps((B, H, W), C, "blobs", seed=5)
    h = dct._lib.lib()
    nbytes = h.dct_boundary_iou_scratch_bytes(C, B, H, W)
    buf = torch.full((nbytes + 4096,), 0xAB, dtype=torch.uint8, device=dev)
    biou = torch.empty((B, C), dtype=torch.float32, device=dev)
    counts = torch.empty((B, C, 3), dtype=torch.int64, device=dev)
    stream = torch.cuda.current_stream(dev).cuda_stream
    for (pp, gg), with_counts, d in (((p, g), True, 3), ((p2, g2), False, 5), ((p, g), True, 9), ((p2, g2), True, 1)):
        biou.fill_(-1.0); counts.fill_(-7)
        assert _abi_call(h, T(pp, dev), T(gg, dev), C, B, H, W, d, -1, biou, counts if with_counts else None, buf,
                         stream) == 0
        torch.cuda.synchronize(dev)
        want = OB.boundary_iou(pp, gg, C, d)
        if with_counts:
            assert_matches({"counts": counts, "biou": biou}, want)
        else:
            assert bool((counts == -7).all())
            assert_matches({"counts": torch.from_numpy(want["counts"]), "biou": biou}, want)
        assert bool((buf[nbytes:] == 0xAB).all())


def test_two_calls_are_bit_identical(dct, dev):
    for kind in ("blobs", "saltpepper"):
        p, g = maps((4, 512, 1024), 19, kind, seed=2)
        pt, gt = T(p, dev), T(g, dev)
        a = dct.boundary_iou(pt, gt, C=19)
        b = dct.boundary_iou(pt, gt, C=19)
        assert torch.equal(a["counts"], b["counts"]) and np.array_equal(bits(a["biou"]), bits(b["biou"]))


def test_cuda_graph_capture_and_replay(dct, dev):
    C = 19
    p0, g0 = maps((4, 96, 160), C, "blobs", seed=9)
    p1, g1 = maps((4, 96, 160), C, "saltpepper", seed=10)
    g1[:, 10:30, 40:90] = 255
    pt, gt = T(p0, dev), T(g0, dev)
    s = torch.cuda.Stream(dev)
    with dct._runtime.check_mode("deferred"):
        s.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(s):
            dct.boundary_iou(pt, gt, C=C, dilation=4, ignore_index=255)   # warm-up on the capture stream
        torch.cuda.current_stream(dev).wait_stream(s)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=s):
            out = dct.boundary_iou(pt, gt, C=C, dilation=4, ignore_index=255)
        for p, g in ((p0, g0), (p1, g1)):
            pt.copy_(T(p, dev)); gt.copy_(T(g, dev))
            graph.replay()
            torch.cuda.synchronize(dev)
            assert_matches(out, OB.boundary_iou(p, g, C, 4, 255))
            eager = dct.boundary_iou(pt, gt, C=C, dilation=4, ignore_index=255)
            assert torch.equal(out["counts"], eager["counts"])
            assert np.array_equal(bits(out["biou"]), bits(eager["biou"]))


def test_argument_errors_leave_outputs_untouched(dct, dev):
    C, (B, H, W) = 4, (2, 16, 16)
    p, g = maps((B, H, W), C, "blobs", seed=6)
    h = dct._lib.lib()
    pt, gt = T(p, dev), T(g, dev)
    buf = torch.zeros(h.dct_boundary_iou_scratch_bytes(C, B, H, W), dtype=torch.uint8, device=dev)
    biou = torch.full((B, C), -1.0, dtype=torch.float32, device=dev)
    counts = torch.full((B, C, 3), -7, dtype=torch.int64, device=dev)
    stream = torch.cuda.current_stream(dev).cuda_stream
    for d, ignore in ((0, -1), (-3, -1), (2, 0), (2, 3)):
        assert _abi_call(h, pt, gt, C, B, H, W, d, ignore, biou, counts, buf, stream) == -1
    assert _abi_call(h, pt, gt, 65, B, H, W, 2, -1, biou, counts, buf, stream) == -2
    assert h.dct_boundary_iou_i64(pt.data_ptr() + 4, gt.data_ptr(), C, B, H, W, 2, -1, biou.data_ptr(),
                                  counts.data_ptr(), None, buf.data_ptr(), stream) == -3
    torch.cuda.synchronize(dev)
    assert bool((biou == -1.0).all()) and bool((counts == -7).all())
    for kw in ({"dilation": 0}, {"dilation": -1}, {"dilation_ratio": 0.0}, {"dilation_ratio": float("nan")},
               {"dilation_ratio": -0.02}, {"dilation_ratio": float("inf")}, {"ignore_index": 2}, {"ignore_index": -1}):
        with pytest.raises(ValueError):
            dct.boundary_iou(pt, gt, C=C, **kw)


def test_largest_accepted_size(dct, dev):
    """B*H*W = 2^31 - 1 (a line: 2^31 - 1 is prime) and a 46340 x 46340 image just below it, on maps of rectangles whose
    bands are known in closed form.  The line (H = 1, so 2d+1 > H and no u bit is ever set) checks the index arithmetic at
    the limit; the 46340 x 46340 image runs the whole decomposition, both run tests and their searches, near it.  Every rectangle differs in class from its four neighbours, so a pixel is interior
    exactly when it lies at least d from each edge of its own rectangle (a rectangle edge on the grid's border included):
    a rectangle of Ly x Lx pixels has max(0, Ly - 2d) * max(0, Lx - 2d) interior pixels."""
    h = dct._lib.lib()
    n = 2 ** 31 - 1
    assert h.dct_boundary_iou_scratch_bytes(3, 1, 1, n) > 0 and h.dct_boundary_iou_scratch_bytes(3, 1, 1, n + 1) == 0
    C = 5

    def closed_form(H, W, sy, sx, d):
        ly = np.bincount(np.arange(H) // sy).astype(np.int64)   # rectangle extents along each axis
        lx = np.bincount(np.arange(W) // sx).astype(np.int64)
        band = np.zeros(C, np.int64)
        for i, a in enumerate(ly):
            for j, b in enumerate(lx):
                inner = max(0, a - 2 * d) * max(0, b - 2 * d) if min(H, W) >= 2 * d + 1 else 0
                band[(i + j) % C] += a * b - inner
        return band

    with dct._runtime.check_mode("deferred"):
        for (H, W, sy, sx, d) in ((1, n, 1, 1000003, 3), (46340, 46340, 3001, 2049, 23)):
            m = ((torch.arange(H, device=dev) // sy)[:, None] + (torch.arange(W, device=dev) // sx)[None, :]) % C
            m = m.reshape(1, H, W)
            got = dct.boundary_iou(m, m, C=C, dilation=d)
            band = closed_form(H, W, sy, sx, d)
            c = got["counts"].cpu().numpy()[0]
            np.testing.assert_array_equal(c, np.stack([band, band, band], 1))
            assert bool((got["biou"][0][torch.from_numpy(band > 0).to(dev)] == 1.0).all())
            del m, got
            torch.cuda.empty_cache()


def test_meter_pools_counts_without_host_sync(dct, dev):
    C = 5
    meter = dct.BoundaryIoUMeter(C, ignore_index=255, report_axises=[1, 2, 3, 4])
    total = np.zeros((C, 3), np.int64)
    batches = []
    for i in range(3):
        p, g = maps((2, 96, 128), C, "blobs", seed=50 + i)
        p[p == 4] = 0; g[g == 4] = 0    # class 4 absent everywhere: NaN, skipped by the mean
        g[:, :5, :] = 255
        batches.append((T(p, dev), T(g, dev)[:, None]))
        total += OB.boundary_iou(p, g, C, OB.dilation_for(96, 128), 255)["counts"].sum(0)
    x = torch.nn.functional.one_hot(batches[0][0], C).permute(0, 3, 1, 2).float()   # scores path of the first batch
    with dct._runtime.check_mode("deferred"):
        meter.add(x, batches[0][1])           # warm-up allocations outside the sync check
        meter.reset()
        torch.cuda.synchronize(dev)
        torch.cuda.set_sync_debug_mode("error")
        try:
            meter.add(x, batches[0][1])
            for p, g in batches[1:]:
                meter.add(p, g)
        finally:
            torch.cuda.set_sync_debug_mode(0)
    acc = meter.device_counts(dev)
    assert acc.device == dev and acc.dtype == torch.int64 and acc.shape == (C, 3)
    np.testing.assert_array_equal(acc.cpu().numpy(), total)
    mean, per_class = meter.value()
    want = np.array([OB.ratio(total[c]) for c in range(C)])
    assert np.isnan(per_class[4].item()) and np.isnan(want[4])
    np.testing.assert_allclose(per_class.numpy()[:4], want[:4], rtol=0, atol=0)
    assert mean.item() == pytest.approx(np.nanmean(want[1:]))
    s = meter.summary()
    assert set(s) == {"mBIoU"} and s["mBIoU"] == pytest.approx(mean.item())
    assert list(meter.detailed_summary()) == [f"BIoU{i}" for i in range(C)]
    meter.reset()
    assert bool((meter.device_counts(dev) == 0).all())
    assert np.isnan(meter.value()[0].item())
