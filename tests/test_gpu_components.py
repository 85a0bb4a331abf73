"""GPU parity of the connected components (dct_components_i64 through ``dct_b200.connected_components`` /
``largest_component``) against the scipy restatement (oracle/oracle_components.py).  Every output is an integer, so
labels, statistics and largest maps must be equal to the oracle, and two calls must give the same bits."""
import ctypes

import numpy as np
import pytest
import torch

import oracle_components as OC
import oracle_hausdorff as OH
import oracle_surface as OS
from test_gpu_hausdorff import CASES as HD_CASES
from test_gpu_surface_distance import assert_matches as assert_surface_matches

pytestmark = pytest.mark.gpu

METHOD_CONN = [("2d", 1), ("2d", 2), ("3d", 1), ("3d", 2), ("3d", 3)]
SPLEEN_VOLUME = ((64, 512, 512), 2)


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


def run(dct, m, C, method, conn, dev):
    """(labels, stats [rows, C, 2], largest) of the device, as numpy."""
    mt = T(m, dev)
    cc = dct.connected_components(mt, C=C, method=method, connectivity=conn)
    largest = dct.largest_component(mt, C=C, method=method, connectivity=conn)
    assert cc["labels"].dtype == torch.int32 and cc["labels"].shape == mt.shape and cc["labels"].device == dev
    assert largest.dtype == torch.int64 and largest.shape == mt.shape
    rows = 1 if method == "3d" else m.shape[0]
    assert cc["count"].shape == (rows, C) and cc["largest"].shape == (rows, C) and cc["count"].dtype == torch.int64
    stats = torch.stack((cc["count"], cc["largest"]), -1)
    return cc["labels"].cpu().numpy(), stats.cpu().numpy(), largest.cpu().numpy()


def assert_equal_to_oracle(got, m, C, method, conn):
    want = OC.components(m, C, method, conn)
    for g, w, name in zip(got, want, ("labels", "stats", "largest")):
        assert g.dtype == w.dtype and g.shape == w.shape, name
        if not np.array_equal(g, w):
            bad = np.argwhere(g != w)
            raise AssertionError(f"{name}: {len(bad)} entries differ, first at {bad[0].tolist()}: "
                                 f"{g[tuple(bad[0])]} vs {w[tuple(bad[0])]}")


def maps(shape, C, kind, seed):
    rng = np.random.default_rng(seed)
    return (OH.blobs if kind == "blobs" else OH.salt_pepper)(rng, shape, C)


def _grid():
    out = [(shape, C, m, c) for shape, C in HD_CASES for m, c in METHOD_CONN]
    out += [(SPLEEN_VOLUME[0], SPLEEN_VOLUME[1], "3d", c) for c in (1, 2, 3)]
    return out


@pytest.mark.parametrize("kind", ["blobs", "saltpepper"])
@pytest.mark.parametrize("shape,C,method,conn", _grid())
def test_components_vs_oracle(shape, C, method, conn, kind, dct, dev):
    m = maps(shape, C, kind, seed=C * 1000 + shape[1] + shape[0])
    assert_equal_to_oracle(run(dct, m, C, method, conn, dev), m, C, method, conn)


# ---- adversarial maps for the union-find -------------------------------------------------------------------------------

def serpentine(shape):
    """Class 1 on a one-pixel-wide path through every row pair of every slice (turning at alternate ends), class 0
    elsewhere; in a volume every odd slice joins the ends of the paths below and above it with a single pixel."""
    B, H, W = shape
    m = np.zeros(shape, np.int64)
    for b in range(0, B, 2):
        m[b, 0::2, :] = 1
        for y in range(1, H, 2):
            m[b, y, W - 1 if y % 4 == 1 else 0] = 1
        if b + 1 < B:
            m[b + 1, H - 1 if (H - 1) % 2 == 0 else H - 2, 0] = 1
    return m


def checkerboard(shape):
    z, y, x = np.indices(shape)
    return ((z + y + x) % 2).astype(np.int64)


def tile_stripes(shape):
    """One-pixel stripes on both sides of every 16- and 32-pixel boundary, along x (class 1) and y (class 2; 3 where they
    cross), and a slice of class 1 on both sides of every 4-slice boundary."""
    z, y, x = np.indices(shape)
    m = np.isin(x % 16, (0, 15)).astype(np.int64) + 2 * np.isin(y % 16, (0, 15))
    m[np.isin(z % 4, (0, 3)) & (m == 0) & (x % 3 == 0)] = 1
    return m


def columns(shape):
    """Isolated pixels of class 1 at the same (y, x) in every slice: one component per pixel for '2d', one per column
    for '3d'."""
    z, y, x = np.indices(shape)
    return ((y % 4 == 1) & (x % 5 == 2)).astype(np.int64)


def corners(shape):
    """Pairs of pixels that touch only through a tile corner: (15, 15) / (16, 16) inside a slice, and across slices
    (3, 15, 15) / (4, 16, 16) of a 4 x 16 x 16 brick, plus the same on the 32-pixel boundaries of the slice tiles."""
    m = np.zeros(shape, np.int64)

    def put(z, y, x, c):
        if z < shape[0] and y < shape[1] and x < shape[2]:
            m[z, y, x] = c

    for z0 in range(0, shape[0], 4):
        put(z0, 15, 15, 1); put(z0, 16, 16, 1)
        put(z0, 31, 31, 1); put(z0, 32, 32, 1)
        put(z0, 31, 32, 2); put(z0, 32, 31, 2)
        put(z0 + 3, 47, 47, 1); put(z0 + 4, 48, 48, 1)
        put(z0 + 3, 48, 47, 2); put(z0 + 4, 47, 48, 2)
    return m


ADVERSARIAL = {"serpentine": serpentine, "checkerboard": checkerboard, "tile_stripes": tile_stripes,
               "columns": columns, "corners": corners}


@pytest.mark.parametrize("method,conn", METHOD_CONN)
@pytest.mark.parametrize("shape", [(8, 96, 160), (13, 67, 41), (5, 256, 512)])
@pytest.mark.parametrize("name", sorted(ADVERSARIAL))
def test_adversarial_maps(name, shape, method, conn, dct, dev):
    m = ADVERSARIAL[name](shape)
    C = 4 if name == "tile_stripes" else 3
    got = run(dct, m, C, method, conn, dev)
    assert_equal_to_oracle(got, m, C, method, conn)
    stats = got[1]
    if name == "serpentine" and method == "3d":
        assert stats[0, 1, 0] == 1 and stats[0, 1, 1] == int((m == 1).sum())   # one path through every tile
    if name == "checkerboard":
        if conn == 1:
            assert np.all(stats[:, 1, 1] == 1)                      # one component per pixel
        else:
            assert np.all(stats[:, :2, 0] == 1)                     # one per colour, joined through diagonals only
    if name == "columns":
        assert np.all(stats[:, 1, 0] == int((m[0] == 1).sum()))   # per slice, or one column per (y, x)
        assert np.all(stats[:, 1, 1] == (shape[0] if method == "3d" else 1))


def test_serpentine_spleen_volume(dct, dev):
    m = serpentine(SPLEEN_VOLUME[0])
    for method, conn in (("3d", 1), ("3d", 3), ("2d", 2)):
        assert_equal_to_oracle(run(dct, m, 2, method, conn, dev), m, 2, method, conn)


def test_tie_goes_to_the_first_component(dct, dev):
    m = np.zeros((2, 40, 70), np.int64)
    m[:, 30, 0:5] = 1        # same size, later first pixel
    m[:, 2, 60:65] = 1       # first in raster order: kept
    m[:, 10:12, 40] = 2
    m[:, 20:22, 10] = 2
    for method, conn in METHOD_CONN:
        got = run(dct, m, 3, method, conn, dev)
        assert_equal_to_oracle(got, m, 3, method, conn)
        assert np.all(got[2][:, 30, 0:5] == 0) and np.all(got[2][:, 2, 60:65] == 1) and np.all(got[2][:, 20:22, 10] == 0)


def test_out_of_range_values_flag_and_pass_through(dct, dev):
    C = 4
    m = maps((4, 37, 29), C, "blobs", seed=5)
    m[0, 3, 4] = C; m[2, 10, 0] = -1; m[3, 36, 28] = C + 7
    st = dct._runtime.state(dev)
    for method, conn in METHOD_CONN:
        with dct._runtime.check_mode("deferred"):
            st.flags.zero_()
            got = run(dct, m, C, method, conn, dev)
            flags = st.flags.cpu().numpy()
            st.flags.zero_()
        assert flags[dct._lib.FLAG_PRED] == 2 * 3   # two calls, three values
        assert flags[dct._lib.FLAG_LABEL] == 0 and flags[dct._lib.FLAG_SIMPLEX] == 0 and flags[dct._lib.FLAG_ONEHOT] == 0
        assert got[0][0, 3, 4] == -1 and got[2][0, 3, 4] == C and got[2][2, 10, 0] == -1 and got[2][3, 36, 28] == C + 7
        assert_equal_to_oracle(got, m, C, method, conn)
    if dct.get_check_mode() == "eager":
        with pytest.raises(AssertionError):
            dct.largest_component(T(m, dev), C=C)


@pytest.mark.parametrize("C", [2, 4, 19])
def test_scores_path_equals_class_map_path(C, dct, dev):
    gen = torch.Generator().manual_seed(C)
    x = (3 * torch.randn(3, C, 45, 38, generator=gen)).to(dev)
    x[0, :, 0, 0] = 0.0   # ties resolve as DiceMeter's arg-max does
    cls = dct.utils._classmap(x, 1, want_cls=True)[0]
    for method, conn in METHOD_CONN:
        a = dct.connected_components(x, method=method, connectivity=conn)
        b = dct.connected_components(cls[:, None], C=C, method=method, connectivity=conn)
        for k in ("labels", "count", "largest"):
            assert torch.equal(a[k], b[k]), k
        assert torch.equal(dct.largest_component(x, method=method, connectivity=conn),
                           dct.largest_component(cls, C=C, method=method, connectivity=conn))


def _abi_buffers(B, H, W, C, volume, dev):
    rows = 1 if volume else B
    return (torch.full((B, H, W), -7, dtype=torch.int32, device=dev),
            torch.full((rows, C, 2), -7, dtype=torch.int64, device=dev),
            torch.full((B, H, W), -7, dtype=torch.int64, device=dev))


@pytest.mark.parametrize("method,conn", [("2d", 2), ("3d", 3)])
def test_every_null_output_combination(method, conn, dct, dev):
    C, (B, H, W) = 4, (6, 70, 90)
    m = maps((B, H, W), C, "blobs", seed=8)
    m[1, 2, 3] = 9
    want = OC.components(m, C, method, conn)
    h = dct._lib.lib()
    volume = int(method == "3d")
    mt = T(m, dev)
    scratch = torch.empty(h.dct_components_scratch_bytes(C, B, H, W, volume), dtype=torch.uint8, device=dev)
    stream = torch.cuda.current_stream(dev).cuda_stream
    for mask in range(8):
        bufs = _abi_buffers(B, H, W, C, volume, dev)
        ptrs = [b.data_ptr() if mask >> i & 1 else None for i, b in enumerate(bufs)]
        rc = h.dct_components_i64(mt.data_ptr(), C, B, H, W, volume, conn, *ptrs, None, scratch.data_ptr(), stream)
        torch.cuda.synchronize(dev)
        if mask == 0:
            assert rc == -1   # DCT_ERR_BAD_ARG: no output asked for
            continue
        assert rc == 0, mask
        for i, (b, w) in enumerate(zip(bufs, want)):
            got = b.cpu().numpy()
            if mask >> i & 1:
                assert np.array_equal(got, w), (mask, i)
            else:
                assert np.all(got == -7), (mask, i)


def test_argument_errors_launch_nothing(dct, dev):
    h = dct._lib.lib()
    B, H, W, C = 2, 8, 8, 3
    mt = T(np.zeros((B, H, W), np.int64), dev)
    labels, stats, largest = _abi_buffers(B, H, W, C, 0, dev)
    scratch = torch.empty(h.dct_components_scratch_bytes(C, B, H, W, 1) + 256, dtype=torch.uint8, device=dev)
    stream = torch.cuda.current_stream(dev).cuda_stream

    def call(C=C, B=B, H=H, W=W, volume=0, conn=1, m=mt.data_ptr(), lab=labels.data_ptr(), st=stats.data_ptr(),
             big=largest.data_ptr(), sc=scratch.data_ptr()):
        return h.dct_components_i64(m, C, B, H, W, volume, conn, lab, st, big, None, sc, stream)

    assert call(conn=0) == -1 and call(conn=3) == -1 and call(volume=1, conn=4) == -1 and call(volume=1, conn=0) == -1
    assert call(C=0) == -1 and call(m=None) == -1 and call(sc=None) == -1 and call(lab=None, st=None, big=None) == -1
    assert call(big=mt.data_ptr()) == -1 and call(big=mt.data_ptr() + 8 * (B * H * W - 1)) == -1   # overlaps the input
    assert call(C=65) == -2 and call(B=1 << 16, H=1 << 8, W=1 << 7) == -2                          # 2^31 pixels
    assert h.dct_components_scratch_bytes(65, B, H, W, 0) == 0
    assert h.dct_components_scratch_bytes(C, 1 << 16, 1 << 8, 1 << 7, 1) == 0
    assert h.dct_components_scratch_bytes(C, 1 << 16, 1 << 8, (1 << 7) - 1, 1) > 0
    assert call(lab=labels.data_ptr() + 2) == -3 and call(big=largest.data_ptr() + 4) == -3
    assert call(st=stats.data_ptr() + 4) == -3 and call(sc=scratch.data_ptr() + 128) == -3
    torch.cuda.synchronize(dev)
    for b in (labels, stats, largest):
        assert bool((b == -7).all())   # nothing was launched
    assert call() == 0 and call(volume=1, conn=3) == 0
    torch.cuda.synchronize(dev)
    assert bool((largest == 0).all()) and bool((labels == 0).all())


def test_two_calls_are_bit_identical(dct, dev):
    for kind in ("blobs", "saltpepper"):
        mt = T(maps((16, 256, 384), 19, kind, seed=2), dev)
        for method, conn in METHOD_CONN:
            a = dct.connected_components(mt, C=19, method=method, connectivity=conn)
            b = dct.connected_components(mt, C=19, method=method, connectivity=conn)
            for k in a:
                assert torch.equal(a[k], b[k]), (kind, method, conn, k)
            assert torch.equal(dct.largest_component(mt, C=19, method=method, connectivity=conn),
                               dct.largest_component(mt, C=19, method=method, connectivity=conn))


@pytest.mark.parametrize("method,conn", [("2d", 1), ("3d", 3)])
def test_cuda_graph_capture_and_replay(method, conn, dct, dev):
    C, shape = 4, (6, 64, 80)
    m0, m1 = maps(shape, C, "blobs", seed=9), maps(shape, C, "saltpepper", seed=10)
    mt = T(m0, dev)
    s = torch.cuda.Stream(dev)
    with dct._runtime.check_mode("deferred"):
        s.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(s):   # warm-up on the capture stream
            dct.connected_components(mt, C=C, method=method, connectivity=conn)
            dct.largest_component(mt, C=C, method=method, connectivity=conn)
        torch.cuda.current_stream(dev).wait_stream(s)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=s):
            cc = dct.connected_components(mt, C=C, method=method, connectivity=conn)
            big = dct.largest_component(mt, C=C, method=method, connectivity=conn)
        for m in (m0, m1):
            mt.copy_(T(m, dev))
            graph.replay()
            torch.cuda.synchronize(dev)
            stats = torch.stack((cc["count"], cc["largest"]), -1)
            assert_equal_to_oracle((cc["labels"].cpu().numpy(), stats.cpu().numpy(), big.cpu().numpy()), m, C, method,
                                   conn)


@pytest.mark.parametrize("method,conn", [("2d", 2), ("3d", 1), ("3d", 3)])
def test_scratch_query_is_sufficient(method, conn, dct, dev):
    """The call stays inside the queried scratch (a canary behind it survives) and needs no initial state in it: the
    scratch starts as 0xAB bytes and is reused as the previous call left it, for another map."""
    C, (B, H, W) = 19, (3, 70, 90)
    h = dct._lib.lib()
    volume = int(method == "3d")
    nbytes = h.dct_components_scratch_bytes(C, B, H, W, volume)
    assert nbytes >= 9 * B * H * W
    buf = torch.full((nbytes + 4096,), 0xAB, dtype=torch.uint8, device=dev)
    stream = torch.cuda.current_stream(dev).cuda_stream
    for seed, kind in ((4, "saltpepper"), (5, "blobs"), (6, "saltpepper")):
        m = maps((B, H, W), C, kind, seed)
        mt = T(m, dev)
        bufs = _abi_buffers(B, H, W, C, volume, dev)
        assert h.dct_components_i64(mt.data_ptr(), C, B, H, W, volume, conn, *[b.data_ptr() for b in bufs], None,
                                    buf.data_ptr(), stream) == 0
        torch.cuda.synchronize(dev)
        assert_equal_to_oracle([b.cpu().numpy() for b in bufs], m, C, method, conn)
        assert bool((buf[nbytes:] == 0xAB).all())


@pytest.mark.parametrize("method", ["2d", "3d"])
def test_surface_distances_of_the_largest_component(method, dct, dev):
    C = 4
    rng = np.random.default_rng(12)
    g = OH.blobs(rng, (10, 96, 96), C)
    p = g.copy()
    noise = rng.random(p.shape) < 0.002    # stray islands far from the organs: HD moves a lot with the post-processing
    p[noise] = rng.integers(1, C, size=int(noise.sum()))
    sp = (10.0, 1.5625, 1.5625) if method == "3d" else (1.5625, 1.5625)
    conn = 3 if method == "3d" else 2
    x = torch.nn.functional.one_hot(T(p, dev), C).permute(0, 3, 1, 2).float() * 4.0   # scores whose arg-max is p
    big = dct.largest_component(x, method=method, connectivity=conn)
    want_big = OC.components(p, C, method, conn)[2]
    assert np.array_equal(big.cpu().numpy(), want_big)
    got = dct.surface_distances(dct.largest_component(x, method=method, connectivity=conn), T(g, dev), C=C,
                                method=method, voxelspacing=sp)
    assert_surface_matches(got, OS.surface(want_big, g, C, method, sp), False)
    got_unit = dct.surface_distances(big, T(g, dev), C=C, method=method)
    assert_surface_matches(got_unit, OS.surface(want_big, g, C, method), True)


def test_invalid_connectivity_raises(dct, dev):
    mt = T(np.zeros((2, 5, 5), np.int64), dev)
    with pytest.raises(dct.DctError):
        dct.largest_component(mt, C=2, method="2d", connectivity=3)
    with pytest.raises(dct.DctError):
        dct.connected_components(mt, C=2, method="3d", connectivity=0)
