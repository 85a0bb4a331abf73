"""Every host-side launch path of the loss and metric families, reached on purpose, named, and checked.

The host dispatch picks a kernel from C, from HW mod 4 / mod 2, from the 16 / 8 / 4-byte alignment of every pointer
(labels and outputs included) and from B.  Tensors straight from the allocator are always 16-byte aligned, so most of
these paths are only reached by shape (odd HW, HW = 2 mod 4, C outside {2, 3, 4, 19}) or by a view that starts inside
a larger buffer: a batch split ``logits[B_l:]``, a row tensor ``(N, C)``, an offset carved out of a flat allocation.

Each matrix row below
  * names the kernel its dispatch must reach and asserts it from a torch.profiler trace of one call (and, for rows
    meant to leave the tile pipeline, that no ``dct::tile_kernel`` ran), so that a dispatch change cannot move a
    test onto another path unnoticed;
  * compares floating results with the float64 oracle at util.RTOL_FP32 and integer results bit-exactly;
  * runs the call twice and requires bit-identical loss sums and maps.

The batch-boundary tests cover the loss sums for B > 8192 (kMaxPartials): the grid of the non-tile kernels is capped
at 8192 CTAs, one workspace partial each, and the kernels stride over images.  DESIGN.md section 3.10 lists the paths
and the rows that reach them.
"""
import ctypes
import zlib

import numpy as np
import pytest
import torch

from util import assert_close, lnK

pytestmark = pytest.mark.gpu

OK, ERR_UNSUPPORTED = 0, -2
IN_PROBS, IN_LOGITS = 0, 1
EPS = 1e-10
TILE = "dct::tile_kernel<"
# Workspace layout (csrc/dct_common.cuh, struct Workspace): a 64-byte header, kMaxPartials doubles of CTA partials,
# then the l2 exchange area (l2_epoch, l2_ticket, padding, l2_slots) that only the one-launch l2 normalisation writes.
WS_HEADER, MAX_PARTIALS = 64, 8192
WS_L2_OFFSET = WS_HEADER + 8 * MAX_PARTIALS
CANARY_BYTES = 512 * 1024


@pytest.fixture(scope="module")
def h():
    import dct_b200
    assert torch.cuda.is_available()
    lib = dct_b200._lib.lib()
    assert lib.dct_device_check(0) == 0
    return lib


DEV = torch.device("cuda:0")


def _s():
    return torch.cuda.current_stream(DEV).cuda_stream


def N(t):
    return t.detach().cpu().numpy()


def carve(a, off):
    """A device copy of `a`, placed `off` elements into a fresh allocation (the caching allocator's blocks are
    512-byte aligned, so the copy's address has exactly the alignment off * itemsize gives)."""
    a = np.ascontiguousarray(a)
    t = torch.from_numpy(a.reshape(-1)).to(DEV)
    buf = torch.zeros(a.size + off, dtype=t.dtype, device=DEV)
    buf[off:] = t
    v = buf[off:]
    assert v.data_ptr() % 16 == (off * a.itemsize) % 16
    return v


def carve_views(arrs, off):
    """K equally shaped float32 views consecutive in ONE flat buffer, the first `off` elements into it."""
    flat = carve(np.concatenate([np.ascontiguousarray(a, np.float32).reshape(-1) for a in arrs]), off)
    n = arrs[0].size
    return [flat[k * n:(k + 1) * n] for k in range(len(arrs))]


def empty(n, off, dtype=torch.float32):
    buf = torch.full((n + off,), float("nan") if dtype.is_floating_point else -1, dtype=dtype, device=DEV)
    return buf[off:]


def ptrs(ts):
    return (ctypes.c_void_p * len(ts))(*[t.data_ptr() for t in ts])


def kernels(fn):
    """Run `fn` once to warm up, then once under torch.profiler; returns (names of the kernels of the profiled call,
    what the warm-up call returned, what the profiled call returned)."""
    from torch.profiler import ProfilerActivity, profile
    first = fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA], acc_events=True) as prof:
        second = fn()
        torch.cuda.synchronize()
    names = sorted({e.key for e in prof.key_averages() if "dct::" in e.key})
    return names, first, second


def assert_path(names, want, off_tile=True):
    wants = [want] if isinstance(want, str) else list(want)
    for w in wants:
        assert any(w in n for n in names), f"expected a launch of {w!r}; the call launched {names}"
    if off_tile:
        assert not any(TILE in n for n in names), f"this row must leave the tile pipeline; launched {names}"


def rng(*key):
    return np.random.default_rng(zlib.crc32(repr(key).encode()))


def logits(r, *shape):
    return (3.0 * r.standard_normal(shape)).astype(np.float32)


def probs_of(z):
    """float32 probabilities (softmax in float64, rounded once)."""
    z = z.astype(np.float64)
    e = np.exp(z - z.max(1, keepdims=True))
    return (e / e.sum(1, keepdims=True)).astype(np.float32)


def f64(a):
    return np.asarray(a, dtype=np.float64)


def close_sum(got, want_map, floor, what):
    """A loss sum against the float64 sum of the oracle's map, scaled per pixel."""
    n = want_map.size
    assert_close(got / n, float(want_map.sum(dtype=np.float64)) / n, floor=floor, what=what)


# ---------------------------------------------------------------------------------------------
# JSD: tile_kernel<JsdOp..> -> jsd_kernel<K, C, VEC, ..> (VEC = jsd_vec<K, C>) -> jsd_kernel_rt
# ---------------------------------------------------------------------------------------------
# id, K, C, H, W, element offset of the views, element offset of the outputs (map, grads), expected kernel
JSD_ROWS = [
    ("k2c19_hw2mod4", 2, 19, 37, 42, 0, 0, "dct::jsd_kernel<2, 19, 2,"),
    ("k2c19_views8B", 2, 19, 32, 32, 2, 0, "dct::jsd_kernel<2, 19, 2,"),
    ("k2c19_out8B", 2, 19, 32, 32, 0, 2, "dct::jsd_kernel<2, 19, 2,"),
    ("k2c19_views4B", 2, 19, 32, 32, 1, 0, "dct::jsd_kernel_rt<"),
    ("k2c19_out4B", 2, 19, 32, 32, 0, 1, "dct::jsd_kernel_rt<"),
    ("k3c19_oddhw", 3, 19, 31, 33, 0, 0, "dct::jsd_kernel<3, 19, 1,"),
    ("k3c19_views4B", 3, 19, 32, 32, 1, 0, "dct::jsd_kernel<3, 19, 1,"),
    ("k4c19_oddhw", 4, 19, 31, 33, 0, 0, "dct::jsd_kernel<4, 19, 1,"),
    ("k4c19_views12B", 4, 19, 32, 32, 3, 0, "dct::jsd_kernel<4, 19, 1,"),
    ("k2c4_hw2mod4", 2, 4, 37, 42, 0, 0, "dct::jsd_kernel_rt<"),
    ("k3c3_views8B", 3, 3, 32, 32, 2, 0, "dct::jsd_kernel_rt<"),
    ("k2c2_out12B", 2, 2, 32, 32, 0, 3, "dct::jsd_kernel_rt<"),
    ("k2c5", 2, 5, 32, 32, 0, 0, "dct::jsd_kernel_rt<"),
    ("k5c4", 5, 4, 32, 32, 0, 0, "dct::jsd_kernel_rt<"),
    ("k2c19_tile", 2, 19, 32, 32, 0, 0, TILE),
]


@pytest.mark.parametrize("mode", ["fwd", "bwd", "fwdbwd"])
@pytest.mark.parametrize("kind", ["probs", "logits"])
@pytest.mark.parametrize("row", JSD_ROWS, ids=[r[0] for r in JSD_ROWS])
def test_jsd_launch_paths(row, kind, mode, h, oracle):
    name, K, C, H, W, voff, ooff, want = row
    B, HW = 2, H * W
    r = rng(name, kind, mode)
    z = [logits(r, B, C, H, W) for _ in range(K)]
    x = [probs_of(t) for t in z] if kind == "probs" else z
    p64 = [f64(t) for t in x] if kind == "probs" else [oracle.softmax(f64(t)) for t in z]
    views = carve_views(x, voff)
    grads = carve_views([np.zeros_like(t) for t in x], ooff) if mode != "fwd" else None
    mp = empty(B * HW, ooff) if mode != "bwd" else None
    gmap = carve(r.standard_normal((B, H, W)).astype(np.float32), 0) if mode == "bwd" else None
    gconst = 0.37
    sm = torch.zeros(1, dtype=torch.float64, device=DEV)
    flags = torch.zeros(4, dtype=torch.int32, device=DEV)
    ws = torch.zeros(int(h.dct_workspace_bytes()), dtype=torch.uint8, device=DEV)
    ik = IN_PROBS if kind == "probs" else IN_LOGITS
    vp = ptrs(views)
    gp = ptrs(grads) if grads is not None else None

    def call():
        if mode == "fwd":
            rc = h.dct_jsd_fwd_f32(vp, K, C, B, HW, ik, mp.data_ptr(), sm.data_ptr(), flags.data_ptr(), ws.data_ptr(), _s())
        elif mode == "bwd":
            rc = h.dct_jsd_bwd_f32(vp, K, C, B, HW, ik, gmap.data_ptr(), None, 1.0, gp, _s())
        else:
            rc = h.dct_jsd_fwdbwd_f32(vp, K, C, B, HW, ik, gconst, mp.data_ptr(), sm.data_ptr(), gp, None, None, 0,
                                      flags.data_ptr(), ws.data_ptr(), _s())
        assert rc == OK, rc
        return (sm.item() if mode != "bwd" else None, N(mp).copy() if mp is not None else None)

    names, (s1, m1), (s2, m2) = kernels(call)
    assert_path(names, want, off_tile=want != TILE)
    assert int(flags.sum()) == 0
    want_map = oracle.jsd_fwd(p64)
    if mode != "bwd":
        assert_close(m2.reshape(B, H, W), want_map, floor=lnK(K), what="map")
        close_sum(s2, want_map, lnK(K), "sum")
        assert s1 == s2 and np.array_equal(m1, m2, equal_nan=True), "two calls on one path differ"
    if mode != "fwd":
        gout = f64(N(gmap)).reshape(B, H, W) if mode == "bwd" else np.full((B, H, W), gconst)
        want_gp = oracle.jsd_bwd(p64, gout)
        if kind == "logits":
            want_gp = [oracle.softmax_bwd(p64[k], want_gp[k]) for k in range(K)]
        got = np.stack([N(g).reshape(B, C, H, W) for g in grads])
        assert_close(got, np.stack(want_gp), floor=float(np.abs(gout).max()), what="grads")


# ---------------------------------------------------------------------------------------------
# KL family, entropy, softmax: tile_kernel<Op..> -> pix_kernel<Op, CT, VEC> -> pix_kernel<Op, 0, 1>
# ---------------------------------------------------------------------------------------------
# id, C, H, W, element offset of the inputs, of the outputs, (CT, VEC) of the expected pix_kernel (None: the tile)
PIX_ROWS = [
    ("c19_hw2mod4", 19, 37, 42, 0, 0, (19, 2)),
    ("c19_in8B", 19, 32, 32, 2, 0, (19, 2)),
    ("c19_out8B", 19, 32, 32, 0, 2, (19, 2)),
    ("c19_in4B", 19, 32, 32, 1, 0, (0, 1)),
    ("c19_oddhw", 19, 31, 33, 0, 0, (0, 1)),
    ("c4_hw2mod4", 4, 37, 42, 0, 0, (0, 1)),
    ("c4_out12B", 4, 32, 32, 0, 3, (0, 1)),
    ("c5", 5, 32, 32, 0, 0, (0, 1)),
    ("c19_tile", 19, 32, 32, 0, 0, None),
]


def _pix_case(op, C, B, H, W, r, g, oracle):
    """The float32 inputs of one op and its float64 reference under the upstream map `g`.  Returns
    (op struct name, inputs, number of outputs, has map, uses gmap, reference() -> (map, [outputs]))."""
    z0, z1 = logits(r, B, C, H, W), logits(r, B, C, H, W)
    p, y = probs_of(z0), probs_of(z1)
    g = f64(g)
    if op == "kl_fwd":
        return "KlProbFwd", [p, y], 0, True, False, lambda: (oracle.kl_fwd(f64(p), f64(y), EPS), [])
    if op == "kl_bwd":
        return "KlProbBwd<true>", [p, y], 2, False, True, lambda: (None, list(oracle.kl_bwd(f64(p), f64(y), g, EPS)))
    if op == "kl_logit_fwd":
        return "KlLogit<false>", [z0, z1], 0, True, False, lambda: (oracle.kl_logit(f64(z0), f64(z1))[0], [])
    if op == "kl_logit_fwdbwd":
        def ref():
            m, gpl, gql = oracle.kl_logit(f64(z0), f64(z1), g)
            return m, [gql, gpl]
        return "KlLogit<true>", [z0, z1], 2, True, True, ref
    if op == "kl_from_logits":
        def ref():
            pp = oracle.softmax(f64(z0))
            gp = oracle.kl_bwd(pp, f64(y), np.full((B, H, W), 0.37), EPS)[0]
            return oracle.kl_fwd(pp, f64(y), EPS), [oracle.softmax_bwd(pp, gp)]
        return "KlFromLogits", [z0, y], 1, True, False, ref
    if op == "kl_div_fwd":
        return "KlDivFwd", [p, y], 0, True, False, lambda: (oracle.kl_div_fwd(f64(p), f64(y), EPS), [])
    if op == "kl_div_bwd":
        return "KlDivBwd<true>", [p, y], 2, False, True, lambda: (None, list(oracle.kl_div_bwd(f64(p), f64(y), g, EPS)))
    if op == "entropy_fwd":
        return "EntropyFwd", [p], 0, True, False, lambda: (oracle.entropy(f64(p)), [])
    if op == "entropy_bwd":
        return "EntropyBwd", [p], 1, False, True, lambda: (None, [oracle.entropy_bwd(f64(p), g)])
    if op == "softmax_fwd":
        return "SoftmaxFwd", [z0], 1, False, False, lambda: (None, [oracle.softmax(f64(z0))])
    if op == "softmax_bwd":
        gpp = r.standard_normal((B, C, H, W)).astype(np.float32)
        return "SoftmaxBwd", [p, gpp], 1, False, False, lambda: (None, [oracle.softmax_bwd(f64(p), f64(gpp))])
    raise AssertionError(op)


PIX_OPS = ["kl_fwd", "kl_bwd", "kl_logit_fwd", "kl_logit_fwdbwd", "kl_from_logits", "kl_div_fwd", "kl_div_bwd",
           "entropy_fwd", "entropy_bwd", "softmax_fwd", "softmax_bwd"]


@pytest.mark.parametrize("op", PIX_OPS)
@pytest.mark.parametrize("row", PIX_ROWS, ids=[r[0] for r in PIX_ROWS])
def test_pixelwise_launch_paths(row, op, h, oracle):
    name, C, H, W, ioff, ooff, ctv = row
    B, HW = 2, H * W
    r = rng(name, op)
    g = r.standard_normal((B, H, W)).astype(np.float32)
    opname, ins, nout, has_map, uses_gmap, ref = _pix_case(op, C, B, H, W, r, g, oracle)
    xs = carve_views(ins, ioff)
    outs = carve_views([np.zeros_like(ins[0])] * nout, ooff) if nout else []
    mp = empty(B * HW, ooff) if has_map else None
    gmap = carve(g, 0) if uses_gmap else None
    sm = torch.zeros(1, dtype=torch.float64, device=DEV)
    flags = torch.zeros(4, dtype=torch.int32, device=DEV)
    ws = torch.zeros(int(h.dct_workspace_bytes()), dtype=torch.uint8, device=DEV)
    P = lambda t: None if t is None else t.data_ptr()  # noqa: E731
    o0 = outs[0] if nout > 0 else None
    o1 = outs[1] if nout > 1 else None
    a0 = xs[0]
    a1 = xs[1] if len(xs) > 1 else None
    s = _s()

    def call():
        if op == "kl_fwd":
            rc = h.dct_kl_fwd_f32(P(a0), P(a1), C, B, HW, EPS, P(mp), P(sm), P(flags), P(ws), s)
        elif op == "kl_bwd":
            rc = h.dct_kl_bwd_f32(P(a0), P(a1), C, B, HW, EPS, P(gmap), None, 1.0, P(o0), P(o1), s)
        elif op == "kl_logit_fwd":
            rc = h.dct_kl_logit_f32(P(a0), P(a1), C, B, HW, P(mp), P(sm), 0, None, None, 1.0, None, None, P(ws), s)
        elif op == "kl_logit_fwdbwd":   # outputs: grad of q_logit (in 0) first, then of p_logit
            rc = h.dct_kl_logit_f32(P(a0), P(a1), C, B, HW, P(mp), P(sm), 1, P(gmap), None, 1.0, P(o1), P(o0), P(ws), s)
        elif op == "kl_from_logits":
            rc = h.dct_kl_from_logits_fwdbwd_f32(P(a0), P(a1), C, B, HW, EPS, 0.37, P(mp), P(sm), P(o0), P(flags), P(ws), s)
        elif op == "kl_div_fwd":
            rc = h.dct_kl_div_fwd_f32(P(a0), P(a1), C, B, HW, EPS, P(mp), P(sm), P(flags), P(ws), s)
        elif op == "kl_div_bwd":
            rc = h.dct_kl_div_bwd_f32(P(a0), P(a1), C, B, HW, EPS, P(gmap), None, 1.0, P(o0), P(o1), s)
        elif op == "entropy_fwd":
            rc = h.dct_entropy_fwd_f32(P(a0), C, B, HW, P(mp), P(sm), P(flags), P(ws), s)
        elif op == "entropy_bwd":
            rc = h.dct_entropy_bwd_f32(P(a0), C, B, HW, P(gmap), None, 1.0, P(o0), s)
        elif op == "softmax_fwd":
            rc = h.dct_softmax_fwd_f32(P(a0), C, B, HW, P(o0), s)
        else:
            rc = h.dct_softmax_bwd_f32(P(a0), P(a1), C, B, HW, P(o0), s)
        assert rc == OK, rc
        return (sm.item() if has_map else None, N(mp).copy() if has_map else None)

    names, (s1, m1), (s2, m2) = kernels(call)
    if ctv is None:
        assert_path(names, TILE, off_tile=False)
    else:
        assert_path(names, f"dct::pix_kernel<dct::{opname}, {ctv[0]}, {ctv[1]}>")
    assert int(flags.sum()) == 0
    want_map, want_outs = ref()
    if has_map:
        assert_close(m2.reshape(B, H, W), want_map, floor=1.0, what="map")
        close_sum(s2, want_map, 1.0, "sum")
        assert s1 == s2 and np.array_equal(m1, m2, equal_nan=True), "two calls on one path differ"
    for k, w in enumerate(want_outs):
        assert_close(N(outs[k]).reshape(w.shape), w, floor=1.0, what=f"output {k}")



# ---------------------------------------------------------------------------------------------
# Cross-entropy: tile_kernel<CeOp..> -> ce_kernel_rt; the Dice counts / confusion of a non-fused call come from a
# second launch (dice_kernel<CT, VEC> / tile_kernel<DiceOp..>, confusion_kernel<CT, VEC>)
# ---------------------------------------------------------------------------------------------
RT, D01, C01 = "dct::ce_kernel_rt<", "dct::dice_kernel<0, 1>", "dct::confusion_kernel<0, 1>"
# id, C, H, W, element offsets of logits / labels / outputs (map, grad), expected kernels of
# fwd and bwd, of fwdbwd with Dice counts, of fwdbwd with the confusion matrix
CE_ROWS = [
    ("c5", 5, 32, 32, 0, 0, 0, [RT], [RT, D01], [RT, C01]),
    ("c4_hw2mod4", 4, 37, 42, 0, 0, 0, [RT], [RT, D01], [RT, C01]),
    ("c4_labels8B", 4, 32, 32, 0, 1, 0, [RT], [RT, D01], [RT, C01]),
    ("c4_logits4B", 4, 32, 32, 1, 0, 0, [RT], [RT, D01], [RT, C01]),
    ("c4_out4B", 4, 32, 32, 0, 0, 1, [RT], [RT, TILE], [RT, "dct::confusion_kernel<4, 4>"]),
    ("c19_hw2mod4", 19, 37, 42, 0, 0, 0, [RT], [RT, "dct::dice_kernel<19, 2>"], [RT, "dct::confusion_kernel<19, 2>"]),
    ("c19_logits8B", 19, 32, 32, 2, 0, 0, [RT], [RT, "dct::dice_kernel<19, 2>"], [RT, "dct::confusion_kernel<19, 2>"]),
    ("c19_labels8B", 19, 32, 32, 0, 1, 0, [RT], [RT, D01], [RT, C01]),
    ("c4_tile", 4, 32, 32, 0, 0, 0, [TILE], [TILE], [TILE]),
]


@pytest.mark.parametrize("mode", ["fwd", "bwd", "fwdbwd_dice", "fwdbwd_conf"])
@pytest.mark.parametrize("row", CE_ROWS, ids=[r[0] for r in CE_ROWS])
def test_cross_entropy_launch_paths(row, mode, h, oracle):
    name, C, H, W, xoff, loff, ooff, k_plain, k_dice, k_conf = row
    B, HW = 2, H * W
    r = rng(name, mode)
    z = logits(r, B, C, H, W)
    gt = r.integers(0, C, (B, H, W)).astype(np.int64)
    if mode != "fwdbwd_dice":   # Dice counting takes labels in [0, C); the other calls also see ignored pixels
        gt[r.random((B, H, W)) < 0.05] = 255
    g = r.standard_normal((B, H, W)).astype(np.float32)
    x = carve(z, xoff)
    lab = carve(gt, loff)
    mp = empty(B * HW, ooff)
    grad = empty(B * C * HW, ooff)
    gmap = carve(g, 0)
    sm = torch.zeros(1, dtype=torch.float64, device=DEV)
    flags = torch.zeros(4, dtype=torch.int32, device=DEV)
    ws = torch.zeros(int(h.dct_workspace_bytes()), dtype=torch.uint8, device=DEV)
    counts = torch.zeros(B * C * 3, dtype=torch.int64, device=DEV)
    conf = torch.zeros(C * C, dtype=torch.int64, device=DEV)
    gconst = 0.37
    s = _s()

    def call():
        if mode == "fwd":
            rc = h.dct_ce_fwd_f32(x.data_ptr(), lab.data_ptr(), C, B, HW, None, 255, mp.data_ptr(), sm.data_ptr(),
                                  flags.data_ptr(), ws.data_ptr(), s)
        elif mode == "bwd":
            rc = h.dct_ce_bwd_f32(x.data_ptr(), lab.data_ptr(), C, B, HW, None, 255, gmap.data_ptr(), None, 1.0,
                                  grad.data_ptr(), flags.data_ptr(), s)
        elif mode == "fwdbwd_dice":
            counts.zero_()
            rc = h.dct_ce_fwdbwd_f32(x.data_ptr(), lab.data_ptr(), C, B, HW, None, 255, None, gconst, mp.data_ptr(),
                                     sm.data_ptr(), grad.data_ptr(), counts.data_ptr(), flags.data_ptr(), ws.data_ptr(), s)
        else:
            conf.zero_()
            rc = h.dct_ce_fwdbwd_conf_f32(x.data_ptr(), lab.data_ptr(), C, B, HW, None, 255, None, gconst, mp.data_ptr(),
                                          sm.data_ptr(), grad.data_ptr(), conf.data_ptr(), flags.data_ptr(), ws.data_ptr(), s)
        assert rc == OK, rc
        return (sm.item(), N(mp).copy(), N(counts).copy(), N(conf).copy())

    names, (s1, m1, c1, f1), (s2, m2, c2, f2) = kernels(call)
    want = {"fwd": k_plain, "bwd": k_plain, "fwdbwd_dice": k_dice, "fwdbwd_conf": k_conf}[mode]
    assert_path(names, want, off_tile=TILE not in want)
    assert int(flags.sum()) == 0
    want_map, want_gmap_grad, _ = oracle.cross_entropy(f64(z), gt, reduction="none", gout=f64(g))
    if mode != "bwd":
        assert_close(m2.reshape(B, H, W), want_map, floor=1.0, what="map")
        close_sum(s2, want_map, 1.0, "sum")
        assert s1 == s2 and np.array_equal(m1, m2, equal_nan=True), "two calls on one path differ"
    if mode == "bwd":
        assert_close(N(grad).reshape(B, C, H, W), want_gmap_grad, floor=float(np.abs(g).max()), what="grad")
    elif mode != "fwd":
        _, want_grad, _ = oracle.cross_entropy(f64(z), gt, reduction="sum", upstream=gconst)
        assert_close(N(grad).reshape(B, C, H, W), want_grad, floor=gconst, what="grad")
    if mode == "fwdbwd_dice":
        oc, bad = oracle.dice_counts(z, gt)
        assert bad == 0 and np.array_equal(c2.reshape(B, C, 3), oc) and np.array_equal(c1, c2)
    if mode == "fwdbwd_conf":
        assert np.array_equal(f2.reshape(C, C), oracle.confusion(z, gt)) and np.array_equal(f1, f2)


# ---------------------------------------------------------------------------------------------
# Fused JSD + Dice with labels that are 8- but not 16-byte aligned: the tile launch drops the counting and the
# counts come from K launches of dice_kernel<0, 1>
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("overwrite", [False, True], ids=["accumulate", "overwrite"])
@pytest.mark.parametrize("K,C", [(2, 2), (2, 4), (3, 4)])
def test_jsd_fused_dice_with_misaligned_labels(K, C, overwrite, h, oracle):
    B, H, W = 2, 32, 32
    HW = H * W
    r = rng("jsd_dice", K, C, overwrite)
    z = [logits(r, B, C, H, W) for _ in range(K)]
    gt = r.integers(0, C, (B, H, W)).astype(np.int64)
    views = carve_views(z, 0)
    grads = carve_views([np.zeros_like(t) for t in z], 0)
    sm = torch.zeros(1, dtype=torch.float64, device=DEV)
    ws = torch.zeros(int(h.dct_workspace_bytes()), dtype=torch.uint8, device=DEV)
    flags = torch.zeros(4, dtype=torch.int32, device=DEV)
    pre = torch.full((K * B * C * 3,), 7 if overwrite else 0, dtype=torch.int64, device=DEV)
    counts = pre.clone()
    results = {}
    for loff in (0, 1):   # 16-byte aligned labels: counted inside the tile launch; 8-byte aligned: separate launches
        lab = carve(gt, loff)

        def call():
            counts.copy_(pre)
            rc = h.dct_jsd_fwdbwd_f32(ptrs(views), K, C, B, HW, IN_LOGITS, 0.5, None, sm.data_ptr(), ptrs(grads),
                                      lab.data_ptr(), counts.data_ptr(), int(overwrite), flags.data_ptr(), ws.data_ptr(),
                                      _s())
            assert rc == OK, rc
            return sm.item(), N(counts).copy()

        names, (s1, c1), (s2, c2) = kernels(call)
        assert_path(names, TILE, off_tile=False)
        if loff:
            assert_path(names, D01, off_tile=False)
        else:
            assert not any("dct::dice_kernel<" in n for n in names), names
        assert s1 == s2 and np.array_equal(c1, c2)
        results[loff] = (s2, c2)
    for k in range(K):
        oc, bad = oracle.dice_counts(z[k], gt)
        assert bad == 0
        assert np.array_equal(results[1][1].reshape(K, B, C, 3)[k], oc), f"separate Dice launches, view {k}"
    assert np.array_equal(results[0][1], results[1][1]), "fused and separate Dice counts differ"
    assert results[0][0] == results[1][0], "the loss sum depends on where the Dice counts are made"
    assert int(flags.sum()) == 0


# ---------------------------------------------------------------------------------------------
# Integer outputs: the same data through every path of dice / confusion / class map / vote, bit-identical and equal
# to the oracle (whose softmax arithmetic is pinned)
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("C", [3, 4, 19])
def test_integer_outputs_identical_across_paths(C, h, oracle):
    B, H, W = 2, 32, 32
    HW = H * W
    r = rng("int", C)
    z = logits(r, B, C, H, W)
    z[:, :, :4, :] = np.round(z[:, :, :4, :])   # exact ties and near-ties take the pinned slow path
    z[0, :, 5, :] = z[0, :1, 5, :]
    gt = r.integers(0, C, (B, H, W)).astype(np.int64)
    want_counts, bad = oracle.dice_counts(z, gt)
    assert bad == 0
    want_conf = oracle.confusion(z, gt)
    want_dice_cls = oracle.predict(z, "dice")
    want_raw_cls = oracle.predict(z, "raw")
    vec = 4 if C <= 8 else 2
    s = _s()
    # (x offset, labels offset) -> the Dice / confusion kernel the dispatch picks
    dice_paths = {(0, 0): TILE if C <= 4 else f"dct::dice_kernel<{C}, {vec}>", (0, 1): D01, (1, 0): D01}
    conf_paths = {(0, 0): f"dct::confusion_kernel<{C}, {vec}>", (0, 1): C01, (1, 0): C01}
    for (xoff, loff), want in dice_paths.items():
        x, lab = carve(z, xoff), carve(gt, loff)
        counts = torch.full((B * C * 3,), 5, dtype=torch.int64, device=DEV)
        names, _, _ = kernels(lambda: h.dct_dice_counts_f32(x.data_ptr(), lab.data_ptr(), C, B, HW, counts.data_ptr(),
                                                            0, None, s))
        assert_path(names, want, off_tile=want != TILE)
        assert np.array_equal(N(counts).reshape(B, C, 3), want_counts), f"dice counts, offsets {(xoff, loff)}"
    for (xoff, loff), want in conf_paths.items():
        x, lab = carve(z, xoff), carve(gt, loff)
        conf = torch.zeros(C * C, dtype=torch.int64, device=DEV)

        def call():
            conf.zero_()
            return h.dct_confusion_f32(x.data_ptr(), lab.data_ptr(), C, B, HW, conf.data_ptr(), s)
        names, _, _ = kernels(call)
        assert_path(names, want)
        assert np.array_equal(N(conf).reshape(C, C), want_conf), f"confusion, offsets {(xoff, loff)}"
    # class maps: <4> needs HW % 4 == 0 and 16-byte scores / int64 map / one-hot; offsets of x and of the map
    for mode, want_cls in ((1, want_dice_cls), (0, want_raw_cls)):   # ABI mode 1: pinned softmax, 0: raw
        for xoff, ooff, v in ((0, 0, 4), (1, 0, 1), (0, 1, 1)):
            x = carve(z, xoff)
            cls = empty(B * HW, ooff, torch.int64)
            oh = empty(B * C * HW, 0, torch.int32)
            names, _, _ = kernels(lambda: h.dct_classmap_f32(x.data_ptr(), C, B, HW, mode, cls.data_ptr(), None,
                                                             oh.data_ptr(), None, s))
            assert_path(names, f"dct::classmap_kernel<{v}, {mode}>")
            assert np.array_equal(N(cls).reshape(B, H, W), want_cls), f"class map mode {mode}, offsets {(xoff, ooff)}"
            want_oh = (want_cls[:, None] == np.arange(C)[None, :, None, None]).astype(np.int32)
            assert np.array_equal(N(oh).reshape(B, C, H, W), want_oh)
    # hard vote of three views: <4> / <1> by the alignment of the views and of the output
    zs = [z, logits(r, B, C, H, W), logits(r, B, C, H, W)]
    raw = np.stack([oracle.predict(t, "raw") for t in zs])
    want_vote = np.empty((B, H, W), np.int64)
    for idx in np.ndindex(B, H, W):
        v = raw[(slice(None),) + idx]
        n = np.bincount(v, minlength=C)
        want_vote[idx] = int(np.flatnonzero(n == n.max())[0])   # most votes, smallest class on ties
    for voff, ooff, v in ((0, 0, 4), (1, 0, 1), (0, 1, 1)):
        views = carve_views(zs, voff)
        cls = empty(B * HW, ooff, torch.int64)
        names, _, _ = kernels(lambda: h.dct_vote_f32(ptrs(views), 3, C, B, HW, 1, None, cls.data_ptr(), None, s))
        assert_path(names, f"dct::vote_hard_kernel<{v}>")
        assert np.array_equal(N(cls).reshape(B, H, W), want_vote), f"hard vote, offsets {(voff, ooff)}"


# ---------------------------------------------------------------------------------------------
# Loss sums for B > kMaxPartials through the C ABI, with a workspace the test owns: zeroed, followed by 512 KiB of
# 0xAB canary.  The workspace bytes after `partials` (the l2 exchange area) must come back unchanged.
# ---------------------------------------------------------------------------------------------
BATCHES = [8191, 8192, 8193, 40000, 65535]
# entry point -> kinds of its two inputs ("p" probabilities, "z" logits, "-" unused)
SUM_OPS = {"jsd_fwd": "pp", "jsd_fwdbwd": "zz", "ce_fwd": "z-", "ce_fwdbwd": "z-", "kl_fwd": "pp", "kl_logit": "zz",
           "kl_from_logits": "zp", "kl_div_fwd": "pp", "entropy_fwd": "p-"}


def _sum_call(op, h, C, B, HW, bufs, ws):
    """Calls `op` with the loss sum into bufs['sum']; returns its status."""
    a, b, g0, g1, lab = bufs["a"], bufs["b"], bufs["g0"], bufs["g1"], bufs["lab"]
    sm, s = bufs["sum"].data_ptr(), _s()
    P = lambda t: t.data_ptr()  # noqa: E731
    if op == "jsd_fwd":
        return h.dct_jsd_fwd_f32(ptrs([a, b]), 2, C, B, HW, IN_PROBS, None, sm, None, ws, s)
    if op == "jsd_fwdbwd":
        return h.dct_jsd_fwdbwd_f32(ptrs([a, b]), 2, C, B, HW, IN_LOGITS, 1.0, None, sm, ptrs([g0, g1]), None, None, 0,
                                    None, ws, s)
    if op == "ce_fwd":
        return h.dct_ce_fwd_f32(P(a), P(lab), C, B, HW, None, 255, None, sm, None, ws, s)
    if op == "ce_fwdbwd":
        return h.dct_ce_fwdbwd_f32(P(a), P(lab), C, B, HW, None, 255, None, 1.0, None, sm, P(g0), None, None, ws, s)
    if op == "kl_fwd":
        return h.dct_kl_fwd_f32(P(a), P(b), C, B, HW, EPS, None, sm, None, ws, s)
    if op == "kl_logit":
        return h.dct_kl_logit_f32(P(a), P(b), C, B, HW, None, sm, 0, None, None, 1.0, None, None, ws, s)
    if op == "kl_from_logits":
        return h.dct_kl_from_logits_fwdbwd_f32(P(a), P(b), C, B, HW, EPS, 1.0, None, sm, P(g0), None, ws, s)
    if op == "kl_div_fwd":
        return h.dct_kl_div_fwd_f32(P(a), P(b), C, B, HW, EPS, None, sm, None, ws, s)
    if op == "entropy_fwd":
        return h.dct_entropy_fwd_f32(P(a), C, B, HW, None, sm, None, ws, s)
    raise AssertionError(op)


def _sum_ref(op, a, b, gt, oracle):
    """float64 sum and pixel count of the op's loss map, from the float64 oracle on the op's own inputs."""
    if op == "jsd_fwd":
        m = oracle.jsd_fwd([a, b])
    elif op == "jsd_fwdbwd":
        m = oracle.jsd_fwd([oracle.softmax(a), oracle.softmax(b)])
    elif op in ("ce_fwd", "ce_fwdbwd"):
        m = oracle.cross_entropy(a, gt, reduction="none", want_grad=False)[0]
    elif op == "kl_fwd":
        m = oracle.kl_fwd(a, b, EPS)
    elif op == "kl_logit":
        m = oracle.kl_logit(a, b)[0]
    elif op == "kl_from_logits":
        m = oracle.kl_fwd(oracle.softmax(a), b, EPS)
    elif op == "kl_div_fwd":
        m = oracle.kl_div_fwd(a, b, EPS)
    else:
        m = oracle.entropy(a)
    return float(m.sum(dtype=np.float64)), m.size


# (C, HW) of shapes that never tile: HW = 1 takes the runtime-C kernels, HW = 2 at C = 19 the register-tiled VEC = 2
# kernels (jsd_kernel<2, 19, 2, ..>, pix_kernel<Op, 19, 2>; cross-entropy has only the runtime-C kernel)
@pytest.mark.parametrize("C,HW", [(5, 1), (19, 2)], ids=["c5_hw1", "c19_hw2"])
@pytest.mark.parametrize("op", list(SUM_OPS))
def test_loss_sums_past_max_partials(op, C, HW, h, oracle):
    wsb = int(h.dct_workspace_bytes())
    assert wsb > WS_L2_OFFSET
    buf = torch.zeros(wsb + CANARY_BYTES, dtype=torch.uint8, device=DEV)
    buf[wsb:] = 0xAB
    ws = buf.data_ptr()
    r = rng("batch", op, C, HW)
    bmax = max(BATCHES)   # inputs of the largest batch; a smaller batch is its leading images
    host = {}
    for name, kind in zip("ab", SUM_OPS[op]):
        z = logits(r, bmax, C, HW)
        host[name] = probs_of(z) if kind == "p" else z
    gt = r.integers(0, C, (bmax, HW)).astype(np.int64)
    bufs = {"a": carve(host["a"], 0), "b": carve(host["b"], 0), "lab": carve(gt, 0),
            "sum": torch.zeros(1, dtype=torch.float64, device=DEV),
            "g0": torch.empty(bmax * C * HW, device=DEV), "g1": torch.empty(bmax * C * HW, device=DEV)}
    for B in BATCHES:
        assert _sum_call(op, h, C, B, HW, bufs, ws) == OK
        got = bufs["sum"].item()
        ws_after = N(buf[:wsb]).tobytes()
        assert _sum_call(op, h, C, B, HW, bufs, ws) == OK
        assert bufs["sum"].item() == got, f"B={B}: two calls give different sums"
        want, n = _sum_ref(op, f64(host["a"][:B]), f64(host["b"][:B]), gt[:B], oracle)
        assert_close(got / n, want / n, floor=1.0, what=f"{op} sum, B={B}")
        tail = N(buf[wsb:])
        assert (tail == 0xAB).all(), f"B={B}: {int((tail != 0xAB).sum())} canary bytes past the workspace overwritten"
        assert not ws_after[WS_L2_OFFSET:].strip(b"\0"), f"B={B}: the l2 exchange area after `partials` was written"
        assert not ws_after[:WS_HEADER].strip(b"\0"), f"B={B}: the workspace header was not re-armed"
    assert _sum_call(op, h, C, 65536, HW, bufs, ws) == ERR_UNSUPPORTED


# ---------------------------------------------------------------------------------------------
# The same through the Python layer and its shared per-stream workspace, followed by the one-launch l2 normalisation
# that keeps its exchange in that workspace's l2 area
# ---------------------------------------------------------------------------------------------
def test_large_batch_losses_leave_the_l2_exchange_intact(h, oracle):
    import dct_b200
    from dct_b200 import _runtime
    ws = _runtime.state(DEV).workspace
    r = rng("python_large_batch")
    d = torch.from_numpy(r.standard_normal((4, 1, 512, 512)).astype(np.float32))
    want_d = oracle.l2_normalize(d.numpy())
    # one l2 normalisation first, so that the l2 area holds a live epoch
    names, _, _ = kernels(lambda: dct_b200.l2_normalize(d.to(DEV).clone()))
    assert any("l2_ll_kernel" in n for n in names), f"expected the one-launch l2 kernel; launched {names}"
    before = N(ws).tobytes()[WS_L2_OFFSET:]
    n, C = 20000, 7
    p = probs_of(logits(r, n, C))
    q = probs_of(logits(r, n, C))
    got = dct_b200.JSD()([torch.from_numpy(p).to(DEV), torch.from_numpy(q).to(DEV)]).item()
    assert_close(got, float(oracle.jsd_fwd([f64(p), f64(q)]).mean()), floor=lnK(2), what="JSD (N, C)")
    got = dct_b200.KL_div(reduce=True)(torch.from_numpy(p).to(DEV), torch.from_numpy(q).to(DEV)).item()
    assert_close(got, float(oracle.kl_div_fwd(f64(p), f64(q), EPS).mean()), floor=1.0, what="KL_div (N, C)")
    z = logits(r, 9000, 5, 2, 2)
    gt = r.integers(0, 5, (9000, 2, 2)).astype(np.int64)
    got = dct_b200.CrossEntropyLoss2d()(torch.from_numpy(z).to(DEV), torch.from_numpy(gt).to(DEV)).item()
    assert_close(got, oracle.cross_entropy(f64(z), gt, want_grad=False)[0], floor=1.0, what="CrossEntropyLoss2d B=9000")
    torch.cuda.synchronize()
    assert N(ws).tobytes()[WS_L2_OFFSET:] == before, "a loss call wrote into the l2 exchange area"
    for _ in range(2):
        got = dct_b200.l2_normalize(d.to(DEV).clone())
        assert_close(N(got), want_d, what="l2_normalize after the large-batch losses")
