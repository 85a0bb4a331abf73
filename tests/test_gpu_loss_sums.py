"""Every loss sum of the training path against the map the same call wrote, across the value range, on the tile
pipeline and off it.

The tile pipeline sums a loss map in 2^-40 fixed point: each consumer thread rounds its fp32 partial (the sum of its
1, 2 or 4 pixels of one tile) to a 64-bit integer and adds it up; the kernels off the tile pipeline add the map in
double.  Whatever the path, a sum must
  * lie within  2^-22 * sum|m_i| + N * 2^-41  of the float64 sum of the map m the call wrote (the fp32 rounding of a
    partial of at most 4 values, plus half a quantum per partial);
  * be finite when every map value is finite with |v| < 2^21, and non-finite when a map value is;
  * be NaN on the tile path when one thread's partial reaches 2^23 (the fixed point's range: |v| >= 2^21 can do that).
A thread's share of a sum used to be one int64, which wraps once it holds 2^23: the range cases put values near
L = 3 * 2^19 on every pixel, at sizes where the busiest CTA's threads hold more than 2^24 each (a wrap is off by 2^24
per wrapped thread).  L is not a power of two, so that no partial sits just under 2^62 and hides the wrap.

Kernels are named from a torch.profiler trace as in test_gpu_launch_paths.py, whose row helpers this file reuses.
"""
import ctypes
import math

import numpy as np
import pytest
import torch

from test_gpu_launch_paths import (DEV, EPS, IN_LOGITS, OK, SUM_OPS, TILE, WS_HEADER, N, _map_ref, _s, _sum_call,
                                   assert_path, carve, f64, h, kernels, logits, probs_of, ptrs, rng)  # noqa: F401
from util import assert_close

pytestmark = pytest.mark.gpu

L = 3 * 2 ** 19                 # per-pixel value of the range cases (exact in fp32 and bf16)
SMS = 148
BF16 = torch.bfloat16
# entry points that write a sum beyond SUM_OPS -> the SUM_OPS entry whose map they compute
BASE = {"ce_fwdbwd_conf": "ce_fwd", "jsd_fwdbwd_pub": "jsd_fwdbwd", "kl_from_logits_pub": "kl_from_logits",
        "jsd_fwdbwd_bf16": "jsd_fwdbwd", "kl_logit_bf16": "kl_logit", "kl_from_logits_bf16": "kl_from_logits",
        "ce_fwdbwd_bf16": "ce_fwdbwd"}
OPS = list(SUM_OPS) + list(BASE)
# the pix_kernel op struct of an entry point, for the name of its kernel off the tile pipeline
PIX = {"kl_fwd": "KlProbFwd", "kl_logit": "KlLogit<false>", "kl_from_logits": "KlFromLogits", "kl_div_fwd": "KlDivFwd",
       "entropy_fwd": "EntropyFwd"}


def base(op):
    return BASE.get(op, op)


def is_bf16(op):
    return op.endswith("_bf16")


@pytest.fixture(scope="module")
def px():
    from dct_b200.distributed import PeerExchange
    x = PeerExchange(DEV, n=4, nslots=8)
    yield x
    x.close()


def off_tile_kernel(op, C):
    """The kernel an entry point reaches for HW = 2 mod 4 (test_gpu_launch_paths.py's *_hw2mod4 rows), and for an odd
    HW at C = 4 (cross-entropy at any C)."""
    b = base(op)
    if b.startswith("jsd"):
        return "dct::jsd_kernel_rt<" if C != 19 else "dct::jsd_kernel<2, 19, 2,"
    if b.startswith("ce"):
        return "dct::ce_kernel_rt<"
    return f"dct::pix_kernel<dct::{PIX[b]}, " + ("0, 1>" if C != 19 else "19, 2>")


def tile_rows(op, C):
    return (1 if base(op).startswith(("ce", "entropy")) else 2) * C


def max_thread_share(rows, B, HW, value):
    """A lower bound on the largest per-thread share of a tile launch's sum when every pixel's value is `value`:
    tile_launch_ct's shape for NIN * C = rows (pixels per thread, consumer warps, CTAs per SM), and the busiest CTA
    holds at least ceil(tiles / grid) tiles whatever the schedule."""
    assert rows <= 24
    ppt, ncw, minb = (4, 8, 2) if rows <= 4 else ((2, 4, 3) if rows <= 16 else (2, 4, 2))
    tiles = B * -(-HW // (ncw * 32 * ppt))
    grid = min(SMS * minb, tiles)
    return -(-tiles // grid) * ppt * value


def sum_bound(m):
    m = f64(m)
    return 2.0 ** -22 * float(np.abs(m).sum()) + m.size * 2.0 ** -41


def assert_sum_of_map(got, m, what):
    want = float(f64(m).sum())
    assert math.isfinite(got), f"{what}: sum {got!r} of a finite map (float64 sum {want!r})"
    assert abs(got - want) <= sum_bound(m), \
        f"{what}: sum {got!r}, float64 sum of its map {want!r}: off by {got - want:.6g} > {sum_bound(m):.6g}"


def run(op, h, C, B, HW, x, ws, px, w=None):
    """Calls `op` twice (the second under the profiler) on host inputs x = {'a', 'b', 'lab'} with a map; returns
    (kernel names, sum, map, the two sums)."""
    dt = BF16 if is_bf16(op) else torch.float32
    dev = lambda a: None if a is None else carve(a, 0).to(dt)  # noqa: E731
    a = dev(x["a"])
    b = dev(x.get("b"))
    sums = torch.zeros(4, dtype=torch.float64, device=DEV)
    bufs = {"a": a, "b": b, "lab": carve(x["lab"], 0), "sum": sums[:1], "map": torch.empty(B * HW, device=DEV),
            "g0": torch.empty(B * C * HW, dtype=dt, device=DEV), "g1": torch.empty(B * C * HW, dtype=dt, device=DEV),
            "w": None if w is None else torch.from_numpy(np.asarray(w, np.float32)).to(DEV)}
    P = lambda t: None if t is None else t.data_ptr()  # noqa: E731
    mp, sm, wp, s = P(bufs["map"]), P(sums), P(bufs["w"]), _s()
    a_, b_, g0, lab = P(a), P(b), P(bufs["g0"]), P(bufs["lab"])
    conf = torch.zeros(C * C, dtype=torch.int64, device=DEV)

    def call():
        if op in SUM_OPS:
            rc = _sum_call(op, h, C, B, HW, bufs, P(ws))
        elif op == "ce_fwdbwd_conf":
            rc = h.dct_ce_fwdbwd_conf_f32(a_, lab, C, B, HW, wp, 255, None, 1.0, mp, sm, g0, P(conf), None, P(ws), s)
        elif op == "jsd_fwdbwd_pub":
            rc = h.dct_jsd_fwdbwd_pub_f32(ptrs([a, b]), 2, C, B, HW, IN_LOGITS, 1.0, mp, sm, ptrs([bufs["g0"], bufs["g1"]]),
                                          None, None, 0, None, P(ws), ctypes.byref(px.descriptor(sums)), s)
        elif op == "kl_from_logits_pub":
            rc = h.dct_kl_from_logits_fwdbwd_pub_f32(a_, b_, C, B, HW, EPS, 1.0, mp, sm, g0, None, P(ws),
                                                     ctypes.byref(px.descriptor(sums)), s)
        elif op == "jsd_fwdbwd_bf16":
            rc = h.dct_jsd_fwdbwd_bf16(ptrs([a, b]), 2, C, B, HW, 1.0, mp, sm, ptrs([bufs["g0"], bufs["g1"]]), None,
                                       None, 0, None, P(ws), s)
        elif op == "kl_logit_bf16":
            rc = h.dct_kl_logit_bf16(a_, b_, C, B, HW, mp, sm, 0, None, None, 1.0, None, None, P(ws), s)
        elif op == "kl_from_logits_bf16":
            rc = h.dct_kl_from_logits_fwdbwd_bf16(a_, b_, C, B, HW, EPS, 1.0, mp, sm, g0, None, P(ws), s)
        elif op == "ce_fwdbwd_bf16":
            rc = h.dct_ce_fwdbwd_bf16(a_, lab, C, B, HW, wp, 255, None, 1.0, mp, sm, g0, None, None, P(ws), s)
        else:
            raise AssertionError(op)
        assert rc == OK, (op, rc)
        return sums[0].item(), N(bufs["map"]).copy()

    names, (s1, _), (s2, m2) = kernels(call)
    return names, s2, m2, (s1, s2)


def as_seen(op, a):
    """The values the kernel reads: bf16 inputs are rounded once."""
    if a is None or not is_bf16(op):
        return a
    return torch.from_numpy(np.ascontiguousarray(a)).to(BF16).float().numpy()


def check_map(oracle, op, x, m, w=None, floor=1.0):
    a, b = as_seen(op, x["a"]), as_seen(op, x.get("b"))
    want = _map_ref(base(op), f64(a), None if b is None else f64(b), x["lab"], oracle, w)
    assert_close(m.reshape(want.shape), want, floor=floor, what=f"{op} map")


def assert_on_path(names, op, C, path):
    if path == "tile":
        assert_path(names, TILE, off_tile=False)
    else:
        assert_path(names, off_tile_kernel(op, C))


def ops_paths(C):
    return [(op, p) for op in OPS for p in ("tile", "off_tile") if not (is_bf16(op) and p == "off_tile")
            and not (is_bf16(op) and C not in (2, 3, 4, 19))]


# ---------------------------------------------------------------------------------------------
# 1. the sum of every entry point against its own map: ragged last tiles, near-zero and mixed-sign maps
# ---------------------------------------------------------------------------------------------
SHAPES = {"tile": (3, 40, 52), "off_tile": (3, 37, 42)}   # HW = 2080: ragged last tiles of 256 and 1024; 1554 = 2 mod 4


def inputs(op, C, B, HW, kind, r):
    """Host inputs of `op`: 'randn' (3 randn logits or their softmax), 'near_zero' (a map of tiny values) or
    'mixed' (the KL ops on positive inputs off the simplex: map values of both signs that largely cancel)."""
    kinds = SUM_OPS[base(op)]
    lab = r.integers(0, C, (B, HW)).astype(np.int64)
    z = logits(r, B, C, HW)
    if kind == "mixed":   # the log-ratio of the two inputs is uniform in (-1, 1): class terms -t*u and t*u cancel
        t = r.uniform(0.05, 1.0, (B, C, HW))
        e = t * np.exp(r.uniform(-1.0, 1.0, (B, C, HW)))
        a, b = (e, t) if op == "kl_fwd" else (t, e)
        return {"a": a.astype(np.float32), "b": b.astype(np.float32), "lab": lab}
    if kind == "near_zero":
        if kinds[1] == "-":   # cross-entropy: the label's logit 40 above the rest; entropy: a near one-hot p
            np.put_along_axis(z, lab[:, None], 40.0, axis=1)
            return {"a": probs_of(z) if kinds[0] == "p" else z, "b": None, "lab": lab}
        z2 = (z + 1e-3 * r.standard_normal(z.shape)).astype(np.float32)
        a = probs_of(z) if kinds[0] == "p" else z
        return {"a": a, "b": probs_of(z2) if kinds[1] == "p" else z2, "lab": lab}
    z2 = logits(r, B, C, HW)
    return {"a": probs_of(z) if kinds[0] == "p" else z,
            "b": None if kinds[1] == "-" else (probs_of(z2) if kinds[1] == "p" else z2), "lab": lab}


CASE1 = [(op, C, path, kind) for C in (4, 19) for op, path in ops_paths(C) for kind in ("randn", "near_zero")] + \
        [(op, 4, path, "mixed") for op in ("kl_fwd", "kl_div_fwd") for path in ("tile", "off_tile")]


@pytest.mark.parametrize("op,C,path,kind", CASE1, ids=[f"{o}-c{c}-{p}-{k}" for o, c, p, k in CASE1])
def test_sum_matches_its_own_map(op, C, path, kind, h, px, oracle):
    B, H, W = SHAPES[path]
    HW = H * W
    x = inputs(op, C, B, HW, kind, rng("own_map", op, C, path, kind))
    ws = torch.zeros(int(h.dct_workspace_bytes()), dtype=torch.uint8, device=DEV)
    names, got, m, (s1, s2) = run(op, h, C, B, HW, x, ws, px)
    assert_on_path(names, op, C, path)
    assert s1 == s2, "two calls give different sums"
    check_map(oracle, op, x, m, floor=math.log(2) if base(op).startswith("jsd") else 1.0)
    assert_sum_of_map(got, m, op)
    if kind == "mixed":
        assert (m < 0).any() and (m > 0).any(), "the map must hold values of both signs"
    assert not N(ws[:WS_HEADER]).any(), "the workspace header was not re-armed"


# ---------------------------------------------------------------------------------------------
# 2. range: per-pixel values near L = 3 * 2^19, at sizes where one thread's share passes 2^23 and 2^24
# ---------------------------------------------------------------------------------------------
def range_inputs(case, C, B, HW):
    """'ce': logits [0, -L, .., -L] with label 1 (loss L); 'ce_w': logits [0, -24, .., -24], label 1 weighted 2^16
    (loss 24 * 2^16 = L); 'kl': q one-hot at class 0 through logits -L elsewhere, p with logit -L at class 0 and 0 at
    class 1 (KL = L).  Returns (inputs, class weights or None)."""
    lab = np.ones((B, HW), np.int64)
    if case in ("ce", "ce_w"):
        z = np.full((B, C, HW), -L if case == "ce" else -24.0, np.float32)
        z[:, 0] = 0.0
        if case == "ce":
            return {"a": z, "b": None, "lab": lab}, None
        w = np.ones(C, np.float32)
        w[1] = 2.0 ** 16
        return {"a": z, "b": None, "lab": lab}, w
    q = np.full((B, C, HW), -L, np.float32)
    q[:, 0] = 0.0
    p = np.full((B, C, HW), -L, np.float32)
    p[:, 1] = 0.0
    return {"a": q, "b": p, "lab": lab}, None


# op, range case, C, B, H, W of the tile launch
RANGE = [("ce_fwd", "ce", 4, 4, 512, 512), ("ce_fwdbwd", "ce", 4, 4, 512, 512),
         ("ce_fwdbwd_conf", "ce", 4, 4, 512, 512), ("ce_fwdbwd_bf16", "ce", 4, 4, 512, 512),
         ("ce_fwd", "ce_w", 4, 4, 512, 512), ("ce_fwdbwd", "ce_w", 4, 4, 512, 512),
         ("ce_fwdbwd_bf16", "ce_w", 4, 4, 512, 512),
         ("ce_fwd", "ce", 19, 2, 512, 512), ("ce_fwdbwd", "ce", 19, 2, 512, 512), ("ce_fwdbwd_bf16", "ce", 19, 2, 512, 512),
         ("kl_logit", "kl", 4, 3, 512, 512), ("kl_logit_bf16", "kl", 4, 3, 512, 512)]
RANGE_PATHS = [r + (p,) for r in RANGE for p in ("tile", "off_tile") if not (is_bf16(r[0]) and p == "off_tile")]


@pytest.mark.parametrize("op,case,C,B,H,W,path", RANGE_PATHS,
                         ids=[f"{r[0]}-{r[1]}-c{r[2]}-{r[6]}" for r in RANGE_PATHS])
def test_sum_of_large_values(op, case, C, B, H, W, path, h, px, oracle):
    if path == "off_tile":
        H, W = H - 1, W - 1   # odd HW: the kernels off the tile pipeline
    HW = H * W
    if path == "tile":
        share = max_thread_share(tile_rows(op, C), B, HW, L)
        assert share >= 2 ** 24, f"a thread's share {share} does not pass 2^24"
    x, w = range_inputs(case, C, B, HW)
    ws = torch.zeros(int(h.dct_workspace_bytes()), dtype=torch.uint8, device=DEV)
    names, got, m, (s1, s2) = run(op, h, C, B, HW, x, ws, px, w)
    assert_on_path(names, op, C, path)
    check_map(oracle, op, x, m, w)
    assert_sum_of_map(got, m, op)
    assert_close(got, float(B * HW) * L, what=f"{op} sum against N * L")
    assert s1 == s2
    assert not N(ws[:WS_HEADER]).any(), "the workspace header was not re-armed"


# ---------------------------------------------------------------------------------------------
# 3. the edge of the fixed point's range at 4 pixels per thread
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("path", ["tile", "off_tile"])
def test_sum_at_the_edge_of_the_range(path, h, px, oracle):
    C, B, H, W = (4, 4, 512, 512) if path == "tile" else (4, 4, 511, 511)
    HW = H * W
    v = 2.0 ** 21 - 64               # every reported value stays below 2^21, so every partial of 4 below 2^23
    x, _ = range_inputs("ce", C, B, HW)
    x["a"][:, 1:] = -v
    ws = torch.zeros(int(h.dct_workspace_bytes()), dtype=torch.uint8, device=DEV)
    names, got, m, _ = run("ce_fwd", h, C, B, HW, x, ws, px)
    assert_on_path(names, "ce_fwd", C, path)
    assert m.max() < 2.0 ** 21 and m.min() > 2.0 ** 20, (m.min(), m.max())
    assert_sum_of_map(got, m, "values just below 2^21")
    assert_close(got, float(B * HW) * v, what="sum against N * v")
    # one pixel of 1.25 * 2^23: its partial leaves the fixed point's range on the tile path
    x["a"][1, 1:, 77] = -1.25 * 2 ** 23
    names, got, m, _ = run("ce_fwd", h, C, B, HW, x, ws, px)
    assert m.max() >= 2.0 ** 23
    if path == "tile":
        assert math.isnan(got), f"a partial >= 2^23 must give NaN on the tile path, got {got!r}"
    else:
        assert_sum_of_map(got, m, "one value of 1.25 * 2^23 off the tile pipeline")
    assert not N(ws[:WS_HEADER]).any(), "the workspace header was not re-armed"


# ---------------------------------------------------------------------------------------------
# 4. non-finite values poison the sum on every path, and the next call on the same workspace is clean
# ---------------------------------------------------------------------------------------------
NONFINITE = [(op, p, "nan") for op, p in ops_paths(4)] + \
            [(op, p, "inf") for op, p in ops_paths(4) if base(op).startswith("ce")]


@pytest.mark.parametrize("op,path,bad", NONFINITE, ids=[f"{o}-{p}-{b}" for o, p, b in NONFINITE])
def test_nonfinite_value_then_clean_call(op, path, bad, h, px, oracle):
    C = 4
    B, H, W = SHAPES[path]
    HW = H * W
    x = inputs(op, C, B, HW, "randn", rng("nonfinite", op, path, bad))
    pix = (1, 1234)
    w = None
    if bad == "nan":
        x_bad = dict(x, a=x["a"].copy())
        x_bad["a"][pix[0], :, pix[1]] = np.nan
    else:   # +inf: the only pixel of class 3 carries an infinite class weight
        lab = np.minimum(x["lab"], 2)
        lab[pix] = 3
        x_bad = dict(x, lab=lab)
        w = np.array([1.0, 1.0, 1.0, np.inf], np.float32)
    ws = torch.zeros(int(h.dct_workspace_bytes()), dtype=torch.uint8, device=DEV)
    names, got, m, _ = run(op, h, C, B, HW, x_bad, ws, px, w)
    assert_on_path(names, op, C, path)
    assert not np.isfinite(m.reshape(B, HW)[pix]), "the map value of the poisoned pixel must be non-finite"
    assert not math.isfinite(got), f"{op}: a non-finite map value gave the finite sum {got!r}"
    assert not N(ws[:WS_HEADER]).any(), "the workspace header was not re-armed"
    _, got, m, _ = run(op, h, C, B, HW, x, ws, px)
    assert_sum_of_map(got, m, f"{op} after a non-finite call")
    assert not N(ws[:WS_HEADER]).any(), "the workspace header was not re-armed"


# ---------------------------------------------------------------------------------------------
# 5. the fused JSD + VAT KL launch: the VAT KL's range and NaN reach kl_sum only
# ---------------------------------------------------------------------------------------------
def test_vat_kl_second_sum(h, oracle):
    K, C, B, H, W = 2, 4, 3, 512, 512
    HW = H * W
    assert max_thread_share((K + 1) * C, B, HW, L) >= 2 ** 24
    r = rng("vat_kl_range")
    q, p = range_inputs("kl", C, B, HW)[0]["a"], range_inputs("kl", C, B, HW)[0]["b"]
    views = [carve(q, 0), carve(logits(r, B, C, HW), 0)]
    grads = [torch.empty(B * C * HW, device=DEV) for _ in range(K)]
    gy = torch.empty(B * C * HW, device=DEV)
    ws = torch.zeros(int(h.dct_workspace_bytes()), dtype=torch.uint8, device=DEV)
    clean = logits(r, B, C, HW)
    nan = clean.copy()
    nan[2, :, 999] = np.nan
    results = {}
    for name, yhat in (("clean", clean), ("large", p), ("nan", nan)):
        y = carve(yhat, 0)
        sums = torch.zeros(2, dtype=torch.float64, device=DEV)

        def call():
            rc = h.dct_jsd_vat_kl_fwdbwd_f32(ptrs(views), K, C, B, HW, 1.0, sums.data_ptr(), ptrs(grads), None, None, 0,
                                             y.data_ptr(), 1.0, sums.data_ptr() + 8, gy.data_ptr(), None, ws.data_ptr(),
                                             None, _s())
            assert rc == OK, rc
            return sums.tolist()

        names, first, second = kernels(call)
        assert_path(names, "JsdVatKlOp", off_tile=False)
        assert np.array_equal(first, second, equal_nan=True)
        results[name] = second
        assert not N(ws[:WS_HEADER]).any(), "the workspace header was not re-armed"
    for name in ("large", "nan"):
        assert results[name][0] == results["clean"][0], f"{name} yhat changed the JSD sum"
    assert math.isnan(results["nan"][1])
    # kl_sum against the map of the stand-alone dct_kl_logit_f32 on the same inputs and the closed form N * L
    mp = torch.empty(B * HW, device=DEV)
    y = carve(p, 0)
    sm = torch.zeros(1, dtype=torch.float64, device=DEV)
    assert h.dct_kl_logit_f32(views[0].data_ptr(), y.data_ptr(), C, B, HW, mp.data_ptr(), sm.data_ptr(), 0, None, None,
                              1.0, None, None, ws.data_ptr(), _s()) == OK
    m = N(mp)
    assert_close(m.reshape(B, HW), oracle.kl_logit(f64(q), f64(p))[0], floor=1.0, what="kl_logit map")
    assert_sum_of_map(sm.item(), m, "stand-alone kl_logit")
    assert_close(results["large"][1], float(m.sum(dtype=np.float64)), what="fused kl_sum against the KL map")
    assert_close(results["large"][1], float(B * HW) * L, what="fused kl_sum against N * L")


# ---------------------------------------------------------------------------------------------
# 6. the Python layer in the range regime, against torch's cross-entropy in float64
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", [torch.float32, BF16], ids=["f32", "bf16"])
@pytest.mark.parametrize("case", ["ce", "ce_w"])
def test_python_cross_entropy_large_values(case, dtype, h):
    import torch.nn.functional as F

    import dct_b200
    C, B, H, W = 4, 4, 512, 512
    x, w = range_inputs(case, C, B, H * W)
    z = torch.from_numpy(x["a"]).reshape(B, C, H, W).to(DEV)
    gt = torch.from_numpy(x["lab"]).reshape(B, H, W).to(DEV)
    wt = None if w is None else torch.from_numpy(w).to(DEV)
    for red, size_average in (("mean", True), ("sum", False)):
        want = F.cross_entropy(z.double(), gt, weight=None if wt is None else wt.double(), reduction=red).item()
        for grad in (False, True):
            zi = z.to(dtype).requires_grad_(grad)
            got = dct_b200.CrossEntropyLoss2d(weight=wt, size_average=size_average)(zi, gt).item()
            assert_close(got, want, what=f"CrossEntropyLoss2d {red}, grad={grad}")
    zi = z.to(dtype).requires_grad_(True)
    got = dct_b200.supervised_from_logits(zi, gt, weight=wt).item()
    want = F.cross_entropy(z.double(), gt, weight=None if wt is None else wt.double()).item()
    assert_close(got, want, what="supervised_from_logits")
