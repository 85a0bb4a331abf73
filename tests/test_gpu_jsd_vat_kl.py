"""GPU: dct_jsd_vat_kl_fwdbwd_f32, the consistency step's JSD launch with the VAT KL folded in.

The entry point is defined as dct_jsd_fwdbwd_f32 (logits) followed by dct_kl_logit_f32(views[0], yhat, grad_p = grad_yhat).
Every test below runs both on the same inputs:
  * shapes with (K + 1) * C <= 16 and C <= 4 run as one tile_kernel<JsdVatKlOp..> launch (asserted from a profiler
    trace); gradients and Dice counts must equal the two calls bit for bit, and so must the two sums where the
    stand-alone launches use the same 256-pixel tiles (C >= 3 and K * C >= 5); elsewhere their per-thread partials
    group 4 pixels instead of 2, so the sums agree within 1e-6 relative;
  * every other shape (rows, C = 19, HW = 2 mod 4, an 8- but not 16-byte aligned yhat or labels) must run the two calls;
  * floating results also match the float64 oracle at util.RTOL_FP32.
"""
import ctypes

import numpy as np
import pytest
import torch

from util import assert_close

pytestmark = pytest.mark.gpu

OK, ERR_BAD_ARG = 0, -1
IN_LOGITS = 1
ACCUMULATE, OVERWRITE = 0, 1
FLAG_LABEL = 1
DEV = torch.device("cuda:0")
FUSED = "JsdVatKlOp"
FUSED_KC = [(2, 2), (2, 3), (2, 4), (3, 2), (3, 3), (3, 4), (4, 2), (4, 3)]


@pytest.fixture(scope="module")
def h():
    import dct_b200
    assert torch.cuda.is_available()
    lib = dct_b200._lib.lib()
    assert lib.dct_device_check(0) == 0
    return lib


def _s():
    return torch.cuda.current_stream(DEV).cuda_stream


def ptrs(ts):
    return (ctypes.c_void_p * len(ts))(*[t.data_ptr() for t in ts])


def carve(t, off):
    """A copy of `t` placed `off` elements into a fresh allocation (off * itemsize sets its alignment mod 16)."""
    flat = t.reshape(-1)
    buf = torch.zeros(flat.numel() + off, dtype=t.dtype, device=DEV)
    buf[off:] = flat
    return buf[off:].view(t.shape)


class Case:
    def __init__(self, K, C, B, H, W, seed=0, yhat_off=0, label_off=0, bad_labels=0):
        g = torch.Generator(device=DEV).manual_seed(seed * 1000 + K * 100 + C * 10 + B)
        self.K, self.C, self.B, self.HW = K, C, B, H * W
        self.n = B * H * W
        self.views = [3 * torch.randn(B, C, H, W, device=DEV, generator=g) for _ in range(K)]
        self.yhat = carve(3 * torch.randn(B, C, H, W, device=DEV, generator=g), yhat_off)
        lab = torch.randint(0, C, (B, H, W), device=DEV, generator=g)
        if bad_labels:
            lab.view(-1)[:bad_labels * 7:7] = C + 3
        self.labels = carve(lab, label_off)

    def outputs(self):
        K, C, B = self.K, self.C, self.B
        f = lambda: torch.full_like(self.views[0], float("nan"))  # noqa: E731
        return dict(grads=[f() for _ in range(K)], gy=f(), sums=torch.zeros(2, dtype=torch.float64, device=DEV),
                    counts=torch.full((K, B, C, 3), -7, dtype=torch.int64, device=DEV),
                    flags=torch.zeros(4, dtype=torch.int32, device=DEV))


def workspace(h):
    return torch.zeros(h.dct_workspace_bytes(), dtype=torch.uint8, device=DEV)


def fused(h, c, o, ws, mode=OVERWRITE, dice=True, pub=None):
    s = o["sums"].data_ptr()
    return h.dct_jsd_vat_kl_fwdbwd_f32(ptrs(c.views), c.K, c.C, c.B, c.HW, 1.0 / c.n, s, ptrs(o["grads"]),
                                       c.labels.data_ptr() if dice else None, o["counts"].data_ptr() if dice else None,
                                       mode, c.yhat.data_ptr(), 1.0 / c.n, s + 8, o["gy"].data_ptr(),
                                       o["flags"].data_ptr(), ws.data_ptr(), pub, _s())


def pair(h, c, o, ws, mode=OVERWRITE, dice=True):
    s = o["sums"].data_ptr()
    rc = h.dct_jsd_fwdbwd_f32(ptrs(c.views), c.K, c.C, c.B, c.HW, IN_LOGITS, 1.0 / c.n, None, s, ptrs(o["grads"]),
                              c.labels.data_ptr() if dice else None, o["counts"].data_ptr() if dice else None, mode,
                              o["flags"].data_ptr(), ws.data_ptr(), _s())
    assert rc == OK
    return h.dct_kl_logit_f32(c.views[0].data_ptr(), c.yhat.data_ptr(), c.C, c.B, c.HW, None, s + 8, 1, None, None,
                              1.0 / c.n, o["gy"].data_ptr(), None, ws.data_ptr(), _s())


def kernels(fn):
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA], acc_events=True) as prof:
        rc = fn()
        torch.cuda.synchronize()
    assert rc == OK
    return sorted({e.key for e in prof.key_averages() if "dct::" in e.key})


def same_tiles(K, C):
    """The stand-alone JSD (K*C rows) and KL (2*C rows) launches run 256-pixel tiles like the fused one (5..16 rows)."""
    return K * C >= 5 and 2 * C >= 5


def assert_same(got, want, sums_exact, dice=True):
    assert all(torch.equal(a, b) for a, b in zip(got["grads"], want["grads"])), "JSD gradients differ"
    assert torch.equal(got["gy"], want["gy"]), "grad yhat differs"
    if dice:
        assert torch.equal(got["counts"], want["counts"]), "Dice counts differ"
    assert torch.equal(got["flags"], want["flags"])
    if sums_exact:
        assert torch.equal(got["sums"], want["sums"]), (got["sums"], want["sums"])
    else:
        rel = ((got["sums"] - want["sums"]).abs() / want["sums"].abs()).max().item()
        assert rel <= 1e-6, (got["sums"], want["sums"])


def check_oracle(oracle, c, o):
    f64 = lambda t: t.detach().double().cpu().numpy()  # noqa: E731
    mean, _, gz = oracle.jsd_logits_fwdbwd([f64(v) for v in c.views], weight=1.0, want_map=False)
    assert_close(o["sums"][0].item() / c.n, mean, floor=np.log(c.K), what="JSD mean")
    scale = 1.0 / c.n
    for k in range(c.K):
        assert_close(f64(o["grads"][k]), gz[k], floor=scale, what=f"JSD grad view {k}")
    m, gpl, _ = oracle.kl_logit(f64(c.views[0]), f64(c.yhat), np.full((c.B,) + tuple(c.views[0].shape[2:]), scale))
    assert_close(o["sums"][1].item() / c.n, float(m.mean()), floor=1.0, what="VAT KL mean")
    assert_close(f64(o["gy"]), gpl, floor=scale, what="grad yhat")


@pytest.mark.parametrize("shape", [(3, 40, 52), (2, 64, 64)])   # ragged last tiles (HW = 2080) and odd B; whole tiles
@pytest.mark.parametrize("kc", FUSED_KC)
def test_fused_shapes_match_the_two_calls_and_the_oracle(h, oracle, kc, shape):
    K, C = kc
    c = Case(K, C, *shape)
    ws = workspace(h)
    got, want = c.outputs(), c.outputs()
    names = kernels(lambda: fused(h, c, got, ws))
    assert any(FUSED in n for n in names) and len(names) == 1, names
    assert pair(h, c, want, ws) == OK
    torch.cuda.synchronize()
    assert_same(got, want, same_tiles(K, C))
    check_oracle(oracle, c, got)
    assert not torch.any(ws[:64]), "workspace header not re-armed"


@pytest.mark.parametrize("kc", [(3, 4), (2, 2)])
def test_without_dice_and_accumulated_counts_and_label_flag(h, kc):
    K, C = kc
    c = Case(K, C, 3, 24, 40, seed=1, bad_labels=5)
    ws = workspace(h)
    got, want = c.outputs(), c.outputs()
    assert fused(h, c, got, ws, dice=False) == OK
    assert pair(h, c, want, ws, dice=False) == OK
    torch.cuda.synchronize()
    assert_same(got, want, same_tiles(K, C), dice=False)
    # overwrite, then accumulate onto it: twice the counts; the out-of-range labels raise the flag on every call
    got, want = c.outputs(), c.outputs()
    for mode in (OVERWRITE, ACCUMULATE):
        assert fused(h, c, got, ws, mode=mode) == OK
        assert pair(h, c, want, ws, mode=mode) == OK
    torch.cuda.synchronize()
    assert_same(got, want, same_tiles(K, C))
    assert int(got["flags"][FLAG_LABEL]) == 2 * 5
    assert not torch.any(ws[:64])


FALLBACK = {
    "K4C4": dict(K=4, C=4, B=2, H=32, W=48),
    "C19": dict(K=2, C=19, B=2, H=32, W=48),
    "HW2mod4": dict(K=3, C=4, B=3, H=6, W=7),
    "yhat_8B": dict(K=3, C=4, B=2, H=32, W=48, yhat_off=2),
    "labels_8B": dict(K=2, C=3, B=2, H=32, W=48, label_off=1),
}


@pytest.mark.parametrize("row", sorted(FALLBACK))
def test_shapes_outside_the_bracket_run_the_two_calls(h, oracle, row):
    c = Case(**FALLBACK[row])
    ws = workspace(h)
    got, want = c.outputs(), c.outputs()
    names = kernels(lambda: fused(h, c, got, ws))
    assert not any(FUSED in n for n in names), names
    assert any("KlLogit" in n for n in names), names
    pair_names = kernels(lambda: pair(h, c, want, ws))
    assert names == pair_names
    assert_same(got, want, True)
    check_oracle(oracle, c, got)


def test_repeatable_and_graph_replay(h):
    c = Case(3, 4, 3, 40, 52, seed=2)
    ws = workspace(h)
    runs = []
    for _ in range(2):
        o = c.outputs()
        assert fused(h, c, o, ws) == OK
        torch.cuda.synchronize()
        runs.append(o)
    assert_same(runs[0], runs[1], True)
    o = c.outputs()
    side = torch.cuda.Stream(device=DEV)
    side.wait_stream(torch.cuda.current_stream(DEV))
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=side):
        assert fused(h, c, o, ws) == OK
    for _ in range(3):
        o["sums"].zero_()
        g.replay()
    torch.cuda.synchronize()
    assert_same(o, runs[0], True)
    assert not torch.any(ws[:64])


def test_refused_arguments_launch_nothing(h):
    c = Case(2, 4, 1, 16, 16)
    ws = workspace(h)
    o = c.outputs()
    s = o["sums"].data_ptr()
    common = (ptrs(c.views), 2, 4, 1, c.HW, 1.0, s, ptrs(o["grads"]), c.labels.data_ptr(), o["counts"].data_ptr(),
              OVERWRITE)
    assert h.dct_jsd_vat_kl_fwdbwd_f32(*common, None, 1.0, s + 8, o["gy"].data_ptr(), None, ws.data_ptr(), None,
                                       _s()) == ERR_BAD_ARG
    assert h.dct_jsd_vat_kl_fwdbwd_f32(*common, c.yhat.data_ptr(), 1.0, s + 8, o["gy"].data_ptr(), None, None, None,
                                       _s()) == ERR_BAD_ARG
    torch.cuda.synchronize()
    assert torch.all(o["counts"] == -7) and torch.all(o["sums"] == 0) and torch.isnan(o["gy"]).all()


@pytest.mark.parametrize("shape", [(3, 4, 2, 64, 64), (2, 2, 2, 128, 128)])   # c2-like (exact) and c3-like (sums 1e-6)
def test_consistency_step_matches_the_separate_entry_points(h, shape):
    from dct_b200.engine import ConsistencyStep, StepBuffers
    K, C, B, H, W = shape
    step = ConsistencyStep(K, C, B, H, W, cin=1, n_global=B * H * W)
    sep = ConsistencyStep(K, C, B, H, W, cin=1, n_global=B * H * W)
    assert step.fused_vat and step.launches_per_step == 4 and step.parts()[1] == "jsd"
    sep.fused_vat = False   # the same step with the VAT KL as its own dct_kl_logit_f32 launch
    bufs = [StepBuffers.allocate(K, C, B, H, W, 1, DEV, torch.Generator(device=DEV).manual_seed(9)) for _ in range(2)]
    step.run(bufs[0])
    sep.run(bufs[1])
    torch.cuda.synchronize()
    a, b = bufs
    for name in ("grad_yhat", "grad_adv", "d", "r_adv", "img_adv", "dice_counts"):
        assert torch.equal(getattr(a, name), getattr(b, name)), name
    assert all(torch.equal(x, y) for x, y in zip(a.grad_logits, b.grad_logits))
    if same_tiles(K, C):
        assert torch.equal(a.sums, b.sums), (a.sums, b.sums)
    else:
        assert torch.equal(a.sums[2:], b.sums[2:])
        assert ((a.sums[:2] - b.sums[:2]).abs() / b.sums[:2].abs()).max().item() <= 1e-6, (a.sums, b.sums)
