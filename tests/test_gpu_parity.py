"""GPU parity tests: the CUDA path (through the C ABI) vs the committed reference fixtures and
the CPU oracle on seeded inputs.  Integer results bit-exact; floating point within 1e-5 scaled
(tests/util.py).  Nothing here reads /root/reference.
"""
import math
import os

import numpy as np
import pytest
import torch

from util import assert_close, cases, lnK

pytestmark = pytest.mark.gpu

GOLDEN = np.load(os.path.join(os.path.dirname(__file__), "golden", "reference_golden.npz"))


def _names(prefix):
    return cases(GOLDEN, prefix)


@pytest.fixture(scope="module")
def dct():
    import dct_b200
    assert torch.cuda.is_available()
    assert dct_b200._lib.lib().dct_device_check(0) == 0
    return dct_b200


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda:0")


def T(a, dev, grad=False):
    t = torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    return t.requires_grad_() if grad else t


def N(t):
    return t.detach().cpu().numpy()


# ---------------------------------------------------------------------------------------------
# JSD against the reference fixtures: probs boundary (drop-in), logits boundary, fused
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", _names("jsd_"))
def test_jsd_dropin_vs_reference(case, dct, dev):
    probs = [T(p, dev, grad=True) for p in GOLDEN[case + "/ref_probs32"]]
    K = len(probs)
    gout = T(GOLDEN[case + "/gout"], dev)
    crit = dct.get_loss_fn("jsd")
    m = crit(probs)
    assert m.shape == gout.shape and m.dtype == torch.float32
    assert_close(N(m), GOLDEN[case + "/ref_map32"], floor=lnK(K), what="map")
    (m * gout).sum().backward()
    got = np.stack([N(p.grad) for p in probs])
    assert_close(got, GOLDEN[case + "/ref_gp32"], floor=float(np.abs(GOLDEN[case + "/gout"]).max()), what="d/dprobs")
    # closer to the fp64 reference than 1e-5 as well
    assert_close(N(m), GOLDEN[case + "/ref_map64"], floor=lnK(K), what="map vs fp64")


@pytest.mark.parametrize("case", _names("jsd_"))
def test_jsd_from_logits_vs_reference(case, dct, dev):
    z = GOLDEN[case + "/z"]
    K, B = z.shape[0], z.shape[1]
    npx = B * z.shape[3] * z.shape[4]
    w = float(GOLDEN[case + "/w"])
    # (a) map with autograd backward (recompute kernel), upstream = w/N everywhere via .mean()
    zs = [T(a, dev, grad=True) for a in z]
    m = dct.jsd_map_from_logits(zs)
    assert_close(N(m), GOLDEN[case + "/ref_map32"], floor=lnK(K), what="map")
    (w * m.mean()).backward()
    assert_close(np.stack([N(t.grad) for t in zs]), GOLDEN[case + "/ref_gz32"], floor=w / npx, what="d/dlogits (bwd)")
    # (b) fused one-pass forward+backward
    zs2 = [T(a, dev, grad=True) for a in z]
    loss = dct.jsd_consistency_from_logits(zs2, weight=w)
    assert_close(loss.item(), w * float(GOLDEN[case + "/ref_mean32"]), floor=w * lnK(K), what="fused loss")
    loss.backward()
    assert_close(np.stack([N(t.grad) for t in zs2]), GOLDEN[case + "/ref_gz32"], floor=w / npx, what="d/dlogits (fused)")
    # (c) a non-unit upstream goes through the scale kernel
    zs3 = [T(a, dev, grad=True) for a in z]
    (2.5 * dct.jsd_consistency_from_logits(zs3, weight=w)).backward()
    assert_close(np.stack([N(t.grad) for t in zs3]), 2.5 * GOLDEN[case + "/ref_gz32"], floor=2.5 * w / npx)
    # (d) no_grad path: forward only
    with torch.no_grad():
        l2 = dct.jsd_consistency_from_logits([T(a, dev) for a in z], weight=w)
    assert_close(l2.item(), loss.item(), floor=w * lnK(K), rtol=1e-6)


@pytest.mark.parametrize("case", [c for c in _names("jsd_") if c.endswith("spread")])
def test_jsd_nd_and_entropy_vs_reference(case, dct, dev):
    probs = [T(p, dev) for p in GOLDEN[case + "/ref_probs32"]]
    K = len(probs)
    assert_close(N(dct.JSD()(probs, reduce=False)), GOLDEN[case + "/ref_JSD_map"], floor=lnK(K))
    assert_close(dct.JSD()(probs, reduce=True).item(), GOLDEN[case + "/ref_JSD_reduce"], floor=lnK(K))
    assert_close(N(dct.Entropy_2D()(probs[0])), GOLDEN[case + "/ref_entropy0"], floor=1.0)
    assert_close(N(dct.Entropy()(probs[0])), GOLDEN[case + "/ref_entropy0"], floor=1.0)


def test_jsd_simplex_assertion(dct, dev):
    bad = [torch.rand(2, 4, 8, 8, device=dev) for _ in range(2)]
    with pytest.raises(AssertionError):
        dct.JSD_2D()(bad)
    with pytest.raises(AssertionError):
        dct.JSD_2D()([torch.rand(2, 4, 8, device=dev)])  # not 4-D
    with pytest.raises(AssertionError):
        dct.KL_Divergence_2D()(bad[0], bad[1])
    old = dct.set_check_mode("deferred")
    try:
        dct.JSD_2D()(bad)  # no sync, no raise
        with pytest.raises(AssertionError):
            dct.raise_if_flagged()
        dct.raise_if_flagged()  # flags were cleared
    finally:
        dct.set_check_mode(old)
    ok = [torch.softmax(torch.randn(2, 4, 8, 8, device=dev), 1) for _ in range(2)]
    dct.JSD_2D()(ok)
    with pytest.raises(ValueError):
        dct.get_loss_fn("jsd", bogus=1)  # ctor errors surface as ValueError like the reference registry


def test_cpu_tensor_is_rejected_loudly(dct):
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        dct.JSD_2D()([torch.softmax(torch.randn(1, 2, 4, 4), 1)] * 2)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        dct.DiceMeter(C=2).add(torch.randn(1, 2, 4, 4), torch.zeros(1, 1, 4, 4, dtype=torch.long))


# ---------------------------------------------------------------------------------------------
# KL family
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", _names("kl_"))
def test_kl_vs_reference(case, dct, dev):
    gout_np = GOLDEN[case + "/gout"]
    gs = float(np.abs(gout_np).max())
    gout = T(gout_np, dev)
    p = T(GOLDEN[case + "/p32"], dev, grad=True); y = T(GOLDEN[case + "/y32"], dev, grad=True)
    m = dct.KL_Divergence_2D(reduce=False)(p, y)
    assert_close(N(m), GOLDEN[case + "/ref_map32"], floor=1.0)
    m.backward(gout)
    assert_close(N(p.grad), GOLDEN[case + "/ref_gp32"], floor=gs)
    assert_close(N(y.grad), GOLDEN[case + "/ref_gy32"], floor=gs)
    red = dct.KL_Divergence_2D(reduce=True)(p_prob=p.detach(), y_prob=y.detach())  # kwargs as vattrainer.py:154
    assert red.dim() == 0
    assert_close(red.item(), GOLDEN[case + "/ref_mean32"], floor=1.0)
    # trainer composite, drop-in form: softmax (ATen) -> KL(reduce=True)(adv, real.detach()) -> backward
    zl = T(GOLDEN[case + "/zp"], dev, grad=True)
    dct.KL_Divergence_2D(reduce=True)(torch.softmax(zl, 1), y.detach()).backward()
    n = gout_np.size
    assert_close(N(zl.grad), GOLDEN[case + "/ref_gzp_mean32"], floor=1.0 / n)
    # trainer composite, fused form
    zl2 = T(GOLDEN[case + "/zp"], dev, grad=True)
    loss = dct.kl_consistency_from_logits(zl2, y.detach(), weight=1.0)
    assert_close(loss.item(), GOLDEN[case + "/ref_mean32"], floor=1.0)
    loss.backward()
    assert_close(N(zl2.grad), GOLDEN[case + "/ref_gzp_mean32"], floor=1.0 / n)
    # logits variants
    ql = T(GOLDEN[case + "/zy"], dev, grad=True); pl = T(GOLDEN[case + "/zp"], dev, grad=True)
    ml = dct.VATGenerator.kl_div_with_logit(ql, pl)
    assert_close(N(ml), GOLDEN[case + "/ref_logit_map32"], floor=1.0)
    ml.backward(gout)
    assert_close(N(pl.grad), GOLDEN[case + "/ref_logit_gpl32"], floor=gs)
    assert_close(N(ql.grad), GOLDEN[case + "/ref_logit_gql32"], floor=gs)
    m2 = dct.KL_Divergence_2D_Logit(reduce=False)(pl.detach(), ql.detach())
    assert_close(N(m2), GOLDEN[case + "/ref_logit2d_map32"], floor=1.0)
    assert_close(N(dct.KL_div(reduce=False)(p.detach(), y.detach())), GOLDEN[case + "/ref_kldiv_map32"], floor=1.0)
    assert_close(N(dct.softmax_dim1(T(GOLDEN[case + "/zp"], dev))), GOLDEN[case + "/p32"], floor=1.0, rtol=2e-7)


# ---------------------------------------------------------------------------------------------
# VAT / FGSM
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", _names("vat_"))
def test_vat_vs_reference(case, dct, dev):
    d = T(GOLDEN[case + "/d"], dev)
    out = dct.VATGenerator._l2_normalize(d)
    assert out.data_ptr() == d.data_ptr()  # in place, returns its argument (AEGenerator.py:73-76)
    assert_close(N(out), GOLDEN[case + "/ref_l2"])
    adv, noise = dct.FSGMGenerator.adversarial_fgsm(T(GOLDEN[case + "/img"], dev), T(GOLDEN[case + "/grad"], dev), epsilon=0.05)
    assert np.array_equal(N(adv), GOLDEN[case + "/ref_fgsm_adv"])
    assert np.array_equal(N(noise), GOLDEN[case + "/ref_fgsm_noise"])


def test_l2_normalize_paths_vs_oracle(dct, dev, oracle):
    g = torch.Generator().manual_seed(7)
    # cluster path (1..16 float4 per thread), the two-launch fallback (large / odd M), scale + clamp tail
    # ... and one cluster of 16 CTAs per sample for 512 KB < sample <= 1 MB (spleen 512 x 512 slices)
    for shape in [(32, 1, 256, 256), (3, 3, 128, 256), (2, 3, 512, 1024), (5, 1, 33, 7), (2, 1, 1, 1), (4, 1, 512, 512),
                  (3, 1, 384, 512)]:
        d = torch.randn(*shape, generator=g)
        img = torch.rand(*shape, generator=g)
        want = oracle.l2_normalize(d.numpy())
        got = dct.l2_normalize(d.to(dev).clone())
        assert_close(N(got), want, what=f"l2 {shape}")
        r, adv = dct.l2_normalize(d.to(dev).clone(), scale=10.0, img=img.to(dev))
        wadv, wr = oracle.vat_apply(img.numpy(), want, 10.0)
        assert_close(N(r), wr, what=f"r_adv {shape}")
        assert_close(N(adv), wadv, floor=1.0, what=f"img_adv {shape}")
        # passes=2: normalise(normalise(d)) then scale, one launch (AEGenerator.py:98 + :103)
        twice = dct.l2_normalize(d.to(dev).clone(), scale=1e-6, passes=2)
        assert_close(N(twice), oracle.l2_normalize(want) * np.float32(1e-6), what=f"l2 x2 {shape}")
        nrm = N(got).reshape(shape[0], -1).astype(np.float64)
        assert np.allclose(np.sqrt((nrm ** 2).sum(1)), 1.0, rtol=1e-3)  # the reference's own assert (:75)


def test_vat_generator_runs(dct, dev):
    torch.manual_seed(0)
    net = torch.nn.Conv2d(1, 4, 3, padding=1).to(dev)
    img = torch.rand(4, 1, 32, 32, device=dev)
    gen = dct.VATGenerator(net, xi=1e-6, eplision=0.03, ip=1, axises=[1, 2, 3])  # kwargs as vattrainer.py:142
    img_adv, r_adv = gen(img, loss_name='kl')
    assert img_adv.shape == img.shape and r_adv.shape == img.shape
    assert float(img_adv.min()) >= 0.0 and float(img_adv.max()) <= 1.0
    nr = r_adv.reshape(4, -1).norm(dim=1)
    assert torch.allclose(nr, torch.full_like(nr, 0.03), rtol=1e-3)
    adv_img, noise, p = dct.FSGMGenerator(net, eplision=0.05)(img.clone(), torch.zeros(4, 1, 32, 32, dtype=torch.long, device=dev),
                                                              torch.nn.CrossEntropyLoss())
    assert float(noise.abs().max()) == pytest.approx(0.05)
    assert p.shape == (4, 4, 32, 32)


# ---------------------------------------------------------------------------------------------
# Dice / confusion: bit-exact
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", [c for c in _names("dice_") if not c.endswith("meter")])
def test_dice_vs_reference_bit_exact(case, dct, dev):
    x = T(GOLDEN[case + "/x"], dev); gt = T(GOLDEN[case + "/gt"], dev)
    C = x.shape[1]
    m2 = dct.DiceMeter(method="2d", C=C); m2.add(x, gt)
    m3 = dct.DiceMeter(method="3d", C=C); m3.add(x, gt)
    assert m2.log.dtype == torch.float32 and m2.log.is_cuda
    assert np.array_equal(N(m2.log), GOLDEN[case + "/ref_2d"])
    assert np.array_equal(N(m3.log), GOLDEN[case + "/ref_3d"])
    if case.endswith("_logits"):
        bad = gt.clone(); bad[0, 0, 0, 0] = C
        with pytest.raises(AssertionError):
            dct.DiceMeter(method="2d", C=C).add(x, bad)


@pytest.mark.parametrize("C", [2, 4, 5, 19])
def test_dice_meter_statistics_vs_reference(C, dct, dev):
    key = f"dice_C{C}_meter"
    m = dct.DiceMeter(method="2d", C=C, report_axises=[1])
    empty = m.value()  # empty-log fallback Tensor([0]*C) (dice_meter.py:68-71)
    assert empty[1][0].shape == (C,)
    for j in range(3):
        m.add(T(GOLDEN[f"{key}/x{j}"], dev), T(GOLDEN[f"{key}/gt{j}"], dev))
    (rm, rs), (ms, ss) = m.value()
    # the rows are bit-exact (test_dice_vs_reference_bit_exact); their mean/std are float reductions
    # whose order differs between ATen CPU (the fixture) and ATen CUDA
    assert_close(N(ms), GOLDEN[key + "/ref_means"], rtol=1e-6)
    assert_close(N(ss), GOLDEN[key + "/ref_stds"], rtol=1e-6)
    assert_close(np.array([rm.item(), rs.item()]), GOLDEN[key + "/ref_report"], rtol=1e-6)
    assert set(m.summary()) == {"mDSC", "mVars"} and set(m.detailed_summary()) == {f"DSC{i}" for i in range(C)}
    m.reset()
    assert m.log.shape == (1, C)


@pytest.mark.parametrize("case", _names("iou_"))
def test_iou_vs_reference_bit_exact(case, dct, dev):
    C = GOLDEN[case + "/x0"].shape[1]
    iou = dct.IoU(C, ignore_index=255)
    for j in range(2):
        iou.add(predicted=T(GOLDEN[f"{case}/x{j}"], dev), target=T(GOLDEN[f"{case}/gt{j}"], dev))
        conf = iou.conf_metric.conf
        assert conf.dtype == np.int32
        assert np.array_equal(conf.astype(np.int64), GOLDEN[f"{case}/ref_conf_after{j}"])
    v = iou.value()
    for k in ("Overall_Acc", "Mean_Acc", "FreqW_Acc", "Validated_Mean_IoU", "Mean_IoU"):
        assert v[k] == GOLDEN[f"{case}/ref_{k}"]
    assert np.array_equal(v["Class_IoU"].numpy(), GOLDEN[case + "/ref_Class_IoU"])
    iou2 = dct.IoU(C)
    iou2.add(T(GOLDEN[case + "/pred_map"], dev), T(GOLDEN[case + "/gt1"], dev).squeeze(1))
    assert np.array_equal(iou2.conf_metric.conf.astype(np.int64), GOLDEN[case + "/ref_conf_from_map"])
    iou2.reset()
    assert iou2.conf_metric.conf.sum() == 0


# ---------------------------------------------------------------------------------------------
# against the oracle on larger seeded inputs (BASELINE configs c1..c4 shapes, scaled to seconds)
# ---------------------------------------------------------------------------------------------
CONFIGS = [  # (name, K, C, B, H, W)
    ("c1", 2, 4, 4, 256, 256),
    ("c2", 3, 4, 8, 256, 256),
    ("c3", 2, 2, 4, 512, 512),
    ("c4", 2, 19, 2, 128, 256),
    ("k4c19", 4, 19, 1, 64, 128),
    ("rt_c5", 3, 5, 2, 40, 52),      # runtime-C fallback
    ("rt_k5", 5, 3, 2, 40, 52),      # runtime-K fallback
    ("odd", 2, 4, 3, 37, 41),        # HW not a multiple of 4: scalar fallback
    ("ragged_c4", 3, 4, 3, 36, 44),   # HW = 6 * 256 + 48: a ragged last tile per image in the 256-pixel tensor-map stages
    ("ragged_c2", 2, 2, 3, 100, 100), # HW = 9 * 1024 + 784: ragged last tile of the 4-row shape (1024-pixel tiles, row copies)
    ("ragged_c19", 2, 19, 2, 36, 44), # the same for the wide tensor-map stages
]


def _inputs(K, C, B, H, W, seed=1234):
    g = torch.Generator().manual_seed(seed)
    z = [3 * torch.randn(B, C, H, W, generator=g) for _ in range(K)]
    gt = torch.randint(0, C, (B, 1, H, W), generator=g)
    return z, gt


@pytest.mark.parametrize("name,K,C,B,H,W", CONFIGS)
def test_consistency_step_vs_oracle(name, K, C, B, H, W, dct, dev, oracle):
    z, gt = _inputs(K, C, B, H, W)
    w = 0.8
    n = B * H * W
    mean, mp, gz = oracle.jsd_logits_fwdbwd([t.numpy() for t in z], w)
    zd = [t.to(dev).requires_grad_() for t in z]
    counts = torch.zeros(K, B, C, 3, dtype=torch.int64, device=dev)
    loss = dct.jsd_consistency_from_logits(zd, weight=w, labels=gt.to(dev), dice_counts=counts)
    loss.backward()
    assert_close(loss.item(), w * mean, floor=w * lnK(K), what="loss")
    assert_close(np.stack([N(t.grad) for t in zd]), np.stack(gz), floor=w / n, what="grad")
    assert_close(N(dct.jsd_map_from_logits([t.to(dev) for t in z])), mp, floor=lnK(K), what="map")
    for k in range(K):
        oc, bad = oracle.dice_counts(z[k].numpy(), gt.numpy())
        assert bad == 0
        assert np.array_equal(N(counts[k]), oc), f"fused dice counts view {k}"
        assert np.array_equal(N(dct.dice_counts(z[k].to(dev), gt.to(dev))), oc), f"dice counts view {k}"
    # probs boundary
    probs = [oracle.softmax(t.numpy()) for t in z]
    pd = [T(p, dev, grad=True) for p in probs]
    m = dct.JSD_2D()(pd)
    assert_close(N(m), oracle.jsd_fwd(probs), floor=lnK(K), what="map from probs")
    gout = torch.randn(B, H, W, generator=torch.Generator().manual_seed(5))
    m.backward(gout.to(dev))
    assert_close(np.stack([N(p.grad) for p in pd]), np.stack(oracle.jsd_bwd(probs, gout.numpy())),
                 floor=float(gout.abs().max()), what="grad probs")
    # dice on probabilities (what the unlabeled meters receive, cotraining_totalloss.py:224)
    assert np.array_equal(N(dct.dice_counts(pd[0].detach(), gt.to(dev))), oracle.dice_counts(probs[0], gt.numpy())[0])
    # KL of view 0 vs view 1
    kl = oracle.kl_fwd(probs[0], probs[1])
    assert_close(N(dct.KL_Divergence_2D()(pd[0].detach(), pd[1].detach())), kl, floor=1.0, what="kl map")
    zl = z[0].to(dev).requires_grad_()
    l2 = dct.kl_consistency_from_logits(zl, pd[1].detach(), weight=w)
    l2.backward()
    assert_close(l2.item(), w * kl.mean(dtype=np.float64), floor=w, what="kl fused loss")
    gp = oracle.kl_bwd(probs[0], probs[1], np.full((B, H, W), w / n, np.float32))[0]
    assert_close(N(zl.grad), oracle.softmax_bwd(probs[0], gp), floor=w / n, what="kl fused grad")
    ml, gpl, gql = oracle.kl_logit(z[1].numpy(), z[0].numpy(), gout.numpy())
    a = z[1].to(dev).requires_grad_(); b_ = z[0].to(dev).requires_grad_()
    out = dct.kl_div_with_logit(a, b_)
    out.backward(gout.to(dev))
    assert_close(N(out), ml, floor=1.0)
    assert_close(N(b_.grad), gpl, floor=float(gout.abs().max()))
    assert_close(N(a.grad), gql, floor=float(gout.abs().max()))
    # confusion with 2% ignore labels
    gi = gt.clone()
    gi[torch.rand(gi.shape, generator=torch.Generator().manual_seed(9)) < 0.02] = 255
    iou = dct.IoU(C)
    iou.add(z[0].to(dev), gi.to(dev))
    assert np.array_equal(iou.conf_metric.conf64, oracle.confusion(z[0].numpy(), gi.numpy()))


@pytest.mark.parametrize("C", [2, 4, 19, 7])
def test_dice_near_ties_bit_exact(C, dct, dev, oracle):
    """Adversarial arg-max inputs: exact ties, 1..64-ulp near-ties, probabilities, NaN/inf rows."""
    g = torch.Generator().manual_seed(C)
    B, H, W = 2, 64, 64
    x = 3 * torch.randn(B, C, H, W, generator=g)
    mx, am = x.max(1, keepdim=True)
    other = (am + 1 + torch.randint(0, max(C - 1, 1), am.shape, generator=g)) % C  # != am
    ulps = torch.randint(0, 65, am.shape, generator=g)
    near = mx.clone()
    for _ in range(64):
        step = torch.nextafter(near, torch.full_like(near, -1e30))
        near = torch.where(ulps > 0, step, near)
        ulps = ulps - 1
    x.scatter_(1, other, near)
    gt = torch.randint(0, C, (B, 1, H, W), generator=g)
    for name, inp in (("logits", x), ("probs", torch.from_numpy(oracle.softmax(x.numpy())))):
        want, _ = oracle.dice_counts(inp.numpy(), gt.numpy())
        got = N(dct.dice_counts(inp.to(dev), gt.to(dev)))
        assert np.array_equal(got, want), name
    # special values
    y = x.clone()
    y[0, 0, 0, :8] = float("nan"); y[0, C - 1, 1, :8] = float("inf"); y[1, :, 2, :8] = float("-inf")
    y[1, 0, 3, :8] = float("inf"); y[1, C - 1, 3, :8] = float("inf")
    assert np.array_equal(N(dct.dice_counts(y.to(dev), gt.to(dev))), oracle.dice_counts(y.numpy(), gt.numpy())[0])
    iou = dct.IoU(C); iou.add(y.to(dev), gt.to(dev))
    assert np.array_equal(iou.conf_metric.conf64, oracle.confusion(y.numpy(), gt.numpy()))
    # on generic inputs the pinned arithmetic agrees with stock ATen on the same device
    z = 3 * torch.randn(B, C, H, W, generator=g)
    pred_aten = torch.softmax(z.to(dev), 1).argmax(1).cpu().numpy()
    assert np.array_equal(pred_aten, oracle.predict(z.numpy(), "dice"))


@pytest.mark.parametrize("K,C", [(3, 4), (2, 2), (4, 4), (2, 4), (3, 3)])
def test_fused_dice_groups_with_adversarial_members(K, C, dct, dev, oracle):
    """The fused K-view Dice path evaluates the fast-path arg-max test of all K x 2 predictions of a pixel pair together and
    redoes the whole group with the pinned arithmetic if ANY member fails it (csrc/dct_tile.cuh).  Inputs where single
    members of a group are exact ties, 1..64-ulp near-ties, NaN / +-inf rows -- next to ordinary members, in either pixel of
    the pair and in any view -- must give the oracle's counts bit for bit, view by view (also through the cross-entropy
    launch: one prediction per pixel)."""
    g = torch.Generator().manual_seed(100 * K + C)
    B, H, W = 2, 48, 44                       # HW = 2112 = 8 * 256 + 64: ragged last tile included
    views = []
    for k in range(K):
        x = 3 * torch.randn(B, C, H, W, generator=g)
        mx, am = x.max(1, keepdim=True)
        other = (am + 1 + torch.randint(0, max(C - 1, 1), am.shape, generator=g)) % C
        ulps = torch.randint(0, 65, am.shape, generator=g)
        hit = torch.rand(am.shape, generator=g) < 0.3          # 30 % of the pixels of this view carry a (near-)tie
        near = mx.clone()
        for _ in range(64):
            near = torch.where(ulps > 0, torch.nextafter(near, torch.full_like(near, -1e30)), near)
            ulps = ulps - 1
        x.scatter_(1, other, torch.where(hit, near, x.gather(1, other)))
        # special rows in a few odd / even pixels of different rows, different per view
        x[0, 0, 1 + k, 1:9:2] = float("nan")
        x[0, C - 1, 5 + k, 0:8:2] = float("inf")
        x[1, :, 9 + k, 3:11] = float("-inf")
        x[1, 0, 13 + k, 2:6] = float("inf"); x[1, C - 1, 13 + k, 2:6] = float("inf")
        x[1, :, 17 + k, 5:7] = float("nan")
        views.append(x)
    gt = torch.randint(0, C, (B, 1, H, W), generator=g)
    want = [oracle.dice_counts(v.numpy(), gt.numpy())[0] for v in views]
    old = dct.set_check_mode("off")          # the loss of these inputs is NaN by construction; only the counts are examined
    try:
        counts = torch.zeros(K, B, C, 3, dtype=torch.int64, device=dev)
        zr = [v.to(dev).requires_grad_() for v in views]
        dct.jsd_consistency_from_logits(zr, weight=1.0, labels=gt.to(dev), dice_counts=counts).backward()
        for k in range(K):
            assert np.array_equal(N(counts[k]), want[k]), f"fused JSD + Dice, view {k}"
            assert np.array_equal(N(dct.dice_counts(views[k].to(dev), gt.to(dev))), want[k]), f"dice_counts, view {k}"
        c1 = torch.zeros(B, C, 3, dtype=torch.int64, device=dev)
        dct.supervised_from_logits(views[0].to(dev).requires_grad_(), gt.to(dev), dice_counts=c1).backward()
        assert np.array_equal(N(c1), want[0]), "fused cross-entropy + Dice"
    finally:
        dct.set_check_mode(old)


def test_flags_and_errors_through_c_abi(dct, dev):
    """Error behaviour of the raw C ABI: bad args return negative codes, nothing is launched."""
    h = dct._lib.lib()
    x = torch.randn(1, 4, 8, 8, device=dev)
    arr = dct._lib.ptr_array([x, x])
    assert h.dct_jsd_fwd_f32(arr, 2, 4, 1, 64, 7, None, None, None, None, None) == -1      # bad in_kind
    assert h.dct_jsd_fwd_f32(arr, 9, 4, 1, 64, 1, None, None, None, None, None) == -2      # K > 8
    assert h.dct_jsd_fwd_f32(arr, 2, 65, 1, 64, 1, None, None, None, None, None) == -2     # C > 64
    assert h.dct_jsd_fwd_f32(None, 2, 4, 1, 64, 1, None, None, None, None, None) == -1
    assert h.dct_dice_counts_f32(x.data_ptr() + 2, x.data_ptr(), 4, 1, 64, x.data_ptr(), 0, None, None) == -3
    assert h.dct_l2_normalize_f32(None, None, 1, 1, 1, 1.0, None, None, None, None) == -1
    d = torch.randn(2, 1, 8, 8, device=dev)
    assert h.dct_l2_normalize_f32(d.data_ptr(), d.data_ptr(), 2, 64, 3, 1.0, None, None, None, None) == -1  # passes in {1,2}
    assert b"misaligned" in h.dct_error_string(-3)
    torch.cuda.synchronize()


# ---------------------------------------------------------------------------------------------
# size-independent properties at BASELINE's full sizes (no oracle: it would take minutes)
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("K,C,B,H,W", [(3, 4, 32, 256, 256), (2, 19, 16, 512, 1024), (2, 2, 32, 512, 512)])
def test_full_size_properties(K, C, B, H, W, dct, dev):
    g = torch.Generator(device=dev).manual_seed(1234)
    z = [3 * torch.randn(B, C, H, W, generator=g, device=dev) for _ in range(K)]
    gt = torch.randint(0, C, (B, 1, H, W), generator=g, device=dev)
    n = B * H * W
    # identical views: K in {2,4}: JSD == 0 exactly and zero gradient; any K: |JSD| tiny
    same = [z[0].clone().requires_grad_() for _ in range(K)]
    l0 = dct.jsd_consistency_from_logits(same, weight=1.0)
    l0.backward()
    assert abs(l0.item()) <= 1e-6
    assert float(max(s.grad.abs().max() for s in same)) <= 1e-5 / n
    # range, symmetry under view permutation, fused == map.mean(), gradient sums to zero over classes
    zr = [t.clone().requires_grad_() for t in z]
    counts = torch.zeros(K, B, C, 3, dtype=torch.int64, device=dev)
    loss = dct.jsd_consistency_from_logits(zr, weight=1.0, labels=gt, dice_counts=counts)
    loss.backward()
    m = dct.jsd_map_from_logits(z)
    assert float(m.min()) >= -1e-6 and float(m.max()) <= math.log(K) + 1e-6
    assert abs(m.double().mean().item() - loss.item()) <= 1e-6 * math.log(K)
    m_perm = dct.jsd_map_from_logits(z[::-1])
    assert float((m - m_perm).abs().max()) <= 2e-6
    for t in zr:
        assert float(t.grad.sum(1).abs().max()) <= 1e-5 / n  # softmax backward: zero class-sum
    # shift invariance of softmax: adding a per-pixel constant changes nothing beyond rounding
    shifted = [t + 5.0 for t in z]
    assert float((dct.jsd_map_from_logits(shifted) - m).abs().max()) <= 2e-5
    # integer conservation laws
    for k in range(K):
        c = counts[k]
        assert torch.equal(c[:, :, 1].sum(1), torch.full((B,), H * W, device=dev))  # every label counted once
        assert torch.equal(c[:, :, 2].sum(1), torch.full((B,), H * W, device=dev))  # every prediction counted once
        assert bool((c[:, :, 0] <= torch.minimum(c[:, :, 1], c[:, :, 2])).all())
        pred = z[k].argmax(1)  # no ties in random data: equals the raw arg-max
        want_p = torch.stack([(pred == cc).flatten(1).sum(1) for cc in range(C)], 1)
        assert torch.equal(c[:, :, 2], want_p)
        want_i = torch.stack([((pred == cc) & (gt.squeeze(1) == cc)).flatten(1).sum(1) for cc in range(C)], 1)
        assert torch.equal(c[:, :, 0], want_i)
    iou = dct.IoU(C)
    gi = gt.clone(); gi[:, :, ::7, ::5] = 255
    iou.add(z[0], gi)
    conf = iou.conf_metric.conf64
    assert conf.sum() == int((gi != 255).sum())
    key = (gi.squeeze(1) * C + z[0].argmax(1))[gi.squeeze(1) != 255]
    assert np.array_equal(conf.reshape(-1), torch.bincount(key, minlength=C * C).cpu().numpy())
    # l2 normalise: idempotent up to rounding, unit norm
    d = torch.randn(B, 1, H, W, generator=g, device=dev)
    d1 = dct.l2_normalize(d.clone())
    nr = d1.flatten(1).double().norm(dim=1)
    assert float((nr - 1).abs().max()) <= 1e-5
    d2 = dct.l2_normalize(d1.clone())
    assert float((d2 - d1).abs().max()) <= 1e-6 * float(d1.abs().max())


# ---------------------------------------------------------------------------------------------
# Dice counters kept in registers across tiles (csrc/dct_tile.cuh, "Fused Dice counters"): images so large that one CTA works
# through hundreds of tiles of the SAME image, so the packed 8-bit fields must be flushed before they overflow
# (every 255 / pixels-per-thread tiles), plus a ragged last tile and a batch of 1 (fewer flushes than warps)
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("C,B,H,W", [(4, 2, 4096, 4096), (2, 1, 4096, 4100), (4, 3, 2048, 2052)])
def test_dice_counters_long_runs_of_one_image(C, B, H, W, dct, dev):
    g = torch.Generator(device=dev).manual_seed(99)
    K = 2
    z = [3 * torch.randn(B, C, H, W, generator=g, device=dev) for _ in range(K)]
    gt = torch.randint(0, C, (B, 1, H, W), generator=g, device=dev)
    gt[:, :, : H // 3] = 0  # unbalanced: class 0 alone would overflow an 8-bit field within 64 tiles

    def want(zk):
        pred = zk.argmax(1)  # random data: no ties, equals argmax softmax
        lab = gt.squeeze(1)
        return torch.stack([torch.stack([((pred == c) & (lab == c)).flatten(1).sum(1), (lab == c).flatten(1).sum(1),
                                         (pred == c).flatten(1).sum(1)], 1) for c in range(C)], 1)   # [B,C,3]

    ref = [want(t) for t in z]
    # the Dice meter's own kernel (one tensor, 4 pixels per thread)
    for k in range(K):
        assert torch.equal(dct.dice_counts(z[k], gt), ref[k])
    # fused into the JSD launch (K count sets, 2 pixels per thread)
    counts = torch.zeros(K, B, C, 3, dtype=torch.int64, device=dev)
    zr = [t.clone().requires_grad_() for t in z]
    dct.jsd_consistency_from_logits(zr, weight=1.0, labels=gt, dice_counts=counts).backward()
    for k in range(K):
        assert torch.equal(counts[k], ref[k])
    del zr
    # fused into the cross-entropy launch
    c1 = torch.zeros(B, C, 3, dtype=torch.int64, device=dev)
    dct.supervised_from_logits(z[0].clone().requires_grad_(), gt, dice_counts=c1).backward()
    assert torch.equal(c1, ref[0])


# ---------------------------------------------------------------------------------------------
# K*C > 40 (K = 3, 4 at C = 19): the one-pixel-per-thread tile shapes, whose K*C values fill most of the register file --
# ragged tails, saturated logits whose exponentials underflow to zero, identical views, confident and agreeing inputs
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("K", [3, 4])
@pytest.mark.parametrize("variant", ["plain", "confident", "agreeing", "saturated", "identical"])
def test_wide_jsd_streaming_body_vs_oracle(K, variant, dct, dev, oracle):
    C, B, H, W = 19, 2, 52, 100          # 5200 pixels per image: the last tile of every image is ragged
    g = torch.Generator().manual_seed(77 + K)
    z0 = torch.randn(B, C, H, W, generator=g)
    if variant == "plain":
        z = [3 * torch.randn(B, C, H, W, generator=g) for _ in range(K)]
    elif variant == "confident":
        z = [10 * torch.randn(B, C, H, W, generator=g) for _ in range(K)]
    elif variant == "agreeing":
        z = [3 * z0 + 0.1 * torch.randn(B, C, H, W, generator=g) for _ in range(K)]
    elif variant == "saturated":
        z = [80.0 * torch.sign(torch.randn(B, C, H, W, generator=g)) for _ in range(K)]   # exp underflows for the -80s
    else:
        z = [(3 * z0).clone() for _ in range(K)]
    w = 0.7
    n = B * H * W
    mean, mp, gz = oracle.jsd_logits_fwdbwd([t.numpy() for t in z], w)
    zd = [t.to(dev).requires_grad_() for t in z]
    loss = dct.jsd_consistency_from_logits(zd, weight=w)
    loss.backward()
    got = np.stack([N(t.grad) for t in zd])
    assert np.isfinite(got).all()
    assert_close(loss.item(), w * mean, floor=w * lnK(K), what="loss")
    assert_close(got, np.stack(gz), floor=w / n, what="grad")
    if variant == "identical":
        assert abs(loss.item()) <= 1e-6 and float(np.abs(got).max()) <= 1e-5 * w / n
