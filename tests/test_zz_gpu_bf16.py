"""GPU parity of the bf16 entry points (networks under autocast): dct_jsd_fwdbwd_bf16, dct_kl_logit_bf16,
dct_kl_from_logits_fwdbwd_bf16, dct_ce_fwdbwd_bf16.

The bf16 kernels read and write 2-byte rows but compute in fp32, so on the SAME (bf16-representable) inputs x every
gradient element is the round-to-nearest-even bf16 of what the fp32 path computes on x.float().  `_check_grad` holds
every bf16 gradient to that, element by element, with three witnesses of the same inputs:
  got  the bf16 gradient,
  gf   the fp32 path's gradient on x.float() (the same values),
  g64  a float64 torch-autograd reference on x.double() with the reference formulas (1e-16 inside the entropies,
       eps = 1e-10 in the adversarial KL, F.cross_entropy with weight and ignore_index), independent of the kernels.
Checks:
  (A) tile shapes, upstream applied in-kernel or equal to 1: every element within 1 bf16 ulp of RNE_bf16(gf) (distance
      of the bit patterns, +0 == -0), and at most max(2, n/100) elements differ at all.  Both paths run the same fp32
      Op::apply in the same tile shape; a differently contracted FMA can only move values lying within a few fp32 ulps
      of a bf16 rounding midpoint, while truncation instead of rounding would move about half of them.
  (B) every element: |got - g64| <= r*|g64| + 2*|gf - g64| + 2^-24 * S_pix + a, S_pix = max_c |g64[b, c, pixel]|;
      r = 2^-8 for one rounding, 2^-7 + 2^-16 when a non-unit upstream is applied afterwards (two roundings).  The
      floor covers underflowed softmax tails and flush-to-zero; a = 2^-134 per rounding is half the spacing of bf16's
      subnormals (at 40*randn whole pixels have gradients near 1e-40).  gf itself is held to g64 at 1e-4 of the largest
      element.
  (C) promoted shapes (the wrapper converts to float32 and runs the fp32 kernels): got == gf.to(bfloat16) bit for bit.
Each check asserts on its own data that it would reject a gradient truncated instead of rounded.
Loss maps (fp32) are bit-equal to the fp32 path's on >= 99 % of the pixels and within 2^-16 * max(1, |mf|) everywhere;
losses are held to the float64 reference at the fp32 bar; integer Dice counts are bit-exact against the CPU oracle,
first-index tie rule included (ties are frequent on bf16's coarse grid).

The shape matrix reaches every tile row class (tile width 1024, 256, 192, 512 forward-only, 160, 224 pixels) with a
ragged last tile, and with >= 10 tiles per CTA of the persistent grid, at 3*randn logits and at 40*randn (softmax
underflow, wide log ranges, many ties).

History: written at the end of round 1 as non-strict xfail (no GPU minutes left); the round-end run showed all 26 cases
passing, so the marker is gone and a regression now fails the suite.  The gradient bar was 1e-2 of the largest element
until the element-wise checker replaced it.
"""
import math

import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

BF = torch.bfloat16
FP32_LOSS_TOL = 1e-5          # losses are accumulated in fp32 / fixed point from identical inputs
R1 = 2.0 ** -8                # one round-to-nearest-even to bf16: |RNE(v) - v| <= 2^-8 |v|
R2 = 2.0 ** -7 + 2.0 ** -16   # RNE(RNE(v) * s) against v * s: two roundings around one fp32 multiply
FLOOR = 2.0 ** -24            # of the pixel's largest |gradient|
SUB_HALF_ULP = 2.0 ** -134    # half the spacing of bf16's subnormals: the absolute error of one rounding down there
GF_TOL = 1e-4                 # the fp32 witness against float64, of the largest |gradient| (its own bar is 1e-5)
EPS_KL = 1e-10
SMS = 148                     # B200


@pytest.fixture(scope="module")
def dct():
    import dct_b200
    assert torch.cuda.is_available()
    return dct_b200


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda:0")


# ------------------------------------------------------------------------------------------------
# the checker
# ------------------------------------------------------------------------------------------------
def _key(t):
    """bf16 bit patterns as ordered integers: neighbouring bf16 values differ by 1, +0 and -0 are both 0."""
    b = t.contiguous().view(torch.int16).to(torch.int32) & 0xffff
    mag = b & 0x7fff
    return torch.where(b >= 0x8000, -mag, mag)


def _bits_equal(a, b):
    return torch.equal(a.contiguous().view(torch.int16), b.contiguous().view(torch.int16))


def _rz(gf):
    """gf truncated to bf16 (what a round-toward-zero store would write)."""
    return (gf.contiguous().view(torch.int32) & -65536).view(torch.float32).to(BF)


def _excess(got, gf, g64, r):
    """(B): per element, |got - g64| minus its bound; > 0 where the bound is broken.  Below 2^-126 bf16 is subnormal
    with a spacing of 2^-133, so each rounding may also be off by up to 2^-134 absolute (half that spacing): 2^-134
    for one rounding, (1 + s) * 2^-134 <= 3 * 2^-134 for RNE(RNE(v) * s) with the upstreams s <= 2 used here."""
    got, gf = got.double(), gf.double()
    s_pix = g64.abs().amax(dim=1, keepdim=True)
    sub = SUB_HALF_ULP * (1.0 if r == R1 else 3.0)
    return (got - g64).abs() - (r * g64.abs() + 2.0 * (gf - g64).abs() + FLOOR * s_pix + sub)


def _check_b(got, gf, g64, r, what):
    ex = _excess(got, gf, g64, r)
    i = int(ex.argmax())
    assert float(ex.flatten()[i]) <= 0.0, \
        f"{what}: bound (B) broken at flat index {i}: got {float(got.flatten()[i])!r}, fp32 path " \
        f"{float(gf.flatten()[i])!r}, float64 {float(g64.flatten()[i])!r}"


def _check_grad(got, gf, g64, what, r=R1, promoted=False):
    """got: bf16 gradient; gf: the fp32 path's gradient of the same values (same upstream); g64: float64 reference."""
    assert got.dtype == BF, f"{what}: gradient dtype {got.dtype}"
    assert got.shape == gf.shape == g64.shape, what
    scale = float(g64.abs().max())
    err = float((gf.double() - g64).abs().max())
    assert err <= GF_TOL * scale, f"{what}: fp32 witness {err:.3e} from float64 (scale {scale:.3e})"
    want = gf.to(BF)
    n = got.numel()
    if promoted:   # (C)
        assert _bits_equal(got, want), f"{what}: promoted gradient is not the bf16 cast of the fp32 path's"
    else:          # (A)
        d = (_key(got) - _key(want)).abs()
        nd = int((d != 0).sum())
        assert int(d.max()) <= 1, f"{what}: {int(d.max())} bf16 ulps from RNE(fp32 path)"
        assert nd <= max(2, n // 100), f"{what}: {nd} of {n} elements differ from RNE(fp32 path)"
        # teeth: truncation would move far more elements than the bar allows
        assert int((_key(_rz(gf)) != _key(want)).sum()) > max(2, n // 100), f"{what}: (A) has no teeth on this data"
    _check_b(got, gf, g64, r, what)
    assert float(_excess(_rz(gf), gf, g64, r).max()) > 0.0, f"{what}: (B) has no teeth on this data"


def _check_map(mb, mf, what):
    """fp32 loss map of the bf16 launch against the fp32 path's on the same values."""
    assert mb.dtype == torch.float32 and mb.shape == mf.shape, what
    eq = mb.contiguous().view(torch.int32) == mf.contiguous().view(torch.int32)
    assert float(eq.double().mean()) >= 0.99, f"{what}: only {float(eq.double().mean()):.4f} of the map bit-equal"
    assert bool(((mb - mf).abs() <= 2.0 ** -16 * mf.abs().clamp_min(1.0)).all()), f"{what}: map off the fp32 path's"


# ------------------------------------------------------------------------------------------------
# shapes and inputs
# ------------------------------------------------------------------------------------------------
def _tile_shape(rows, nout):
    """(pixels per tile, CTAs per SM) of the tile pipeline for NIN*C = rows (dct_tile.cuh, tile_launch_ct)."""
    if rows <= 4:
        return 1024, 2
    if rows <= 16:
        return 256, 3
    if rows <= 24:
        return 256, 2
    if rows <= 40:
        return (512, 1) if nout == 0 else (192, 2)
    if rows <= 60:
        return 160, 2
    return 224, 1


def _hw(rows, nout, size):
    """'tail': one whole tile and a ragged one of 8 pixels per image; 'many': with B = 2, >= 10 tiles per CTA."""
    tpx, minb = _tile_shape(rows, nout)
    return tpx + 8 if size == "tail" else 5 * SMS * minb * tpx + 8


def _logits(K, C, B, H, W, dev, seed, amp=3.0):
    g = torch.Generator(device=dev).manual_seed(seed)
    return [(amp * torch.randn(B, C, H, W, generator=g, device=dev)).to(BF) for _ in range(K)]


def _simplex(C, B, H, W, dev, seed):
    """Probabilities bf16 holds exactly (the kernel asserts a simplex to 1e-5, which a rounded bf16 softmax is not):
    half the mass on each of two random classes, all of it when they agree."""
    g = torch.Generator(device=dev).manual_seed(seed)
    c1 = torch.randint(0, C, (B, 1, H, W), generator=g, device=dev)
    c2 = torch.randint(0, C, (B, 1, H, W), generator=g, device=dev)
    y = torch.zeros(B, C, H, W, device=dev).scatter_add_(1, c1, torch.full_like(c1, 0.5, dtype=torch.float32))
    y.scatter_add_(1, c2, torch.full_like(c2, 0.5, dtype=torch.float32))
    assert torch.equal(y.to(BF).float(), y)
    return y.to(BF)


# ------------------------------------------------------------------------------------------------
# float64 references (torch autograd on the same values)
# ------------------------------------------------------------------------------------------------
def _jsd64(zs, weight):
    p = [torch.softmax(z, 1) for z in zs]
    m = sum(p) / len(p)
    ent = lambda q: -(q * torch.log(q + 1e-16)).sum(1)
    return weight * (ent(m) - sum(ent(q) for q in p) / len(p)).mean()


def _kl_logit_map64(q, p):
    return (torch.softmax(q, 1) * (torch.log_softmax(q, 1) - torch.log_softmax(p, 1))).sum(1)


def _klc64(a, y, weight):
    p = torch.softmax(a, 1)
    return weight * (y * torch.log(y + EPS_KL) - y * torch.log(p + EPS_KL)).sum(1).mean()


def _ce64(z, gt, w, reduction):
    return F.cross_entropy(z, gt.squeeze(1), weight=None if w is None else w.double(), ignore_index=255,
                           reduction=reduction)


def _grad64(fn, xs):
    """(value, gradients) of fn(*xd) at xd = x.double()."""
    xd = [x.detach().double().requires_grad_() for x in xs]
    v = fn(*xd)
    return v.detach(), torch.autograd.grad(v, xd)


def _jsd_mean_f64(zs):
    return float(_jsd64([z.double() for z in zs], 1.0))


# ------------------------------------------------------------------------------------------------
# the original cases (their loss and count assertions unchanged; gradients through the checker)
# ------------------------------------------------------------------------------------------------
# H*W % 8 == 0 -> the bf16 tile pipeline; (5, 7) and (9, 12) are not -> promotion to the fp32 kernels inside the wrapper
@pytest.mark.parametrize("K,C,B,H,W", [(2, 4, 3, 64, 72), (3, 4, 2, 40, 40), (2, 2, 2, 128, 64), (2, 19, 2, 32, 40),
                                       (3, 19, 1, 24, 40), (4, 4, 2, 16, 24), (2, 4, 2, 5, 7), (3, 19, 1, 9, 12)])
def test_jsd_consistency_bf16(K, C, B, H, W, dct, dev, oracle):
    zb = _logits(K, C, B, H, W, dev, 11)
    zf = [z.float().requires_grad_() for z in zb]
    lf = dct.jsd_consistency_from_logits(zf, weight=0.7)
    lf.backward()
    zr = [z.clone().requires_grad_() for z in zb]
    lb = dct.jsd_consistency_from_logits(zr, weight=0.7)
    lb.backward()
    assert abs(lb.item() - lf.item()) <= FP32_LOSS_TOL * math.log(K)
    assert abs(lb.item() - 0.7 * _jsd_mean_f64(zb)) <= FP32_LOSS_TOL * math.log(K)
    omean, _, _ = oracle.jsd_logits_fwdbwd([z.float().cpu().numpy() for z in zb], 0.7, want_map=False)
    assert abs(lb.item() - 0.7 * omean) <= FP32_LOSS_TOL * math.log(K)
    _, g64 = _grad64(lambda *z: _jsd64(z, 0.7), zb)
    promoted = (H * W) % 8 != 0
    for k in range(K):
        _check_grad(zr[k].grad, zf[k].grad, g64[k], f"view {k}", promoted=promoted)


@pytest.mark.parametrize("K,C,B,H,W", [(3, 4, 4, 64, 64), (2, 2, 2, 96, 80), (2, 4, 1, 8, 8), (2, 19, 2, 32, 40)])
def test_jsd_consistency_bf16_with_dice_counts(K, C, B, H, W, dct, dev, oracle):
    zb = _logits(K, C, B, H, W, dev, 12)
    g = torch.Generator(device=dev).manual_seed(5)
    gt = torch.randint(0, C, (B, 1, H, W), generator=g, device=dev)
    cf = torch.zeros(K, B, C, 3, dtype=torch.int64, device=dev)
    zf = [z.float().requires_grad_() for z in zb]
    lf = dct.jsd_consistency_from_logits(zf, labels=gt, dice_counts=cf)
    lf.backward()
    cb = torch.zeros(K, B, C, 3, dtype=torch.int64, device=dev)
    zr = [z.clone().requires_grad_() for z in zb]
    lb = dct.jsd_consistency_from_logits(zr, labels=gt, dice_counts=cb)
    lb.backward()
    assert torch.equal(cb, cf), "Dice counts of the bf16 launch differ from the fp32 launch on the same values"
    for k in range(K):   # and from a plain count (bf16 values tie often: first index wins, as argmax softmax does)
        assert torch.equal(cb[k, :, :, 1].sum(1), torch.full((B,), H * W, device=dev))
        assert torch.equal(cb[k, :, :, 2].sum(1), torch.full((B,), H * W, device=dev))
    assert abs(lb.item() - lf.item()) <= FP32_LOSS_TOL * math.log(K)
    _, g64 = _grad64(lambda *z: _jsd64(z, 1.0), zb)
    for k in range(K):
        _check_grad(zr[k].grad, zf[k].grad, g64[k], f"view {k}")
        oc, bad = oracle.dice_counts(zb[k].float().cpu().numpy(), gt.cpu().numpy())
        assert bad == 0 and np.array_equal(cb[k].cpu().numpy(), oc), "Dice counts of the bf16 launch differ from the oracle"


@pytest.mark.parametrize("C,B,H,W", [(4, 3, 64, 72), (2, 2, 128, 64), (19, 2, 32, 40), (4, 2, 5, 7)])
def test_kl_div_with_logit_bf16(C, B, H, W, dct, dev, oracle):
    qb, pb = _logits(2, C, B, H, W, dev, 13)
    g = torch.Generator(device=dev).manual_seed(6)
    up = torch.rand(B, H, W, generator=g, device=dev)   # a per-pixel upstream, as `.mean()` or a weighting would send
    qf, pf = qb.float().requires_grad_(), pb.float().requires_grad_()
    mf = dct.kl_div_with_logit(qf, pf)
    (mf * up).sum().backward()
    qr, pr = qb.clone().requires_grad_(), pb.clone().requires_grad_()
    mb = dct.kl_div_with_logit(qr, pr)
    (mb * up).sum().backward()
    assert mb.dtype == torch.float32 and mb.shape == (B, H, W)
    assert float((mb - mf).detach().abs().max()) <= FP32_LOSS_TOL * max(1.0, float(mf.detach().abs().max()))
    want = (torch.softmax(qb.double(), 1) * (torch.log_softmax(qb.double(), 1) - torch.log_softmax(pb.double(), 1))).sum(1)
    assert float((mb.detach().double() - want).abs().max()) <= 2e-5 * max(1.0, float(want.abs().max()))
    _, (gq64, gp64) = _grad64(lambda q, p: (_kl_logit_map64(q, p) * up.double()).sum(), (qb, pb))
    promoted = (H * W) % 8 != 0
    if not promoted:
        _check_map(mb.detach(), mf.detach(), "map")
    _check_grad(pr.grad, pf.grad, gp64, "p_logit", promoted=promoted)
    _check_grad(qr.grad, qf.grad, gq64, "q_logit", promoted=promoted)
    omap, _, _ = oracle.kl_logit(qb.float().cpu().numpy(), pb.float().cpu().numpy(), up.cpu().numpy())
    assert float(np.abs(mb.detach().cpu().numpy() - omap).max()) <= 2e-5 * max(1.0, float(np.abs(omap).max()))


@pytest.mark.parametrize("C,B,H,W", [(4, 3, 64, 72), (2, 2, 128, 64), (19, 2, 32, 40), (4, 2, 5, 7)])
def test_kl_consistency_from_logits_bf16(C, B, H, W, dct, dev, oracle):
    (ab,) = _logits(1, C, B, H, W, dev, 14)
    real_b = _simplex(C, B, H, W, dev, 8)
    af = ab.float().requires_grad_()
    lf = dct.kl_consistency_from_logits(af, real_b.float(), weight=1.3)
    lf.backward()
    ar = ab.clone().requires_grad_()
    lb = dct.kl_consistency_from_logits(ar, real_b, weight=1.3)
    lb.backward()
    assert abs(lb.item() - lf.item()) <= FP32_LOSS_TOL * max(1.0, abs(lf.item()))
    a_np, y_np = ab.float().cpu().numpy(), real_b.float().cpu().numpy()
    p_np = oracle.softmax(a_np)
    assert abs(lb.item() - 1.3 * float(oracle.kl_fwd(p_np, y_np).mean(dtype=np.float64))) <= 2e-5 * max(1.0, abs(lf.item()))
    _, (g64,) = _grad64(lambda a: _klc64(a, real_b.double(), 1.3), (ab,))
    _check_grad(ar.grad, af.grad, g64, "adv_logit", promoted=(H * W) % 8 != 0)


@pytest.mark.parametrize("C,B,H,W,weighted", [(4, 3, 64, 72, False), (4, 2, 40, 40, True), (2, 2, 128, 64, False),
                                              (19, 2, 32, 40, True), (4, 2, 5, 7, False)])
def test_supervised_from_logits_bf16(C, B, H, W, weighted, dct, dev, oracle):
    (zb,) = _logits(1, C, B, H, W, dev, 15)
    g = torch.Generator(device=dev).manual_seed(7)
    gt = torch.randint(0, C, (B, 1, H, W), generator=g, device=dev)
    if C == 19:
        gt[:, :, ::5, ::3] = 255      # ignore_index
    w = (0.5 + torch.rand(C, generator=g, device=dev)) if weighted else None
    dice = C <= 4
    cf = torch.zeros(B, C, 3, dtype=torch.int64, device=dev) if dice else None
    cb = torch.zeros(B, C, 3, dtype=torch.int64, device=dev) if dice else None
    zf = zb.float().requires_grad_()
    lf = dct.supervised_from_logits(zf, gt, weight=w, dice_counts=cf)
    lf.backward()
    zr = zb.clone().requires_grad_()
    lb = dct.supervised_from_logits(zr, gt, weight=w, dice_counts=cb)
    lb.backward()
    want = torch.nn.functional.cross_entropy(zb.double(), gt.squeeze(1), weight=None if w is None else w.double(),
                                             ignore_index=255)
    assert abs(lb.item() - lf.item()) <= FP32_LOSS_TOL * max(1.0, abs(lf.item()))
    assert abs(lb.item() - float(want)) <= 2e-5 * max(1.0, abs(float(want)))
    _, (g64,) = _grad64(lambda z: _ce64(z, gt, w, "mean"), (zb,))
    _check_grad(zr.grad, zf.grad, g64, "logits", promoted=(H * W) % 8 != 0)
    oloss, _, _ = oracle.cross_entropy(zb.float().cpu().numpy(), gt.cpu().numpy(),
                                       weight=None if w is None else w.cpu().numpy(), ignore_index=255)
    assert abs(lb.item() - oloss) <= 2e-5 * max(1.0, abs(oloss))
    if dice:
        assert torch.equal(cb, cf)
        oc, bad = oracle.dice_counts(zb.float().cpu().numpy(), gt.cpu().numpy())
        assert bad == 0 and np.array_equal(cb.cpu().numpy(), oc)


def test_mixed_precision_views_are_promoted(dct, dev):
    """One bf16 view next to a float32 view: promoted to the fp32 kernels, each gradient in its input's dtype."""
    zb = _logits(2, 4, 2, 32, 32, dev, 16)
    a, b = zb[0].clone().requires_grad_(), zb[1].float().requires_grad_()
    loss = dct.jsd_consistency_from_logits([a, b])
    loss.backward()
    af, bf = zb[0].float().requires_grad_(), zb[1].float().requires_grad_()
    lf = dct.jsd_consistency_from_logits([af, bf])
    lf.backward()
    assert abs(loss.item() - lf.item()) <= FP32_LOSS_TOL
    assert a.grad.dtype == torch.bfloat16 and b.grad.dtype == torch.float32
    _, g64 = _grad64(lambda *z: _jsd64(z, 1.0), zb)
    _check_grad(a.grad, af.grad, g64[0], "bf16 view", promoted=True)
    assert float((b.grad - bf.grad).abs().max()) <= 1e-6 * float(bf.grad.abs().max())


# ------------------------------------------------------------------------------------------------
# the tile shape matrix
# ------------------------------------------------------------------------------------------------
JSD_KC = [(2, 2), (2, 3), (3, 3), (4, 3), (4, 4), (2, 19), (3, 19), (4, 19)]   # rows 4, 6, 9, 12, 16, 38, 57, 76
KL_C = [2, 3, 4, 19]


def _jsd_cases():
    out = []
    for K, C in JSD_KC:
        for dice in (("none", "acc", "over") if C <= 4 else ("none",)):
            out.append((K, C, "tail", dice, 3.0))
        out.append((K, C, "many", "over" if C <= 4 else "none", 3.0))
    return out + [(2, 2, "tail", "acc", 40.0), (2, 19, "tail", "none", 40.0), (4, 19, "tail", "none", 40.0)]


@pytest.mark.parametrize("K,C,size,dice,amp", _jsd_cases())
def test_jsd_consistency_bf16_tiles(K, C, size, dice, amp, dct, dev, oracle):
    B, HW = 2, _hw(K * C, K, size)
    H, W = HW // 8, 8
    zb = _logits(K, C, B, H, W, dev, 100 * K + C, amp)
    g = torch.Generator(device=dev).manual_seed(31)
    gt = torch.randint(0, C, (B, 1, H, W), generator=g, device=dev) if dice != "none" else None
    base = None
    if dice == "acc":
        base = torch.randint(0, 1000, (K, B, C, 3), generator=g, device=dev)
    elif dice == "over":
        base = torch.full((K, B, C, 3), 12345, dtype=torch.int64, device=dev)   # must be overwritten

    def run(zs):
        cnt = None if base is None else base.clone()
        zr = [z.detach().clone().requires_grad_() for z in zs]
        loss = dct.jsd_consistency_from_logits(zr, weight=0.7, labels=gt, dice_counts=cnt, accumulate=dice != "over")
        loss.backward()
        return loss.item(), [z.grad for z in zr], cnt

    lb, gb, cb = run(zb)
    lf, gf, cf = run([z.float() for z in zb])
    l64, g64 = _grad64(lambda *z: _jsd64(z, 0.7), zb)
    assert abs(lb - lf) <= FP32_LOSS_TOL * math.log(K)
    assert abs(lb - float(l64)) <= FP32_LOSS_TOL * math.log(K)
    for k in range(K):
        _check_grad(gb[k], gf[k], g64[k], f"view {k}")
    if base is not None:
        assert torch.equal(cb, cf), "Dice counts of the bf16 launch differ from the fp32 launch"
        gt_np = gt.cpu().numpy()
        for k in range(K):
            oc, bad = oracle.dice_counts(zb[k].float().cpu().numpy(), gt_np)
            if dice == "acc":
                oc = oc + base[k].cpu().numpy()
            assert bad == 0 and np.array_equal(cb[k].cpu().numpy(), oc), f"view {k}: Dice counts differ from the oracle"


@pytest.mark.parametrize("K,C", JSD_KC)
@pytest.mark.parametrize("with_labels", [False, True])
def test_jsd_consistency_bf16_forward_only(K, C, with_labels, dct, dev, oracle):
    """Evaluation: no input requires a gradient, so the forward-only instantiation runs (at 38 rows a 512-pixel tile)."""
    B, HW = 2, _hw(K * C, 0, "tail")
    H, W = HW // 8, 8
    zb = _logits(K, C, B, H, W, dev, 200 + 10 * K + C)
    g = torch.Generator(device=dev).manual_seed(32)
    gt = torch.randint(0, C, (B, 1, H, W), generator=g, device=dev) if with_labels else None

    def run(zs):
        cnt = torch.full((K, B, C, 3), -1, dtype=torch.int64, device=dev) if with_labels else None
        with torch.no_grad():
            loss = dct.jsd_consistency_from_logits(zs, weight=0.7, labels=gt, dice_counts=cnt, accumulate=False)
        return loss.item(), cnt

    lb, cb = run(zb)
    lf, cf = run([z.float() for z in zb])
    assert abs(lb - lf) <= FP32_LOSS_TOL * math.log(K)
    assert abs(lb - 0.7 * _jsd_mean_f64(zb)) <= FP32_LOSS_TOL * math.log(K)
    if with_labels:
        assert torch.equal(cb, cf)
        for k in range(K):
            oc, bad = oracle.dice_counts(zb[k].float().cpu().numpy(), gt.cpu().numpy())
            assert bad == 0 and np.array_equal(cb[k].cpu().numpy(), oc), f"view {k}: Dice counts differ from the oracle"


def _kl_cases():
    out = [(C, size, mode, 3.0) for C in KL_C for size, mode in (("tail", "fwd"), ("tail", "gmap"), ("many", "gmap"),
                                                                  ("tail", "reduce"))]
    return out + [(4, "tail", "gmap", 40.0), (19, "tail", "gmap", 40.0), (19, "tail", "reduce", 40.0)]


@pytest.mark.parametrize("C,size,mode,amp", _kl_cases())
def test_kl_div_with_logit_bf16_tiles(C, size, mode, amp, dct, dev):
    """mode 'fwd': the map alone; 'gmap': backward with a per-pixel upstream map; 'reduce': KL_Divergence_2D_Logit
    (reduce=True) scaled by 0.3, the upstream applied inside the backward launch (gscalar)."""
    B, HW = 2, _hw(2 * C, 0 if mode == "fwd" else 2, size)
    H, W = HW // 8, 8
    qb, pb = _logits(2, C, B, H, W, dev, 300 + C, amp)
    g = torch.Generator(device=dev).manual_seed(33)
    up = torch.rand(B, H, W, generator=g, device=dev)
    m64 = _kl_logit_map64(qb.double(), pb.double())
    if mode == "fwd":
        with torch.no_grad():
            mb = dct.kl_div_with_logit(qb, pb)
            mf = dct.kl_div_with_logit(qb.float(), pb.float())
        _check_map(mb, mf, "map")
        assert float((mb.double() - m64).abs().max()) <= 2e-5 * max(1.0, float(m64.abs().max()))
        return

    def run(q, p):
        qr, pr = q.detach().clone().requires_grad_(), p.detach().clone().requires_grad_()
        if mode == "gmap":
            out = dct.kl_div_with_logit(qr, pr)
            (out * up).sum().backward()
        else:
            out = dct.KL_Divergence_2D_Logit(reduce=True)(pr, qr)
            (out * 0.3).backward()
        return out.detach(), qr.grad, pr.grad

    ob, gqb, gpb = run(qb, pb)
    of, gqf, gpf = run(qb.float(), pb.float())
    if mode == "gmap":
        _check_map(ob, of, "map")
        assert float((ob.double() - m64).abs().max()) <= 2e-5 * max(1.0, float(m64.abs().max()))
        _, (gq64, gp64) = _grad64(lambda q, p: (_kl_logit_map64(q, p) * up.double()).sum(), (qb, pb))
    else:
        assert abs(ob.item() - of.item()) <= FP32_LOSS_TOL * max(1.0, abs(of.item()))
        assert abs(ob.item() - float(m64.mean())) <= 2e-5 * max(1.0, abs(float(m64.mean())))
        _, (gq64, gp64) = _grad64(lambda q, p: 0.3 * _kl_logit_map64(q, p).mean(), (qb, pb))
    _check_grad(gqb, gqf, gq64, "q_logit")
    _check_grad(gpb, gpf, gp64, "p_logit")


@pytest.mark.parametrize("C,size,amp", [(C, s, 3.0) for C in KL_C for s in ("tail", "many")] + [(19, "tail", 40.0)])
def test_kl_consistency_from_logits_bf16_tiles(C, size, amp, dct, dev):
    B, HW = 2, _hw(2 * C, 1, size)
    H, W = HW // 8, 8
    (ab,) = _logits(1, C, B, H, W, dev, 400 + C, amp)
    real = _simplex(C, B, H, W, dev, 34)

    def run(a, y):
        ar = a.detach().clone().requires_grad_()
        loss = dct.kl_consistency_from_logits(ar, y, weight=1.3)
        loss.backward()
        return loss.item(), ar.grad

    lb, gb = run(ab, real)
    lf, gf = run(ab.float(), real.float())
    l64, (g64,) = _grad64(lambda a: _klc64(a, real.double(), 1.3), (ab,))
    assert abs(lb - lf) <= FP32_LOSS_TOL * max(1.0, abs(lf))
    assert abs(lb - float(l64)) <= 2e-5 * max(1.0, abs(float(l64)))
    _check_grad(gb, gf, g64, "adv_logit")


def _ce_cases():
    out = []
    for C in KL_C:
        for v in ("mean", "mean_w", "sum") + (("dice",) if C <= 4 else ()):
            out.append((C, v, "tail", 3.0))
        out.append((C, "mean", "many", 3.0))
    return out + [(19, "mean_w", "tail", 40.0), (4, "dice", "tail", 40.0)]


@pytest.mark.parametrize("C,variant,size,amp", _ce_cases())
def test_supervised_bf16_tiles(C, variant, size, amp, dct, dev, oracle):
    """supervised_from_logits (mean; class weights; Dice counts) and CrossEntropyLoss2d(size_average=False) (sum).
    Every variant but the Dice one ignores a grid of pixels (label 255); their gradient must be exactly 0."""
    B, HW = 2, _hw(C, 1, size)
    H, W = HW // 8, 8
    (zb,) = _logits(1, C, B, H, W, dev, 500 + C, amp)
    g = torch.Generator(device=dev).manual_seed(35)
    gt = torch.randint(0, C, (B, 1, H, W), generator=g, device=dev)
    if variant != "dice":   # the fused meter flags every label outside [0, C)
        gt[:, :, ::5, ::3] = 255
    w = 0.5 + torch.rand(C, generator=g, device=dev) if variant == "mean_w" else None
    red = "sum" if variant == "sum" else "mean"

    def run(z):
        zr = z.detach().clone().requires_grad_()
        cnt = torch.zeros(B, C, 3, dtype=torch.int64, device=dev) if variant == "dice" else None
        if variant == "sum":
            loss = dct.CrossEntropyLoss2d(size_average=False)(zr, gt.squeeze(1))
        else:
            loss = dct.supervised_from_logits(zr, gt, weight=w, dice_counts=cnt)
        loss.backward()
        return loss.item(), zr.grad, cnt

    lb, gb, cb = run(zb)
    lf, gf, cf = run(zb.float())
    l64, (g64,) = _grad64(lambda z: _ce64(z, gt, w, red), (zb,))
    assert abs(lb - lf) <= FP32_LOSS_TOL * max(1.0, abs(lf))
    assert abs(lb - float(l64)) <= 2e-5 * max(1.0, abs(float(l64)))
    _check_grad(gb, gf, g64, "logits")
    ign = (gt == 255).expand(B, C, H, W)
    if variant != "dice":
        assert bool(ign.any()) and bool((gb[ign] == 0).all()), "an ignored pixel has a non-zero gradient"
    else:
        assert torch.equal(cb, cf)
        oc, bad = oracle.dice_counts(zb.float().cpu().numpy(), gt.cpu().numpy())
        assert bad == 0 and np.array_equal(cb.cpu().numpy(), oc)


# ------------------------------------------------------------------------------------------------
# promoted shapes: the fp32 kernels followed by the cast (check C)
# ------------------------------------------------------------------------------------------------
def _leaves(vals, offset):
    """Leaf tensors holding `vals` and the (input, gradient getter) pairs the op sees: with offset, each input is a
    view at storage offset 1 element (2 bytes for bf16: never 16-byte aligned)."""
    out = []
    for v in vals:
        if offset:
            buf = torch.zeros(v.numel() + 1, dtype=v.dtype, device=v.device)
            buf[1:].copy_(v.flatten())
            buf.requires_grad_()
            x = buf[1:].view(v.shape)
            assert x.data_ptr() % 16 != 0
            out.append((x, lambda b=buf, s=v.shape: b.grad[1:].view(s)))
        else:
            leaf = v.detach().clone().requires_grad_()
            out.append((leaf, lambda l=leaf: l.grad))
    return out


def _op_loss(op, dct, xs, aux, s=1.0):
    """One of the fused ops on the inputs xs (bf16 or float32), scaled by s, as a scalar to differentiate."""
    gt, up, y, w = aux["gt"], aux["up"], aux["y"], aux["w"]
    if op == "jsd":
        return dct.jsd_consistency_from_logits(xs, weight=0.7) * s
    if op == "kl":
        return (dct.kl_div_with_logit(xs[0], xs[1]) * up).sum() * s
    if op == "klc":
        return dct.kl_consistency_from_logits(xs[0], y.to(xs[0].dtype), weight=1.3) * s
    if op == "ce_mean":
        return dct.supervised_from_logits(xs[0], gt, weight=w) * s
    if op == "ce_sum":
        return dct.CrossEntropyLoss2d(size_average=False)(xs[0], gt.squeeze(1)) * s
    if op == "ce_conf":
        conf = torch.zeros(xs[0].shape[1], xs[0].shape[1], dtype=torch.int64, device=xs[0].device)
        return dct.supervised_from_logits(xs[0], gt, confusion=conf) * s
    if op == "ce_none":
        return (dct.CrossEntropyLoss2d(reduce=False)(xs[0], gt.squeeze(1)) * up).sum() * s
    raise AssertionError(op)


def _op_loss64(op, xs, aux, s=1.0):
    gt, up, y, w = aux["gt"], aux["up"], aux["y"], aux["w"]
    if op == "jsd":
        return _jsd64(xs, 0.7) * s
    if op == "kl":
        return (_kl_logit_map64(xs[0], xs[1]) * up.double()).sum() * s
    if op == "klc":
        return _klc64(xs[0], y.double(), 1.3) * s
    if op in ("ce_mean", "ce_conf"):
        return _ce64(xs[0], gt, w, "mean") * s
    if op == "ce_sum":
        return _ce64(xs[0], gt, None, "sum") * s
    if op == "ce_none":
        return (_ce64(xs[0], gt, None, "none") * up.double()).sum() * s
    raise AssertionError(op)


def _op_inputs(op, K, C, B, H, W, dev, seed):
    n_in = K if op == "jsd" else (2 if op == "kl" else 1)
    vals = _logits(n_in, C, B, H, W, dev, seed)
    g = torch.Generator(device=dev).manual_seed(seed + 1)
    gt = torch.randint(0, C, (B, 1, H, W), generator=g, device=dev)
    gt[:, :, ::5, ::3] = 255
    aux = {"gt": gt, "up": torch.rand(B, H, W, generator=g, device=dev), "y": _simplex(C, B, H, W, dev, seed + 2),
           "w": 0.5 + torch.rand(C, generator=g, device=dev) if op == "ce_mean" else None}
    return vals, aux


def _op_grads(op, dct, vals, aux, s=1.0, offset=False):
    lv = _leaves(vals, offset)
    _op_loss(op, dct, [x for x, _ in lv], aux, s).backward()
    return [get() for _, get in lv]


PROMO = [("jsd", 5, 4, 8, "plain"), ("jsd", 8, 2, 8, "plain"), ("jsd", 2, 5, 8, "plain"), ("jsd", 2, 64, 8, "plain"),
         ("jsd", 2, 4, 4, "plain"), ("jsd", 2, 19, 8, "offset"),
         ("kl", 2, 5, 8, "plain"), ("kl", 2, 4, 4, "plain"), ("kl", 2, 19, 8, "offset"),
         ("klc", 1, 5, 8, "plain"), ("klc", 1, 4, 4, "plain"), ("klc", 1, 4, 8, "offset"),
         ("ce_mean", 1, 5, 8, "plain"), ("ce_mean", 1, 19, 4, "plain"), ("ce_mean", 1, 4, 8, "offset"),
         ("ce_conf", 1, 4, 8, "plain"), ("ce_none", 1, 19, 8, "plain")]


@pytest.mark.parametrize("op,K,C,hw_mod,layout", PROMO)
def test_promoted_shapes_bf16(op, K, C, hw_mod, layout, dct, dev):
    """Shapes the bf16 tile pipeline does not take (K >= 5, C outside {2, 3, 4, 19}, K*C > 80, HW % 8 == 4, a view at
    an odd storage offset) and the CE calls that always run in fp32 (confusion counts, reduction 'none')."""
    B, H = 2, 33
    W = 8 if hw_mod == 8 else 4          # HW = 264 (% 8 == 0) or 132 (% 8 == 4, % 4 == 0)
    vals, aux = _op_inputs(op, K, C, B, H, W, dev, 600 + C)
    gb = _op_grads(op, dct, vals, aux, offset=layout == "offset")
    gf = _op_grads(op, dct, [v.float() for v in vals], aux)
    _, g64 = _grad64(lambda *x: _op_loss64(op, x, aux), vals)
    for k in range(len(vals)):
        _check_grad(gb[k], gf[k], g64[k], f"{op} input {k}", promoted=True)


# ------------------------------------------------------------------------------------------------
# a non-unit upstream: one fp32 multiply of the stored bf16 gradient, one rounding
# ------------------------------------------------------------------------------------------------
UP_SHAPES = {"jsd": (2, 3), "klc": (1, 4), "ce_mean": (1, 19), "ce_sum": (1, 4)}


@pytest.mark.parametrize("op", list(UP_SHAPES))
@pytest.mark.parametrize("s", [0.3, 1.0 / 3.0, 2.0, 1.0])
@pytest.mark.parametrize("layout", ["tile", "promoted"])
def test_nonunit_upstream_bf16(op, s, layout, dct, dev):
    """(loss * s).backward() against the same call at s = 1.  Tile shapes: the gradient is RNE_bf16(float(grad_at_1) * s)
    bit for bit and within bound (B) at two roundings; promoted shapes: RNE_bf16(fp32 gradient at 1 * s)."""
    K, C = UP_SHAPES[op]
    B, W = 2, 8 if layout == "tile" else 4
    H = 257                              # HW = 2056 (% 8 == 0) or 1028 (% 8 == 4)
    vals, aux = _op_inputs(op, K, C, B, H, W, dev, 700 + C)
    g1 = _op_grads(op, dct, vals, aux)
    gs = _op_grads(op, dct, vals, aux, s)
    gf1 = _op_grads(op, dct, [v.float() for v in vals], aux)
    gfs = _op_grads(op, dct, [v.float() for v in vals], aux, s)
    _, g64 = _grad64(lambda *x: _op_loss64(op, x, aux, s), vals)
    s_bf16 = torch.tensor(s, dtype=torch.float32, device=dev).to(BF)
    for k in range(len(vals)):
        what = f"{op} input {k}, s = {s:.6g}"
        if layout == "promoted":
            assert _bits_equal(gs[k], (gf1[k] * s).to(BF)), what
            _check_b(gs[k], gfs[k], g64[k], R1, what)
            continue
        want = (g1[k].float() * s).to(BF)
        assert _bits_equal(gs[k], want), f"{what}: not RNE_bf16(float(gradient at 1) * s)"
        _check_b(gs[k], gfs[k], g64[k], R2, what)
        if s not in (1.0, 2.0):
            # teeth: a bf16-rounded upstream times the bf16 gradient, rounded again, is caught on this data
            old = g1[k] * s_bf16
            assert not _bits_equal(old, want), f"{what}: the data cannot tell a bf16-rounded upstream apart"
            if s == 0.3:
                assert float(_excess(old, gfs[k], g64[k], R2).max()) > 0.0, f"{what}: (B) has no teeth on this data"


# ------------------------------------------------------------------------------------------------
# an upstream map at any 4-byte offset
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("C", [4, 19])
def test_kl_div_with_logit_bf16_unaligned_upstream_map(C, dct, dev):
    """Autograd may hand the backward a slice of a larger buffer as the upstream map (the gradient of a torch.cat of
    the map after a tensor whose size is not a multiple of 4): every 4-byte offset gives the aligned call's bits."""
    B, HW = 2, _hw(2 * C, 2, "tail")
    H, W = HW // 8, 8
    qb, pb = _logits(2, C, B, H, W, dev, 800 + C)
    g = torch.Generator(device=dev).manual_seed(36)
    up = torch.rand(B, H, W, generator=g, device=dev)

    def run(q, p, off):
        qr, pr = q.detach().clone().requires_grad_(), p.detach().clone().requires_grad_()
        m = dct.kl_div_with_logit(qr, pr)
        if off == "cat":
            x = torch.ones(5, device=dev, requires_grad=True)
            wts = torch.cat([torch.ones(5, device=dev), up.flatten()])
            (torch.cat([x, m.flatten()]) * wts).sum().backward()
        else:
            buf = torch.zeros(up.numel() + off, device=dev)
            gmap = buf[off:].view(up.shape)
            gmap.copy_(up)
            assert gmap.is_contiguous() and gmap.data_ptr() % 16 == 4 * off
            m.backward(gmap)
        return qr.grad, pr.grad

    ref = run(qb, pb, 0)
    for off in (1, 2, 3, "cat"):
        got = run(qb, pb, off)
        for a, b, what in zip(got, ref, ("q_logit", "p_logit")):
            assert _bits_equal(a, b), f"offset {off}: {what} gradient differs from the aligned call's"
    gf = run(qb.float(), pb.float(), 0)
    _, (gq64, gp64) = _grad64(lambda q, p: (_kl_logit_map64(q, p) * up.double()).sum(), (qb, pb))
    _check_grad(ref[0], gf[0], gq64, "q_logit")
    _check_grad(ref[1], gf[1], gp64, "p_logit")
