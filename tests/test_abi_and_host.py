"""CPU: the C-ABI library loads and exports every symbol include/dct_b200.h declares, the ctypes
table matches the header, host-side logic (alias import, check modes, install rebinding)."""
import ctypes
import os
import re

import numpy as np
import pytest
import ref_shim
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
# the original project's source tree is not part of this repository: oracle/ref_shim.py finds it through
# $DCT_REFERENCE_ROOT or a copy staged into baseline/_ref (tools/stage_reference.sh)
needs_reference = pytest.mark.skipif(not ref_shim.reference_available(),
                                     reason="original project's source tree not found ($DCT_REFERENCE_ROOT or baseline/_ref)")


def _header_symbols():
    txt = open(os.path.join(ROOT, "include", "dct_b200.h")).read()
    return sorted(set(re.findall(r"DCT_API\s+[\w\s\*]+?\b(dct_\w+)\s*\(", txt)))


def test_header_symbols_are_exported_and_bound():
    import dct_b200
    names = _header_symbols()
    assert len(names) >= 24
    h = ctypes.CDLL(dct_b200.library_path())
    for n in names:
        assert hasattr(h, n), f"{n} declared in include/dct_b200.h but not exported"
    assert sorted(dct_b200._lib.EXPORTED_SYMBOLS) == names  # ctypes table covers the whole header, nothing else


def test_header_prototype_arity_matches_ctypes_table():
    import dct_b200
    txt = open(os.path.join(ROOT, "include", "dct_b200.h")).read()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    for name, argtypes in dct_b200._lib._SIGNATURES.items():
        m = re.search(r"\b" + name + r"\s*\((.*?)\)\s*;", txt, flags=re.S)
        assert m, name
        params = m.group(1).strip()
        n = 0 if params in ("", "void") else len(params.split(","))
        assert n == len(argtypes), f"{name}: header has {n} params, ctypes table {len(argtypes)}"


def test_library_basics_without_gpu():
    import dct_b200
    h = dct_b200._lib.lib()
    assert h.dct_abi_version() == 2
    assert h.dct_workspace_bytes() >= 8 * 8192
    assert h.dct_error_string(0) == b"ok"
    assert b"unsupported" in h.dct_error_string(-2)
    if not torch.cuda.is_available():
        assert h.dct_device_check(0) == -5
    # argument errors are detected before anything touches the device: publication variants without a descriptor
    assert h.dct_jsd_fwdbwd_pub_f32(None, 2, 4, 1, 64, 1, 1.0, None, None, None, None, None, 0, None, None, None, None) == -1
    assert h.dct_exchange_publish(None, None) == -1
    assert h.dct_dev_tile_image(0, 0) == -1


def test_tile_schedule_division_is_exact():
    """The tile pipeline never divides on the device: the producer lane derives a tile's image index through a multiply-shift
    (csrc/dct_tile.cuh tile_set_geometry / tile_image).  Host-side check of that exact code against integer division: every
    divisor up to 4096 plus large and power-of-two-adjacent ones, tiles at the edges of every image boundary and of int32."""
    import dct_b200
    f = dct_b200._lib.lib().dct_dev_tile_image
    divisors = list(range(1, 4097)) + [4097, 65535, 65536, 65537, 1 << 20, (1 << 20) + 1, 3 ** 12, (1 << 24) - 1, 1 << 24,
                                       (1 << 30) - 1, 1 << 30, (1 << 31) - 1]
    rng = np.random.default_rng(7)
    top = (1 << 31) - 1
    for d in divisors:
        tiles = {0, 1, d - 1, d, d + 1, 2 * d - 1, 2 * d, 7 * d - 1, 7 * d, top, top - 1, top // d * d, max(top // d * d - 1, 0)}
        tiles |= {int(t) for t in rng.integers(0, top, size=6)}
        for t in tiles:
            if 0 <= t <= top:
                assert f(d, t) == t // d, (d, t)
    assert f(0, 1) < 0 and f(4, -1) < 0


def test_exchange_descriptor_layout_matches_header():
    """dct_peer_pub (include/dct_b200.h) is built word by word in distributed.PeerExchange._descriptor."""
    import dct_b200
    L = dct_b200._lib
    txt = open(os.path.join(ROOT, "include", "dct_b200.h")).read()
    defs = {k: int(v) for k, v in re.findall(r"#define\s+(DCT_\w+)\s+(\d+)\s*$", txt, flags=re.M)}
    assert (defs["DCT_MAX_PEERS"], defs["DCT_PUB_ROW_WORDS"], defs["DCT_PUB_MAX_VALUES"], defs["DCT_IPC_HANDLE_BYTES"]) == \
        (L.MAX_PEERS, L.PUB_ROW_WORDS, L.PUB_MAX_VALUES, L.IPC_HANDLE_BYTES)
    assert L.lib().dct_peer_pub_bytes() == ctypes.sizeof(L.PeerPub) == 40   # 3 pointers + 4 int32
    assert 2 * L.PUB_MAX_VALUES <= L.PUB_ROW_WORDS                 # two tagged words per published double


def test_alias_import_shares_modules():
    import dct_b200
    import dct_b200.loss as L
    from dct_b200.metrics import DiceMeter
    assert L.JSD_2D is dct_b200.JSD_2D and DiceMeter is dct_b200.DiceMeter
    assert dct_b200.get_loss_fn("jsd").__class__ is dct_b200.JSD_2D
    with pytest.raises(ValueError):
        dct_b200.get_loss_fn("nope")


def test_no_cpu_fallback():
    import dct_b200
    p = torch.softmax(torch.randn(1, 3, 4, 4), 1)
    for call in (lambda: dct_b200.JSD_2D()([p, p]),
                 lambda: dct_b200.KL_Divergence_2D()(p, p),
                 lambda: dct_b200.Entropy_2D()(p),
                 lambda: dct_b200.jsd_consistency_from_logits([p, p]),
                 lambda: dct_b200.DiceMeter(C=3).add(p, torch.zeros(1, 1, 4, 4, dtype=torch.long)),
                 lambda: dct_b200.IoU(3).add(p, torch.zeros(1, 1, 4, 4, dtype=torch.long)),
                 lambda: dct_b200.l2_normalize(torch.randn(2, 1, 4, 4))):
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            call()


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "deep-co-training-for-semi-supervised-image-segmentation_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert "import oracle" not in src and "dct_oracle" not in src and "libdct_oracle" not in src, f


def test_check_mode_switch():
    import dct_b200
    old = dct_b200.set_check_mode("deferred")
    assert dct_b200.get_check_mode() == "deferred"
    dct_b200.set_check_mode(old)
    with pytest.raises(ValueError):
        dct_b200.set_check_mode("sometimes")


def test_meter_host_logic_matches_reference_structures():
    import dct_b200
    m = dct_b200.DiceMeter(method="2d", C=4, report_axises=[1, 2, 3])
    (rm, rs), (ms, ss) = m.value()           # empty log fallback, dice_meter.py:68-71
    assert ms.shape == (4,) and float(ms.sum()) == 0.0
    m.diceLog.append(torch.tensor([[1.0, 0.5, 0.25, 0.75], [1.0, 0.0, 0.5, 0.25]]))   # the public list, behind add()'s back
    (rm, rs), (ms, ss) = m.value()
    assert torch.allclose(ms, torch.tensor([1.0, 0.25, 0.375, 0.5]))
    assert abs(rm.item() - (0.5 + 0.25) / 2) < 1e-7
    assert m.value()[1][0] is ms                                   # unchanged log: the kept result
    m.diceLog.append(torch.tensor([[0.0, 0.0, 0.0, 0.0]]))
    assert torch.allclose(m.value()[1][0], torch.tensor([2.0, 0.5, 0.75, 1.0]) / 3)   # changed log: recomputed
    m.reset()
    assert float(m.value()[1][0].sum()) == 0.0 and m.value()[1][0].shape == (4,)
    iou = dct_b200.IoU(3)
    iou.conf_metric._host[:] = np.array([[5, 1, 0], [2, 3, 0], [0, 0, 0]])
    v = iou.value()
    assert v["Overall_Acc"] == 8 / 11 and np.isnan(v["Class_IoU"][2].item())
    assert v["Validated_Mean_IoU"] == np.mean([5 / 8, 3 / 6])


@needs_reference
def test_install_rebinds_reference_call_sites():
    import ref_shim
    ref_shim.install()
    import generalframework.loss as gl
    import generalframework.trainer.cotraining_totalloss as ct
    import dct_b200
    orig = gl.LOSS["jsd"]
    n = dct_b200.install()
    try:
        assert n > 0
        assert gl.get_loss_fn("jsd").__class__ is dct_b200.JSD_2D          # registry path, loss/__init__.py:12-16
        assert ct.KL_Divergence_2D is dct_b200.KL_Divergence_2D            # trainer global, cotraining_totalloss.py:13
        assert ct.DiceMeter is dct_b200.DiceMeter and ct.FSGMGenerator is dct_b200.FSGMGenerator
        # functional Dice of the supervised baseline (trainer/trainer.py:171-175): rebound in trainer modules only
        import generalframework.trainer.trainer as tr
        import generalframework.utils.utils as gu
        assert tr.dice_coef is dct_b200.utils.dice_coef and tr.probs2one_hot is dct_b200.utils.probs2one_hot
        assert gu.class2one_hot is not dct_b200.utils.class2one_hot       # dataset workers keep the host version
    finally:
        dct_b200.uninstall()
    assert gl.LOSS["jsd"] is orig and ct.DiceMeter is not dct_b200.DiceMeter


@needs_reference
def test_install_keeps_the_metrics2_flavour():
    """generalframework.metrics2.DiceMeter (user: trainer/mean_teacher_trainer.py:18) differs from metrics.DiceMeter on the
    host side (metrics2/dice_meter.py:43,82-84); install() must hand each module its own flavour and uninstall() must
    restore both (round-1 defect: both were replaced by the metrics/ flavour)."""
    import ref_shim
    ref_shim.install()
    import generalframework.metrics as gm
    import generalframework.metrics2 as gm2
    import generalframework.metrics2.dice_meter as gm2d
    import generalframework.trainer.mean_teacher_trainer as mt
    import dct_b200
    ref1, ref2, refk2 = gm.DiceMeter, gm2.DiceMeter, gm2.KappaMetrics
    assert ref1 is not ref2
    want1 = ref1(method="2d", C=4)
    want2 = ref2(method="2d", C=4)
    log = torch.tensor([[1.0, 0.5, 0.25, 0.75], [1.0, 0.0, 0.5, 0.25]])
    want1.diceLog.append(log); want2.diceLog.append(log)
    dct_b200.install()
    try:
        dct_b200.install()   # idempotent: a second call must not re-dispatch our own classes
        assert gm.DiceMeter is dct_b200.DiceMeter and gm2.DiceMeter is dct_b200.DiceMeter2
        assert gm2d.DiceMeter is dct_b200.DiceMeter2 and mt.DiceMeter is dct_b200.DiceMeter2
        assert gm2.KappaMetrics is dct_b200.KappaMetrics2 and gm.KappaMetrics is dct_b200.KappaMetrics
        a, b = gm.DiceMeter(method="2d", C=4), gm2.DiceMeter(method="2d", C=4)
        assert a.report_axis == want1.report_axis == "all" and b.report_axis == want2.report_axis == [0, 1, 2, 3]
        a.diceLog.append(log); b.diceLog.append(log)
        assert a.summary() == want1.summary() and set(a.summary()) == {"mDSC", "mVars"}
        assert b.summary() == want2.summary() and set(b.summary()) == {"DSC0", "DSC1", "DSC2", "DSC3"}
        assert b.detailed_summary() == want2.detailed_summary()
        c = gm2.DiceMeter(method="3d", C=4, report_axises=[1, 3])
        c.diceLog.append(log)
        w = ref2(method="3d", C=4, report_axises=[1, 3]); w.diceLog.append(log)
        assert c.summary() == w.summary() and set(c.summary()) == {"DSC1", "DSC3"}
        (rm, rs), _ = c.value(); (wm, ws), _ = w.value()
        assert rm.item() == wm.item() and rs.item() == ws.item()
    finally:
        dct_b200.uninstall()
    assert gm.DiceMeter is ref1 and gm2.DiceMeter is ref2 and gm2.KappaMetrics is refk2 and mt.DiceMeter is ref2
