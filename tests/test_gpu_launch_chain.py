"""GPU: consecutive tile-pipeline launches on ONE workspace, chained by programmatic dependent launch in one CUDA graph.

Every launch's last CTA re-arms the workspace header (ticket, pool counter, Dice-clear flag, sum accumulators) for the
next launch, which reads it once its griddepcontrol.wait has returned.  Each launch of the chain must give the bits the
same launch gives alone on a fresh workspace, on every replay.  The shape draws tiles from the dynamic pool and clears
its own Dice counters, so every part of the header is used by every launch.
"""
import pytest
import torch

from test_gpu_jsd_vat_kl import DEV, OK, Case, assert_same, fused, h, workspace  # noqa: F401  (h: the fixture)

pytestmark = pytest.mark.gpu


def test_graph_of_consecutive_launches_on_one_workspace(h):  # noqa: F811
    cases = [Case(3, 4, 16, 256, 256, seed=s) for s in (5, 6)]   # c2's per-pixel shape at half its batch
    want = []
    for c in cases:
        o = c.outputs()
        assert fused(h, c, o, workspace(h)) == OK
        want.append(o)
    torch.cuda.synchronize()
    ws = workspace(h)
    outs = [cases[i % 2].outputs() for i in range(8)]
    side = torch.cuda.Stream(device=DEV)
    side.wait_stream(torch.cuda.current_stream(DEV))
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=side):
        for i, o in enumerate(outs):
            assert fused(h, cases[i % 2], o, ws) == OK
    for _ in range(2):
        for o in outs:   # what a launch that wrote nothing would leave
            for t in o["grads"] + [o["gy"]]:
                t.fill_(float("nan"))
            o["sums"].zero_()
            o["counts"].fill_(-7)
        g.replay()
        torch.cuda.synchronize()
        for i, o in enumerate(outs):
            assert_same(o, want[i % 2], True)
        assert not torch.any(ws[:64]), "the workspace header was not re-armed"
