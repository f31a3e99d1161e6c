"""Edge tiles folded into the panel launch store exactly what the separate edge launch stores.

Dense formats of wide nets write the MIXED / GENERAL edge tiles (slivers, band corners, x_1 / x_K coupling) as work
items of the panel-ordered launch.  NNSDP_PANEL_FOLD=0 (read when a batch is created) keeps them in a launch of their
own.  Every test runs the same queries through one batch of each form and compares every ring slot after every pass
bit for bit.
"""
import os
import sys

import numpy as np
import pytest

import nnsdp_b200 as nb
from helpers import rand_net, rand_query, to_numeric_batch

pytestmark = pytest.mark.gpu

WIDE = [2, 300, 270, 280, 2]
RADII = (0.0, 0.6, 0.001, 0.6, 0.0, 0.6, 0.002, 0.6)   # small radii: Gram-active layers; large: none


def _batch(dnet, beta, fold, **kw):
    old = os.environ.get("NNSDP_PANEL_FOLD")
    os.environ["NNSDP_PANEL_FOLD"] = "1" if fold else "0"
    try:
        return nb.Batch(dnet, beta, **kw)
    finally:
        if old is None:
            del os.environ["NNSDP_PANEL_FOLD"]
        else:
            os.environ["NNSDP_PANEL_FOLD"] = old


def _ring_bits(b, nslots):
    """The first nslots ring slots on the device, as int64 (bit patterns)."""
    torch = pytest.importorskip("torch")
    ptr, per = b.ring_ptr()

    class _Dev:
        __cuda_array_interface__ = {"shape": (nslots * per,), "typestr": "<i8", "data": (ptr, False), "strides": None,
                                    "version": 2}

    b.sync()
    return torch.as_tensor(_Dev(), device="cuda")


def _same_passes(a, b, passes):
    import torch

    for q0, nq in passes:
        for x in (a, b):
            x.emit(q0, nq)
        ra, rb = _ring_bits(a, nq), _ring_bits(b, nq)
        torch.cuda.synchronize()
        assert torch.equal(ra, rb), (q0, nq, int((ra != rb).sum()))


def _pair(net, dnet, beta, qs, ring, **kw):
    out = []
    for fold in (True, False):
        b = _batch(dnet, beta, fold, Qcap=len(qs), ring=ring, **kw)
        b.set_inputs(to_numeric_batch(nb, net, qs))
        b.bounds()
        b.prepare()
        out.append(b)
    return out


@pytest.fixture(scope="module")
def wide(ctx):
    net = rand_net(WIDE, seed=41, sigma=0.12)
    dnet = nb.Net(ctx, net.xdims, net.Ms)
    yield net, dnet
    dnet.close()


def test_the_folded_form_has_no_edge_launch(wide):
    net, dnet = wide
    rng = np.random.default_rng(1)
    qs = [rand_query(net, 2, rng, radius=r) for r in RADII]
    a, b = _pair(net, dnet, 2, qs, ring=8)
    for x in (a, b):
        x.stage_reset()
        x.emit(0, 8)
        x.sync()
    # the separate form has one launch more, the edge kernel; the band launch is left in the edge span of both
    assert a.stage_ms("emit")[1] == b.stage_ms("emit")[1] - 1
    assert a.stage_ms("emit_edge")[1] == 1 and b.stage_ms("emit_edge")[1] == 2
    assert a.emitted_bytes() == b.emitted_bytes()
    a.close()
    b.close()


@pytest.mark.parametrize("beta", [1, 2, 4])
@pytest.mark.parametrize("kind", ["safety", "hplaneS"])
def test_slots_after_every_pass_equal_the_separate_launches(wide, beta, kind):
    """Ring of 3 slots, Gram activity alternating per query (a slot sees active -> inactive -> active for the same
    block); output QCs with (safety) and without (hplaneS) an S22 part."""
    net, dnet = wide
    rng = np.random.default_rng(3 + beta)
    qs = [rand_query(net, beta, rng, kind=kind, radius=r) for r in RADII]
    a, b = _pair(net, dnet, beta, qs, ring=3)
    ncon, _ = a.gram_stats()
    assert 0 < ncon < len(qs) * (len(net.xdims) - 2)
    _same_passes(a, b, [(0, 3), (3, 3), (6, 2), (5, 3), (1, 1), (2, 3), (7, 1), (0, 2), (4, 3)])
    a.close()
    b.close()


def test_run_into_ring_halves_and_ring_reset(wide):
    """nnsdp_batch_run with a host buffer (the ring as two halves), then nnsdp_batch_ring_reset and a pass."""
    net, dnet = wide
    rng = np.random.default_rng(7)
    qs = [rand_query(net, 2, rng, radius=r) for r in RADII]
    outs = []
    for fold in (True, False):
        b = _batch(dnet, 2, fold, Qcap=len(qs), ring=4)
        out = np.full((len(qs), b.per_query), np.nan)
        for order, flags in ((np.arange(8), nb.RUN_DENSE_COPY), (np.roll(np.arange(8), 3), 0)):
            b.set_inputs(to_numeric_batch(nb, net, [qs[i] for i in order]))
            b.run(out, flags=flags)
            outs.append(out.copy())
        b.ring_reset()
        b.emit(0, 4)
        outs.append(_ring_bits(b, 4).cpu().numpy())
        b.close()
    for x, y in zip(outs[:3], outs[3:]):
        assert np.array_equal(x.view(np.int64), y.view(np.int64))


def test_stress_shape_ring_32(ctx):
    """W1000-D20, beta = 2 (the bench.py stress workload), 96 queries through 32 ring slots, two sweeps."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    if root not in sys.path:
        sys.path.insert(0, root)
    import bench

    name = bench.DEFAULT_WORKLOAD
    xdims, Ms, beta, inp = bench.make_workload(name, 0, Q=96)
    dnet = nb.Net(ctx, xdims, Ms)
    bs = []
    for fold in (True, False):
        b = _batch(dnet, beta, fold, Qcap=96, ring=32)
        b.set_inputs(bench.numeric_batch(nb, name, inp), Q=96)
        b.bounds()
        b.prepare()
        bs.append(b)
    _same_passes(bs[0], bs[1], [(0, 32), (32, 32), (64, 32), (0, 32), (40, 32)])
    for b in bs:
        b.close()
    dnet.close()
