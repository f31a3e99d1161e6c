"""Ring slots that are reused keep exactly the dense output of their current query.

The emitter zeroes a ring slot once and afterwards stores only the entries that can differ from what the slot holds:
structural zeros are never stored again, and the diagonal block of a layer only while the slot's current or previous
query has a non-zero bulk there (Gram of a stably-active neuron, W_K' S22 W_K).  Every test compares ring slots, bit
for bit, with the same query emitted into a fresh batch; each one fails when the library's record of what a slot holds
is wrong.
"""
import numpy as np
import pytest

import nnsdp_b200 as nb
from helpers import rand_net, rand_query, to_numeric_batch

pytestmark = pytest.mark.gpu

BETA = 2
WIDE = [2, 300, 270, 280, 2]        # hidden layers >= 256: panel launch, band kernel after bulk-only strips
NARROW = [2, 20, 24, 20, 20, 2]     # band added inside the DIAG strips (band_inline)
RADII = (0.0, 0.6, 0.001, 0.6, 0.0, 0.6, 0.002, 0.6)   # tiny: Gram-active layers; wide: none


@pytest.fixture(scope="module", params=["wide", "narrow"])
def model(request, ctx):
    xdims = WIDE if request.param == "wide" else NARROW
    net = rand_net(xdims, seed=41, sigma=0.12 if request.param == "wide" else None)
    dnet = nb.Net(ctx, net.xdims, net.Ms)
    yield net, dnet
    dnet.close()


def _queries(net, kind, seed=3):
    rng = np.random.default_rng(seed)
    return [rand_query(net, BETA, rng, kind=kind, radius=r) for r in RADII]


def _fresh(net, dnet, dense, qs):
    """Each query alone in a new batch of one slot."""
    out = []
    for q in qs:
        b = nb.Batch(dnet, BETA, Qcap=1, ring=1, dense=dense)
        b.set_inputs(to_numeric_batch(nb, net, [q]), Q=1)
        b.run(None)
        out.append(b.get_slot(0))
        b.close()
    return out


def _emit_and_check(b, ref, passes):
    for q0, nq in passes:
        b.emit(q0, nq)
        b.sync()
        for i in range(nq):
            assert np.array_equal(b.get_slot(i), ref[q0 + i]), (q0, nq, i)


@pytest.mark.parametrize("fmt", ["blocks", "dense_z"])
def test_slots_after_every_pass_equal_fresh_batches(model, fmt):
    """Ring of 3 slots, 8 queries alternating Gram-active and inactive: a slot sees active -> inactive -> active for
    the same block; passes with any q0 and nq (nnsdp_batch_emit always starts at slot 0)."""
    net, dnet = model
    dense = fmt == "dense_z"
    qs = _queries(net, "safety")
    ref = _fresh(net, dnet, dense, qs)
    b = nb.Batch(dnet, BETA, Qcap=len(qs), ring=3, dense=dense)
    b.set_inputs(to_numeric_batch(nb, net, qs))
    b.bounds()
    b.prepare()
    ncon, _ = b.gram_stats()
    assert 0 < ncon < len(qs) * (len(net.xdims) - 2)   # some (query, layer) pairs are Gram-active, not all
    _emit_and_check(b, ref, [(0, 3), (3, 3), (6, 2), (5, 3), (1, 1), (2, 3), (7, 1), (0, 2), (4, 3)])
    b.close()


def test_output_qc_switching_its_s22_part(model):
    """set_inputs on the same batch: an output QC with an S22 part (x_K block non-zero), then one without, then back."""
    net, dnet = model
    with_s22 = _queries(net, "safety", seed=5)[:4]
    without = _queries(net, "hplaneS", seed=6)[:4]
    b = nb.Batch(dnet, BETA, Qcap=4, ring=4)
    for qs in (with_s22, without, with_s22, without):
        ref = _fresh(net, dnet, False, qs)
        b.set_inputs(to_numeric_batch(nb, net, qs))
        b.bounds()
        b.prepare()
        _emit_and_check(b, ref, [(0, 4)])
    b.close()


def test_run_into_host_buffer_twice(model):
    """nnsdp_batch_run with a host buffer uses the ring as two halves; two runs with the queries in a different order,
    copied verbatim (NNSDP_RUN_DENSE_COPY) and through the sparse gather."""
    net, dnet = model
    qs = _queries(net, "safety", seed=7)
    ref = np.stack(_fresh(net, dnet, False, qs))
    b = nb.Batch(dnet, BETA, Qcap=len(qs), ring=4)
    out = np.full((len(qs), b.per_query), np.nan)
    for order, flags in ((np.arange(8), nb.RUN_DENSE_COPY), (np.arange(8)[::-1], nb.RUN_DENSE_COPY),
                         (np.roll(np.arange(8), 3), 0)):
        b.set_inputs(to_numeric_batch(nb, net, [qs[i] for i in order]))
        b.run(out, flags=flags)
        assert np.array_equal(out, ref[order])
    b.close()


def test_ring_reset_after_writing_into_the_ring(model):
    """Garbage written into the ring through its device pointer, then nnsdp_batch_ring_reset: the next pass gives the
    complete output again."""
    torch = pytest.importorskip("torch")
    net, dnet = model
    qs = _queries(net, "safety", seed=9)[:4]
    ref = _fresh(net, dnet, False, qs)
    b = nb.Batch(dnet, BETA, Qcap=4, ring=4)
    b.set_inputs(to_numeric_batch(nb, net, qs))
    b.bounds()
    b.prepare()
    _emit_and_check(b, ref, [(0, 4)])
    ptr, per = b.ring_ptr()

    class _Dev:
        __cuda_array_interface__ = {"shape": (4 * per,), "typestr": "<f8", "data": (ptr, False), "strides": None,
                                    "version": 2}

    b.sync()
    torch.as_tensor(_Dev(), device="cuda").fill_(12345.0)
    torch.cuda.synchronize()
    b.ring_reset()
    _emit_and_check(b, ref, [(0, 4)])
    b.close()


def test_emitted_bytes_count_what_a_pass_stores(model):
    """Dense formats: the bytes the last run stored hold no structural zero."""
    net, dnet = model
    qs = _queries(net, "safety", seed=11)
    b = nb.Batch(dnet, BETA, Qcap=len(qs), ring=8)
    b.set_inputs(to_numeric_batch(nb, net, qs))
    b.run(None)
    full = len(qs) * b.per_query * 8
    stored = b.emitted_bytes()
    st = nb.plan_stats(net.xdims, BETA)
    assert 0 < stored <= full - 8 * len(qs) * st["entries"]["ZERO"]
    b.close()

