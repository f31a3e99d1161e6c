#!/usr/bin/env python
"""Bytes the emitter stores per pass of a bench workload (default: the stress batch, dense clique blocks), checked
against the count the ring-slot rules predict, with the emitter time and the achieved write bandwidth.

A slot is zeroed when it is first used; after that a pass stores, for every query, all launched strips and tiles except
the structurally zero ones, plus the SAME / DIAG strips of block Br when the query or the slot's previous query has a
non-zero bulk there (a stably-active neuron in layer Br + 1, or the S22 part of the output QC for Br = K - 1).  The
prediction below rebuilds those sets from nnsdp_plan_tiles and the bounds of the batch, independently of the library's
own bookkeeping, and must equal what nnsdp_batch_emit_stats reports for every pass.

  python tools/ring_bytes.py [--workload NAME] [--sweeps 2] [--summary-only]
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "nn-sdp_b200"))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402

import bench  # noqa: E402
import nnsdp_b200 as nb  # noqa: E402

PROG = dict(ZERO=0, SAME=1, RC=2, CR=3, MIXED=4, GENERAL=5, DIAG=6, AFF=7)


def plan_counts(xdims, beta):
    """(entries every query of a pass stores, entries of the bulk strips per block), from the plan's tile list."""
    t = nb.plan_tiles(xdims, beta)
    F = {n: i for i, n in enumerate(nb.core.TILE_FIELDS)}
    K = len(xdims) - 1
    prog, rblk, cblk = t[:, F["prog"]], t[:, F["rblk"]], t[:, F["cblk"]]
    ent = t[:, F["nrows"]].astype(np.int64) * t[:, F["ncols"]]
    diag_like = ((prog == PROG["SAME"]) | (prog == PROG["DIAG"])) & (rblk >= 1) & (rblk == cblk)
    # the square range of every (matrix, block) the SAME / DIAG strips cover: band_inline when the widest is < 256
    boxes = {}
    for i in np.flatnonzero(diag_like):
        key = (int(t[i, F["mat"]]), int(rblk[i]))
        g0, c0 = int(t[i, F["grow0"]]), int(t[i, F["gcol0"]])
        lo, hi, band = boxes.get(key, (1 << 62, -1, False))
        boxes[key] = (min(lo, g0, c0), max(hi, g0 + int(t[i, F["nrows"]]) - 1, c0 + int(t[i, F["ncols"]]) - 1),
                      band or prog[i] == PROG["DIAG"])
    band_inline = not boxes or max(hi - lo + 1 for lo, hi, _ in boxes.values()) < 256
    bulk_sel = diag_like & ((prog == PROG["SAME"]) | (not band_inline))
    bulk = np.zeros(K, dtype=np.int64)
    np.add.at(bulk, rblk[bulk_sel], ent[bulk_sel])
    every = int(ent[(prog != PROG["ZERO"]) & ~bulk_sel].sum())
    if not band_inline:  # the band kernel re-writes the (2 beta + 1)-wide band of every DIAG range in place
        every += sum((hi - lo + 1) * (2 * beta + 1) - beta * (beta + 1) for lo, hi, band in boxes.values() if band)
    return every, bulk


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default=bench.DEFAULT_WORKLOAD, choices=sorted(bench.WORKLOADS))
    ap.add_argument("--sweeps", type=int, default=2, help="passes over all queries of the batch")
    ap.add_argument("--summary-only", action="store_true")
    args = ap.parse_args()
    w = bench.WORKLOADS[args.workload]
    xdims, Ms, beta, inp = bench.make_workload(args.workload, 0)
    Q, ring = w["Q"], min(w["ring"], w["Q"])
    K = len(xdims) - 1
    ctx = nb.Context([0])
    net = nb.Net(ctx, xdims, Ms)
    sz = net.sizes(beta)
    b = nb.Batch(net, beta, Qcap=Q, ring=ring)
    b.set_inputs(bench.numeric_batch(nb, args.workload, inp), Q=Q)
    b.bounds()
    b.prepare()
    # Gram-active (query, block): some neuron of layer blk + 1 has smin = smax = 1 (d11 != 0); no S22 part in the
    # output QCs of the bench workloads (checked below against the library's count)
    bnd = b.get_bounds()
    on = bnd["smin"] * bnd["smax"] != 0
    noff = np.concatenate([[0], np.cumsum(xdims[1:-1])])
    active = np.zeros((Q, K), dtype=bool)
    for blk in range(K - 1):
        active[:, blk] = on[:, noff[blk]:noff[blk + 1]].any(axis=1)
    ncon, _ = b.gram_stats()
    assert ncon == int(active[:, : K - 1].sum()), (ncon, int(active.sum()))
    S = inp.get("out_S")
    has_s22 = S is not None and np.any(S[:, xdims[0]:xdims[0] + xdims[-1], xdims[0]:xdims[0] + xdims[-1]] != 0)
    every, bulk = plan_counts(xdims, beta)
    peak, peak_src = bench.measured_peaks()
    held = np.zeros((ring, K), dtype=bool)
    rows = []
    for p in range(args.sweeps * (-(-Q // ring))):
        q0 = (p * ring) % (ring * (-(-Q // ring)))
        nq = min(ring, Q - q0)
        pred = every * nq
        for i in range(nq):
            for blk in range(1, K):
                now = bool(active[q0 + i, blk]) if blk <= K - 2 else bool(has_s22)
                if bulk[blk] and (now or held[i, blk]):
                    pred += int(bulk[blk])
                held[i, blk] = now
        e0 = b.emitted_bytes()
        b.stage_reset()
        b.emit(q0, nq)
        b.sync()
        got = b.emitted_bytes() - e0
        ms = b.stage_ms("emit")[0]
        row = {"pass": p, "q0": q0, "queries": nq, "stored_bytes": got, "predicted_bytes": 8 * pred,
               "dense_block_bytes": 8 * sz["sum_ck_sq"] * nq, "emitter_ms": ms, "achieved_gbs": got / (ms * 1e-3) / 1e9,
               "frac_of_peak": got / (ms * 1e-3) / 1e9 / peak}
        rows.append(row)
        if not args.summary_only:
            print(json.dumps(row), flush=True)
        assert got == 8 * pred, row
    steady = rows[-(-(-Q // ring)):]  # the last sweep: every slot reused
    ms = float(np.mean([r["emitter_ms"] for r in steady]))
    stored = float(np.mean([r["stored_bytes"] for r in steady]))
    print(json.dumps({"workload": args.workload, "ring_slots": ring, "queries": Q,
                      "env": {k: v for k, v in os.environ.items() if k.startswith("NNSDP_")},
                      "steady_state_pass": {"emitter_ms": ms, "stored_bytes": stored,
                                            "stored_per_query_mb": stored / ring / 1e6,
                                            "dense_block_bytes": 8.0 * sz["sum_ck_sq"] * ring,
                                            "achieved_gbs": stored / (ms * 1e-3) / 1e9, "peak_gbs": peak,
                                            "frac_of_peak": stored / (ms * 1e-3) / 1e9 / peak, "peak_source": peak_src},
                      "gram_active_pairs": int(active.sum()), "all_passes_match_prediction": True}), flush=True)
    b.close()
    net.close()


if __name__ == "__main__":
    main()
