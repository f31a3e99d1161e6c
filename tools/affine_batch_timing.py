"""Affine-coefficient hand-off of a whole reach polytope / vnnlib property: one nnsdp_affine_create per query plus the
scipy canonicalisation of its COO (what every consumer had to do), against one nnsdp_affine_create_batch plus
csc_matrix built from its arrays (no sort).  Bounds are CROWN bounds computed once with nnsdp_bounds_crown and passed as
the caller's bounds (with IBP the deep nets have no stably-active neuron at all).

Workloads: the reference's W20-D100 net (tests/golden) and a seeded W20-D50 net, beta = 2, box [0.5, 1.5]^2, 64
hyperplane directions theta_i = 2 pi (i - 1) / 64; an ACAS-shaped [5, 50 x 6, 5] net, beta = 2, 9 boxes x 5 output
half-spaces.  Every call ends in a device synchronise (both calls are blocking); one warm-up, median of --reps.

    python tools/affine_batch_timing.py [--reps 7] [--out FILE]
"""
import argparse
import os
import statistics
import subprocess
import sys
import time

import numpy as np
import scipy.sparse as sp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "nn-sdp_b200"))
sys.path.insert(0, os.path.join(ROOT, "oracle"))

import nnsdp_b200 as nb  # noqa: E402
import nnsdp_oracle as o  # noqa: E402


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown (nvidia-smi failed)"


def crown_bounds(dnet, lo, hi):
    r = nb.bounds_crown(dnet, lo, hi)
    n1, ac = lo.shape[1], r["acxmin"].shape[1]
    smin, smax = nb.sector_minmax(dnet.ctx, r["acxmin"], r["acxmax"])
    return r["xmin"][:, n1:n1 + ac], r["xmax"][:, n1:n1 + ac], smin, smax


def polytope(dnet, lo, hi):
    ymin, ymax, smin, smax = crown_bounds(dnet, lo[None], hi[None])
    th = 2 * np.pi * np.arange(64) / 64
    vec = np.stack([np.cos(th), np.sin(th)], axis=1)
    batch = nb.NumericBatch(x1min=lo, x1max=hi, ymin=ymin[0], ymax=ymax[0], smin=smin[0], smax=smax[0],
                            out_kind=nb.OUT_HPLANE, out_vec=vec)
    singles = [nb.NumericBatch(x1min=lo, x1max=hi, ymin=ymin, ymax=ymax, smin=smin, smax=smax, out_kind=nb.OUT_HPLANE,
                               out_vec=vec[q:q + 1]) for q in range(64)]
    return batch, singles


def acas(dnet, net, rng):
    boxes = []
    for _ in range(9):
        c = rng.uniform(-0.5, 0.5, 5)
        boxes.append((c - 0.05, c + 0.05))
    lo = np.stack([b[0] for b in boxes])
    hi = np.stack([b[1] for b in boxes])
    ymin, ymax, smin, smax = crown_bounds(dnet, lo, hi)
    S = [o.hplaneS(rng.standard_normal(5), 0.7, net) for _ in range(5)]
    box_of = np.repeat(np.arange(9), 5)
    Ss = np.stack([S[i % 5] for i in range(45)])
    batch = nb.NumericBatch(x1min=lo[box_of], x1max=hi[box_of], ymin=ymin[box_of], ymax=ymax[box_of],
                            smin=smin[box_of], smax=smax[box_of], out_kind=nb.OUT_SAFETY, out_S=Ss)
    singles = [nb.NumericBatch(x1min=lo[b:b + 1], x1max=hi[b:b + 1], ymin=ymin[b:b + 1], ymax=ymax[b:b + 1],
                               smin=smin[b:b + 1], smax=smax[b:b + 1], out_kind=nb.OUT_SAFETY, out_S=Ss[q:q + 1])
               for q, b in enumerate(box_of)]
    return batch, singles


def loop_once(dnet, beta, singles):
    """per query: nnsdp_affine_create / get, then coo -> csc with duplicates summed; returns (total, library) seconds"""
    t_lib = 0.0
    t0 = time.perf_counter()
    for b in singles:
        t1 = time.perf_counter()
        A = nb.affine_form(dnet, beta, b)
        t_lib += time.perf_counter() - t1
        M = sp.coo_matrix((A["coo_val"], (A["coo_ent"] - 1, A["coo_var"] - 1)), shape=(A["nent"], A["nvar"])).tocsc()
        M.sum_duplicates()
    return time.perf_counter() - t0, t_lib


def batch_once(dnet, beta, batch, Q):
    t0 = time.perf_counter()
    B = nb.affine_form_batch(dnet, beta, batch, Q=Q)
    mats = [sp.csc_matrix((g["val"], g["ent_idx"] - 1, g["var_ptr"] - 1), shape=(B["nent"], B["nvar"]))
            for g in B["groups"]]
    return time.perf_counter() - t0, B, mats


def check(dnet, beta, B, mats, singles):
    """every query's canonicalised single call equals its group's matrix (values to 1e-12: the two calls run the
    same kernels on the same bounds, so in practice bit for bit) and its z0"""
    worst = 0.0
    for q in (0, len(singles) // 2, len(singles) - 1):
        A = nb.affine_form(dnet, beta, singles[q])
        M = sp.coo_matrix((A["coo_val"], (A["coo_ent"] - 1, A["coo_var"] - 1)), shape=(A["nent"], A["nvar"])).tocsc()
        M.sum_duplicates()
        G = mats[B["group_of"][q]]
        assert np.array_equal(M.indptr, G.indptr) and np.array_equal(M.indices, G.indices)
        worst = max(worst, np.abs(M.data - G.data).max() / max(np.abs(M.data).max(), 1e-300))
        assert np.array_equal(A["z0"], B["z0"][q])
    assert worst <= 1e-12, worst
    return worst


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if nb.device_count() < 1:
        raise SystemExit("no CUDA device: nothing to measure")
    lines = [f"card: {card()}", f"reps: {args.reps} (median; one warm-up first)"]
    ctx = nb.Context([0])
    gold = os.path.join(ROOT, "tests", "golden")
    rng = np.random.default_rng(2024)
    work = []
    xd, Ms = nb.read_nnet(os.path.join(gold, "scale-I2-O2-W20-D100.nnet"))
    work.append(("W20-D100 polytope (64 directions)", xd, Ms, "poly"))
    net50 = o.random_network([2] + [20] * 50 + [2], 2.0 / np.sqrt(20 * np.log(20)), np.random.default_rng(50))
    work.append(("W20-D50 polytope (64 directions)", net50.xdims, net50.Ms, "poly"))
    netA = o.random_network([5] + [50] * 6 + [5], 2.0 / np.sqrt(50 * np.log(50)), np.random.default_rng(12))
    work.append(("ACAS [5, 50x6, 5] (9 boxes x 5 half-spaces)", netA.xdims, netA.Ms, "acas"))
    beta = 2
    for name, xdims, Ms, kind in work:
        dnet = nb.Net(ctx, list(xdims), list(Ms))
        if kind == "poly":
            batch, singles = polytope(dnet, np.full(2, 0.5), np.full(2, 1.5))
        else:
            batch, singles = acas(dnet, netA, rng)
        Q = len(singles)
        loop_once(dnet, beta, singles)
        _, B, mats = batch_once(dnet, beta, batch, Q)
        worst = check(dnet, beta, B, mats, singles)
        loops, libs, bats = [], [], []
        for _ in range(args.reps):  # alternate the two so that drift hits both alike
            t, tl = loop_once(dnet, beta, singles)
            loops.append(t)
            libs.append(tl)
            bats.append(batch_once(dnet, beta, batch, Q)[0])
        ml, mb = statistics.median(loops), statistics.median(bats)
        lines += [
            f"{name}: Q = {Q}, groups = {B['ngroups']}, nvar = {B['nvar']}, nent = {B['nent']}, "
            f"nnz per group max = {B['nnz_max']}, total = {B['nnz_total']}, batch vs single values max rel diff {worst:.1e}",
            f"  loop of affine_form + scipy coo->csc: median {ml * 1e3:9.2f} ms  ({ml / Q * 1e3:.2f} ms/query; library "
            f"calls {statistics.median(libs) * 1e3:.2f} ms, scipy {(ml - statistics.median(libs)) * 1e3:.2f} ms)  "
            f"min {min(loops) * 1e3:.2f} max {max(loops) * 1e3:.2f}",
            f"  affine_form_batch + csc_matrix:       median {mb * 1e3:9.2f} ms  min {min(bats) * 1e3:.2f} "
            f"max {max(bats) * 1e3:.2f}   speed-up {ml / mb:.1f}x",
        ]
        print("\n".join(lines[-3:]), flush=True)
        dnet.close()
    ctx.close()
    text = "\n".join(lines) + "\n"
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        open(args.out, "w").write(text)


if __name__ == "__main__":
    main()
