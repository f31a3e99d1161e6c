"""Timing of nnsdp_batch_certify (the sound eigmax(Z) <= tau certificate) against the Lanczos check of the same batch
and numpy.linalg.eigvalsh on the dense Z (the reference's eigmax), where the dense Z fits.  Prints one line per
configuration and the FP64 tensor-core rate of the trailing-update kernel (torch.profiler, a run of its own).

    python tools/certify_timing.py [--out DIR]      (DIR/certify_timing.json gets the rows as well)
"""
import argparse
import json
import os
import re
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (os.path.join(ROOT, "nn-sdp_b200"), os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")):
    sys.path.insert(0, p)

import nnsdp_b200 as nb  # noqa: E402
from helpers import rand_net, rand_query, to_numeric_batch  # noqa: E402

CONFIGS = [
    ("stress W1000-D20", [2] + [1000] * 19 + [2], 2, 4),
    ("W100-D50", [2] + [100] * 49 + [2], 2, 16),
    ("W20-D100", [2] + [20] * 99 + [2], 2, 16),
    ("ACAS 5x50x6", [5] + [50] * 6 + [5], 2, 45),
]


def update_flops(xdims, beta):
    """2 * (lower-triangle entries) * panel width, summed over the panels of every front."""
    f = 0
    for _, n, npriv, _, _, _ in nb.certify_plan(xdims, beta):
        for j0 in range(0, npriv, 32):   # CHOL_NB
            w = min(32, npriv - j0)
            m = n - j0 - w
            f += m * (m + 1) * w
    return f


def setup(ctx, xdims, beta, Q):
    net = rand_net(xdims, seed=5)
    rng = np.random.default_rng(5)
    qs = [rand_query(net, beta, rng, kind="safety") for _ in range(Q)]
    dnet = nb.Net(ctx, net.xdims, net.Ms)
    nbq = to_numeric_batch(nb, net, qs)
    b = nb.Batch(dnet, beta, Qcap=Q, ring=min(Q, 4 if max(xdims) >= 500 else 16))
    b.set_inputs(nbq)
    b.bounds()
    b.prepare()
    return net, dnet, to_numeric_batch(nb, net, qs[:1]), b


def timed(fn, reps=3):
    fn()
    t = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        t.append(time.perf_counter() - t0)
    return float(np.median(t)), fn()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    print("GPU:", gpu)
    ctx = nb.Context([0])
    rows = []
    for name, xdims, beta, Q in CONFIGS:
        net, dnet, nbq, b = setup(ctx, xdims, beta, Q)
        lo = b.lambda_max(max_iters=300, tol=1e-10, full=True)[0]
        t_cert, (cert, bound, _, _) = timed(lambda: b.certify(lo + 1e-6 * np.maximum(np.abs(lo), 1.0)))
        t_lan, _ = timed(lambda: b.lambda_max(max_iters=300, tol=1e-10, full=True), reps=1)
        row = dict(config=name, Q=Q, Zdim=int(net.Zdim) if hasattr(net, "Zdim") else sum(xdims[:-1]) + 1,
                   certify_ms_per_query=1e3 * t_cert / Q, lanczos300_ms_per_query=1e3 * t_lan / Q,
                   certified=int(cert.sum()), update_gflop_per_query=update_flops(xdims, beta) / 1e9)
        if row["Zdim"] <= 6000:
            Z = nb.assemble_dense(dnet, beta, nbq, Q=1)[0]
            n = row["Zdim"]
            Z = Z.reshape(n, n, order="F")
            t0 = time.perf_counter()
            np.linalg.eigvalsh(Z)
            row["eigvalsh_ms_per_query"] = 1e3 * (time.perf_counter() - t0)
        print(json.dumps(row))
        rows.append(row)
        b.close()
    # the update kernel's rate: torch.profiler around one certify call of the stress batch
    try:
        import torch
        from torch.profiler import ProfilerActivity, profile

        name, xdims, beta, Q = CONFIGS[0]
        _, _, _, b = setup(ctx, xdims, beta, Q)
        b.certify(1e6)                       # far above lambda_max: every query runs the whole factorisation
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            b.certify(1e6)
        us = {}
        for e in prof.key_averages():
            m = re.search(r"chol_\w+_kernel", e.key)
            if m:
                us[m.group(0)] = us.get(m.group(0), 0.0) + getattr(e, "device_time_total", 0.0)
        upd = sum(v for k, v in us.items() if "update" in k)
        fl = update_flops(xdims, beta) * Q
        line = dict(kernel_us=us, update_tflops=fl / (upd * 1e-6) / 1e12 if upd else None)
        print(json.dumps(line))
        rows.append(line)
        b.close()
    except Exception as e:  # the measurement above stands without the profiler
        print("profiler:", repr(e))
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "certify_timing.json"), "w") as f:
            json.dump(dict(gpu=gpu, rows=rows), f, indent=1)


if __name__ == "__main__":
    main()
