"""Cost of the certificate for the exact Z(γ): nnsdp_batch_assembly_error alone (the bound e_q), and
nnsdp_batch_certify_gamma against nnsdp_batch_certify on the same batch, the two alternated in one session.  Also the
rate of the |W|' G products (zerr_gemv_kernel) from torch.profiler in a run of its own, and the kernels' share.

    python tools/certify_gamma_timing.py [--out DIR]      (DIR/certify_gamma_timing.json gets the rows as well)
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

# (name, xdims, beta, Q of the bound alone, Q of the certify pair)
CONFIGS = [
    ("stress W1000-D20", [2] + [1000] * 19 + [2], 2, 1024, 8),
    ("W100-D50", [2] + [100] * 49 + [2], 2, 1024, 16),
    ("ACAS 5x50x6", [5] + [50] * 6 + [5], 2, 1024, 45),
]


def setup(ctx, xdims, beta, Q, ring):
    net = rand_net(xdims, seed=5)
    rng = np.random.default_rng(5)
    qs = [rand_query(net, beta, rng, kind="safety") for _ in range(min(Q, 64))]
    qs = [qs[i % len(qs)] for i in range(Q)]
    dnet = nb.Net(ctx, net.xdims, net.Ms)
    b = nb.Batch(dnet, beta, Qcap=Q, ring=ring)
    b.set_inputs(to_numeric_batch(nb, net, qs))
    b.bounds()
    b.prepare()
    return dnet, b


def gemv_flops(xdims, Q):
    """One fma (2 flops) per weight of layers 1 .. K-1 and query."""
    return 2 * sum(xdims[k] * xdims[k + 1] for k in range(len(xdims) - 2)) * Q


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=5)
    a = ap.parse_args()
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    print("GPU:", gpu, flush=True)
    ctx = nb.Context([0])
    rows = []
    for name, xdims, beta, Qb, Qc in CONFIGS:
        # the bound alone, Qb queries (ring 1: nothing is emitted)
        dnet, b = setup(ctx, xdims, beta, Qb, 1)
        b.assembly_error()
        t = []
        for _ in range(a.reps):
            t0 = time.perf_counter()
            e = b.assembly_error()
            t.append(time.perf_counter() - t0)
        tb = float(np.median(t))
        b.close()
        # certify vs certify_gamma, alternated, Qc queries
        dnet, b = setup(ctx, xdims, beta, Qc, min(Qc, 8 if max(xdims) >= 500 else 16))
        lo = b.lambda_max(max_iters=300, tol=1e-10, full=True)[0]
        tau = lo + 1e-6 * np.maximum(np.abs(lo), 1.0)
        b.certify(tau)
        b.certify_gamma(tau)
        tc, tg = [], []
        for _ in range(max(1, a.reps // 2)):
            t0 = time.perf_counter()
            c1 = b.certify(tau)
            tc.append(time.perf_counter() - t0)
            t0 = time.perf_counter()
            c2 = b.certify_gamma(tau)
            tg.append(time.perf_counter() - t0)
        b.close()
        row = dict(config=name, bound_Q=Qb, assembly_error_ms=1e3 * tb, assembly_error_ms_per_1024=1e3 * tb * 1024 / Qb,
                   gemv_tflops_end_to_end=gemv_flops(xdims, Qb) / tb / 1e12, e_max=float(np.max(e)),
                   certify_Q=Qc, certify_ms_per_query=1e3 * float(np.median(tc)) / Qc,
                   certify_gamma_ms_per_query=1e3 * float(np.median(tg)) / Qc,
                   certified=int(c1[0].sum()), certified_gamma=int(c2[0].sum()))
        print(json.dumps(row), flush=True)
        rows.append(row)
    # kernel times of one bound call at the stress size (torch.profiler, a run of its own)
    try:
        import torch
        from torch.profiler import ProfilerActivity, profile

        name, xdims, beta, Qb, _ = CONFIGS[0]
        _, b = setup(ctx, xdims, beta, Qb, 1)
        b.assembly_error()
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            b.assembly_error()
            torch.cuda.synchronize()
        us = {}
        for ev in prof.key_averages():
            m = re.search(r"zerr_\w+_kernel", ev.key)
            if m:
                us[m.group(0)] = us.get(m.group(0), 0.0) + getattr(ev, "device_time_total", 0.0)
        g = us.get("zerr_gemv_kernel", 0.0)
        line = dict(kernel_us=us, gemv_tflops=gemv_flops(xdims, Qb) / (g * 1e-6) / 1e12 if g else None)
        print(json.dumps(line), flush=True)
        rows.append(line)
        b.close()
    except Exception as ex:  # the measurement above stands without the profiler
        print("profiler:", repr(ex))
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "certify_gamma_timing.json"), "w") as f:
            json.dump(dict(gpu=gpu, rows=rows), f, indent=1)


if __name__ == "__main__":
    main()
