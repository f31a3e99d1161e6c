#!/usr/bin/env python
"""bench.py -- throughput of the Chordal-DeepSDP constraint-construction path on B200.

Metric (BASELINE.json): clique LMI blocks assembled/sec and queries/sec.  `value` is queries/s
(blocks/s = value * cliques per query, reported in `config`), whole job over all ranks.

Workload (BASELINE.json configs[4], "synthetic stress"): random ReLU net xdims = [2, 1000 x 20, 2],
beta = 2, 1024 batched queries with distinct input boxes and numeric multipliers.  A step = one
pass of the hot path over the 1024 queries of a rank: IBP bounds -> sector slopes -> QC
diagonals / affine column -> Gram contractions -> emission of all dense clique blocks into a ring
of device slots.

  python bench.py [--gpus N] [--steps K] [--warmup W]          our arm
  python bench.py --impl reference ...                          CPU restatement of the reference
  python bench.py ... --dump-outputs DIR                        also save what the last timed step computed
Under torchrun every rank drives one GPU with its own 1024 queries (weak scaling, no collective).
Each GPU line (headline, packed, end to end, CROWN bounds, other workloads) times --steps steps.

--dump-outputs DIR writes DIR/dense_blocks.npy (float64), the dense clique blocks that the headline loop
(nnsdp_batch_run into the device ring) left in its ring slots after its last step: row i is query Q - n + i of
rank 0, n = the queries of the last pass, each row the flat blocks of one query (nnsdp_batch_get_slot layout), or
the same fixed, seeded sample of its entries when all n rows would exceed DUMP_BYTES.  The inputs depend on the
arguments only, so two builds run with the same arguments can be compared entry for entry.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "nn-sdp_b200"))

WORKLOADS = {
    # name: (width, depth, beta, queries, ring slots)
    "stress-W1000-D20-beta2-Q1024": dict(W=1000, D=20, beta=2, Q=1024, ring=32),   # 32 slots = 42.6 GB of blocks in HBM
    "mid-W100-D50-beta2-Q1024": dict(W=100, D=50, beta=2, Q=1024, ring=256),
    "tiny-W10-D10-beta1-Q64": dict(W=10, D=10, beta=1, Q=64, ring=64),
    # BASELINE configs[2]: experiments/reach.jl / findReach2Dpoly (src/NnSdp.jl:73-95): one net and box, 64 hyperplane
    # directions -- a reach batch (shared bounds and multipliers, per-query normal and gamma_out)
    "reach-W20-D10-beta2-Q64": dict(W=20, D=10, beta=2, Q=64, ring=64, kind="reach"),
    # BASELINE configs[3]: ACAS Xu shape 5 x (6 x 50) x 5 (exts/nnet_parser.jl), 45 safety queries (one vnnlib property
    # flattened over its boxes and half-spaces, experiments/vnnlib_utils.jl:18-56)
    "acas-5x50x6-beta2-Q45": dict(xdims=[5] + [50] * 6 + [5], beta=2, Q=45, ring=45, kind="acas"),
    # alignment probe (profiles/r2_experiments.txt): clique blocks with ld = 3000, a multiple of four doubles
    "probe-W999-D20-beta2-Q1024": dict(W=999, D=20, beta=2, Q=1024, ring=32),
}
EXTRA_WORKLOADS = ("mid-W100-D50-beta2-Q1024", "tiny-W10-D10-beta1-Q64", "reach-W20-D10-beta2-Q64", "acas-5x50x6-beta2-Q45")
DEFAULT_WORKLOAD = "stress-W1000-D20-beta2-Q1024"
DUMP_BYTES = 60_000_000          # --dump-outputs: size cap of the dumped arrays (one stress query alone is 1.33 GB)


def make_workload(name: str, rank: int, Q: int | None = None, radius_scale: float = 1.0):
    """Seeded synthetic inputs (SURVEY.md section 8d, config 5).  Returns (xdims, Ms, inputs)."""
    w = WORKLOADS[name]
    beta = w["beta"]
    Q = Q or w["Q"]
    xdims = w.get("xdims") or [2] + [w["W"]] * w["D"] + [2]
    W, D = max(xdims[1:-1]), len(xdims) - 2
    n_in, n_out = xdims[0], xdims[-1]
    rng = np.random.default_rng(1000 * D + W)          # net: the same on every rank
    sigma = 2.0 / np.sqrt(W * np.log(W))               # scripts/make_networks.jl:44
    Ms = []
    for k in range(len(xdims) - 1):
        Ms.append(sigma * rng.standard_normal((xdims[k + 1], xdims[k] + 1)))
    rq = np.random.default_rng(777 + rank)             # queries: distinct per rank
    acdim = sum(xdims[1:-1])
    lamdim = sum(range(acdim - beta, acdim + 1))
    kind = w.get("kind", "safety")
    if kind == "reach":                                # shared box and multipliers, one hyperplane normal per query
        th = 2 * np.pi * np.arange(Q) / Q
        inputs = dict(x1min=np.full((1, n_in), 0.5), x1max=np.full((1, n_in), 1.5), gamma_in=rq.random((1, n_in)),
                      gamma_bnd=rq.random((1, acdim)), gamma_sec=rq.random((1, lamdim + 2 * acdim)),
                      out_vec=np.stack([np.cos(th), np.sin(th)], 1), gamma_out=rq.random((Q, 1)))
        return xdims, Ms, beta, inputs
    centre = rq.uniform(0.5, 1.5, (Q, n_in))
    radius = rq.uniform(0.01, 0.5, (Q, 1)) * radius_scale   # radius_scale << 1: stable ReLUs, Gram-heavy
    sd = n_in + n_out + 1
    if kind == "acas":                                 # one half-space per query: hplaneS(-A_i, -b_i - 1e-4)
        normals = rq.standard_normal((Q, n_out))
        S = np.zeros((Q, sd, sd))
        S[:, n_in:n_in + n_out, sd - 1] = normals
        S[:, sd - 1, n_in:n_in + n_out] = normals
        S[:, sd - 1, sd - 1] = -2.0 * rq.random(Q)
        radius = radius * 0.1
    else:
        normal = np.zeros(n_out)
        normal[0] = 1.0
        S = np.zeros((1, sd, sd))
        S[0, n_in:n_in + n_out, sd - 1] = normal
        S[0, sd - 1, n_in:n_in + n_out] = normal
        S[0, sd - 1, sd - 1] = -2.0 * 1.0              # hplaneS([1,0], 1.0) (src/Utils/qc.jl:27-38)
    inputs = dict(
        x1min=centre - radius, x1max=centre + radius,
        gamma_in=rq.random((Q, n_in)), gamma_bnd=rq.random((Q, acdim)),
        gamma_sec=rq.random((Q, lamdim + 2 * acdim)), out_S=S)
    return xdims, Ms, beta, inputs


def numeric_batch(nb, name, inp):
    kind = nb.OUT_HPLANE if WORKLOADS[name].get("kind") == "reach" else nb.OUT_SAFETY
    return nb.NumericBatch(out_kind=kind, **inp)


def ncu_traffic(kernel):
    """dram__bytes_read.sum + dram__bytes_write.sum of ONE launch of `kernel` from the committed `ncu --set full`
    summary of this round (profiles/r2_emit_full.summary.csv: a 32-query pass of the stress workload), or None.
    Fails loudly when the capture does not hold the kernel: a stale table must not go unnoticed."""
    import csv

    path = os.path.join(ROOT, "profiles", "r2_emit_full.summary.csv")
    if not os.path.exists(path):
        return None
    unit = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
    # the default pass (panel-ordered launch), then the capture with NNSDP_PANEL=0 (fill and window kernels on their own)
    for p in (path, os.path.join(ROOT, "profiles", "r2_emit_full_separate_kernels.summary.csv")):
        if not os.path.exists(p):
            continue
        rows = list(csv.reader(open(p)))
        hdr = rows[0]

        def col(prefix):
            i = [j for j, h in enumerate(hdr) if h.startswith(prefix)][0]
            return i, unit[hdr[i].split("[")[1].rstrip("]")]

        (ir, ur), (iw, uw) = col("dram__bytes_read.sum"), col("dram__bytes_write.sum")
        for r in rows[1:]:
            if r[0].split("<")[0] == kernel:
                return float(r[ir]) * ur + float(r[iw]) * uw
    if os.environ.get("NNSDP_BENCH_RECAPTURE") == "1":   # the run that re-captures the profile itself
        print(f"bench.py: {path} holds no launch of {kernel}; traffic = null in this run", file=sys.stderr)
        return None
    raise RuntimeError(f"{path} holds no launch of {kernel}: re-capture the profile (tools/ncu_summary.py)")


def quick_measure(nb, torch, name, peak, steps, warmup=3):
    """Device-timed dense and packed passes of one of the other BASELINE configs (single GPU, short)."""
    w = WORKLOADS[name]
    xdims, Ms, beta, inp = make_workload(name, 0)
    Q = w["Q"]
    ctx = nb.Context([torch.cuda.current_device()])
    net = nb.Net(ctx, xdims, Ms)
    sz = net.sizes(beta)
    out = {"workload": name, "xdims": f"{xdims[0]}, {max(xdims[1:-1])} x {len(xdims) - 2}, {xdims[-1]}", "beta": beta, "queries": Q,
           "cliques_per_query": sz["ncliques"], "dense_block_bytes_per_query": 8 * sz["sum_ck_sq"]}
    nbatch = numeric_batch(nb, name, inp)
    for fmt in ("dense", "packed"):
        b = nb.Batch(net, beta, Qcap=Q, ring=min(w["ring"], Q), packed=(fmt == "packed"))
        b.set_inputs(nbatch, Q=Q)
        run = (lambda: b.run_packed(None)) if fmt == "packed" else (lambda: b.run(None))
        for _ in range(warmup):
            run()
        b.stage_reset()
        b.sync()
        torch.cuda.synchronize()
        b.event_record(0)
        for _ in range(steps):
            run()
        b.event_record(1)
        b.sync()
        torch.cuda.synchronize()
        ms = b.elapsed_ms() / steps
        emit_ms = b.stage_ms("emit")[0] / steps
        nbytes = b.packed_stats()["emitted_bytes"] if fmt == "packed" else 8.0 * sz["sum_ck_sq"] * Q
        launches = sum(b.stage_ms(k)[1] for k in ("bounds", "prepare", "gram", "emit")) / steps
        out[fmt] = {"queries_per_s": Q / (ms * 1e-3), "ms_per_step": ms, "us_per_query": 1e3 * ms / Q,
                    "emitter_ms": emit_ms, "emitted_bytes_per_step": nbytes,
                    "emitter_gbs": nbytes / max(emit_ms, 1e-9) / 1e6, "emitter_frac_of_peak": nbytes / max(emit_ms, 1e-9) / 1e6 / peak,
                    "launches_per_step": launches,
                    "stage_ms": {k: b.stage_ms(k)[0] / steps for k in ("bounds", "prepare", "gram", "emit")}}
        b.close()
    net.close()
    return out


def crown_line(nb, torch, net, name, beta, inp, Q, steps):
    """The stress workload with the reference's DEFAULT bounds (IntervalsAutoLirpa -> CROWN on the device) instead of
    interval arithmetic: realistic bounds leave stably-active neurons in every layer, so the FP64 tensor-core Gram
    contractions (K3) run on wide layers.  Bounded sample of Q queries; packed records left in HBM."""
    sub = {k: (v[:Q] if v.shape[0] >= Q and v.shape[0] != 1 else v) for k, v in inp.items()}
    b = nb.Batch(net, beta, Qcap=Q, ring=min(Q, 16), packed=True)
    b.set_inputs(numeric_batch(nb, name, sub), Q=Q)
    b.set_bounds_method("crown")
    b.run_packed(None)
    b.stage_reset()
    b.sync()
    torch.cuda.synchronize()
    b.event_record(0)
    for _ in range(steps):
        b.run_packed(None)
    b.event_record(1)
    b.sync()
    torch.cuda.synchronize()
    ms = b.elapsed_ms() / steps
    st = {k: b.stage_ms(k)[0] / steps for k in ("bounds", "prepare", "gram", "emit")}
    ncon, nact = b.gram_stats()
    W = WORKLOADS[name]["W"]
    flops = float(W) * (W + 128) * nact          # executed: upper 128 x 128 tile pairs, 2 flops per (entry, active neuron)
    full = 2.0 * W * W * nact                    # algorithmic: the full W' diag W product over the active neurons
    dgemm_peak = 36.06                           # TFLOP/s, cuBLAS DGEMM 8192^3 on this pool (profiles/r1_probe_dgemm.txt)
    out = {"bounds": "crown (nnsdp_batch_set_bounds_method: the reference's default IntervalsAutoLirpa)", "queries": Q,
           "queries_per_s": Q / (ms * 1e-3), "ms_per_step": ms, "stage_ms": st,
           "gram_contractions_per_step": ncon, "gram_active_rows_per_step": nact,
           "present_diag_cells_per_query": b.packed_stats()["present_optional_cells"] / Q,
           "roofline": {"bound": "tensor", "kernel": "gram_kernel (FP64 DMMA)", "achieved": flops / max(st["gram"], 1e-9) / 1e9,
                        "achieved_algorithmic": full / max(st["gram"], 1e-9) / 1e9, "peak": dgemm_peak, "unit": "TFLOP/s",
                        "frac": flops / max(st["gram"], 1e-9) / 1e9 / dgemm_peak,
                        "peak_source": "measured cuBLAS DGEMM on this pool (tools/probe_dgemm.cu, profiles/r1_probe_dgemm.txt); "
                                       "MEASURED_PEAKS.json has no FP64 figure"}}
    b.close()
    return out


class _DeviceDoubles:
    """A float64 device range seen through __cuda_array_interface__, so torch can index it in place."""

    def __init__(self, ptr: int, n: int):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": "<f8", "data": (ptr, False), "strides": None,
                                         "version": 2}


def last_pass_outputs(torch, batch, Q: int, ring: int, nbytes: int) -> np.ndarray:
    """The ring slots a device-only run (batch.run(None)) left behind: a pass writes queries q0 .. q0 + n - 1 into
    slots 0 .. n - 1, so after the last pass slot i holds query Q - n + i.  Returns them as an (n, per_query) array,
    or (n, m) with the same seeded sample of m entries per slot when n whole slots exceed `nbytes`.  Gathered on the
    device: copying whole slots to the host would move 1.33 GB per stress query."""
    n = Q - ring * ((Q - 1) // ring)
    ptr, per = batch.ring_ptr()
    batch.sync()
    slots = torch.as_tensor(_DeviceDoubles(ptr, n * per)).view(n, per)
    m = min(per, nbytes // (8 * n))
    if m < per:
        idx = np.sort(np.random.default_rng(0).choice(per, size=m, replace=False))
        slots = slots[:, torch.from_numpy(idx).to(slots.device)]
    return slots.cpu().numpy()


# ------------------------------------------------------------------------------------------
# clocks sampler (nvidia-smi during the timed region)
# ------------------------------------------------------------------------------------------
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu, self.rows, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "100",
                 "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([t.strip() for t in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.th.join(timeout=2)
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            if len(r) < 6:
                continue
            try:
                sm.append(float(r[0]))
                smax.append(float(r[1]))
            except ValueError:
                continue
            for n, v in zip(names, r[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md, MEASURED_PEAKS.json absent)"


# ------------------------------------------------------------------------------------------
# CPU arm: the oracle's closed-form restatement on all host cores.  The reference is single-threaded
# Julia; the port gets the strongest fair treatment: P worker processes (spawned, one BLAS thread each)
# assemble P different queries of the workload at the same time, P = host cores (memory permitting).
# ------------------------------------------------------------------------------------------
_W = {}


_BLAS_ENV = ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS")


def _blas_threads():
    """Largest BLAS/OpenMP thread-pool size of this process, as the libraries report it (threadpoolctl)."""
    from threadpoolctl import threadpool_info

    return max([int(i.get("num_threads", 1)) for i in threadpool_info()] or [1])


def _cpu_worker_init(name, root):
    # The thread-pool size is fixed when numpy's BLAS is loaded, and a spawned child re-imports this module
    # (numpy included) BEFORE the initializer runs: the variables must already be in the environment the
    # child inherits (CpuPool sets them in the parent).  Here the result is only checked.
    nt = _blas_threads()
    if nt != 1:
        raise RuntimeError(f"CPU arm worker runs {nt} BLAS threads, expected 1 (environment not inherited)")
    sys.path.insert(0, os.path.join(root, "oracle"))
    import nnsdp_oracle as o

    xdims, Ms, beta, inp = make_workload(name, 0, Q=64)
    _W.update(o=o, net=o.FeedFwdNet(xdims, Ms), beta=beta, inp=inp)


def _cpu_worker_threads(_):
    return _blas_threads()


def _cpu_worker_query(i):
    o, inp = _W["o"], _W["inp"]
    i = i % inp["x1min"].shape[0]
    q = o.NumericQuery(x1min=inp["x1min"][i], x1max=inp["x1max"][i], gin=inp["gamma_in"][i],
                       gbnd=inp["gamma_bnd"][i], gsec=inp["gamma_sec"][i], qc_out=o.QcSafety(S=inp["out_S"][0]))
    r = o.run_query(_W["net"], _W["beta"], q, form="closed")
    n = len(r["blocks"])
    del r
    return n


class CpuPool:
    """P spawned worker processes holding the network; map() assembles a list of queries in parallel."""

    def __init__(self, name):
        import multiprocessing as mp

        w = WORKLOADS[name]
        cores = os.cpu_count() or 1
        per_proc_gb = 8.0 if w["W"] >= 500 else 0.5     # dense Z + blocks + temporaries of one query
        try:
            avail_gb = os.sysconf("SC_AVPHYS_PAGES") * os.sysconf("SC_PAGE_SIZE") / 2**30
        except (ValueError, OSError):
            avail_gb = 32.0
        self.procs = int(max(1, min(cores, 0.6 * avail_gb / per_proc_gb)))
        saved = {v: os.environ.get(v) for v in _BLAS_ENV}
        for v in _BLAS_ENV:                                      # inherited by the spawned workers
            os.environ[v] = "1"
        try:
            self.pool = mp.get_context("spawn").Pool(self.procs, initializer=_cpu_worker_init, initargs=(name, ROOT))
            self.blas_threads = max(self.pool.map(_cpu_worker_threads, range(self.procs)))   # verified, not assumed
        finally:
            for v, old in saved.items():
                if old is None:
                    os.environ.pop(v, None)
                else:
                    os.environ[v] = old
        assert self.blas_threads == 1, self.blas_threads
        self.pool.map(_cpu_worker_query, range(self.procs))      # warm-up: imports, page faults

    def run(self, n_queries):
        t0 = time.perf_counter()
        self.pool.map(_cpu_worker_query, range(n_queries), chunksize=1)
        return time.perf_counter() - t0

    def close(self):
        self.pool.close()
        self.pool.join()


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    name = args.workload
    w = WORKLOADS[name]
    pool = CpuPool(name)
    per_step = pool.procs if w["W"] >= 500 else 16 * pool.procs
    for _ in range(args.warmup):
        pool.run(per_step)
    times = [pool.run(per_step) for _ in range(args.steps)]
    pool.close()
    sec_per_step = float(np.mean(times))
    value = per_step / sec_per_step
    line = {
        "impl": "reference", "metric": "queries/sec (clique LMI blocks assembled: value * cliques_per_query)",
        "value": value, "unit": "queries/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * sec_per_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": name, "queries_per_step": per_step, "cliques_per_query": w["D"] - 1,
                   "note": "CPU restatement of the reference algorithm (Julia/JuMP/MOSEK are not installable here); "
                           "the reference itself is single-threaded, the port runs one query per worker process"},
        "cpu_baseline": {"value": value, "unit": "queries/s", "cores": pool.procs, "kind": "port",
                         "sample": f"{per_step} queries per step x {args.steps} steps of the same workload, numpy closed form, "
                                   f"{pool.procs} worker processes x {pool.blas_threads} BLAS thread (verified with threadpoolctl in the workers) "
                                   f"on {os.cpu_count()} host cores"},
        "e2e": {"value": value, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist

    import nnsdp_b200 as nb

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    name = args.workload
    w = WORKLOADS[name]
    Q = args.queries or w["Q"]
    if args.scaling == "strong":                         # BASELINE config 5 read literally: 1024 queries in total
        from nnsdp_b200.dist import shard_range
        _, Q = shard_range(Q, world, rank)
    xdims, Ms, beta, inp = make_workload(name, rank, Q=Q, radius_scale=args.radius_scale)
    ctx = nb.Context([local])
    net = nb.Net(ctx, xdims, Ms)
    sz = net.sizes(beta)
    ring = min(args.ring or w["ring"], Q)
    batch = nb.Batch(net, beta, Qcap=Q, ring=ring)
    nbatch = numeric_batch(nb, name, inp)
    batch.set_inputs(nbatch, Q=Q)

    def barrier():
        if world > 1:
            dist.barrier()
        batch.sync()
        torch.cuda.synchronize()

    def step():
        batch.run(None)

    for _ in range(args.warmup):
        step()
    batch.stage_reset()
    sampler = ClockSampler(local)
    barrier()
    if rank == 0:
        sampler.start()
    batch.event_record(0)
    for _ in range(args.steps):
        step()
    batch.event_record(1)
    barrier()
    ms = batch.elapsed_ms()
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "dense_blocks.npy"), last_pass_outputs(torch, batch, Q, ring, DUMP_BYTES))
    stage = {k: batch.stage_ms(k) for k in ("bounds", "prepare", "gram", "emit")}  # emit = its three kernels
    ncon, nact = batch.gram_stats()
    if world > 1:
        t = torch.tensor([ms], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    ms_per_step = ms / args.steps
    Qtot = Q
    if world > 1:
        t = torch.tensor([Q], device="cuda", dtype=torch.int64)
        dist.all_reduce(t)
        Qtot = int(t.item())
    else:
        Qtot = Q
    value = Qtot / (ms_per_step * 1e-3)

    # ---- roofline of the emitter (HBM-write bound).  One pass = emit_fill_kernel, emit_window_kernel,
    # emit_edge_kernel back to back over `ring` queries; each kernel is timed with its own CUDA-event
    # span on the launching stream.  Algorithmic bytes of a kernel = 8 B x the output entries of the
    # tiles it owns (host plan), x the queries of the pass; the three add up to 8 * sum|Ck|^2 per query.
    ps = nb.plan_stats(xdims, beta)
    ent = ps["entries"]
    kernel_entries = {"emit_fill_kernel": ent["ZERO"] + ent["SAME"] + ent["DIAG"] + ent["AFF"],
                      "emit_window_kernel": ent["RC"] + ent["CR"], "emit_edge_kernel": ent["MIXED"] + ent["GENERAL"]}
    assert sum(kernel_entries.values()) == sz["sum_ck_sq"]
    peak, peak_src = measured_peaks()
    q_per_pass = Q / max(1, -(-Q // ring))          # average queries per emitter pass
    kernels = []
    # dense formats of wide nets: the fill strips and the window tiles go out as ONE launch in panel order
    # (emit_panel_kernel, timed in the fill span; the window span stays empty)
    if kernel_entries["emit_window_kernel"] > 0 and batch.stage_ms("emit_window")[1] == 0 and batch.stage_ms("emit_fill")[1] > 0:
        kernel_entries["emit_panel_kernel"] = kernel_entries.pop("emit_fill_kernel") + kernel_entries.pop("emit_window_kernel")
    for kname, stage_name in (("emit_panel_kernel", "emit_fill"), ("emit_fill_kernel", "emit_fill"),
                              ("emit_window_kernel", "emit_window"), ("emit_edge_kernel", "emit_edge")):
        if kname not in kernel_entries:
            continue
        kms, kl = batch.stage_ms(stage_name)
        if kl == 0:
            continue
        b_launch = 8.0 * kernel_entries[kname] * q_per_pass
        avg = kms / kl
        kernels.append({"kernel": kname, "launches": kl, "avg_launch_ms": avg, "algorithmic_bytes_per_launch": b_launch,
                        "achieved": b_launch / (avg * 1e-3) / 1e9, "share_of_step": kms / ms if ms > 0 else None})
    emit_ms, _ = stage["emit"]
    n_pass = max(1, -(-Q // ring)) * args.steps
    if not kernels:  # kernels of a pass were not timed one by one (overlapped launch experiment)
        kernels = [{"kernel": "emitter pass (overlapped kernels)", "launches": n_pass, "avg_launch_ms": emit_ms / n_pass,
                    "algorithmic_bytes_per_launch": 8.0 * sz["sum_ck_sq"] * q_per_pass,
                    "achieved": 8.0 * sz["sum_ck_sq"] * q_per_pass / (emit_ms / n_pass * 1e-3) / 1e9,
                    "share_of_step": emit_ms / ms if ms > 0 else None}]
    dom = max(kernels, key=lambda k: k["share_of_step"])
    passes = n_pass
    pass_bytes = 8.0 * sz["sum_ck_sq"] * q_per_pass
    pass_gbs = pass_bytes / (emit_ms / passes * 1e-3) / 1e9
    roofline = {"bound": "hbm", "kernel": dom["kernel"], "achieved": dom["achieved"], "peak": peak, "unit": "GB/s",
                "frac": dom["achieved"] / peak,
                "traffic": (ncu_traffic(dom["kernel"]) * q_per_pass / 32.0) if name == DEFAULT_WORKLOAD and ncu_traffic(dom["kernel"]) else None,
                "traffic_source": "profiles/r2_emit_full.summary.csv (ncu --set full, one 32-query pass), scaled to the queries of a pass",
                "peak_source": peak_src,
                "algorithmic_bytes_per_launch": dom["algorithmic_bytes_per_launch"], "avg_launch_ms": dom["avg_launch_ms"],
                "share_of_step": dom["share_of_step"],
                "emitter_pass": {"kernels": kernels, "algorithmic_bytes": pass_bytes, "ms": emit_ms / passes,
                                 "achieved": pass_gbs, "frac": pass_gbs / peak, "share_of_step": emit_ms / ms if ms > 0 else None,
                                 "note": "8*sum|Ck|^2 bytes per query over the kernels of a pass"}}

    # ---- the same pass with packed records (NNSDP_FORMAT_PACKED): the block-sparse upper triangle of Z, every
    # region once, no structural zero written.  Same bounds / prepare / Gram work, same values (bit-identical to the
    # dense blocks, tests/test_gpu_packed.py); the emitter writes `emitted_bytes` instead of 8 * sum|Ck|^2 per query.
    batch.close()
    pring = min(int(os.environ.get("NNSDP_BENCH_PRING", 4 * ring)), Q)
    pb = nb.Batch(net, beta, Qcap=Q, ring=pring, packed=True)
    pb.set_inputs(nbatch, Q=Q)
    for _ in range(args.warmup):
        pb.run_packed(None)
    pb.stage_reset()
    barrier_p = lambda: (dist.barrier() if world > 1 else None, pb.sync(), torch.cuda.synchronize())
    barrier_p()
    pb.event_record(0)
    for _ in range(args.steps):
        pb.run_packed(None)
    pb.event_record(1)
    barrier_p()
    pms = pb.elapsed_ms()
    if world > 1:
        t = torch.tensor([pms], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        pms = float(t.item())
    pst = pb.packed_stats()
    pstage = {k: pb.stage_ms(k) for k in ("bounds", "prepare", "gram", "emit", "emit_fill", "emit_window", "emit_edge")}
    p_emit_ms = pstage["emit"][0] / args.steps
    packed = {"value": Qtot / (pms / args.steps * 1e-3), "unit": "queries/s", "ms_per_step": pms / args.steps,
              "record_bytes": 8 * pst["record_doubles"], "cells": pst["ncells"],
              "emitted_bytes_per_step": pst["emitted_bytes"], "ring_slots": pring,
              "stage_ms_per_step": {k: pstage[k][0] / args.steps for k in pstage},
              "emitter": {"ms": p_emit_ms, "achieved": pst["emitted_bytes"] / max(p_emit_ms, 1e-9) / 1e6, "unit": "GB/s",
                          "frac": pst["emitted_bytes"] / max(p_emit_ms, 1e-9) / 1e6 / peak},
              "note": "device-timed like `value`, records left in HBM; dense blocks are recovered by views / nnsdp_packed_unpack"}
    pb.close()

    # ---- end-to-end through the public API with host buffers (bounded sample of the same workload), on
    # EVERY rank at the same time: the ranks share the host's memory bandwidth and PCIe root complexes,
    # so the whole-job figure is world * Qe / (slowest rank's time), not N times a single-GPU number.
    if args.no_e2e:
        if rank == 0:
            print(json.dumps({"value": value, "ms_per_step": ms_per_step, "roofline": roofline, "packed": packed,
                              "stage_ms_per_step": {k: stage[k][0] / args.steps for k in stage}}), flush=True)
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return
    Qe = min(Q, args.e2e_queries)
    # host worker threads of the gather: share the box's cores between the ranks of this node
    os.environ.setdefault("NNSDP_HOST_THREADS", str(max(2, min(16, (os.cpu_count() or 16) // max(world, 1)))))
    pin = nb.PinnedBuffer(Qe * sz["sum_ck_sq"])
    eb = nb.Batch(net, beta, Qcap=Qe, ring=min(ring, Qe))
    sub = {k: (v[:Qe] if v.shape[0] == Q and Q > 1 else v) for k, v in inp.items()}
    ebatch = numeric_batch(nb, name, sub)
    h2d = sum(int(np.asarray(v).nbytes) for v in sub.values())
    d2h = Qe * sz["sum_ck_sq"] * 8

    def e2e_step(flags=0):
        eb.set_inputs(ebatch, Q=Qe)            # host -> device copy of this step's inputs
        eb.run(pin.array, flags=flags)         # compute + gather of every dense block into host memory

    def time_e2e(flags):
        e2e_step(flags)
        nrep = args.steps
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        for _ in range(nrep):
            e2e_step(flags)
        dt = (time.perf_counter() - t0) / nrep
        if world > 1:
            t = torch.tensor([dt], device="cuda", dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt = float(t.item())
        return dt

    e2e_s = time_e2e(0)
    gs = eb.gather_stats()
    e2e = {"value": world * Qe / e2e_s, "unit": "queries/s", "h2d_bytes_per_step": world * h2d,
           "d2h_bytes_per_step": world * (gs["dma_bytes"] + gs["thin_bytes"]),
           "queries_per_step": world * Qe, "ms_per_step": 1e3 * e2e_s, "host_result_bytes_per_step": world * d2h,
           "host_zero_filled_bytes_per_step": world * gs["zeroed_bytes"], "sparse_gather": gs["sparse"],
           "note": "bounded sample of the workload on every rank concurrently; the complete dense blocks (1.33 GB/query) "
                   "land in pinned host memory: dense cells by strided DMA, thin entries packed + scattered, "
                   "structural / value-dependent zeros filled by host threads"}
    # variants, for the record: caller-zeroed buffers (NNSDP_RUN_HOST_PREZEROED) and the plain dense copy
    t_pre = time_e2e(nb.RUN_HOST_PREZEROED)
    gs_pre = eb.gather_stats()
    t_dense = time_e2e(nb.RUN_DENSE_COPY)
    e2e["variants"] = {
        "host_prezeroed": {"value": world * Qe / t_pre, "d2h_bytes_per_step": world * (gs_pre["dma_bytes"] + gs_pre["thin_bytes"]),
                           "host_zero_filled_bytes_per_step": world * gs_pre["zeroed_bytes"]},
        "dense_copy": {"value": world * Qe / t_dense, "d2h_bytes_per_step": world * d2h}}
    eb.close()
    pin.close()

    # packed records end to end: nnsdp_batch_set_inputs + nnsdp_batch_run_packed with pinned host buffers; the D2H moves
    # the always-written part of every record plus the DIAG cells a query carries, nothing is filled on the host
    Qp = min(Q, args.e2e_packed_queries)
    epb = nb.Batch(net, beta, Qcap=Qp, ring=min(pring, Qp), packed=True)
    ppin = nb.PinnedBuffer(Qp * epb.per_query)
    ppresent = np.zeros((Qp, epb.ncells), dtype=np.uint8)
    psub = {k: (v[:Qp] if v.shape[0] == Q and Q > 1 else v) for k, v in inp.items()}
    pebatch = numeric_batch(nb, name, psub)
    ph2d = sum(int(np.asarray(v).nbytes) for v in psub.values())

    def e2e_packed_step(flags=0):
        epb.set_inputs(pebatch, Q=Qp)
        epb.run_packed(ppin.array, ppresent, flags=flags)

    e2e_step = e2e_packed_step
    tp = time_e2e(0)
    pst2 = epb.packed_stats()
    e2e_dense = e2e
    e2e = {"value": world * Qp / tp, "unit": "queries/s", "format": "packed", "h2d_bytes_per_step": world * ph2d,
           "d2h_bytes_per_step": world * pst2["d2h_bytes"], "queries_per_step": world * Qp, "ms_per_step": 1e3 * tp,
           "host_result_bytes_per_step": world * pst2["d2h_bytes"],
           "d2h_gbs": world * pst2["d2h_bytes"] / tp / 1e9,
           "note": "nnsdp_batch_set_inputs + nnsdp_batch_run_packed with pinned host buffers on every rank concurrently "
                   "(bounded sample of the workload): packed records = the block-sparse upper triangle of Z, from which "
                   "every Z[C_k, C_k] is a set of views (bit-identical to the dense blocks); `dense` = the same through "
                   "nnsdp_batch_run with complete dense blocks in host memory",
           "dense": e2e_dense}
    epb.close()
    ppin.close()

    extras, crown = None, None
    if rank == 0 and world == 1 and name == DEFAULT_WORKLOAD and not args.no_extras:
        crown = crown_line(nb, torch, net, name, beta, inp, Q=min(Q, args.crown_queries), steps=args.steps)
        extras = [quick_measure(nb, torch, n, peak, steps=args.steps) for n in EXTRA_WORKLOADS]
    line = None
    if rank == 0:
        # ---- CPU baseline on this box's host cores (bounded sample)
        cpu = None
        if not args.no_cpu and world == 1:
            pool = CpuPool(name)
            nq_cpu = (2 if w["W"] >= 500 else 32) * pool.procs
            dt = pool.run(nq_cpu)
            pool.close()
            cpu = {"value": nq_cpu / dt, "unit": "queries/s", "cores": pool.procs, "kind": "port",
                   "sample": f"{nq_cpu} queries of the same workload in {dt:.1f} s, numpy closed-form oracle, "
                             f"{pool.procs} worker processes x {pool.blas_threads} BLAS thread (verified with threadpoolctl in the "
                             f"workers) on {os.cpu_count()} host cores"}
        launches_per_step = sum(stage[k][1] for k in stage) / max(args.steps, 1)
        line = {
            "metric": "queries/sec (clique LMI blocks assembled: value * cliques_per_query)",
            "value": value, "unit": "queries/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": name, "output_format": "dense clique blocks (value); packed records in `packed` and `e2e`", "xdims": f"[2, {w['W']} x {w['D']}, 2]", "beta": beta,
                       "queries_per_gpu_per_step": Q, "cliques_per_query": sz["ncliques"],
                       "blocks_per_sec": value * sz["ncliques"],
                       "dense_block_bytes_per_query": 8 * sz["sum_ck_sq"], "ring_slots": ring,
                       "l2": "outputs (ring) and inputs are far larger than the 126 MB L2",
                       "gram_contractions_per_step": ncon, "gram_active_rows_per_step": nact,
                       "radius_scale": args.radius_scale,
                       "parallelism": f"queries sharded over {world} GPU(s), no collective"},
            "roofline": roofline, "packed": packed, "crown_bounds": crown, "other_workloads": extras,
            "cpu_baseline": cpu, "e2e": e2e, "clocks": clocks,
            "gpu_launches": int(round(launches_per_step * args.steps)),
            "stage_ms_per_step": {k: stage[k][0] / args.steps for k in stage},
        }
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if line is not None and world > 1:
        line["ctx_multi_device"] = multi_device_context_check(nb, world)
    if line is not None:
        print(json.dumps(line), flush=True)


def multi_device_context_check(nb, ndev):
    """The second multi-GPU form of SURVEY.md 8e on the box's GPUs: ONE nnsdp_ctx over `ndev` devices (what a Julia
    process would hold) shards the queries of a one-shot call over them; the gathered result is compared with the
    single-device result, for the dense blocks and for the packed records.  Which bounds / affine kernels run depends
    on how many queries a device gets (<= 8, 9..32, more: different summation orders), so bit-identity is asserted on
    a net whose kernels do not depend on the query count (widths <= 256) and the wide net is compared to rounding."""
    out = {"devices": ndev}
    try:
        rng = np.random.default_rng(42)
        for tag, xdims in (("narrow", [2, 200, 180, 2]), ("wide", [2, 300, 270, 2])):
            beta, nq = 2, 2 * ndev + 1
            Ms = [0.1 * rng.standard_normal((xdims[k + 1], xdims[k] + 1)) for k in range(len(xdims) - 1)]
            acdim = sum(xdims[1:-1])
            lamdim = sum(range(acdim - beta, acdim + 1))
            c = rng.uniform(0.5, 1.5, (nq, 2))
            r = rng.uniform(0.0, 0.05, (nq, 1))
            A = rng.standard_normal((nq, 5, 5))
            b = nb.NumericBatch(x1min=c - r, x1max=c + r, gamma_in=rng.random((nq, 2)), gamma_bnd=rng.random((nq, acdim)),
                                gamma_sec=rng.random((nq, lamdim + 2 * acdim)), out_kind=nb.OUT_SAFETY,
                                out_S=A + np.transpose(A, (0, 2, 1)))
            c1 = nb.Context([0])
            one = nb.assemble_blocks(nb.Net(c1, xdims, Ms), beta, b)
            cn = nb.Context(list(range(ndev)))
            netn = nb.Net(cn, xdims, Ms)
            many = nb.assemble_blocks(netn, beta, b)
            rec, present, _ = nb.assemble_packed(netn, beta, b)
            unp = np.stack([nb.packed_unpack(xdims, beta, rec[i], present[i]) for i in range(nq)])
            scale = np.abs(one).max()
            out[tag] = {"queries": nq, "bit_identical": bool(np.array_equal(one, many)),
                        "packed_equals_dense_of_the_same_context": bool(np.array_equal(unp, many)),
                        "max_abs_diff_over_scale": float(np.abs(one - many).max() / scale)}
        out["bit_identical"] = out["narrow"]["bit_identical"] and out["narrow"]["packed_equals_dense_of_the_same_context"]
        out["wide_equal_to_rounding"] = out["wide"]["max_abs_diff_over_scale"] <= 1e-12
    except Exception as e:  # reported, never fatal for the bench line
        out.update({"bit_identical": False, "error": repr(e)[:300]})
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=DEFAULT_WORKLOAD, choices=sorted(WORKLOADS))
    ap.add_argument("--queries", type=int, default=None, help="override queries per GPU per step")
    ap.add_argument("--e2e-queries", type=int, default=8)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-e2e", action="store_true", help="developer runs: device-timed figures only")
    ap.add_argument("--no-extras", action="store_true", help="skip the CROWN-bounds line and the other BASELINE configs")
    ap.add_argument("--crown-queries", type=int, default=16)
    ap.add_argument("--ring", type=int, default=None, help="override the number of device-resident output slots")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: --queries per GPU (default); strong: --queries in total, sharded over the ranks")
    ap.add_argument("--e2e-packed-queries", type=int, default=24)
    ap.add_argument("--radius-scale", type=float, default=1.0,
                    help="scale of the input-box radii (default 1 = BASELINE config 5); small values make every ReLU stable (Gram-heavy)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="save what the last timed step computed as DIR/<name>.npy (see the module docstring)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs saves the outputs of the GPU arm (--impl ours)")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
