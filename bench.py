#!/usr/bin/env python
"""bench.py -- headline benchmark of the splpak fit-and-evaluate hot path on B200.

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K --warmup W   # CPU restatement of the reference

Workload (BASELINE.json configs[2], the config the metric is quoted on; it fits one GPU):
  3-D splcw weighted fit of 1e8 scattered points on 24^3 nodes (xtrap = 1) + splfe at 1e9 points,
  real64, PER GPU ("weak" scaling: every rank holds its own 1e8-point / 1e9-query shard of one global
  problem; the partial normal equations are summed with ONE NCCL all-reduce before the replicated solve).
A step = one fit (assembly + all-reduce + constraints + Cholesky solve) followed by one evaluation
pass, inputs resident in HBM.  Inputs (4 GB + 24 GB per GPU) are far larger than the 126 MB L2, so no
L2 flush is needed between steps.

One JSON line on stdout (rank 0).  `value` = data points fitted per second (whole job), `evals_per_s`
= spline evaluations per second; `e2e` = the same metric through the host-array C-ABI entry points
(pinned host buffers, H2D/D2H inside the timed region).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

NDIM = 3
NODES = [24, 24, 24]
XMIN = [0.0, 0.0, 0.0]
XMAX = [1.0, 1.0, 1.0]
XTRAP = 1.0
NCOL = 24 ** 3
WORKLOAD = "cfg3: 3-D splcw weighted fit, 1e8 points/GPU on 24^3 nodes (xtrap=1) + splfe at 1e9 points/GPU, real64"
# ONE metric string for both arms (the driver compares them literally before it computes the ratio)
METRIC = "data points fitted/s (3-D splcw, 24^3 nodes; points / fit_ms)"


def load_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the two dominant kernels, from the committed
    `ncu --set full` capture of this same command (profiles/r01_traffic.json, written by scripts/gpu_profile.sh)."""
    for name in ("r02_traffic.json", "r01_traffic.json"):
        try:
            return json.load(open(os.path.join(ROOT, "profiles", name)))
        except Exception:
            continue
    return {}


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20", "-i",
                 str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [t.strip() for t in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for name, val in zip(names, f[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# -------------------------------------------------------------------------------------------------
# CPU baseline: the oracle (C restatement of the reference), steady-state sample
# -------------------------------------------------------------------------------------------------
def cpu_fit_sample(m_rows, seed=42):
    """Seconds for m_rows real cfg3 data rows entering a FULL 13,824-column triangle through the
    restated splcw row loop + suprls Householder update (the reference's steady state: ~2*ncol^2 flops
    per point).  The fill phase (first ncol rows, ~1.8e12 flops) is excluded -- it would take tens of
    minutes on one core -- so this is an optimistic per-point cost for the reference."""
    from oracle import Oracle
    from splpak_b200 import synth

    o = Oracle()
    x, y, w = synth.points_numpy(NDIM, m_rows, start=0, seed=seed)
    return o.suprls_steady_sample(NDIM, x, y, w, m_rows, XMIN, XMAX, NODES)


def cpu_eval_sample(nq, seed=43):
    from oracle import Oracle
    from splpak_b200 import synth

    o = Oracle()
    q = synth.queries_numpy(NDIM, nq, seed=seed)
    coef = np.random.default_rng(0).standard_normal(NCOL)
    t0 = time.perf_counter()
    o.evaluate_batch(NDIM, q, coef, XMIN, XMAX, NODES)
    return time.perf_counter() - t0


def cpu_matched_sample(n_sample, npts_total, seed=42):
    """BASELINE.md section 3's optional 'algorithm-matched' CPU row: the GPU path's ALGORITHM (sparse normal equations by
    window + LAPACK band Cholesky, oracle/cpu_matched.py) on the host's cores via numpy/BLAS/LAPACK.  Assembly is
    timed on n_sample cfg3 points and extrapolated linearly to npts_total; the solve is timed in full."""
    from oracle import cpu_matched
    from splpak_b200 import synth

    x, y, w = synth.points_numpy(NDIM, n_sample, start=0, seed=seed)
    _, t_asm, t_solve = cpu_matched.fit(NDIM, x, y, w, XMIN, XMAX, NODES)
    total = t_asm * (npts_total / n_sample) + t_solve
    return {"value": npts_total / total, "unit": "points/s", "cores": os.cpu_count(), "kind": "port (algorithm-matched)",
            "assembly_s_sample": t_asm, "solve_s": t_solve,
            "sample": f"sparse normal equations + scipy.linalg.cholesky_banded: assembly of {n_sample} cfg3 points "
                      f"({t_asm:.2f} s, extrapolated linearly to {npts_total}) + full 13,824 x 1,803 band solve ({t_solve:.2f} s); "
                      f"numpy/BLAS/LAPACK threads on {os.cpu_count()} cores"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    from oracle import build_oracle

    build_oracle()
    m = args.cpu_rows
    for _ in range(args.warmup):
        cpu_fit_sample(m)
    ts = []
    t_wall0 = time.perf_counter()
    for _ in range(args.steps):
        ts.append(cpu_fit_sample(m))
    t_wall = time.perf_counter() - t_wall0
    sec = sum(ts) / len(ts)
    value = m / sec
    te = cpu_eval_sample(200_000)
    sample = (f"{m} cfg3 data rows per step entering a full {NCOL}-column triangle (steady-state suprls "
              f"Householder update, fill phase excluded; one full batch of the reference is ~{NCOL // 2} rows = 2.6e12 flops "
              f"= ~10 min on one core, so a bounded sample of rows is timed; the per-row cost of an {m}-row batch is "
              f"(1 + 1/{m}) x that of a full batch); 1 thread, the reference is serial")
    line = {
        "impl": "reference", "metric": METRIC, "value": value,
        "unit": "points/s", "evals_per_s": 200_000 / te, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * sec, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": WORKLOAD, "reference_arm": "C restatement of src/splpak.F90 (oracle/); no Fortran "
                   "compiler exists in the image so the reference itself cannot be built"},
        "cpu_baseline": {"value": value, "unit": "points/s", "cores": 1, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "points/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "wall_s": t_wall,
    }
    print(json.dumps(line), flush=True)
    return 0


# -------------------------------------------------------------------------------------------------
# this repo's CUDA path
# -------------------------------------------------------------------------------------------------
DUMP_VALUES = 1 << 21          # sampled evaluations: 16 MB of values + 16 MB of indices


def dump_outputs(dirname, dcoef, out):
    """Write what a caller of the timed path receives from its last step, so that two builds can be compared
    output for output on the same seeded inputs: coef.npy (all coefficients), values.npy (the evaluated values at a
    fixed, seeded sample of the queries, or all of them when there are at most DUMP_VALUES) and values_index.npy
    (the query index of each sampled value, as float64).  The inputs are seeded, but the default fit adds in a
    run-dependent order, so two runs differ in the last digits (about 1e-12 relative in the coefficients) unless
    SPLPAK_B200_DETERMINISTIC=1."""
    import torch

    os.makedirs(dirname, exist_ok=True)
    nq = out.numel()
    if nq <= DUMP_VALUES:
        idx = np.arange(nq)
    else:
        idx = np.sort(np.random.default_rng(0).choice(nq, DUMP_VALUES, replace=False))
    values = out[torch.from_numpy(idx).to(out.device)]
    np.save(os.path.join(dirname, "coef.npy"), dcoef.cpu().numpy())
    np.save(os.path.join(dirname, "values.npy"), values.cpu().numpy())
    np.save(os.path.join(dirname, "values_index.npy"), idx.astype(np.float64))


def run_ours(args):
    import torch
    import torch.distributed as dist

    import splpak_b200 as sp
    from splpak_b200 import synth

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world == 1:
        sp.build()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
        if rank == 0:
            sp.build()                       # one builder; the others wait (no-op when the .so is current)
        dist.barrier()

    def barrier():
        if world > 1:
            dist.barrier()

    def reduce_max(v):
        if world == 1:
            return v
        t = torch.tensor([v], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def reduce_sum(v):
        if world == 1:
            return v
        t = torch.tensor([v], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    npts, nq = args.npoints, args.nqueries
    hbm_peak, peak_src = load_peaks()

    # ---- synthetic shard of this rank (counter-based: global point index = rank*npts + i) ----
    x, y, w = synth.points_torch(NDIM, npts, start=rank * npts, seed=42, device=dev)
    q = synth.queries_torch(NDIM, nq, start=rank * nq, seed=43, device=dev)
    out = torch.empty(nq, dtype=torch.float64, device=dev)
    dcoef = torch.zeros(NCOL, dtype=torch.float64, device=dev)
    torch.cuda.synchronize()

    h = sp.FitHandle(NDIM, XMIN, XMAX, NODES, XTRAP)
    if h.ierror != 0:
        raise SystemExit(f"fit_create failed: {h.ierror}")
    stream = torch.cuda.ExternalStream(h.stream(), device=dev)
    part = h.partial_tensor()

    def fit_step():
        h.reset()
        rc = h.add_points_device(x, NDIM, y, w, npts, True)
        if rc != 0:
            raise SystemExit(f"add_points_device failed: {rc}")
        if world > 1:
            dist.all_reduce(part)            # one NCCL all-reduce (sum) of [G | g | histogram | totals]
        ierr = h.compute_device(dcoef)
        if ierr != 0:
            raise SystemExit(f"compute failed: ierror {ierr}")

    def eval_step():
        ierr = sp.eval_batch_device(NDIM, q, NDIM, nq, dcoef, XMIN, XMAX, NODES, out, stream=stream)
        if ierr != 0:
            raise SystemExit(f"eval failed: ierror {ierr}")

    with torch.cuda.stream(stream):
        for _ in range(args.warmup):
            fit_step()
            eval_step()
        torch.cuda.synchronize()
        barrier()
        torch.cuda.synchronize()
        sampler = ClockSampler(local)
        if rank == 0:
            sampler.start()
        launches0 = sp.total_launches()
        evs = []
        stage_ms = {}
        t_wall0 = time.perf_counter()
        for _ in range(args.steps):
            e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
            e0.record(stream)
            fit_step()
            e1.record(stream)
            eval_step()
            e2.record(stream)
            evs.append((e0, e1, e2))
            for k, v in h.timings().items():
                stage_ms[k] = stage_ms.get(k, 0.0) + v
        torch.cuda.synchronize()
        barrier()
        torch.cuda.synchronize()
        t_wall = time.perf_counter() - t_wall0
        launches = sp.total_launches() - launches0
        clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, dcoef, out)      # before the sub-records below overwrite dcoef and out

    fit_all = [a.elapsed_time(b) for a, b, _ in evs]
    eval_all = [b.elapsed_time(c) for _, b, c in evs]
    fit_ms = reduce_max(sum(fit_all) / args.steps)          # contract: total over EXACTLY K steps / K, max over ranks
    eval_ms = reduce_max(sum(eval_all) / args.steps)
    fit_med, eval_med = reduce_max(statistics.median(fit_all)), reduce_max(statistics.median(eval_all))
    fit_min, eval_min = reduce_max(min(fit_all)), reduce_max(min(eval_all))
    stage_ms = {k: reduce_max(v / args.steps) for k, v in stage_ms.items()}
    launches_total = reduce_sum(float(launches))
    checksum = float(out[:: max(1, nq // 1000)].sum().item())

    # ---- the north star's TARGET JOB at N > 1: ONE problem of npts points + nq queries in total, sharded over the
    #      ranks (strong scaling).  Reported as a sub-record; the contract line above stays the weak-scaling one. ----
    strong = None
    if world > 1:
        ns, qs = npts // world, nq // world
        xs, ys, wsd, qsd, outs = x[:ns], y[:ns], w[:ns], q[:qs], out[:qs]

        def strong_fit():
            h.reset()
            rc = h.add_points_device(xs, NDIM, ys, wsd, ns, True)
            if rc != 0:
                raise SystemExit(f"add_points_device failed: {rc}")
            dist.all_reduce(part)
            ierr = h.compute_device(dcoef)
            if ierr != 0:
                raise SystemExit(f"compute failed: ierror {ierr}")

        with torch.cuda.stream(stream):
            for _ in range(3):
                strong_fit()
                sp.eval_batch_device(NDIM, qsd, NDIM, qs, dcoef, XMIN, XMAX, NODES, outs, stream=stream)
            torch.cuda.synchronize()
            barrier()
            torch.cuda.synchronize()
            sev = []
            ssteps = max(3, min(args.steps, 10))
            for _ in range(ssteps):
                e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
                e0.record(stream)
                strong_fit()
                e1.record(stream)
                sp.eval_batch_device(NDIM, qsd, NDIM, qs, dcoef, XMIN, XMAX, NODES, outs, stream=stream)
                e2.record(stream)
                sev.append((e0, e1, e2))
                sstages = h.timings()
            torch.cuda.synchronize()
            barrier()
            torch.cuda.synchronize()
        sfit = reduce_max(sum(a.elapsed_time(b) for a, b, _ in sev) / ssteps)
        sevl = reduce_max(sum(b.elapsed_time(c) for _, b, c in sev) / ssteps)
        strong = {"scaling": "strong", "points_total": ns * world, "queries_total": qs * world, "steps": ssteps,
                  "fit_ms": sfit, "eval_ms": sevl, "ms_per_step": sfit + sevl,
                  "value": ns * world / (sfit * 1e-3), "unit": "points/s", "evals_per_s": qs * world / (sevl * 1e-3),
                  "stages_ms_rank0_last": sstages,
                  "note": "the north star's target job (1e8 points + 1e9 evaluations IN TOTAL) sharded over the ranks; "
                          "the solve is replicated, so the fit's strong scaling is bounded by it"}

    # ---- end to end through the host-array C ABI (host buffers, copies inside the timed region): once with PINNED
    #      buffers (torch pin_memory) and once with plain PAGEABLE numpy arrays, which is what a Fortran caller's
    #      arrays are (src/splpak.F90:537-559); the library stages those through its own pinned ring ----
    nq_e2e = min(nq, args.e2e_queries)
    e2e = None
    e2e_pageable = None
    if not args.no_e2e:
        import ctypes as C
        lib = sp.load()

        def e2e_leg(xa, ya, wa, qa, out_ptr, label):
            def e2e_step():
                h.reset()
                rc = h.add_points(xa, ya, wa, weighted=True)              # chunked H2D overlapped with the kernels
                if rc != 0:
                    raise SystemExit(f"add_points failed: {rc}")
                if world > 1:
                    with torch.cuda.stream(stream):                       # the handle's own stream: ordered, no host sync
                        dist.all_reduce(part)
                coef, ierr = h.compute()                                   # D2H of the coefficients
                if ierr != 0:
                    raise SystemExit(f"compute failed: {ierr}")
                t_mid = time.perf_counter()
                ie = C.c_int(0)
                mn = (C.c_double * 3)(*XMIN); mx = (C.c_double * 3)(*XMAX); no = (C.c_int * 3)(*NODES)
                lib.splpak_b200_eval(NDIM, C.c_void_p(qa.ctypes.data), NDIM, nq_e2e, None,
                                     C.c_void_p(coef.ctypes.data), mn, mx, no, C.c_void_p(out_ptr), C.byref(ie))
                if ie.value != 0:
                    raise SystemExit(f"eval failed: {ie.value}")
                return t_mid

            e2e_step()                                                     # warm-up
            barrier()
            fit_s, eval_s = [], []
            for _ in range(args.e2e_steps):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                t_mid = e2e_step()
                t1 = time.perf_counter()
                fit_s.append(t_mid - t0)
                eval_s.append(t1 - t_mid)
            print(f"[bench rank {rank}] e2e ({label}) per-step fit {[round(1e3 * v, 1) for v in fit_s]} ms, "
                  f"eval {[round(1e3 * v, 1) for v in eval_s]} ms", file=sys.stderr, flush=True)
            e2e_fit = reduce_max(sum(fit_s) / len(fit_s))
            e2e_eval = reduce_max(sum(eval_s) / len(eval_s))
            return {
                "value": world * npts / e2e_fit, "unit": "points/s",
                "evals_per_s": world * nq_e2e / e2e_eval,
                "h2d_bytes_per_step": int(npts * (NDIM + 2) * 8 + nq_e2e * NDIM * 8 + NCOL * 8),
                "d2h_bytes_per_step": int(NCOL * 8 + nq_e2e * 8),
                "fit_ms": 1e3 * e2e_fit, "eval_ms": 1e3 * e2e_eval, "steps": args.e2e_steps, "host_memory": label,
                "note": f"host API: FitHandle.add_points+compute on {npts} {label} host points, splpak_b200_eval on "
                        f"{nq_e2e} {label} host queries (bounded sample of the {nq} device-resident queries)",
            }

        hx = torch.empty((npts, NDIM), dtype=torch.float64, pin_memory=True)
        hy = torch.empty(npts, dtype=torch.float64, pin_memory=True)
        hw = torch.empty(npts, dtype=torch.float64, pin_memory=True)
        hq = torch.empty((nq_e2e, NDIM), dtype=torch.float64, pin_memory=True)
        hx.copy_(x); hy.copy_(y); hw.copy_(w); hq.copy_(q[:nq_e2e])
        torch.cuda.synchronize()
        hout = torch.empty(nq_e2e, dtype=torch.float64, pin_memory=True)
        # ceiling of every e2e number: pinned host -> device bandwidth with ALL ranks copying at once (at N = 8 the
        # eight ranks share one socket's memory controllers and PCIe root: topology "CPU Affinity 0-31, NUMA 0")
        barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(2):
            x.copy_(hx, non_blocking=True)
        torch.cuda.synchronize()
        h2d_s = reduce_max(time.perf_counter() - t0)
        h2d_gbs = world * 2 * hx.numel() * 8 / h2d_s / 1e9
        e2e = e2e_leg(hx.numpy(), hy.numpy(), hw.numpy(), hq.numpy(), hout.data_ptr(), "pinned")
        e2e["h2d_gbs_all_ranks_concurrent"] = h2d_gbs
        e2e["fit_ms_at_that_bandwidth"] = 1e3 * world * npts * (NDIM + 2) * 8 / (h2d_gbs * 1e9)
        if not args.no_pageable:
            px, py, pw, pq = (np.array(t.numpy(), copy=True) for t in (hx, hy, hw, hq))     # ordinary malloc'ed arrays
            pout = np.empty(nq_e2e, dtype=np.float64)
            del hx, hy, hw, hq, hout
            e2e_pageable = e2e_leg(px, py, pw, pq, pout.ctypes.data, "pageable")
            del px, py, pw, pq, pout
        else:
            del hx, hy, hw, hq, hout

    # ---- the same 1e9 evaluations on a regular 1000^3 output grid (fit-then-grid, the upstream use case) ----
    grid = None
    try:
        ng = 1000 if nq >= 1_000_000_000 else max(8, int(round(nq ** (1.0 / 3.0))))
        ax = torch.linspace(0.0, 1.0, ng, dtype=torch.float64, device=dev)
        d_axes = torch.cat([ax, ax, ax])
        gout = out[: ng ** 3]
        with torch.cuda.stream(stream):
            best = None
            for rep in range(4):
                g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                g0.record(stream)
                ierr = sp.eval_grid_device(NDIM, d_axes, [ng] * 3, dcoef, XMIN, XMAX, NODES, gout, stream=stream)
                g1.record(stream)
                torch.cuda.synchronize()
                if ierr != 0:
                    raise RuntimeError(f"eval_grid failed: {ierr}")
                if rep:
                    t = g0.elapsed_time(g1)
                    best = t if best is None else min(best, t)
        gms = reduce_max(best)
        grid = {"grid": [ng] * 3, "ms": gms, "points_per_s": world * ng ** 3 / (gms * 1e-3),
                "hbm_written_gbs": ng ** 3 * 8 / (gms * 1e-3) / 1e9, "hbm_frac": ng ** 3 * 8 / (gms * 1e-3) / 1e9 / hbm_peak,
                "note": "splpak_b200_eval_grid_device: separable contraction, bit-identical to point-wise splfe; "
                        "best of 3, outside the timed steps"}
    except Exception as exc:                                    # reported, never fatal for the contract line
        grid = {"error": str(exc)}

    h.destroy()

    if rank == 0:
        # ---- rooflines ----
        try:
            dfma_tf, dmma_tf, copy_gbs = sp.measure_peaks()
        except Exception:
            dfma_tf = dmma_tf = copy_gbs = None
        acc_ms = stage_ms.get("accumulate", 0.0)
        eval_bytes = nq * (NDIM + 1) * 8
        asm_bytes = npts * (NDIM + 2) * 8
        traffic = load_traffic()

        def traffic_for(kernel, units):
            t = traffic.get(kernel)
            # the capture is per launch at t["units"] units (points or queries); DRAM traffic is linear in them
            return None if not t else t["dram_bytes"] * (units / t["units"])

        eval_roof = {"kernel": "spl_eval_regroup_kernel<3,1> (chosen by spl_eval_probe_kernel for scattered queries)",
                     "bound": "hbm", "achieved": eval_bytes / (eval_ms * 1e-3) / 1e9,
                     "peak": hbm_peak, "unit": "GB/s",
                     "traffic": traffic_for("spl_eval_regroup_kernel<3>", nq) or traffic_for("spl_eval_kernel<3>", nq),
                     "algorithmic_bytes": eval_bytes,
                     "note": "uniform-random 3-D real64 queries, uniform (phantom-node) form of the basis: conflict-free "
                             "shared-memory gathers through warp-private bank-class FIFOs.  NOT HBM-bound: the kernel "
                             "saturates the shared-memory crossbar (ncu l1tex data pipe 95.6 % of peak: 5.84 shared "
                             "wavefronts per query -- 4.0 are the 64 coefficients x 8 B at 128 B/clk/SM, i.e. a 13.8 ms "
                             "floor per 1e9 queries on 148 SMs -- plus FIFO traffic and 13 % idle lanes); FP64 pipe 33 %: "
                             "DESIGN.md 4.5, profiles/r02_eval_uniform.md",
                     "smem_crossbar": {"wavefronts_per_query_floor": 4.0, "wavefronts_per_query_measured": 5.84,
                                       "floor_ms_per_1e9": 13.8,
                                       "frac_of_floor": 13.8 / (eval_ms * 1e9 / nq) if eval_ms > 0 else None}}
        eval_roof["frac"] = eval_roof["achieved"] / hbm_peak
        # accumulate stage = spl_moments_kernel (+ the per-cell change of basis, ~2% of it).  It gathers the
        # cell-sorted points through the 4-byte permutation: on uniform-random data every gather of x / y / w pulls
        # its own 128-byte line, so the kernel moves ~390 B of DRAM traffic per point for 44 algorithmic bytes
        # (40 B point + 4 B permutation entry) and runs at the HBM roof on that TRAFFIC (DESIGN.md 4.3).
        # FP64: 9 DMMA.8x8x4 tiles per 4 points = 576 FMA per point executed (407 needed).
        asm_bytes = npts * ((NDIM + 2) * 8 + 4)
        acc_flops = npts * 2.0 * 576
        acc_traffic = traffic_for("spl_moments_kernel", npts)
        acc_roof = {"kernel": "spl_moments_kernel", "bound": "hbm (gather traffic)", "unit": "TFLOP/s",
                    "achieved": acc_flops / (acc_ms * 1e-3) / 1e12 if acc_ms > 0 else None,
                    "peak": dmma_tf, "peak_source": "DMMA micro-benchmark in this run (splpak_b200_measure_peaks)",
                    "traffic": acc_traffic, "algorithmic_bytes": asm_bytes,
                    "hbm_achieved_gbs": asm_bytes / (acc_ms * 1e-3) / 1e9 if acc_ms > 0 else None,
                    "hbm_frac": (asm_bytes / (acc_ms * 1e-3) / 1e9) / hbm_peak if acc_ms > 0 else None,
                    "traffic_gbs": acc_traffic / (acc_ms * 1e-3) / 1e9 if (acc_ms > 0 and acc_traffic) else None,
                    "traffic_frac": (acc_traffic / (acc_ms * 1e-3) / 1e9) / hbm_peak if (acc_ms > 0 and acc_traffic) else None}
        if acc_roof["achieved"] and dmma_tf:
            acc_roof["frac"] = acc_roof["achieved"] / dmma_tf
        dominant = eval_roof if eval_ms >= acc_ms else {
            "kernel": acc_roof["kernel"], "bound": "hbm", "achieved": acc_roof["hbm_achieved_gbs"], "peak": hbm_peak,
            "unit": "GB/s", "frac": acc_roof["hbm_frac"], "traffic": acc_roof["traffic"],
            "note": "bound by the DRAM traffic of the permutation gathers; see roofline_fp64.traffic_frac"}
        dominant = dict(dominant)
        dominant["peak_source"] = peak_src

        cpu = None
        if world == 1 and not args.no_cpu:
            sec = cpu_fit_sample(args.cpu_rows)
            te = cpu_eval_sample(1_000_000)
            cpu = {"value": args.cpu_rows / sec, "unit": "points/s", "cores": 1, "kind": "port",
                   "evals_per_s": 1_000_000 / te,
                   "sample": f"{args.cpu_rows} cfg3 data rows entering a full {NCOL}-column triangle through the "
                             f"restated splcw row loop + suprls Householder update ({sec:.2f} s; steady state, fill "
                             f"phase excluded); eval: 1e6 scalar splfe calls ({te:.2f} s)"}

        cpu_matched = None
        if world == 1 and not args.no_cpu:
            try:
                cpu_matched = cpu_matched_sample(args.cpu_matched_points, npts)
            except Exception as exc:                                # optional row: reported, never fatal
                cpu_matched = {"error": str(exc)}

        line = {
            "metric": METRIC,
            "value": world * npts / (fit_ms * 1e-3), "unit": "points/s",
            "evals_per_s": world * nq / (eval_ms * 1e-3),
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": fit_ms + eval_ms, "fit_ms": fit_ms, "eval_ms": eval_ms,
            # identical launches on these shared boxes show sporadic 1.5-5x slowdowns at constant clocks
            # (profiles/r01_eval_jitter.md); the per-step median / minimum are given beside the mean
            "per_step_ms": {"fit_median": fit_med, "fit_min": fit_min, "eval_median": eval_med, "eval_min": eval_min,
                            "eval_all_rank0": [round(v, 2) for v in eval_all]},
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": WORKLOAD, "ndim": NDIM, "nodes": NODES, "points_per_gpu": npts,
                       "queries_per_gpu": nq, "e2e_queries_per_gpu": nq_e2e, "xtrap": XTRAP, "query_order": "uniform random",
                       "l2": "inputs (4 GB points + 24 GB queries per GPU) exceed the 126 MB L2; no flush needed",
                       "parallelism": f"point-sharded x{world}, one all-reduce, replicated solve"},
            "stages_ms": stage_ms,
            "roofline": dominant, "roofline_eval": eval_roof, "roofline_fp64": acc_roof,
            "fp64_peaks": {"dfma_tflops": dfma_tf, "dmma_tflops": dmma_tf, "copy_gbs": copy_gbs},
            "eval_grid": grid,
            "cpu_baseline": cpu, "cpu_baseline_algorithm_matched": cpu_matched,
            "e2e": e2e, "e2e_pageable": e2e_pageable, "strong": strong, "gpu_launches": int(launches_total),
            "clocks": clocks, "checksum": checksum, "wall_s": t_wall,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--npoints", type=int, default=100_000_000, help="data points per GPU (cfg3: 1e8)")
    ap.add_argument("--nqueries", type=int, default=1_000_000_000, help="evaluation points per GPU (cfg3: 1e9)")
    ap.add_argument("--e2e-queries", type=int, default=100_000_000)
    ap.add_argument("--e2e-steps", type=int, default=2)
    ap.add_argument("--cpu-rows", type=int, default=16)
    ap.add_argument("--cpu-matched-points", type=int, default=1_000_000)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-pageable", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write rank 0's coefficients and a seeded sample of its evaluated values from the last timed "
                         "step to DIR/*.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the CUDA path's results; it does not apply to --impl reference")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3                       # timing rule: W >= 3
    if args.impl == "reference":
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
