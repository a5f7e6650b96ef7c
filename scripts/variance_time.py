"""Cost of the posterior variances (splpak_b200_fit_prepare_variance / _fit_variance_device) on one GPU.

For cfg3 (3-D, 24^3 nodes, 1e8 fit points) and cfg4 (4-D, 12^4 nodes, 1e7 fit points), weighted, xtrap = 1, curvature
penalty, device-resident points (splpak_b200.synth.points_torch):
  * prepare_variance with a score (the handle's lambda was not scored yet) and without one (smoothing_score of the same
    lambda just ran, so only the tables are built); host clock around the call, which ends in a synchronisation;
  * variance_device over nq queries (CUDA events on the handle's stream), random and raster order (a regular grid
    walked with dimension 1 fastest), nderiv 0 and one second derivative, against eval_device of the fitted spline on
    the same queries;
  * bytes per query (the window's table, the coordinates, the output) and the effective table bandwidth.
The card name, power limit and clocks are read in the same process.
usage: python scripts/variance_time.py [out.md] [reps] [scale]   (scale < 1 shrinks the point counts, for a dry run)
"""
import os
import statistics
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

import splpak_b200 as sp  # noqa: E402
from splpak_b200 import synth  # noqa: E402

# name, ndim, nodes, fit points, queries
CONFIGS = [("cfg3", 3, [24, 24, 24], 1e8, 1e8), ("cfg4", 4, [12, 12, 12, 12], 1e7, 1e7)]
HBM_TBS = 7.7          # data-sheet HBM3e bandwidth of one B200


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader",
                            "-i", "0"], capture_output=True, text=True, timeout=60).stdout.strip()
    except Exception as e:
        q = f"{torch.cuda.get_device_name(0)}, unknown ({e})"
    return q


def events_ms(stream, fn, reps):
    out = []
    for rep in range(reps + 1):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        rc = fn()
        b.record(stream)
        b.synchronize()
        assert rc == 0, rc
        if rep:
            out.append(a.elapsed_time(b))
    return statistics.median(out)


def raster(ndim, nq, lo=-0.05, hi=1.05):
    k = int(round(nq ** (1.0 / ndim)))
    ax = torch.linspace(lo, hi, k, dtype=torch.float64, device="cuda")
    grids = torch.meshgrid(*([ax] * ndim), indexing="ij")
    # dimension 1 fastest: the last meshgrid index varies fastest, so dimension d takes grid ndim - 1 - d
    return torch.stack([grids[ndim - 1 - d].reshape(-1) for d in range(ndim)], dim=1).contiguous()


def main():
    path = sys.argv[1] if len(sys.argv) > 1 else "variance_time.md"
    reps = int(sys.argv[2]) if len(sys.argv) > 2 else 5
    scale = float(sys.argv[3]) if len(sys.argv) > 3 else 1.0
    info = card()
    print("card", info, flush=True)
    out = ["# Posterior variances: cost of prepare_variance and variance_device", "",
           f"Measured on one GPU: `{info}` (name, power limit, current SM clock, max SM clock; read in the same run) with "
           f"`scripts/variance_time.py`: weighted synthetic fit points (`splpak_b200.synth.points_torch`), "
           f"device-resident, xtrap = 1, curvature penalty; one warm-up, then {reps} repetitions, median shown.  "
           f"Queries: uniform random in [-0.05, 1.05]^ndim, or a regular grid over the same box walked with dimension 1 "
           f"fastest (raster).  The HBM figure is the data-sheet {HBM_TBS} TB/s.", ""]
    for cfg, ndim, nodes, npts, nqf in CONFIGS:
        n, nq = int(npts * scale), int(nqf * scale)
        mn, mx = [0.0] * ndim, [1.0] * ndim
        x, y, w = synth.points_torch(ndim, n, seed=42)
        ncol = int(np.prod(nodes))
        nwin = int(np.prod([k - 3 for k in nodes]))
        ent = 10 ** ndim
        lam = 1e-3 * (n / ncol) * (1.0 / (nodes[0] - 1)) ** 3
        h = sp.FitHandle(ndim, mn, mx, nodes, 1.0)
        assert h.enable_gcv() == 0
        assert h.add_points_device(x, ndim, y, w, n) == 0
        h.synchronize()
        with_score, build_only = [], []
        for rep in range(reps + 1):
            lam_r = lam * (1.0 + 1e-3 * rep)                 # a lambda not scored yet: prepare scores once
            assert h.set_smoothing(lam_r, "curvature") == 0
            t0 = time.perf_counter()
            h.prepare_variance()
            t1 = time.perf_counter()
            h.smoothing_score(lam_r, "curvature")            # the same system: prepare only builds the tables
            t2 = time.perf_counter()
            h.prepare_variance()
            t3 = time.perf_counter()
            if rep:
                with_score.append(1e3 * (t1 - t0))
                build_only.append(1e3 * (t3 - t2))
        coef = torch.empty(ncol, dtype=torch.float64, device="cuda")
        c, ierr = h.compute()
        assert ierr == 0
        coef.copy_(torch.from_numpy(c))
        st = torch.cuda.ExternalStream(h.stream())
        qs = {"random": (torch.rand((nq, ndim), dtype=torch.float64, device="cuda",
                                    generator=torch.Generator(device="cuda").manual_seed(7)) * 1.1 - 0.05)}
        if ndim == 3:
            qs["raster"] = raster(ndim, nq)
        d_out = torch.empty(max(len(v) for v in qs.values()), dtype=torch.float64, device="cuda")
        rows = []
        nds = [None, [2] + [0] * (ndim - 1)]
        for order, qx in qs.items():
            m = len(qx)
            for nd in nds:
                tv = events_ms(st, lambda: h.variance_device(qx, ndim, m, d_out, nderiv=nd), reps)
                te = events_ms(st, lambda: sp.eval_batch_device(ndim, qx, ndim, m, coef, mn, mx, nodes, d_out, nderiv=nd,
                                                                stream=st), reps)
                tb = m * 8.0 * ent
                rows.append((order, m, "0" if nd is None else ",".join(map(str, nd)), tv, te, tb / (tv * 1e-3) / 1e12))
                print(cfg, rows[-1], flush=True)
        tbytes = 8.0 * ent * nwin
        qbytes = 8 * ent + 8 * ndim + 8
        out += [f"## {cfg}: {ndim}-D {nodes[0]}^{ndim} nodes ({ncol:,} columns, {nwin:,} windows), {n:.0e} fit points", "",
                f"* tables: {ent:,} doubles per window, {tbytes / 1e6:.0f} MB in all (L2: 126 MB).",
                f"* `prepare_variance` with its score: {statistics.median(with_score):.2f} ms; table build alone (the "
                f"selected inverse of the same lambda already held, as after `select_smoothing`): "
                f"{statistics.median(build_only):.2f} ms.  Host clock; both end in a synchronisation.",
                f"* bytes per query: {8 * ent:,} of table + {8 * ndim} of coordinates + 8 of output = {qbytes:,}.", "",
                "| queries | nq | nderiv | variance_device ms | eval_device ms | table bytes / time, TB/s | "
                "HBM bound (table bytes / 7.7 TB/s) ms |",
                "|---|---:|---|---:|---:|---:|---:|"]
        for order, m, nds_, tv, te, bw in rows:
            out.append(f"| {order} | {m:.0e} | {nds_} | {tv:.2f} | {te:.2f} | {bw:.1f} | "
                       f"{m * 8.0 * ent / (HBM_TBS * 1e12) * 1e3:.1f} |")
        out.append("")
        h.destroy()
        del x, y, w, qs, d_out
        torch.cuda.empty_cache()
    text = "\n".join(out) + "\n"
    with open(path, "w") as f:
        f.write(text)
    print(text)


if __name__ == "__main__":
    main()
