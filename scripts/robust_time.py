"""Cost of the robust fit (splpak_b200_fit_robust_device), one GPU.

For cfg3 (3-D, 24^3 nodes, 1e8 points) and cfg4 (4-D, 12^4 nodes, 1e7 points), weighted, xtrap = 1, device-resident
points (splpak_b200.synth.points_torch) with 5 % gross outliers (+-50 x the noise), bisquare, tol = 1e-6:
  * the whole call (host clock around it; it ends in a device synchronisation), its iteration count, and the time per
    iteration, (call - plain fit) / iterations, against add_points_device + fit_compute_device of the same points;
  * a per-kernel split of one call from torch.profiler, in a separate pass (kernel names grouped by prefix).
The card name, power limit and clocks are read in the same process.
usage: python scripts/robust_time.py [out.md] [reps] [scale]   (scale < 1 shrinks the point counts, for a dry run)
"""
import os
import statistics
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

import splpak_b200 as sp  # noqa: E402
from splpak_b200 import synth  # noqa: E402
from gcv_time import card  # noqa: E402

CONFIGS = [("cfg3", 3, [24, 24, 24], 1e8), ("cfg4", 4, [12, 12, 12, 12], 1e7)]
GROUPS = [("spl_robust_key", "keys and selection"), ("spl_robust_hist", "keys and selection"),
          ("spl_robust_select", "keys and selection"), ("spl_robust_weight", "reweighting"),
          ("spl_robust_stats", "reweighting"), ("spl_robust_change", "reweighting"),
          ("spl_eval", "evaluation"), ("spl_to_double", "evaluation"), ("spl_from_double", "evaluation"),
          ("spl_constraints", "constraints and penalty"), ("spl_penalty", "constraints and penalty"),
          ("spl_fx_", "binning and assembly"), ("spl_classify", "binning and assembly"), ("spl_scan", "binning and assembly"),
          ("spl_perm", "binning and assembly"), ("spl_part", "binning and assembly"), ("spl_items", "binning and assembly"),
          ("spl_hist", "binning and assembly"), ("spl_wmax", "binning and assembly"), ("spl_moments", "binning and assembly"),
          ("spl_cell", "binning and assembly"), ("spl_accumulate", "binning and assembly"),
          ("spl_segsort", "binning and assembly"), ("spl_residual", "refinement"), ("spl_axpy", "refinement")]


def group_of(name):
    for prefix, g in GROUPS:
        if prefix in name:
            return g
    if "emcpy" in name or "emset" in name:
        return "copies and memsets"
    return "factor and solve"


def main():
    path = sys.argv[1] if len(sys.argv) > 1 else "robust_time.md"
    reps = int(sys.argv[2]) if len(sys.argv) > 2 else 3
    scale = float(sys.argv[3]) if len(sys.argv) > 3 else 1.0
    info = card()
    print("card", info, flush=True)
    out = ["# Robust fit: cost per iteration", "",
           f"Measured on one GPU: `{info}` (name, power limit, current SM clock, max SM clock; read in the same run) with "
           f"`scripts/robust_time.py`: weighted synthetic points (`splpak_b200.synth.points_torch`), device-resident, "
           f"xtrap = 1, 5 % gross outliers of +-50 x the noise, bisquare, tol = 1e-6; one warm-up, then {reps} "
           f"repetitions alternating the plain fit and the robust call, median shown.", ""]
    for cfg, ndim, nodes, npts in CONFIGS:
        n = int(npts * scale)
        mn, mx = [0.0] * ndim, [1.0] * ndim
        x, y, w = synth.points_torch(ndim, n, seed=42)
        gen = torch.Generator(device="cuda")
        gen.manual_seed(5)
        bad = torch.rand(n, dtype=torch.float64, device="cuda", generator=gen) < 0.05
        y += bad * 50 * 0.03 * torch.sign(torch.randn(n, dtype=torch.float64, device="cuda", generator=gen))
        del bad
        ncol = int(torch.tensor(nodes).prod())
        coef = torch.empty(ncol, dtype=torch.float64, device="cuda")
        plain_ms, rob_ms, iters = [], [], None
        for rep in range(reps + 1):
            h = sp.FitHandle(ndim, mn, mx, nodes, 1.0)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            assert h.add_points_device(x, ndim, y, w, n) == 0
            assert h.compute_device(coef) == 0
            t1 = time.perf_counter()
            h.destroy()
            h = sp.FitHandle(ndim, mn, mx, nodes, 1.0)
            torch.cuda.synchronize()
            t2 = time.perf_counter()
            res, ierr = h.robust_fit_device(x, ndim, y, w, n, coef, psi="bisquare", max_iter=50, tol=1e-6)
            t3 = time.perf_counter()
            assert ierr == 0, (ierr, res)
            h.destroy()
            if rep:
                plain_ms.append(1e3 * (t1 - t0))
                rob_ms.append(1e3 * (t3 - t2))
                iters = res
        h = sp.FitHandle(ndim, mn, mx, nodes, 1.0)
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            res, ierr = h.robust_fit_device(x, ndim, y, w, n, coef, psi="bisquare", max_iter=50, tol=1e-6)
            torch.cuda.synchronize()
        h.destroy()
        split = {}
        for ev in prof.key_averages():
            dt = getattr(ev, "device_time_total", None)
            if dt is None:
                dt = ev.cuda_time_total
            if dt <= 0:
                continue
            g = group_of(ev.key)
            split[g] = split.get(g, 0.0) + dt / 1e3
        k = iters["iterations"]
        pm, rm = statistics.median(plain_ms), statistics.median(rob_ms)
        per_it = (rm - pm) / max(k, 1)
        print(cfg, pm, rm, iters, split, flush=True)
        out += [f"## {cfg}: {ndim}-D {nodes[0]}^{ndim} nodes (n = {ncol:,} columns), {n:.0e} points", "",
                f"* plain fit (`add_points_device` + `fit_compute_device`): {pm:.2f} ms; robust call: {rm:.2f} ms for "
                f"{k} iterations to tol = 1e-6 (converged {iters['converged']}, sigma {iters['sigma']:.4g}, "
                f"{iters['n_rejected']:,} points with u = 0); per iteration {per_it:.2f} ms.",
                f"* per iteration, from the profile below divided by {k} (the plain fit's kernels included once): "
                + ", ".join(f"{g} {ms / max(k, 1):.3f} ms" for g, ms in sorted(split.items(), key=lambda kv: -kv[1])), "",
                f"| kernels of one robust call ({k} iterations; torch.profiler) | ms |", "|---|---:|"]
        for g, ms in sorted(split.items(), key=lambda kv: -kv[1]):
            out.append(f"| {g} | {ms:.3f} |")
        out += [""]
        del x, y, w
        torch.cuda.empty_cache()
    text = "\n".join(out) + "\n"
    with open(path, "w") as f:
        f.write(text)
    print(text)


if __name__ == "__main__":
    main()
