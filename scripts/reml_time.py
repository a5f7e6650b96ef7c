"""Cost of the REML score (splpak_b200_fit_reml_score / select_smoothing_reml) against the GCV score, one GPU.

For cfg3 (3-D, 24^3 nodes, 1e8 points) and cfg4 (4-D, 12^4 nodes, 1e7 points), weighted, xtrap = 1, device-resident
points (splpak_b200.synth.points_torch):
  * one reml_score, one smoothing_score (host clock around each call, which ends in a device synchronisation) and
    fit_compute_device of a handle with the same lambda on the same points (CUDA events), alternating;
  * a per-kernel split of one REML score from torch.profiler, in a separate pass (kernel names grouped by prefix);
  * select_smoothing_reml against select_smoothing over the default range: total time and evaluations.
Then a replicate study (reported, not gated): 50 seeded 2-D data sets with a known truth, the spread of the selected
log10 lambda and the RMS error against the truth on a test grid under both criteria.
The card name, power limit and clocks are read in the same process.
usage: python scripts/reml_time.py [out.md] [reps] [scale]   (scale < 1 shrinks the point counts, for a dry run)
"""
import os
import statistics
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

import splpak_b200 as sp  # noqa: E402
from splpak_b200 import synth  # noqa: E402
from gcv_time import card, timed  # noqa: E402

CONFIGS = [("cfg3", 3, [24, 24, 24], 1e8), ("cfg4", 4, [12, 12, 12, 12], 1e7)]
GROUPS = [("spl_penalty", "penalty"), ("spl_constraints", "constraint rows"), ("spl_expand_band", "band expansion"),
          ("spl_reml", "REML reductions"), ("spl_gcv", "REML reductions"),
          ("spl_panel", "factor and substitutions"), ("spl_syrk", "factor and substitutions"),
          ("spl_factor", "factor and substitutions"), ("spl_backsolve", "factor and substitutions"),
          ("spl_forwardsolve", "factor and substitutions")]


def group_of(name):
    for prefix, g in GROUPS:
        if prefix in name:
            return g
    if "emcpy" in name or "emset" in name:
        return "copies and memsets"
    return "other"


def host_ms(h, fn):
    h.synchronize()
    t0 = time.perf_counter()
    fn()
    return 1e3 * (time.perf_counter() - t0)


def replicate_study(nsets=50):
    """2-D, 14 x 14 nodes, 1,500 points, sigma = 0.2, thin plate; truth sin(4 x) + cos(3 y) x."""
    nodes = [14, 14]
    mn, mx = np.zeros(2), np.ones(2)
    truth = lambda p: np.sin(4 * p[:, 0]) + np.cos(3 * p[:, 1]) * p[:, 0]
    g = np.stack(np.meshgrid(np.linspace(0, 1, 41), np.linspace(0, 1, 41)), -1).reshape(-1, 2)
    res = {"gcv": ([], []), "reml": ([], [])}
    for seed in range(nsets):
        rng = np.random.default_rng(1000 + seed)
        x = rng.random((1500, 2))
        y = truth(x) + 0.2 * rng.standard_normal(len(x))
        for crit in ("gcv", "reml"):
            h = sp.FitHandle(2, mn, mx, nodes, 0.0)
            assert h.enable_gcv() == 0
            assert h.add_points(x, y) == 0
            lam, _, _ = h.select_smoothing("thin_plate", criterion=crit)
            c, ierr = h.compute()
            assert ierr == 0
            h.destroy()
            v = sp.eval_batch(2, g, c, mn, mx, nodes)
            v = v[0] if isinstance(v, tuple) else v
            res[crit][0].append(np.log10(lam))
            res[crit][1].append(float(np.sqrt(np.mean((v - truth(g)) ** 2))))
    return res


def main():
    path = sys.argv[1] if len(sys.argv) > 1 else "reml_time.md"
    reps = int(sys.argv[2]) if len(sys.argv) > 2 else 5
    scale = float(sys.argv[3]) if len(sys.argv) > 3 else 1.0
    info = card()
    print("card", info, flush=True)
    out = ["# REML: cost of the restricted-likelihood score against the GCV score and compute", "",
           f"Measured on one GPU: `{info}` (name, power limit, current SM clock, max SM clock; read in the same run) with "
           f"`scripts/reml_time.py`: weighted synthetic points (`splpak_b200.synth.points_torch`), device-resident, "
           f"xtrap = 1, curvature penalty; one warm-up, then {reps} repetitions alternating the three calls, median shown.",
           ""]
    for cfg, ndim, nodes, npts in CONFIGS:
        n = int(npts * scale)
        mn, mx = [0.0] * ndim, [1.0] * ndim
        x, y, w = synth.points_torch(ndim, n, seed=42)
        ncol = int(torch.tensor(nodes).prod())
        coef = torch.empty(ncol, dtype=torch.float64, device="cuda")
        lam = 1e-3 * (n / ncol) * (1.0 / (nodes[0] - 1)) ** 3
        plain = sp.FitHandle(ndim, mn, mx, nodes, 1.0)
        h = sp.FitHandle(ndim, mn, mx, nodes, 1.0)
        assert h.enable_gcv() == 0
        assert plain.set_smoothing(lam, "curvature") == 0
        assert h.add_points_device(x, ndim, y, w, n) == 0
        comp, reml, gcv = [], [], []
        for rep in range(reps + 1):
            assert plain.reset() == 0
            assert plain.add_points_device(x, ndim, y, w, n) == 0
            plain.synchronize()
            ms_c = timed(plain, lambda: plain.compute_device(coef))
            ms_r = host_ms(h, lambda: h.reml_score(lam, "curvature"))
            ms_g = host_ms(h, lambda: h.smoothing_score(lam, "curvature"))
            if rep:
                comp.append(ms_c)
                reml.append(ms_r)
                gcv.append(ms_g)
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            h.reml_score(lam, "curvature")
            torch.cuda.synchronize()
        split = {}
        for ev in prof.key_averages():
            dt = getattr(ev, "device_time_total", None)
            if dt is None:
                dt = ev.cuda_time_total
            if dt <= 0:
                continue
            g = group_of(ev.key)
            split[g] = split.get(g, 0.0) + dt / 1e3
        sel = {}
        for crit in ("reml", "gcv"):
            h.synchronize()
            t0 = time.perf_counter()
            lam_best, best, trace = h.select_smoothing("curvature", criterion=crit)
            sel[crit] = (time.perf_counter() - t0, len(trace), lam_best)
        row = {"cfg": cfg, "n": n, "ncol": ncol, "compute": statistics.median(comp), "reml": statistics.median(reml),
               "gcv": statistics.median(gcv), "split": split, "select": sel}
        print(row, flush=True)
        ratio = row["reml"] / row["compute"]
        out += [f"## {cfg}: {ndim}-D {nodes[0]}^{ndim} nodes (n = {ncol:,} columns), {n:.0e} points", "",
                f"* one `reml_score`: {row['reml']:.2f} ms, {ratio:.2f}x `fit_compute_device` of the same smoothed system "
                f"({row['compute']:.2f} ms, CUDA events); one `smoothing_score` (GCV): {row['gcv']:.2f} ms.",
                f"* `select_smoothing_reml` over the default range: {sel['reml'][0]:.3f} s for {sel['reml'][1]} evaluations "
                f"(selected lambda {sel['reml'][2]:.3e}); `select_smoothing` (GCV): {sel['gcv'][0]:.3f} s for "
                f"{sel['gcv'][1]} evaluations (selected lambda {sel['gcv'][2]:.3e}).", "",
                "| kernels of one REML score (torch.profiler) | ms |", "|---|---:|"]
        for g, ms in sorted(split.items(), key=lambda kv: -kv[1]):
            out.append(f"| {g} | {ms:.3f} |")
        out += ["", "Kernel times are summed over streams: where the factor runs kernel per phase on two streams (cfg4), "
                "their sum exceeds the call's wall time.", ""]
        plain.destroy()
        h.destroy()
        del x, y, w
        torch.cuda.empty_cache()
    res = replicate_study(max(2, int(50 * min(1.0, scale * 10))))
    out += ["## Replicate study (reported, not gated)", "",
            f"{len(res['gcv'][0])} seeded 2-D data sets: 14 x 14 nodes, 1,500 uniform points, sigma = 0.2, thin-plate "
            "penalty, truth sin(4 x) + cos(3 y) x; RMS error against the truth on a 41 x 41 grid.", "",
            "| criterion | log10 lambda: median | std | min | max | RMS error: median | mean | max |",
            "|---|---:|---:|---:|---:|---:|---:|---:|"]
    for crit in ("gcv", "reml"):
        t, e = np.array(res[crit][0]), np.array(res[crit][1])
        out.append(f"| {crit.upper()} | {np.median(t):.2f} | {t.std():.2f} | {t.min():.2f} | {t.max():.2f} | "
                   f"{np.median(e):.4f} | {e.mean():.4f} | {e.max():.4f} |")
    out.append("")
    text = "\n".join(out) + "\n"
    with open(path, "w") as f:
        f.write(text)
    print(text)


if __name__ == "__main__":
    main()
