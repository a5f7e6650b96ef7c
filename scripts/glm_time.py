"""Cost of the GLM fit (splpak_b200_fit_glm_device), one GPU.

For cfg3 (3-D, 24^3 nodes, 1e8 points) and cfg4 (4-D, 12^4 nodes, 1e7 points), xtrap = 1, device-resident points
(splpak_b200.synth.points_torch) with Poisson counts of rate exp(0.5 + f(x)), f the synthetic response, tol = 1e-8:
  * the whole call (host clock around it; it ends in a device synchronisation), its iteration count, and the time per
    iteration, call / iterations, against add_points_device + fit_compute_device of the same points;
  * a per-kernel split of one call from torch.profiler, in a separate pass (kernel names grouped by prefix), with the
    share of the GLM kernels (domain check, working pass, deviance sum, halving) in it.
cfg4 runs again with SPLPAK_B200_DETERMINISTIC=1.  The card name, power limit and clocks are read in the same process.
usage: python scripts/glm_time.py [out.md] [reps] [scale]   (scale < 1 shrinks the point counts, for a dry run)
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
from robust_time import group_of  # noqa: E402

CONFIGS = [("cfg3", 3, [24, 24, 24], 1e8, False), ("cfg4", 4, [12, 12, 12, 12], 1e7, False),
           ("cfg4", 4, [12, 12, 12, 12], 1e7, True)]


def glm_group(name):
    return "GLM kernels" if "spl_glm_" in name else group_of(name)


def main():
    path = sys.argv[1] if len(sys.argv) > 1 else "glm_time.md"
    reps = int(sys.argv[2]) if len(sys.argv) > 2 else 3
    scale = float(sys.argv[3]) if len(sys.argv) > 3 else 1.0
    info = card()
    print("card", info, flush=True)
    out = ["# GLM fit: cost per iteration", "",
           f"Measured on one GPU: `{info}` (name, power limit, current SM clock, max SM clock; read in the same run) with "
           f"`scripts/glm_time.py`: synthetic points (`splpak_b200.synth.points_torch`), device-resident, Poisson counts "
           f"of rate exp(0.5 + f(x)), xtrap = 1, tol = 1e-8; one warm-up, then {reps} repetitions alternating the plain "
           f"fit and the GLM call, median shown.", ""]
    for cfg, ndim, nodes, npts, det in CONFIGS:
        if det:
            os.environ["SPLPAK_B200_DETERMINISTIC"] = "1"
        else:
            os.environ.pop("SPLPAK_B200_DETERMINISTIC", None)
        n = int(npts * scale)
        mn, mx = [0.0] * ndim, [1.0] * ndim
        x, f, _ = synth.points_torch(ndim, n, seed=42, weighted=False)
        gen = torch.Generator(device="cuda")
        gen.manual_seed(5)
        y = torch.poisson(torch.exp(0.5 + f), generator=gen)
        del f
        ncol = int(torch.tensor(nodes).prod())
        coef = torch.empty(ncol, dtype=torch.float64, device="cuda")
        plain_ms, glm_ms, res = [], [], None
        for rep in range(reps + 1):
            h = sp.FitHandle(ndim, mn, mx, nodes, 1.0)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            assert h.add_points_device(x, ndim, y, None, n) == 0
            assert h.compute_device(coef) == 0
            t1 = time.perf_counter()
            h.destroy()
            h = sp.FitHandle(ndim, mn, mx, nodes, 1.0)
            torch.cuda.synchronize()
            t2 = time.perf_counter()
            r, ierr = h.glm_fit_device(x, ndim, y, None, n, coef, family="poisson", max_iter=50, tol=1e-8)
            t3 = time.perf_counter()
            assert ierr == 0, (ierr, r)
            h.destroy()
            if rep:
                plain_ms.append(1e3 * (t1 - t0))
                glm_ms.append(1e3 * (t3 - t2))
                res = r
        h = sp.FitHandle(ndim, mn, mx, nodes, 1.0)
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            r, ierr = h.glm_fit_device(x, ndim, y, None, n, coef, family="poisson", max_iter=50, tol=1e-8)
            torch.cuda.synchronize()
        h.destroy()
        split, glm_rows = {}, []
        for ev in prof.key_averages():
            dt = getattr(ev, "device_time_total", None)
            if dt is None:
                dt = ev.cuda_time_total
            if dt <= 0:
                continue
            g = glm_group(ev.key)
            split[g] = split.get(g, 0.0) + dt / 1e3
            if g == "GLM kernels":
                glm_rows.append((ev.key.split("(")[0], ev.count, dt / 1e3))
        k = res["iterations"]
        pm, gm = statistics.median(plain_ms), statistics.median(glm_ms)
        total = sum(split.values())
        share = split.get("GLM kernels", 0.0) / total if total > 0 else 0.0
        mode = "deterministic mode" if det else "default mode"
        print(cfg, mode, pm, gm, res, split, flush=True)
        out += [f"## {cfg}, {mode}: {ndim}-D {nodes[0]}^{ndim} nodes (n = {ncol:,} columns), {n:.0e} points", "",
                f"* plain fit (`add_points_device` + `fit_compute_device`): {pm:.2f} ms; GLM call: {gm:.2f} ms for "
                f"{k} iterations to tol = 1e-8 (converged {res['converged']}, deviance {res['deviance']:.6g}, "
                f"Pearson X^2 {res['pearson']:.6g}, last change {res['change']:.2e}, {res['halvings']} halvings); "
                f"{gm / max(k, 1):.2f} ms per iteration.",
                f"* GLM kernels: {100 * share:.2f} % of the kernel time of the profiled call.",
                f"* per iteration, from the profile below divided by {k}: "
                + ", ".join(f"{g} {ms / max(k, 1):.3f} ms" for g, ms in sorted(split.items(), key=lambda kv: -kv[1])), "",
                f"| kernels of one GLM call ({k} iterations; torch.profiler) | ms |", "|---|---:|"]
        for g, ms in sorted(split.items(), key=lambda kv: -kv[1]):
            out.append(f"| {g} | {ms:.3f} |")
        out += ["", "| GLM kernel | launches | ms | ms per launch |", "|---|---:|---:|---:|"]
        for name, cnt, ms in sorted(glm_rows, key=lambda t: -t[2]):
            out.append(f"| `{name}` | {cnt} | {ms:.3f} | {ms / max(cnt, 1):.3f} |")
        out += [""]
        del x, y
        torch.cuda.empty_cache()
    os.environ.pop("SPLPAK_B200_DETERMINISTIC", None)
    text = "\n".join(out) + "\n"
    with open(path, "w") as f:
        f.write(text)
    print(text)


if __name__ == "__main__":
    main()
