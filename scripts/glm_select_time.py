"""Cost of the GLM fit with lambda selection (splpak_b200_fit_glm_select_device), one GPU.

For cfg3 (3-D, 24^3 nodes, 1e8 points) and cfg4 (4-D, 12^4 nodes, 1e7 points), xtrap = 1, device-resident points
(splpak_b200.synth.points_torch) with Poisson counts of rate exp(0.5 + f(x)), f the synthetic response, tol = 1e-8,
for both criteria (REML; UBRE, the prediction criterion of a Poisson response):
  * the whole call (host clock around it; it ends in a device synchronisation), PIRLS iterations, selecting
    iterations and the scores each selecting iteration evaluated (from the trace);
  * a split of the call: the PIRLS work is a plain glm_fit_device at the selected lambda with the same number of
    iterations (tol = 0); the final score is one assembly of the points plus one smoothing_score at that lambda on a
    GCV handle; the score loop is the rest of the call, and is divided by the scores evaluated.
The card name, power limit and clocks are read in the same process.
usage: python scripts/glm_select_time.py [out.md] [reps] [scale]   (scale < 1 shrinks the point counts, for a dry run)
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


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    r = fn()
    torch.cuda.synchronize()
    return 1e3 * (time.perf_counter() - t0), r


def main():
    path = sys.argv[1] if len(sys.argv) > 1 else "glm_select_time.md"
    reps = int(sys.argv[2]) if len(sys.argv) > 2 else 3
    scale = float(sys.argv[3]) if len(sys.argv) > 3 else 1.0
    info = card()
    print("card", info, flush=True)
    out = ["# GLM fit with lambda selection: cost of the call", "",
           f"Measured on one GPU: `{info}` (name, power limit, current SM clock, max SM clock; read in the same run) with "
           f"`scripts/glm_select_time.py`: synthetic points (`splpak_b200.synth.points_torch`), device-resident, "
           f"Poisson counts of rate exp(0.5 + f(x)), xtrap = 1, tol = 1e-8, default range and max_select = 10; one "
           f"warm-up, then {reps} repetitions, median shown.  The PIRLS work is a plain `glm_fit_device` at the "
           f"selected lambda with the same iteration count (tol = 0); the final score is one assembly plus one "
           f"`smoothing_score` at that lambda; the score loop is the rest of the call.", ""]
    for cfg, ndim, nodes, npts in CONFIGS:
        n = int(npts * scale)
        mn, mx = [0.0] * ndim, [1.0] * ndim
        x, f, _ = synth.points_torch(ndim, n, seed=42, weighted=False)
        gen = torch.Generator(device="cuda")
        gen.manual_seed(5)
        y = torch.poisson(torch.exp(0.5 + f), generator=gen)
        del f
        ncol = int(torch.tensor(nodes).prod())
        coef = torch.empty(ncol, dtype=torch.float64, device="cuda")
        out += [f"## {cfg}: {ndim}-D {nodes[0]}^{ndim} nodes (n = {ncol:,} columns), {n:.0e} points", "",
                "| criterion | call ms | PIRLS iterations | selecting | scores per selecting iteration | "
                "score loop ms | ms per score | PIRLS work ms | final score ms | lambda | edf | settled |",
                "|---|---:|---:|---:|---|---:|---:|---:|---:|---:|---:|---|"]
        for crit in ("reml", "prediction"):
            calls, res = [], None
            for rep in range(reps + 1):
                h = sp.FitHandle(ndim, mn, mx, nodes, 1.0)
                ms, r = timed(lambda: h.glm_select_device(x, ndim, y, None, n, coef, family="poisson", criterion=crit,
                                                          max_iter=50, tol=1e-8))
                assert r[2] == 0, r
                h.destroy()
                if rep:
                    calls.append(ms)
                    res = r
            sel, trace, _ = res
            k, lam = sel["iterations"], sel["lam"]
            pirls, final = [], []
            for rep in range(reps + 1):
                h = sp.FitHandle(ndim, mn, mx, nodes, 1.0)
                assert h.set_smoothing(lam, "curvature") == 0
                ms, r = timed(lambda: h.glm_fit_device(x, ndim, y, None, n, coef, family="poisson", max_iter=k,
                                                       tol=0.0))
                assert r[1] == 0, r
                h.destroy()
                h = sp.FitHandle(ndim, mn, mx, nodes, 1.0)
                assert h.enable_gcv() == 0
                ms2, _ = timed(lambda: (h.add_points_device(x, ndim, y, None, n), h.smoothing_score(lam)))
                h.destroy()
                if rep:
                    pirls.append(ms)
                    final.append(ms2)
            cm, pm, fm = statistics.median(calls), statistics.median(pirls), statistics.median(final)
            scores = [int(v) for v in trace[:, 2] if v > 0]
            loop = cm - pm - fm
            print(cfg, crit, cm, pm, fm, sel, scores, flush=True)
            out.append(f"| {crit} | {cm:.1f} | {k} | {sel['select_iterations']} | {scores} | {loop:.1f} | "
                       f"{loop / max(sum(scores), 1):.2f} | {pm:.1f} | {fm:.1f} | {lam:.4e} | {sel['edf']:.2f} | "
                       f"{sel['settled']} |")
        out.append("")
        del x, y
        torch.cuda.empty_cache()
    text = "\n".join(out) + "\n"
    with open(path, "w") as f:
        f.write(text)
    print(text)


if __name__ == "__main__":
    main()
