"""Cost of smoothing (splpak_b200_fit_set_smoothing) on the streaming Cholesky fit, device-resident, one GPU.

For cfg3 (3-D, 24^3 nodes, 1e8 points) and cfg4 (4-D, 12^4 nodes, 1e7 points), weighted, xtrap = 1: one handle per mode
(lambda = 0, curvature, thin plate), the same points.  Every repetition resets the handle, adds the points and times
splpak_b200_fit_compute_device with CUDA events on the handle's stream; the modes alternate inside a repetition.  One
warm-up of each mode, then REPS repetitions; best and median are reported.  The "constraints" slot of fit_timings holds
the constraint rows and, with smoothing, the penalty kernels (tables + S += lambda R); its growth over lambda = 0 is the
penalty's cost.  One refinement step (splpak_b200_fit_refine_*_device, residual pass over the same points + re-solve with
the stored factor) is timed with and without smoothing.  The card name and its power limit are read in the same process.
usage: python scripts/smoothing_time.py [out.md] [reps] [scale]   (scale < 1 shrinks the point counts, for a dry run)
"""
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

import splpak_b200 as sp  # noqa: E402
from splpak_b200 import synth  # noqa: E402

CONFIGS = [("cfg3", 3, [24, 24, 24], 1e8), ("cfg4", 4, [12, 12, 12, 12], 1e7)]
MODES = [("lambda = 0", None), ("curvature", "curvature"), ("thin plate", "thin_plate")]


def card():
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                            capture_output=True, text=True, timeout=60).stdout.strip()
    except Exception as e:                      # the number is still worth having; say why the limit is missing
        pl = f"unknown ({e})"
    return name, pl


def timed(h, fn):
    """fn() on the handle's stream between two CUDA events; milliseconds."""
    s = torch.cuda.ExternalStream(h.stream())
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(s)
    rc = fn()
    b.record(s)
    b.synchronize()
    assert rc == 0, rc
    return a.elapsed_time(b)


def main():
    path = sys.argv[1] if len(sys.argv) > 1 else "smoothing_time.md"
    reps = int(sys.argv[2]) if len(sys.argv) > 2 else 5
    scale = float(sys.argv[3]) if len(sys.argv) > 3 else 1.0
    name, power = card()
    print("card", name, "power limit", power, flush=True)
    rows = []
    for cfg, ndim, nodes, npts in CONFIGS:
        n = int(npts * scale)
        mn, mx = [0.0] * ndim, [1.0] * ndim
        x, y, w = synth.points_torch(ndim, n, seed=42)
        ncol = int(torch.tensor(nodes).prod())
        coef = torch.empty(ncol, dtype=torch.float64, device="cuda")
        # lambda at the scale of the data Gram matrix (n / ncol points per node) against R's (dxin^3): its size does not
        # change the work, only the solution
        lam = 1e-3 * (n / ncol) * (1.0 / (nodes[0] - 1)) ** 3
        handles = {}
        for label, pen in MODES:
            h = sp.FitHandle(ndim, mn, mx, nodes, 1.0)
            if pen is not None:
                assert h.set_smoothing(lam, pen) == 0
            handles[label] = h
        torch.cuda.synchronize()
        res = {label: {"compute": [], "constraints": [], "refine": []} for label, _ in MODES}
        for rep in range(reps + 1):
            for label, _ in MODES:
                h = handles[label]
                assert h.reset() == 0
                assert h.add_points_device(x, ndim, y, w, n) == 0
                h.synchronize()
                ms = timed(h, lambda: h.compute_device(coef))
                t = h.timings()
                rms = None
                if label != "thin plate":
                    rms = timed(h, lambda: h.refine_device(x, ndim, y, w, n, coef))
                if rep == 0:
                    continue                                         # warm-up
                res[label]["compute"].append(ms)
                res[label]["constraints"].append(t["constraints"])
                if rms is not None:
                    res[label]["refine"].append(rms)
        for label, _ in MODES:
            r = res[label]
            row = {"cfg": cfg, "ndim": ndim, "nodes": nodes, "n": n, "mode": label, "lambda": 0.0 if label == "lambda = 0" else lam,
                   "compute_best": min(r["compute"]), "compute_med": statistics.median(r["compute"]),
                   "constraints_med": statistics.median(r["constraints"]),
                   "refine_best": min(r["refine"]) if r["refine"] else None,
                   "refine_med": statistics.median(r["refine"]) if r["refine"] else None,
                   "stencil_entries": ncol * 4 ** ndim}
            rows.append(row)
            print(row, flush=True)
        for h in handles.values():
            h.destroy()
        del x, y, w
        torch.cuda.empty_cache()

    lines = ["# Smoothing: cost of the roughness penalty on the streaming Cholesky fit", "",
             f"Measured on one {name} at a {power} power limit (`scripts/smoothing_time.py`: device-resident points, "
             f"CUDA events around `splpak_b200_fit_compute_device` on the handle's stream, one warm-up of each mode, then "
             f"{reps} repetitions with the modes alternating; best and median shown).  Weighted synthetic points "
             f"(`splpak_b200.synth.points_torch`), xtrap = 1.  \"constraints\" is the `fit_timings` slot that holds the "
             f"constraint rows and, with smoothing, the penalty kernels (1-D tables + `S += lambda R`): its growth over "
             f"lambda = 0 is the penalty's cost.  \"refine\" is one refinement step (residual pass over the same points, "
             f"constraint and penalty residuals, re-solve with the stored factor).", "",
             "| config | points | mode | compute best ms | compute median ms | constraints slot median ms | "
             "refine best ms | refine median ms |",
             "|---|---:|---|---:|---:|---:|---:|---:|"]
    for r in rows:
        rb = "" if r["refine_best"] is None else f"{r['refine_best']:.3f}"
        rm = "" if r["refine_med"] is None else f"{r['refine_med']:.3f}"
        lines.append(f"| {r['cfg']} {r['ndim']}-D {r['nodes'][0]}^{r['ndim']} | {r['n']:.0e} | {r['mode']} | "
                     f"{r['compute_best']:.3f} | {r['compute_med']:.3f} | {r['constraints_med']:.3f} | {rb} | {rm} |")
    lines.append("")
    for cfg, ndim, nodes, _ in CONFIGS:
        sub = {r["mode"]: r for r in rows if r["cfg"] == cfg}
        base = sub["lambda = 0"]
        for label in ("curvature", "thin plate"):
            r = sub[label]
            lines.append(f"* {cfg}, {label}: penalty kernels {r['constraints_med'] - base['constraints_med']:.3f} ms "
                         f"(median constraints slot minus lambda = 0) for {r['stencil_entries']:,} stencil entries; compute "
                         f"{r['compute_med'] - base['compute_med']:+.3f} ms median over lambda = 0.")
        rc = sub["curvature"]
        if rc["refine_med"] is not None and base["refine_med"] is not None:
            lines.append(f"* {cfg}, one refinement step: {base['refine_med']:.3f} ms without smoothing, "
                         f"{rc['refine_med']:.3f} ms with the curvature penalty (median).")
    text = "\n".join(lines) + "\n"
    with open(path, "w") as f:
        f.write(text)
    print(text)


if __name__ == "__main__":
    main()
