"""Cost of the GCV score (splpak_b200_fit_smoothing_score / select_smoothing) on the streaming Cholesky fit, one GPU.

For cfg3 (3-D, 24^3 nodes, 1e8 points) and cfg4 (4-D, 12^4 nodes, 1e7 points), weighted, xtrap = 1, device-resident
points (splpak_b200.synth.points_torch):
  * add_points_device with and without enable_gcv (CUDA events on the handle's stream, modes alternating);
  * one smoothing_score call (host clock around the call, which ends in a device synchronisation) against
    fit_compute_device of a handle with the same lambda on the same points (CUDA events);
  * a per-kernel split of one score call from torch.profiler, in a separate pass (kernel names grouped by prefix);
  * the selected inverse's FP64 rate, counted as 2 n b^2 over its kernels' time;
  * select_smoothing over the default range: total time and evaluations.
The card name, power limit and clocks are read in the same process.
usage: python scripts/gcv_time.py [out.md] [reps] [scale]   (scale < 1 shrinks the point counts, for a dry run)
"""
import os
import statistics
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

import splpak_b200 as sp  # noqa: E402
from splpak_b200 import synth  # noqa: E402

CONFIGS = [("cfg3", 3, [24, 24, 24], 1e8), ("cfg4", 4, [12, 12, 12, 12], 1e7)]
GROUPS = [("spl_penalty", "penalty"), ("spl_constraints", "constraint rows"), ("spl_expand_band", "band expansion"),
          ("spl_selinv", "selected inverse"), ("spl_gcv", "trace and misfit"),
          ("spl_panel", "factor and substitutions"), ("spl_syrk", "factor and substitutions"),
          ("spl_factor", "factor and substitutions"), ("spl_backsolve", "factor and substitutions"),
          ("spl_forwardsolve", "factor and substitutions")]


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader",
                            "-i", "0"], capture_output=True, text=True, timeout=60).stdout.strip()
    except Exception as e:
        q = f"{torch.cuda.get_device_name(0)}, unknown ({e})"
    return q


def half_bandwidth(nodes):
    b, s = 0, 1
    for n in nodes:
        b += 3 * s
        s *= n
    return b


def timed(h, fn):
    s = torch.cuda.ExternalStream(h.stream())
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(s)
    rc = fn()
    b.record(s)
    b.synchronize()
    assert rc == 0, rc
    return a.elapsed_time(b)


def group_of(name):
    for prefix, g in GROUPS:
        if prefix in name:
            return g
    return "other"


def main():
    path = sys.argv[1] if len(sys.argv) > 1 else "gcv_time.md"
    reps = int(sys.argv[2]) if len(sys.argv) > 2 else 5
    scale = float(sys.argv[3]) if len(sys.argv) > 3 else 1.0
    info = card()
    print("card", info, flush=True)
    out = ["# GCV: cost of the smoothing score and the selected inverse", "",
           f"Measured on one GPU: `{info}` (name, power limit, current SM clock, max SM clock; read in the same run) with "
           f"`scripts/gcv_time.py`: weighted synthetic points (`splpak_b200.synth.points_torch`), device-resident, "
           f"xtrap = 1, curvature penalty; one warm-up, then {reps} repetitions, median shown.", ""]
    for cfg, ndim, nodes, npts in CONFIGS:
        n = int(npts * scale)
        mn, mx = [0.0] * ndim, [1.0] * ndim
        x, y, w = synth.points_torch(ndim, n, seed=42)
        ncol = int(torch.tensor(nodes).prod())
        bw = min(half_bandwidth(nodes), ncol - 1)
        coef = torch.empty(ncol, dtype=torch.float64, device="cuda")
        lam = 1e-3 * (n / ncol) * (1.0 / (nodes[0] - 1)) ** 3
        plain = sp.FitHandle(ndim, mn, mx, nodes, 1.0)
        gcv = sp.FitHandle(ndim, mn, mx, nodes, 1.0)
        assert gcv.enable_gcv() == 0
        assert plain.set_smoothing(lam, "curvature") == 0
        add = {"plain": [], "gcv": []}
        comp, score = [], []
        for rep in range(reps + 1):
            for label, h in (("plain", plain), ("gcv", gcv)):
                assert h.reset() == 0
                h.synchronize()
                ms = timed(h, lambda: h.add_points_device(x, ndim, y, w, n))
                if rep:
                    add[label].append(ms)
            ms = timed(plain, lambda: plain.compute_device(coef))
            gcv.synchronize()
            t0 = time.perf_counter()
            gcv.smoothing_score(lam, "curvature")
            t1 = time.perf_counter()
            if rep:
                comp.append(ms)
                score.append(1e3 * (t1 - t0))
        # per-kernel split of one score call (separate pass: tracing slows the host)
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            gcv.smoothing_score(lam, "curvature")
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
        flops = 2.0 * ncol * bw * bw
        sel_ms = split.get("selected inverse", float("nan"))
        fac_ms = split.get("factor and substitutions", float("nan"))
        gcv.synchronize()
        t0 = time.perf_counter()
        lam_best, best, trace = gcv.select_smoothing("curvature")
        t_sel = time.perf_counter() - t0
        row = {"cfg": cfg, "n": n, "ncol": ncol, "b": bw, "add_plain": statistics.median(add["plain"]),
               "add_gcv": statistics.median(add["gcv"]), "compute": statistics.median(comp),
               "score": statistics.median(score), "split": split, "selinv_tflops": flops / (sel_ms * 1e-3) / 1e12,
               "select_s": t_sel, "evals": len(trace), "lam": lam_best, "edf": best["edf"]}
        print(row, flush=True)
        out += [f"## {cfg}: {ndim}-D {nodes[0]}^{ndim} nodes (n = {ncol:,} columns, half bandwidth b = {bw:,}), "
                f"{n:.0e} points", "",
                f"* `add_points_device`: {row['add_plain']:.3f} ms without `enable_gcv`, {row['add_gcv']:.3f} ms with it.",
                f"* one `smoothing_score`: {row['score']:.2f} ms (host clock, ends in a synchronisation); "
                f"`fit_compute_device` of the same smoothed system: {row['compute']:.2f} ms (CUDA events).",
                f"* selected inverse: {sel_ms:.2f} ms for 2 n b^2 = {flops:.2e} flop, {row['selinv_tflops']:.2f} TFLOP/s "
                f"FP64; {sel_ms / fac_ms:.2f}x the factor and substitutions of the same call ({fac_ms:.2f} ms).",
                f"* `select_smoothing` over the default range: {t_sel:.2f} s for {len(trace)} evaluations "
                f"(selected lambda {lam_best:.3e}, edf {best['edf']:.1f}).", "",
                "| kernels of one score call (torch.profiler) | ms |", "|---|---:|"]
        for g, ms in sorted(split.items(), key=lambda kv: -kv[1]):
            out.append(f"| {g} | {ms:.3f} |")
        out.append("")
        plain.destroy()
        gcv.destroy()
        del x, y, w
        torch.cuda.empty_cache()
    text = "\n".join(out) + "\n"
    with open(path, "w") as f:
        f.write(text)
    print(text)


if __name__ == "__main__":
    main()
