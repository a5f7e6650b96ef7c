"""Fused derivative sets against the separate single-component calls they replace, device-resident, one GPU.

For every row: one splpak_b200_eval_derivs_device call (order 1 or 2, ncomp outputs per query) against ncomp
splpak_b200_eval_device calls with the nderiv of each component, on the same queries and the same table.  CUDA events,
one warm-up of each, then REPS alternating A/B repetitions; the best and median of each side are reported.  The fused
outputs are checked to be bit-identical to the separate ones.  The card name and its power limit are read in the same
process.
usage: python scripts/eval_derivs_time.py [out.json] [reps] [scale]   (scale < 1 shrinks every row, for a dry run)
"""
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

import splpak_b200 as sp  # noqa: E402
from splpak_b200 import synth  # noqa: E402

# (ndim, nodes, nq, raster order, derivative order): the named configurations, at sizes whose inputs plus both
# outputs fit in 180 GB
ROWS = [
    (2, [64, 64], 1e9, False, 1), (2, [64, 64], 1e9, False, 2),
    (3, [24, 24, 24], 1e9, False, 1), (3, [24, 24, 24], 5e8, False, 2),
    (3, [24, 24, 24], 1e9, True, 1), (3, [24, 24, 24], 5e8, True, 2),
    (4, [12, 12, 12, 12], 1e8, False, 1), (4, [12, 12, 12, 12], 1e8, False, 2),
]


def components(ndim, order):
    comps = [[0] * ndim] + [[int(e == d) for e in range(ndim)] for d in range(ndim)]
    if order == 2:
        for i in range(ndim):
            for j in range(i, ndim):
                nd = [0] * ndim
                nd[i] += 1
                nd[j] += 1
                comps.append(nd)
    return comps


def card():
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                            capture_output=True, text=True, timeout=60).stdout.strip()
    except Exception as e:                      # the number is still worth having; say why the limit is missing
        pl = f"unknown ({e})"
    return name, pl


def main():
    path = sys.argv[1] if len(sys.argv) > 1 else "eval_derivs_time.json"
    reps = int(sys.argv[2]) if len(sys.argv) > 2 else 5
    scale = float(sys.argv[3]) if len(sys.argv) > 3 else 1.0
    name, power = card()
    print("card", name, "power limit", power, flush=True)
    st = torch.cuda.current_stream()
    results = []
    for ndim, nodes, nq, raster, order in ROWS:
        nq = int(nq * scale)
        mn, mx = [0.0] * ndim, [1.0] * ndim
        g = torch.Generator(device="cuda").manual_seed(5)
        coef = torch.randn(int(torch.tensor(nodes).prod()), dtype=torch.float64, device="cuda", generator=g)
        q = synth.queries_torch(ndim, nq, raster=raster)
        comps = components(ndim, order)
        nc = len(comps)
        fused = torch.empty((nq, nc), dtype=torch.float64, device="cuda")
        sep = torch.empty((nc, nq), dtype=torch.float64, device="cuda")

        def run_fused():
            return sp.eval_derivs_device(ndim, q, ndim, nq, coef, mn, mx, nodes, fused, order=order, stream=st)

        def run_sep():
            rc = 0
            for k, nd in enumerate(comps):
                rc |= sp.eval_batch_device(ndim, q, ndim, nq, coef, mn, mx, nodes, sep[k], nderiv=nd, stream=st)
            return rc

        times = {"fused": [], "separate": []}
        for rep in range(reps + 1):
            for key, fn in (("fused", run_fused), ("separate", run_sep)) if rep % 2 == 0 else \
                    (("separate", run_sep), ("fused", run_fused)):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(st)
                assert fn() == 0
                e1.record(st)
                torch.cuda.synchronize()
                if rep > 0:                        # rep 0 warms up both
                    times[key].append(e0.elapsed_time(e1))
        same = all(torch.equal(fused[:, k], sep[k]) for k in range(nc))
        row = {"ndim": ndim, "nodes": nodes, "nq": nq, "order": order, "ncomp": nc,
               "queries": "raster" if raster else "random", "bit_identical": bool(same)}
        for key in times:
            ts = sorted(times[key])
            row[key + "_ms_best"] = round(ts[0], 3)
            row[key + "_ms_median"] = round(ts[len(ts) // 2], 3)
            row[key + "_outputs_per_s"] = nq * nc / (ts[0] * 1e-3)
        row["speedup"] = round(row["separate_ms_best"] / row["fused_ms_best"], 3)
        results.append(row)
        print(json.dumps(row), flush=True)
        del q, fused, sep, coef
        torch.cuda.empty_cache()
    with open(path, "w") as f:
        json.dump({"card": name, "power_limit": power, "reps": reps, "rows": results}, f, indent=1)


if __name__ == "__main__":
    main()
