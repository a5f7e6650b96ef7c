"""Time of the 3-D moment kernel (spl_moments_kernel) alone at cfg3, one GPU.

cfg3 as bench.py runs it: 3-D, 24^3 nodes, xtrap = 1, 1e8 weighted device-resident points
(splpak_b200.synth.points_torch, seed 42), one handle reused with reset() per step.  Two passes:
  * the accumulate stage (moment kernel + cell transform) from the handle's own CUDA event pairs, mean over the steps;
  * the moment kernel's device time per fit from torch.profiler's CUDA activity records, in a separate pass.
Achieved DMMA rate = 576 FMA per point (72 DMMA.8x8x4 per 32 points, 256 FMA each, 2 flop per FMA) over the kernel
time, against the DMMA peak measured in the same process (splpak_b200_measure_peaks).  Card name, power limit and
clocks are read in the same process.
usage: python scripts/moments_time.py [steps] [npoints]
"""
import os
import statistics
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

import splpak_b200 as sp  # noqa: E402
from splpak_b200 import synth  # noqa: E402
from gcv_time import card  # noqa: E402

NODES = [24, 24, 24]
FMA_PER_POINT = 576


def main():
    steps = int(sys.argv[1]) if len(sys.argv) > 1 else 10
    n = int(float(sys.argv[2])) if len(sys.argv) > 2 else 100_000_000
    if not torch.cuda.is_available():
        raise SystemExit("moments_time.py: no CUDA device")
    print("card", card(), flush=True)
    x, y, w = synth.points_torch(3, n, seed=42)
    coef = torch.empty(24 ** 3, dtype=torch.float64, device="cuda")
    h = sp.FitHandle(3, [0.0] * 3, [1.0] * 3, NODES, 1.0)

    def fit():
        h.reset()
        assert h.add_points_device(x, 3, y, w, n, True) == 0
        assert h.compute_device(coef) == 0

    for _ in range(3):
        fit()
    torch.cuda.synchronize()
    acc = []
    for _ in range(steps):
        fit()
        torch.cuda.synchronize()
        acc.append(h.timings()["accumulate"])

    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        for _ in range(steps):
            fit()
        torch.cuda.synchronize()
    kern_us = [e.time_range.elapsed_us() for e in prof.events()
               if "spl_moments_kernel" in e.name and e.device_type == torch.autograd.DeviceType.CUDA]
    if len(kern_us) % steps:
        raise SystemExit(f"{len(kern_us)} moment-kernel launches over {steps} steps")
    per = len(kern_us) // steps
    per_step_ms = [sum(kern_us[i * per:(i + 1) * per]) / 1e3 for i in range(steps)]
    kern_ms = statistics.median(per_step_ms)
    _, dmma_tf, _ = sp.measure_peaks()
    tflops = 2.0 * FMA_PER_POINT * n / (kern_ms * 1e-3) / 1e12
    print(f"accumulate stage ms: mean {statistics.mean(acc):.3f} median {statistics.median(acc):.3f} "
          f"min {min(acc):.3f}")
    print(f"spl_moments_kernel ms per fit ({per} launch(es)): median {kern_ms:.3f} min {min(per_step_ms):.3f} "
          f"max {max(per_step_ms):.3f}")
    print(f"DMMA: {tflops:.2f} TFLOP/s achieved at {FMA_PER_POINT} FMA/point; measured peak {dmma_tf:.2f} TFLOP/s "
          f"({100 * tflops / dmma_tf:.1f} %)")
    h.destroy()


if __name__ == "__main__":
    main()
