"""splpak_b200 -- B200-native (sm_100a) fit-and-evaluate hot path of jacobwilliams/splpak.

Host-side mirror of the reference's `splpak_type` (initialize / evaluate / destroy, with the
splcc / splcw / splfe / splde entry points) over the C ABI in include/splpak_b200.h.
All compute runs in hand-written CUDA kernels (splpak_b200/csrc); there is no CPU fallback.
"""
from ._lib import SYMBOLS, build, lib_path, load  # noqa: F401
from .api import (  # noqa: F401
    FitHandle,
    SplpakError,
    SplpakType,
    cfaerr_text,
    derivs_ncomp,
    eval_batch,
    eval_batch_device,
    eval_derivs,
    eval_derivs_device,
    eval_grid,
    eval_grid_device,
    measure_peaks,
    splcc,
    splcw,
    splde,
    splfe,
    total_launches,
)

__all__ = [
    "SplpakType", "FitHandle", "SplpakError", "splcc", "splcw", "splfe", "splde", "eval_batch",
    "eval_batch_device", "eval_derivs", "eval_derivs_device", "eval_grid", "eval_grid_device", "measure_peaks",
    "total_launches", "cfaerr_text", "derivs_ncomp", "build", "load", "lib_path", "SYMBOLS",
]
