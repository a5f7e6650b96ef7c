"""ctypes loader of the product library (splpak_b200/lib/libsplpak_b200*.so).

The library is built in-tree by `__graft_entry__.build()` / `splpak_b200.build()` with nvcc for
sm_100a.  There is no fallback: if the library is missing the import of any compute entry point
raises, and every compute call returns 201 when no CUDA device is usable.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_HERE, "csrc")
LIBDIR = os.path.join(_HERE, "lib")
HEADER = os.path.join(os.path.dirname(_HERE), "include", "splpak_b200.h")

# every symbol include/splpak_b200.h declares (tests check the header against this list)
SYMBOLS = [
    "splpak_b200_sizeof_real",
    "splpak_b200_strerror",
    "splpak_b200_splcw",
    "splpak_b200_splcc",
    "splpak_b200_splde",
    "splpak_b200_splfe",
    "splpak_b200_eval",
    "splpak_b200_eval_device",
    "splpak_b200_eval_derivs",
    "splpak_b200_eval_derivs_device",
    "splpak_b200_eval_grid",
    "splpak_b200_eval_grid_device",
    "splpak_b200_fit_create",
    "splpak_b200_fit_add_points",
    "splpak_b200_fit_add_points_device",
    "splpak_b200_fit_partial_buffer",
    "splpak_b200_fit_allreduce",
    "splpak_b200_fit_allreduce_rhs",
    "splpak_b200_comm_init_all",
    "splpak_b200_comm_unique_id",
    "splpak_b200_comm_init_rank",
    "splpak_b200_comm_destroy",
    "splpak_b200_comm_group_start",
    "splpak_b200_comm_group_end",
    "splpak_b200_fit_compute",
    "splpak_b200_fit_compute_device",
    "splpak_b200_fit_refine_begin",
    "splpak_b200_fit_refine_add_points",
    "splpak_b200_fit_refine_add_points_device",
    "splpak_b200_fit_refine_compute",
    "splpak_b200_fit_refine_compute_device",
    "splpak_b200_fit_set_solver",
    "splpak_b200_fit_get_solver",
    "splpak_b200_fit_set_smoothing",
    "splpak_b200_fit_enable_gcv",
    "splpak_b200_fit_smoothing_score",
    "splpak_b200_fit_select_smoothing",
    "splpak_b200_fit_get_selected_inverse",
    "splpak_b200_fit_reml_score",
    "splpak_b200_fit_select_smoothing_reml",
    "splpak_b200_fit_robust_device",
    "splpak_b200_fit_robust",
    "splpak_b200_fit_glm_device",
    "splpak_b200_fit_glm",
    "splpak_b200_fit_glm_select_device",
    "splpak_b200_fit_glm_select",
    "splpak_b200_fit_prepare_variance",
    "splpak_b200_fit_variance",
    "splpak_b200_fit_variance_device",
    "splpak_b200_fit_get_orthogonal_factor",
    "splpak_b200_fit_get_cholesky_factor",
    "splpak_b200_fit_condition_estimate",
    "splpak_b200_fit_constraints_fired",
    "splpak_b200_fit_rhs_buffer",
    "splpak_b200_fit_reset",
    "splpak_b200_fit_stream",
    "splpak_b200_fit_timings",
    "splpak_b200_fit_launch_count",
    "splpak_b200_fit_get_normal_equations",
    "splpak_b200_fit_destroy",
    "splpak_b200_measure_peaks",
    "splpak_b200_total_launches",
]


def lib_path(real32: bool = False) -> str:
    return os.path.join(LIBDIR, "libsplpak_b200_r32.so" if real32 else "libsplpak_b200.so")


def _sources():
    out = [HEADER, os.path.join(CSRC, "Makefile")]
    for f in os.listdir(CSRC):
        if f.endswith((".cu", ".cuh", ".hpp")):
            out.append(os.path.join(CSRC, f))
    return out


def build(force: bool = False, verbose: bool = False) -> None:
    """Compile the CUDA library for sm_100a with nvcc (csrc/Makefile).  Cross-compiles without a GPU."""
    newest = max(os.path.getmtime(p) for p in _sources())
    stale = any((not os.path.exists(p)) or os.path.getmtime(p) < newest for p in (lib_path(False), lib_path(True)))
    if not (force or stale):
        return
    cmd = ["make", "-C", CSRC, "-j8", "all"]
    if force:
        subprocess.run(["make", "-C", CSRC, "clean"], check=True, capture_output=not verbose)
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("splpak_b200: nvcc build failed\n" + r.stdout[-4000:] + r.stderr[-4000:])
    if verbose:
        print(r.stdout)


_cache = {}


def load(real32: bool = False) -> C.CDLL:
    """Load the product library; raises (loudly) when it has not been built."""
    if real32 in _cache:
        return _cache[real32]
    path = lib_path(real32)
    if not os.path.exists(path):
        raise ImportError(
            f"splpak_b200: {path} is missing. Build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a). There is no CPU fallback.")
    lib = C.CDLL(path)
    real = C.c_float if real32 else C.c_double
    rp, ip, vp = C.POINTER(real), C.POINTER(C.c_int), C.c_void_p
    i64 = C.c_int64
    sig = {
        "splpak_b200_sizeof_real": (C.c_int, []),
        "splpak_b200_strerror": (C.c_char_p, [C.c_int, C.c_int]),
        "splpak_b200_splcw": (C.c_int, [C.c_int, vp, C.c_int, vp, vp, i64, rp, rp, ip, real, vp, i64, vp, i64, ip]),
        "splpak_b200_splcc": (C.c_int, [C.c_int, vp, C.c_int, vp, i64, rp, rp, ip, real, vp, i64, vp, i64, ip]),
        "splpak_b200_splde": (real, [C.c_int, rp, ip, vp, rp, rp, ip, ip]),
        "splpak_b200_splfe": (real, [C.c_int, rp, vp, rp, rp, ip, ip]),
        "splpak_b200_eval": (C.c_int, [C.c_int, vp, C.c_int, i64, ip, vp, rp, rp, ip, vp, ip]),
        "splpak_b200_eval_device": (C.c_int, [C.c_int, vp, C.c_int, i64, ip, vp, rp, rp, ip, vp, vp, ip]),
        "splpak_b200_eval_derivs": (C.c_int, [C.c_int, vp, C.c_int, i64, C.c_int, vp, rp, rp, ip, vp, ip]),
        "splpak_b200_eval_derivs_device": (C.c_int, [C.c_int, vp, C.c_int, i64, C.c_int, vp, rp, rp, ip, vp, vp, ip]),
        "splpak_b200_eval_grid": (C.c_int, [C.c_int, vp, C.POINTER(i64), ip, vp, rp, rp, ip, vp, ip]),
        "splpak_b200_eval_grid_device": (C.c_int, [C.c_int, vp, C.POINTER(i64), ip, vp, rp, rp, ip, vp, vp, ip]),
        "splpak_b200_fit_create": (C.c_int, [C.c_int, rp, rp, ip, real, C.POINTER(vp), ip]),
        "splpak_b200_fit_add_points": (C.c_int, [vp, vp, C.c_int, vp, vp, C.c_int, i64]),
        "splpak_b200_fit_add_points_device": (C.c_int, [vp, vp, C.c_int, vp, vp, C.c_int, i64]),
        "splpak_b200_fit_partial_buffer": (C.c_int, [vp, C.POINTER(vp), C.POINTER(i64)]),
        "splpak_b200_fit_allreduce": (C.c_int, [vp, vp]),
        "splpak_b200_fit_allreduce_rhs": (C.c_int, [vp, vp]),
        "splpak_b200_comm_init_all": (C.c_int, [C.c_int, ip, C.POINTER(vp)]),
        "splpak_b200_comm_unique_id": (C.c_int, [C.c_char_p]),
        "splpak_b200_comm_init_rank": (C.c_int, [C.c_int, C.c_int, C.c_char_p, C.POINTER(vp)]),
        "splpak_b200_comm_destroy": (C.c_int, [vp]),
        "splpak_b200_comm_group_start": (C.c_int, []),
        "splpak_b200_comm_group_end": (C.c_int, []),
        "splpak_b200_fit_compute": (C.c_int, [vp, vp, i64, i64, ip]),
        "splpak_b200_fit_compute_device": (C.c_int, [vp, vp, i64, i64, ip]),
        "splpak_b200_fit_refine_begin": (C.c_int, [vp]),
        "splpak_b200_fit_refine_add_points": (C.c_int, [vp, vp, C.c_int, vp, vp, C.c_int, i64]),
        "splpak_b200_fit_refine_add_points_device": (C.c_int, [vp, vp, C.c_int, vp, vp, C.c_int, i64]),
        "splpak_b200_fit_refine_compute": (C.c_int, [vp, vp, i64, ip]),
        "splpak_b200_fit_refine_compute_device": (C.c_int, [vp, vp, i64, ip]),
        "splpak_b200_fit_set_solver": (C.c_int, [vp, C.c_int]),
        "splpak_b200_fit_get_solver": (C.c_int, [vp]),
        "splpak_b200_fit_set_smoothing": (C.c_int, [vp, C.c_double, C.c_int]),
        "splpak_b200_fit_enable_gcv": (C.c_int, [vp]),
        "splpak_b200_fit_smoothing_score": (C.c_int, [vp, C.c_double, C.c_int, vp, C.c_int, ip]),
        "splpak_b200_fit_select_smoothing": (C.c_int, [vp, C.c_int, C.c_double, C.c_double, C.POINTER(C.c_double), vp,
                                                       C.c_int, vp, i64, C.POINTER(i64), ip]),
        "splpak_b200_fit_get_selected_inverse": (C.c_int, [vp, vp, i64, C.POINTER(i64)]),
        "splpak_b200_fit_reml_score": (C.c_int, [vp, C.c_double, C.c_int, vp, C.c_int, ip]),
        "splpak_b200_fit_select_smoothing_reml": (C.c_int, [vp, C.c_int, C.c_double, C.c_double, C.POINTER(C.c_double),
                                                            vp, C.c_int, vp, i64, C.POINTER(i64), ip]),
        "splpak_b200_fit_robust_device": (C.c_int, [vp, vp, C.c_int, vp, vp, C.c_int, i64, C.c_int, C.c_double, C.c_int,
                                                    C.c_double, vp, vp, i64, vp, vp, C.c_int, ip]),
        "splpak_b200_fit_robust": (C.c_int, [vp, vp, C.c_int, vp, vp, C.c_int, i64, C.c_int, C.c_double, C.c_int,
                                             C.c_double, vp, vp, i64, vp, vp, C.c_int, ip]),
        "splpak_b200_fit_glm_device": (C.c_int, [vp, vp, C.c_int, vp, vp, C.c_int, vp, i64, C.c_int, C.c_int, C.c_double,
                                                 vp, vp, i64, vp, vp, C.c_int, ip]),
        "splpak_b200_fit_glm": (C.c_int, [vp, vp, C.c_int, vp, vp, C.c_int, vp, i64, C.c_int, C.c_int, C.c_double, vp,
                                          vp, i64, vp, vp, C.c_int, ip]),
        "splpak_b200_fit_glm_select_device": (C.c_int, [vp, vp, C.c_int, vp, vp, C.c_int, vp, i64, C.c_int, C.c_int,
                                                        C.c_int, C.c_double, C.c_double, C.c_int, C.c_int, C.c_int,
                                                        C.c_double, vp, vp, i64, vp, vp, C.c_int, vp, i64,
                                                        C.POINTER(i64), ip]),
        "splpak_b200_fit_glm_select": (C.c_int, [vp, vp, C.c_int, vp, vp, C.c_int, vp, i64, C.c_int, C.c_int, C.c_int,
                                                 C.c_double, C.c_double, C.c_int, C.c_int, C.c_int, C.c_double, vp, vp,
                                                 i64, vp, vp, C.c_int, vp, i64, C.POINTER(i64), ip]),
        "splpak_b200_fit_prepare_variance": (C.c_int, [vp, vp, C.c_int, ip]),
        "splpak_b200_fit_variance": (C.c_int, [vp, vp, C.c_int, i64, ip, vp, ip]),
        "splpak_b200_fit_variance_device": (C.c_int, [vp, vp, C.c_int, i64, ip, vp, vp, ip]),
        "splpak_b200_fit_get_orthogonal_factor": (C.c_int, [vp, C.c_int, vp, i64, C.POINTER(i64)]),
        "splpak_b200_fit_get_cholesky_factor": (C.c_int, [vp, C.c_int, i64, i64, vp, i64, C.POINTER(i64)]),
        "splpak_b200_fit_condition_estimate": (C.c_int, [vp, C.POINTER(C.c_double)]),
        "splpak_b200_fit_constraints_fired": (C.c_int, [vp]),
        "splpak_b200_fit_rhs_buffer": (C.c_int, [vp, C.POINTER(vp), C.POINTER(i64)]),
        "splpak_b200_fit_reset": (C.c_int, [vp]),
        "splpak_b200_fit_stream": (vp, [vp]),
        "splpak_b200_fit_timings": (C.c_int, [vp, C.POINTER(C.c_double), C.c_int]),
        "splpak_b200_fit_launch_count": (i64, [vp]),
        "splpak_b200_fit_get_normal_equations": (C.c_int, [vp, vp, vp, vp, vp]),
        "splpak_b200_fit_destroy": (C.c_int, [vp]),
        "splpak_b200_measure_peaks": (C.c_int, [C.POINTER(C.c_double), C.c_int]),
        "splpak_b200_total_launches": (i64, []),
    }
    for name, (res, args) in sig.items():
        fn = getattr(lib, name)          # AttributeError here == a declared symbol is not exported
        fn.restype = res
        fn.argtypes = args
    lib._real = real
    _cache[real32] = lib
    return lib
