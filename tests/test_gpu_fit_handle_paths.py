"""The fit handle's shared host paths: the host staging loop of a refinement step, checked entry by entry, and the
handle state after the error returns of compute and refine_compute.

  * Refinement with HOST points across two 2^22-point staging chunks, with a leading dimension of 5 (NaN padding): the
    right-hand side after splpak_b200_fit_refine_add_points against B^T W^2 (y - B c) on the host, with the tolerance
    and the one-point-out check of test_gpu_assembly_routes.test_refinement_rhs_reassembly.
  * compute: 104 before the finalized check (the handle stays open), 203 once finalized, 204 when the band does not fit
    (the handle stays open), 107 from an orthogonal handle without points (finalized).
  * refine_compute: 203 without refine_begin, 104 for a small ncf (the step stays open for a valid call).
"""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")
import splpak_b200 as sp  # noqa: E402
import test_gpu_assembly_routes as routes  # noqa: E402


def _refine_compute(h, ncf):
    coef = np.zeros(max(ncf, 1))
    ierr = C.c_int(-1)
    rc = h.lib.splpak_b200_fit_refine_compute(h.h, coef.ctypes.data, int(ncf), C.byref(ierr))
    assert rc == ierr.value
    return coef, rc


def _small_fit(xtrap=1.0, solver=None):
    rng = np.random.default_rng(7)
    x = rng.random((20000, 3))
    y = np.sin(3.0 * x).sum(axis=1) + 0.01 * rng.standard_normal(len(x))
    w = 0.5 + rng.random(len(x))
    return sp.FitHandle(3, [0.0] * 3, [1.0] * 3, [6, 5, 7], xtrap, solver=solver), x, y, w


def test_host_refinement_rhs_across_host_chunks(monkeypatch, oracle):
    """6.3e6 skewed points (two host chunks) through refine_add_points with l1x = 5; rhs read before refine_compute."""
    d = routes.reference("3d12_skew")
    routes._set_env(monkeypatch, {})
    n = len(d["y"])
    h = sp.FitHandle(3, d["xmin"], d["xmax"], d["nodes"], 0.0)
    assert h.add_points(d["x"], d["y"], d["w"]) == 0
    c, ierr = h.compute()
    assert ierr == 0
    x5 = np.full((n, 5), np.nan)                                  # the padding must never be read
    x5[:, :3] = d["x"]
    assert h.lib.splpak_b200_fit_refine_begin(h.h) == 0
    assert h.lib.splpak_b200_fit_refine_add_points(h.h, x5.ctypes.data, 5, d["y"].ctypes.data, d["w"].ctypes.data, 1,
                                                   n) == 0
    h.synchronize()
    rhs = h.rhs_tensor().cpu().numpy().copy()
    _, rc = _refine_compute(h, h.ncol)
    assert rc == 0
    h.destroy()
    routes.check_refine_rhs("3d12_skew", "refine rhs_only, host l1x=5", d, c, rhs, oracle)
    routes._REF.pop("3d12_skew", None)


def test_compute_state_after_errors():
    """104 leaves the handle open, a valid compute then succeeds; a second compute is refused with 203, and a small ncf
    is still 104 (checked first)."""
    h, x, y, w = _small_fit()
    assert h.add_points(x, y, w) == 0
    coef, ierr = h.compute(ncf=h.ncol - 1)
    assert ierr == 104
    assert h.set_smoothing(0.0) == 0                              # still open: set_smoothing refuses a finalized handle
    coef, ierr = h.compute()
    assert ierr == 0 and np.all(np.isfinite(coef))
    assert h.set_smoothing(0.0) == 203
    assert h.compute()[1] == 203
    assert h.compute(ncf=h.ncol - 1)[1] == 104
    h.destroy()


def test_compute_band_allocation_failure_keeps_handle_open():
    """A 100^3 grid: the band needs ~240 GB, so compute returns 204 and the handle stays open."""
    h = sp.FitHandle(3, [0.0] * 3, [1.0] * 3, [100] * 3, 0.0)
    assert h.ierror == 0
    assert h.compute()[1] == 204
    assert h.set_smoothing(0.0) == 0
    h.destroy()


def test_refine_compute_state_after_errors():
    """refine_compute without refine_begin: 203; with a small ncf: 104, and the step stays open for a valid call, whose
    coefficients match those of the same step on a second handle."""
    h, x, y, w = _small_fit()
    assert h.add_points(x, y, w) == 0
    c0, ierr = h.compute()
    assert ierr == 0
    assert _refine_compute(h, h.ncol)[1] == 203
    assert h.lib.splpak_b200_fit_refine_begin(h.h) == 0
    assert h.lib.splpak_b200_fit_refine_add_points(h.h, x.ctypes.data, 3, y.ctypes.data, w.ctypes.data, 1, len(x)) == 0
    assert _refine_compute(h, h.ncol - 1)[1] == 104
    c1, rc = _refine_compute(h, h.ncol)
    assert rc == 0
    assert _refine_compute(h, h.ncol)[1] == 203                   # the step is used up
    h.destroy()
    h2, _, _, _ = _small_fit()
    assert h2.add_points(x, y, w) == 0
    assert h2.compute()[1] == 0
    c2, ierr = h2.refine(x, y, w)
    assert ierr == 0
    h2.destroy()
    assert np.abs(c1 - c2).max() <= 1e-8 * np.abs(c0).max()


def test_orthogonal_compute_without_points():
    """An orthogonal handle that never saw a point: 107 and finalized, then 203."""
    h, _, _, _ = _small_fit(xtrap=0.0, solver="orthogonal")
    assert h.compute()[1] == 107
    assert h.compute()[1] == 203
    h.destroy()
