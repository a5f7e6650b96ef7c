"""Host-side mirror of the reference interface (src/splpak.F90:45-127) over the C ABI.

`SplpakType` keeps the reference's names, argument order, argument meaning and error behaviour:
    s = SplpakType()
    coef, ierror = s.initialize(ndim, xdata, l1xdat, ydata, [wdata,] ndata, xmin, xmax, nodes,
                                xtrap, ncf, nwrk)            # -> splcw / splcc
    f, ierror    = s.evaluate(ndim, x, [nderiv,] coef, xmin, xmax, nodes)   # -> splde / splfe
    s.destroy()
Fortran `intent(out)` arguments (coef, ierror, the function result) are returned instead of being
written through references; `work` is dropped (the GPU path needs no host scratch) but `nwrk` is
still validated exactly as the reference validates it.  Like the reference, nothing raises on a
numerical/argument error: the integer `ierror` is returned and, unless quiet, ' IERR=nnnnn' and the
reference's message are printed (cfaerr, :399-407).

Array convention: xdata is passed as a C-ordered numpy array of shape (ndata, l1xdat) -- the
memory image of Fortran's xdata(l1xdat, ndata).  coef is 1-D, dimension 1 fastest (:661-666).

New, non-reference entry points (named by the north star): `FitHandle.add_points / compute`
(streaming assembly / solve split), `eval_batch` (batched splfe/splde), `eval_derivs` (every partial derivative up
to order 1 or 2 in one pass) and device-pointer variants
that take torch CUDA tensors so benchmarks can run device-resident.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib


class SplpakError(RuntimeError):
    """Raised only for misuse of this Python layer (wrong dtype/shape), never for ierror codes."""


def _np_dtype(real32):
    return np.float32 if real32 else np.float64


def cfaerr_text(ierr: int, evaluation: bool, real32: bool = False) -> str:
    """What the reference's cfaerr would print for this code (:399-407)."""
    lib = _lib.load(real32)
    msg = lib.splpak_b200_strerror(int(ierr), 1 if evaluation else 0).decode()
    out = ""
    if ierr != 0:
        out += " IERR=%5d\n" % ierr
    return out + msg.rstrip() + "\n"


def _report(ierr, evaluation, quiet, real32=False):
    if ierr != 0 and not quiet:
        print(cfaerr_text(ierr, evaluation, real32), end="")


def _vec(a, dtype, n=None):
    a = np.ascontiguousarray(a, dtype=dtype).reshape(-1)
    if n is not None and a.size < n:
        raise SplpakError(f"expected at least {n} entries, got {a.size}")
    return a


def _ptr(a):
    return C.c_void_p(a.ctypes.data)


def _grid_args(lib, ndim, xmin, xmax, nodes, real32):
    dt = _np_dtype(real32)
    nd = max(int(ndim), 1)
    mn = _vec(xmin, dt, nd if ndim >= 1 else None)
    mx = _vec(xmax, dt, nd if ndim >= 1 else None)
    no = _vec(nodes, np.int32, nd if ndim >= 1 else None)
    rp = C.POINTER(lib._real)
    return (mn, mx, no), (mn.ctypes.data_as(rp), mx.ctypes.data_as(rp), no.ctypes.data_as(C.POINTER(C.c_int)))


def _ncol(ndim, nodes):
    if ndim < 1:
        return 1
    return int(np.prod(np.asarray(nodes, dtype=np.int64).reshape(-1)[:ndim]))


# ---------------------------------------------------------------------------------------------
# one-shot procedures (exact replacements)
# ---------------------------------------------------------------------------------------------
def splcw(ndim, xdata, l1xdat, ydata, wdata, ndata, xmin, xmax, nodes, xtrap, ncf=None, nwrk=None,
          *, quiet=False, real32=False):
    """splcw (src/splpak.F90:512).  Returns (coef[ncf], ierror)."""
    lib = _lib.load(real32)
    dt = _np_dtype(real32)
    ncol = _ncol(ndim, nodes) if ndim >= 1 and all(n >= 1 for n in np.asarray(nodes).reshape(-1)[:max(ndim, 0)]) else 1
    if ncf is None:
        ncf = ncol
    if nwrk is None:
        nwrk = ncol * (ncol + 1) + 1
    x = np.ascontiguousarray(xdata, dtype=dt)
    y = _vec(ydata, dt)
    w = _vec(wdata, dt) if wdata is not None else np.array([-1.0], dtype=dt)
    keep, (mnp, mxp, nop) = _grid_args(lib, ndim, xmin, xmax, nodes, real32)
    coef = np.zeros(max(int(ncf), 1), dtype=dt)
    if ndata >= 1 and l1xdat >= 1:
        # the C ABI trusts (ndata, l1xdat) as Fortran explicit-shape dummies do: check the buffers here
        if x.size < int(ndata) * int(l1xdat) or y.size < int(ndata) or (w[0] >= 0 and w.size < int(ndata)):
            raise SplpakError(f"xdata/ydata/wdata are smaller than ndata={ndata} x l1xdat={l1xdat} requires")
    ierr = C.c_int(0)
    rc = lib.splpak_b200_splcw(int(ndim), _ptr(x), int(l1xdat), _ptr(y), _ptr(w), int(ndata), mnp, mxp, nop,
                               lib._real(xtrap), _ptr(coef), int(ncf), None, int(nwrk), C.byref(ierr))
    ie = ierr.value if ierr.value != 0 else int(rc)          # a failure that could not write ierror still surfaces
    _report(ie, False, quiet, real32)
    return coef[:int(ncf)] if ncf >= 1 else coef[:0], ie


def splcc(ndim, xdata, l1xdat, ydata, ndata, xmin, xmax, nodes, xtrap, ncf=None, nwrk=None, *,
          quiet=False, real32=False):
    """splcc (src/splpak.F90:421): splcw with all weights 1.  Returns (coef, ierror)."""
    return splcw(ndim, xdata, l1xdat, ydata, None, ndata, xmin, xmax, nodes, xtrap, ncf, nwrk,
                 quiet=quiet, real32=real32)


def splde(ndim, x, nderiv, coef, xmin, xmax, nodes, *, quiet=False, real32=False):
    """splde (src/splpak.F90:1089): one value / partial derivative.  Returns (value, ierror)."""
    lib = _lib.load(real32)
    dt = _np_dtype(real32)
    xv = _vec(np.atleast_1d(x), dt)
    nd = _vec(nderiv, np.int32)
    cf = _vec(coef, dt)
    keep, (mnp, mxp, nop) = _grid_args(lib, ndim, xmin, xmax, nodes, real32)
    ierr = C.c_int(0)
    v = lib.splpak_b200_splde(int(ndim), xv.ctypes.data_as(C.POINTER(lib._real)),
                              nd.ctypes.data_as(C.POINTER(C.c_int)), _ptr(cf), mnp, mxp, nop, C.byref(ierr))
    _report(ierr.value, True, quiet, real32)
    return float(v), ierr.value


def splfe(ndim, x, coef, xmin, xmax, nodes, *, quiet=False, real32=False):
    """splfe (src/splpak.F90:1258): one spline value.  Returns (value, ierror)."""
    lib = _lib.load(real32)
    dt = _np_dtype(real32)
    xv = _vec(np.atleast_1d(x), dt)
    cf = _vec(coef, dt)
    keep, (mnp, mxp, nop) = _grid_args(lib, ndim, xmin, xmax, nodes, real32)
    ierr = C.c_int(0)
    v = lib.splpak_b200_splfe(int(ndim), xv.ctypes.data_as(C.POINTER(lib._real)), _ptr(cf), mnp, mxp, nop,
                              C.byref(ierr))
    _report(ierr.value, True, quiet, real32)
    return float(v), ierr.value


def eval_batch(ndim, x, coef, xmin, xmax, nodes, nderiv=None, *, quiet=True, real32=False):
    """Batched splfe/splde over HOST points x (nq, l1x).  Returns (values[nq], ierror)."""
    lib = _lib.load(real32)
    dt = _np_dtype(real32)
    xa = np.ascontiguousarray(x, dtype=dt)
    if xa.ndim == 1:
        xa = xa.reshape(-1, 1)
    nq, l1x = xa.shape
    cf = _vec(coef, dt)
    out = np.zeros(nq, dtype=dt)
    keep, (mnp, mxp, nop) = _grid_args(lib, ndim, xmin, xmax, nodes, real32)
    ndp = None
    if nderiv is not None:
        nd = _vec(nderiv, np.int32)
        ndp = nd.ctypes.data_as(C.POINTER(C.c_int))
    ierr = C.c_int(0)
    lib.splpak_b200_eval(int(ndim), _ptr(xa), int(l1x), int(nq), ndp, _ptr(cf), mnp, mxp, nop, _ptr(out),
                         C.byref(ierr))
    _report(ierr.value, True, quiet, real32)
    return out, ierr.value


def eval_batch_device(ndim, d_x, l1x, nq, d_coef, xmin, xmax, nodes, d_out, nderiv=None, stream=None,
                      *, real32=False):
    """Batched evaluation with torch CUDA tensors (or raw device pointers) for x, coef, out.
    Asynchronous on `stream` (a torch.cuda.Stream, a raw cudaStream_t int, or None)."""
    lib = _lib.load(real32)
    keep, (mnp, mxp, nop) = _grid_args(lib, ndim, xmin, xmax, nodes, real32)
    ndp = None
    if nderiv is not None:
        nd = _vec(nderiv, np.int32)
        ndp = nd.ctypes.data_as(C.POINTER(C.c_int))
    ierr = C.c_int(0)
    lib.splpak_b200_eval_device(int(ndim), _dev_ptr(d_x), int(l1x), int(nq), ndp, _dev_ptr(d_coef), mnp, mxp,
                                nop, _dev_ptr(d_out), _stream_ptr(stream), C.byref(ierr))
    return ierr.value


def derivs_ncomp(ndim, order):
    """Outputs per query of eval_derivs: ndim + 1 (order 1) or (ndim + 1)(ndim + 2) / 2 (order 2); 0 for another order."""
    n = max(int(ndim), 0)
    return {1: n + 1, 2: (n + 1) * (n + 2) // 2}.get(int(order), 0)


def eval_derivs(ndim, x, coef, xmin, xmax, nodes, order=1, *, quiet=True, real32=False):
    """Every partial derivative up to total order `order` (1 or 2) at HOST points x (nq, l1x), in one pass.
    Returns (out[nq, ncomp], ierror).  Columns: the value, d/dx1 .. d/dxn, then (order 2) d2/dxi dxj for i <= j in row
    order.  Column k is bit-identical to eval_batch with the nderiv it names; an order other than 1 or 2 gives 104."""
    lib = _lib.load(real32)
    dt = _np_dtype(real32)
    xa = np.ascontiguousarray(x, dtype=dt)
    if xa.ndim == 1:
        xa = xa.reshape(-1, 1)
    nq, l1x = xa.shape
    cf = _vec(coef, dt)
    out = np.zeros((nq, derivs_ncomp(ndim, order)), dtype=dt)
    keep, (mnp, mxp, nop) = _grid_args(lib, ndim, xmin, xmax, nodes, real32)
    ierr = C.c_int(0)
    lib.splpak_b200_eval_derivs(int(ndim), _ptr(xa), int(l1x), int(nq), int(order), _ptr(cf), mnp, mxp, nop, _ptr(out),
                                C.byref(ierr))
    _report(ierr.value, True, quiet, real32)
    return out, ierr.value


def eval_derivs_device(ndim, d_x, l1x, nq, d_coef, xmin, xmax, nodes, d_out, order=1, stream=None, *, real32=False):
    """eval_derivs with torch CUDA tensors (or raw device pointers); d_out holds nq * ncomp values, the ncomp of one
    query contiguous.  Asynchronous on `stream`.  Returns ierror."""
    lib = _lib.load(real32)
    keep, (mnp, mxp, nop) = _grid_args(lib, ndim, xmin, xmax, nodes, real32)
    ierr = C.c_int(0)
    lib.splpak_b200_eval_derivs_device(int(ndim), _dev_ptr(d_x), int(l1x), int(nq), int(order), _dev_ptr(d_coef), mnp,
                                       mxp, nop, _dev_ptr(d_out), _stream_ptr(stream), C.byref(ierr))
    return ierr.value


def eval_grid(ndim, axes, coef, xmin, xmax, nodes, nderiv=None, *, quiet=True, real32=False):
    """Spline (or partial derivative) on the tensor grid spanned by `axes` (a list of ndim 1-D arrays).
    Returns (values with shape (len(axes[ndim-1]), ..., len(axes[0])), i.e. dimension 1 fastest; ierror)."""
    lib = _lib.load(real32)
    dt = _np_dtype(real32)
    ax = [np.ascontiguousarray(a, dtype=dt).reshape(-1) for a in axes]
    cat = np.concatenate(ax) if ax else np.zeros(0, dtype=dt)
    na = (C.c_int64 * max(len(ax), 1))(*[len(a) for a in ax])
    keep, (mnp, mxp, nop) = _grid_args(lib, ndim, xmin, xmax, nodes, real32)
    ca = _vec(coef, dt)
    ndp = None
    if nderiv is not None:
        nd = _vec(nderiv, np.int32)
        ndp = nd.ctypes.data_as(C.POINTER(C.c_int))
    out = np.zeros(int(np.prod([len(a) for a in ax])) if ax else 0, dtype=dt)
    ierr = C.c_int(0)
    lib.splpak_b200_eval_grid(int(ndim), _ptr(cat), na, ndp, _ptr(ca), mnp, mxp, nop, _ptr(out), C.byref(ierr))
    _report(ierr.value, True, quiet, real32)
    return out.reshape([len(a) for a in reversed(ax)]), ierr.value


def eval_grid_device(ndim, d_axes, naxis, d_coef, xmin, xmax, nodes, d_out, nderiv=None, stream=None, *, real32=False):
    """Same with device arrays: d_axes = the axes concatenated, naxis = their lengths, d_out = prod(naxis) values."""
    lib = _lib.load(real32)
    keep, (mnp, mxp, nop) = _grid_args(lib, ndim, xmin, xmax, nodes, real32)
    na = (C.c_int64 * len(naxis))(*[int(v) for v in naxis])
    ndp = None
    if nderiv is not None:
        nd = _vec(nderiv, np.int32)
        ndp = nd.ctypes.data_as(C.POINTER(C.c_int))
    ierr = C.c_int(0)
    lib.splpak_b200_eval_grid_device(int(ndim), _dev_ptr(d_axes), na, ndp, _dev_ptr(d_coef), mnp, mxp, nop,
                                     _dev_ptr(d_out), _stream_ptr(stream), C.byref(ierr))
    return ierr.value


def _dev_ptr(t):
    if t is None:
        return None
    if hasattr(t, "data_ptr"):
        return C.c_void_p(t.data_ptr())
    return C.c_void_p(int(t))


def _stream_ptr(s):
    if s is None:
        return None
    if hasattr(s, "cuda_stream"):
        return C.c_void_p(s.cuda_stream)
    return C.c_void_p(int(s))


def measure_peaks():
    """(DFMA TFLOP/s, DMMA TFLOP/s, copy GB/s) measured on the current device."""
    lib = _lib.load(False)
    out = (C.c_double * 3)()
    rc = lib.splpak_b200_measure_peaks(out, 3)
    if rc != 0:
        raise SplpakError(f"measure_peaks failed: {rc}")
    return out[0], out[1], out[2]


def total_launches():
    return int(_lib.load(False).splpak_b200_total_launches())


# ---------------------------------------------------------------------------------------------
# streaming handle (add_points / compute) -- new entry points
# ---------------------------------------------------------------------------------------------
class FitHandle:
    """create -> add_points* -> [all-reduce partial buffer] -> compute."""

    def __init__(self, ndim, xmin, xmax, nodes, xtrap, *, real32=False, solver=None):
        """solver: None / "cholesky" (band Cholesky of the normal equations, default) or "orthogonal" (Householder
        path matching the reference's suprls numerics; 1-D..3-D)."""
        self.lib = _lib.load(real32)
        self.real32 = real32
        self.dt = _np_dtype(real32)
        self.ndim = int(ndim)
        self.nodes = np.asarray(nodes, dtype=np.int32).reshape(-1)[:max(self.ndim, 0)].copy()
        self.ncol = _ncol(self.ndim, self.nodes)
        keep, (mnp, mxp, nop) = _grid_args(self.lib, ndim, xmin, xmax, nodes, real32)
        h = C.c_void_p()
        ierr = C.c_int(0)
        self.lib.splpak_b200_fit_create(int(ndim), mnp, mxp, nop, self.lib._real(xtrap), C.byref(h), C.byref(ierr))
        self.ierror = ierr.value
        self.h = h if ierr.value == 0 else None
        if self.h is not None and solver is not None:
            code = {"cholesky": 0, "orthogonal": 1}[solver]
            rc = self.lib.splpak_b200_fit_set_solver(self.h, code)
            if rc != 0:
                raise SplpakError(f"solver {solver!r} is not available for this grid (rc {rc})")

    def solver(self):
        self._check()
        return {0: "cholesky", 1: "orthogonal"}.get(self.lib.splpak_b200_fit_get_solver(self.h))

    PENALTIES = {"curvature": 0, "thin_plate": 1}

    def set_smoothing(self, lam, penalty="curvature"):
        """Smoothing of the Cholesky fit: minimise the weighted squared residuals (+ the constraint rows) + lam times the
        integral over [xmin, xmax] of the penalty, "curvature" (sum of squared second derivatives d2s/dx_d^2) or
        "thin_plate" (that + 2 x the squared mixed second derivatives).  Any time before compute; persists across reset.
        Returns the library code: 203 for lam < 0, NaN or inf, an unknown penalty code, a finalized handle, or lam > 0
        with the orthogonal solver.  An unknown penalty name raises SplpakError."""
        self._check()
        if isinstance(penalty, str):
            if penalty not in self.PENALTIES:
                raise SplpakError(f"unknown penalty {penalty!r}: expected one of {sorted(self.PENALTIES)}")
            penalty = self.PENALTIES[penalty]
        return self.lib.splpak_b200_fit_set_smoothing(self.h, float(lam), int(penalty))

    def _penalty_code(self, penalty):
        if isinstance(penalty, str):
            if penalty not in self.PENALTIES:
                raise SplpakError(f"unknown penalty {penalty!r}: expected one of {sorted(self.PENALTIES)}")
            return self.PENALTIES[penalty]
        return int(penalty)

    def enable_gcv(self):
        """Generalized cross-validation: before the first add_points (203 otherwise).  Every chunk then also sums
        (w y)^2 into one more slot at the end of the partial buffer.  Persists across reset.  Returns the library code."""
        self._check()
        return self.lib.splpak_b200_fit_enable_gcv(self.h)

    _SCORE_KEYS = ("gcv", "rss", "edf", "n", "ywy")

    def smoothing_score(self, lam, penalty="curvature"):
        """GCV score of the fit with smoothing `lam`, after the (all-reduced) assembly and before compute; changes
        nothing a later compute sees.  Returns {gcv, rss, edf, n, ywy}; raises SplpakError on a non-zero code (107: a
        non-positive pivot, 203: refused)."""
        self._check()
        out = np.zeros(5)
        ierr = C.c_int(0)
        rc = self.lib.splpak_b200_fit_smoothing_score(self.h, float(lam), self._penalty_code(penalty), _ptr(out), 5,
                                                      C.byref(ierr))
        if rc != 0:
            raise SplpakError(f"smoothing_score failed: {rc}", rc)
        return dict(zip(self._SCORE_KEYS, (float(v) for v in out)))

    _REML_KEYS = ("reml", "dp", "logdet", "n", "ywy", "phi")

    def reml_score(self, lam, penalty="curvature"):
        """REML score of the fit with smoothing `lam` > 0, after the (all-reduced) assembly and before compute; changes
        nothing a later compute sees.  Returns {reml, dp, logdet, n, ywy, phi}: V_R (-2 x the profiled restricted
        log-likelihood up to terms that do not depend on lam), the penalised deviance, log|M|, the rows counted
        (constraint rows included), ywy and phi = dp / (n - Mp), the REML estimate of the noise variance.  Raises
        SplpakError on a non-zero code (107: a non-positive pivot, 203: refused)."""
        self._check()
        out = np.zeros(6)
        ierr = C.c_int(0)
        rc = self.lib.splpak_b200_fit_reml_score(self.h, float(lam), self._penalty_code(penalty), _ptr(out), 6,
                                                 C.byref(ierr))
        if rc != 0:
            raise SplpakError(f"reml_score failed: {rc}", rc)
        return dict(zip(self._REML_KEYS, (float(v) for v in out)))

    CRITERIA = ("gcv", "reml")

    def _criterion_is_reml(self, criterion):
        if criterion not in self.CRITERIA:
            raise SplpakError(f"unknown criterion {criterion!r}: expected one of {list(self.CRITERIA)}")
        return criterion == "reml"

    def select_smoothing(self, penalty="curvature", lo=None, hi=None, trace_cap=512, criterion="gcv"):
        """lambda minimising the GCV score (criterion="gcv") or the REML score (criterion="reml") over [lo, hi]
        (default: rho * [1e-10, 1e4], rho = tr G0 / tr R); sets it on the handle (set_smoothing), so the next compute is
        the selected fit.  Returns (lam, score dict, trace), trace: (k, 4) rows in evaluation order, [lambda, V, RSS, edf]
        for GCV, [lambda, V_R, dp, logdet] for REML; the score dict is that of smoothing_score or reml_score.  Raises
        SplpakError on a non-zero code or an unknown criterion."""
        reml = self._criterion_is_reml(criterion)
        self._check()
        fn = self.lib.splpak_b200_fit_select_smoothing_reml if reml else self.lib.splpak_b200_fit_select_smoothing
        keys = self._REML_KEYS if reml else self._SCORE_KEYS
        lam = C.c_double(0.0)
        out = np.zeros(len(keys))
        trace = np.zeros((int(trace_cap), 4))
        nt = C.c_int64(0)
        ierr = C.c_int(0)
        rc = fn(self.h, self._penalty_code(penalty), 0.0 if lo is None else float(lo), 0.0 if hi is None else float(hi),
                C.byref(lam), _ptr(out), len(keys), _ptr(trace), int(trace_cap), C.byref(nt), C.byref(ierr))
        if rc != 0:
            raise SplpakError(f"select_smoothing failed: {rc}", rc)
        return lam.value, dict(zip(keys, (float(v) for v in out))), trace[: min(nt.value, int(trace_cap))]

    def selected_inverse(self):
        """Parity hook, after a score call: (ncol, b + 1), row i = Sigma(i, i..i+b), Sigma = (G0 + C + lambda R)^-1."""
        self._check()
        n = C.c_int64(0)
        if self.lib.splpak_b200_fit_get_selected_inverse(self.h, None, 0, C.byref(n)) != 0:
            raise SplpakError("no selected inverse on this handle (call smoothing_score first)")
        out = np.zeros(n.value)
        rc = self.lib.splpak_b200_fit_get_selected_inverse(self.h, _ptr(out), n.value, C.byref(n))
        if rc != 0:
            raise SplpakError(f"get_selected_inverse failed: {rc}")
        return out.reshape(self.ncol, -1)

    def prepare_variance(self):
        """Posterior variances: after the (all-reduced) assembly and before compute, with the handle's current (lambda,
        penalty).  Reuses the selected inverse select_smoothing left behind, otherwise scores once, then builds the
        per-window tables the variance calls read.  Returns the smoothing_score dict plus sigma2 = rss / (n - edf) (+inf
        when n <= edf); raises SplpakError on a non-zero code (107, 203, 204)."""
        self._check()
        out = np.zeros(6)
        ierr = C.c_int(0)
        rc = self.lib.splpak_b200_fit_prepare_variance(self.h, _ptr(out), 6, C.byref(ierr))
        if rc != 0:
            raise SplpakError(f"prepare_variance failed: {rc}", rc)
        return dict(zip(self._SCORE_KEYS + ("sigma2",), (float(v) for v in out)))

    PSI = {"huber": 0, "bisquare": 1}
    _ROBUST_KEYS = ("iterations", "sigma", "change", "sum_u", "n_rejected", "converged")

    def _psi_code(self, psi):
        if psi not in self.PSI:
            raise SplpakError(f"unknown psi {psi!r}: expected one of {sorted(self.PSI)}")
        return self.PSI[psi]

    def _robust_info(self, out):
        info = dict(zip(self._ROBUST_KEYS, (float(v) for v in out)))
        for k in ("iterations", "n_rejected"):
            info[k] = int(info[k])
        info["converged"] = bool(info["converged"])
        return info

    def robust_fit(self, x, y, w=None, psi="bisquare", tuning=None, max_iter=20, tol=1e-6, return_weights=False):
        """Robust fit of HOST points on a fresh (or reset) handle by iteratively reweighted least squares: Huber or
        Tukey bisquare weights from the residuals scaled by their exact median absolute value (header:
        splpak_b200_fit_robust_device).  tuning None: 1.345 (Huber) / 4.685 (bisquare).  Returns (coef, info, ierror),
        info = {iterations, sigma, change, sum_u, n_rejected, converged} and, with return_weights, "u": the weights u_i
        of the final solve.  An unknown psi name raises SplpakError."""
        self._check()
        code = self._psi_code(psi)
        xa = np.ascontiguousarray(x, dtype=self.dt)
        if xa.ndim == 1:
            xa = xa.reshape(-1, 1)
        ya = _vec(y, self.dt)
        wa = _vec(w, self.dt) if w is not None else None
        n = xa.shape[0]
        coef = np.zeros(self.ncol, dtype=self.dt)
        u = np.zeros(max(n, 1), dtype=self.dt) if return_weights else None
        out = np.zeros(6)
        ierr = C.c_int(0)
        self.lib.splpak_b200_fit_robust(self.h, _ptr(xa), xa.shape[1], _ptr(ya), _ptr(wa) if wa is not None else None,
                                        int(wa is not None), n, code, 0.0 if tuning is None else float(tuning),
                                        int(max_iter), float(tol), None, _ptr(coef), self.ncol,
                                        _ptr(u) if u is not None else None, _ptr(out), 6, C.byref(ierr))
        info = self._robust_info(out)
        if return_weights:
            info["u"] = u[:n]
        return coef, info, ierr.value

    def robust_fit_device(self, d_x, l1x, d_y, d_w, n, d_coef, psi="bisquare", tuning=None, max_iter=20, tol=1e-6,
                          d_u=None, comm=None):
        """robust_fit with torch CUDA tensors or raw device pointers (d_w None: all weights 1; d_u None: no weights
        returned).  comm: a raw ncclComm_t (splpak_b200_comm_*) when every rank passes its shard, None on one GPU.
        Returns (info, ierror)."""
        self._check()
        code = self._psi_code(psi)
        out = np.zeros(6)
        ierr = C.c_int(0)
        self.lib.splpak_b200_fit_robust_device(self.h, _dev_ptr(d_x), int(l1x), _dev_ptr(d_y), _dev_ptr(d_w),
                                               int(d_w is not None), int(n), code,
                                               0.0 if tuning is None else float(tuning), int(max_iter), float(tol),
                                               comm, _dev_ptr(d_coef), self.ncol, _dev_ptr(d_u), _ptr(out), 6,
                                               C.byref(ierr))
        return self._robust_info(out), ierr.value

    FAMILY = {"poisson": 0, "binomial": 1, "gamma": 2}
    _GLM_KEYS = ("iterations", "deviance", "pearson", "change", "halvings", "converged", "m")

    def _family_code(self, family):
        if family not in self.FAMILY:
            raise SplpakError(f"unknown family {family!r}: expected one of {sorted(self.FAMILY)}")
        return self.FAMILY[family]

    def _glm_info(self, out):
        info = dict(zip(self._GLM_KEYS, (float(v) for v in out)))
        for k in ("iterations", "halvings", "m"):
            info[k] = int(info[k])
        info["converged"] = bool(info["converged"])
        return info

    def glm_fit(self, x, y, w=None, family="poisson", offset=None, max_iter=25, tol=1e-8, return_mu=False):
        """Generalized smoothing fit of HOST points on a fresh (or reset) handle by penalized IRLS: Poisson (log link),
        binomial (logit; y a proportion, w = sqrt(trials)) or Gamma (log) responses, eta = s(x) + offset (header:
        splpak_b200_fit_glm_device).  Returns (coef, info, ierror), info = {iterations, deviance, pearson, change,
        halvings, converged, m} and, with return_mu, "mu": the fitted means at the points.  An unknown family name
        raises SplpakError."""
        code = self._family_code(family)
        self._check()
        xa = np.ascontiguousarray(x, dtype=self.dt)
        if xa.ndim == 1:
            xa = xa.reshape(-1, 1)
        n = xa.shape[0]
        ya = _vec(y, self.dt, n)
        wa = _vec(w, self.dt, n) if w is not None else None
        oa = _vec(offset, self.dt, n) if offset is not None else None
        coef = np.zeros(self.ncol, dtype=self.dt)
        mu = np.zeros(max(n, 1), dtype=self.dt) if return_mu else None
        out = np.zeros(7)
        ierr = C.c_int(0)
        self.lib.splpak_b200_fit_glm(self.h, _ptr(xa), xa.shape[1], _ptr(ya), _ptr(wa) if wa is not None else None,
                                     int(wa is not None), _ptr(oa) if oa is not None else None, n, code,
                                     int(max_iter), float(tol), None, _ptr(coef), self.ncol,
                                     _ptr(mu) if mu is not None else None, _ptr(out), 7, C.byref(ierr))
        info = self._glm_info(out)
        if return_mu:
            info["mu"] = mu[:n]
        return coef, info, ierr.value

    def glm_fit_device(self, d_x, l1x, d_y, d_w, n, d_coef, family="poisson", d_offset=None, max_iter=25, tol=1e-8,
                       d_mu=None, comm=None):
        """glm_fit with torch CUDA tensors or raw device pointers (d_w None: all weights 1; d_offset None: no offset;
        d_mu None: no fitted means returned).  comm: a raw ncclComm_t (splpak_b200_comm_*) when every rank passes its
        shard, None on one GPU.  Returns (info, ierror)."""
        code = self._family_code(family)
        self._check()
        out = np.zeros(7)
        ierr = C.c_int(0)
        self.lib.splpak_b200_fit_glm_device(self.h, _dev_ptr(d_x), int(l1x), _dev_ptr(d_y), _dev_ptr(d_w),
                                            int(d_w is not None), _dev_ptr(d_offset), int(n), code, int(max_iter),
                                            float(tol), comm, _dev_ptr(d_coef), self.ncol, _dev_ptr(d_mu), _ptr(out), 7,
                                            C.byref(ierr))
        return self._glm_info(out), ierr.value

    GLM_CRITERIA = {"reml": 0, "prediction": 1}
    _GLM_SELECT_KEYS = ("lam", "score", "edf", "scale", "select_iterations", "settled")

    def _glm_select_args(self, family, criterion, penalty, lo, hi):
        code = self._family_code(family)
        if criterion not in self.GLM_CRITERIA:
            raise SplpakError(f"unknown criterion {criterion!r}: expected one of {sorted(self.GLM_CRITERIA)}")
        return (code, self.GLM_CRITERIA[criterion], self._penalty_code(penalty), 0.0 if lo is None else float(lo),
                0.0 if hi is None else float(hi))

    def _glm_select_info(self, out):
        info = self._glm_info(out[:7])
        info.update(zip(self._GLM_SELECT_KEYS, (float(v) for v in out[7:13])))
        info["select_iterations"] = int(info["select_iterations"])
        info["settled"] = bool(info["settled"])
        return info

    def glm_select(self, x, y, w=None, family="poisson", offset=None, criterion="reml", penalty="curvature", lo=None,
                   hi=None, max_select=10, variance=False, max_iter=25, tol=1e-8, return_mu=False, trace_cap=64):
        """glm_fit with lambda chosen on each PIRLS working system (header: splpak_b200_fit_glm_select_device):
        criterion "reml" or "prediction" (UBRE for Poisson / binomial, GCV for Gamma) over [lo, hi] (default rho *
        [1e-10, 1e4]).  With variance=True the variance calls then return q(x) of the final working system; scale * q
        is the posterior variance of eta(x).  Returns (coef, info, trace, ierror), info = the glm_fit keys plus {lam,
        score, edf, scale, select_iterations, settled} (and "mu" with return_mu), trace: (k, 5) rows [lambda,
        criterion (NaN when frozen), scores, deviance, halvings].  Unknown family, criterion or penalty names raise
        SplpakError."""
        code, crit, pen, lo, hi = self._glm_select_args(family, criterion, penalty, lo, hi)
        self._check()
        xa = np.ascontiguousarray(x, dtype=self.dt)
        if xa.ndim == 1:
            xa = xa.reshape(-1, 1)
        n = xa.shape[0]
        ya = _vec(y, self.dt, n)
        wa = _vec(w, self.dt, n) if w is not None else None
        oa = _vec(offset, self.dt, n) if offset is not None else None
        coef = np.zeros(self.ncol, dtype=self.dt)
        mu = np.zeros(max(n, 1), dtype=self.dt) if return_mu else None
        out = np.zeros(13)
        trace = np.zeros((max(int(trace_cap), 1), 5))
        nt = C.c_int64(0)
        ierr = C.c_int(0)
        self.lib.splpak_b200_fit_glm_select(self.h, _ptr(xa), xa.shape[1], _ptr(ya),
                                            _ptr(wa) if wa is not None else None, int(wa is not None),
                                            _ptr(oa) if oa is not None else None, n, code, crit, pen, lo, hi,
                                            int(max_select), int(bool(variance)), int(max_iter), float(tol), None,
                                            _ptr(coef), self.ncol, _ptr(mu) if mu is not None else None, _ptr(out), 13,
                                            _ptr(trace), int(trace_cap), C.byref(nt), C.byref(ierr))
        info = self._glm_select_info(out)
        if return_mu:
            info["mu"] = mu[:n]
        return coef, info, trace[: nt.value].copy(), ierr.value

    def glm_select_device(self, d_x, l1x, d_y, d_w, n, d_coef, family="poisson", d_offset=None, criterion="reml",
                          penalty="curvature", lo=None, hi=None, max_select=10, variance=False, max_iter=25, tol=1e-8,
                          d_mu=None, trace_cap=64, comm=None):
        """glm_select with torch CUDA tensors or raw device pointers (d_w None: all weights 1; d_offset None: no offset;
        d_mu None: no fitted means returned).  comm: a raw ncclComm_t (splpak_b200_comm_*) when every rank passes its
        shard, None on one GPU.  Returns (info, trace, ierror)."""
        code, crit, pen, lo, hi = self._glm_select_args(family, criterion, penalty, lo, hi)
        self._check()
        out = np.zeros(13)
        trace = np.zeros((max(int(trace_cap), 1), 5))
        nt = C.c_int64(0)
        ierr = C.c_int(0)
        self.lib.splpak_b200_fit_glm_select_device(self.h, _dev_ptr(d_x), int(l1x), _dev_ptr(d_y), _dev_ptr(d_w),
                                                   int(d_w is not None), _dev_ptr(d_offset), int(n), code, crit, pen,
                                                   lo, hi, int(max_select), int(bool(variance)), int(max_iter),
                                                   float(tol), comm, _dev_ptr(d_coef), self.ncol, _dev_ptr(d_mu),
                                                   _ptr(out), 13, _ptr(trace), int(trace_cap), C.byref(nt),
                                                   C.byref(ierr))
        return self._glm_select_info(out), trace[: nt.value].copy(), ierr.value

    def variance(self, x, nderiv=None):
        """q(x) = b(x)^T Sigma b(x) at HOST points x (nq, l1x), after prepare_variance: the posterior variance of the
        fitted value (nderiv: of that partial derivative) divided by sigma2.  Returns (q[nq], ierror)."""
        self._check()
        xa = np.ascontiguousarray(x, dtype=self.dt)
        if xa.ndim == 1:
            xa = xa.reshape(-1, 1)
        nq, l1x = xa.shape
        out = np.zeros(nq, dtype=self.dt)
        nd = _vec(nderiv, np.int32, self.ndim) if nderiv is not None else None
        ierr = C.c_int(0)
        self.lib.splpak_b200_fit_variance(self.h, _ptr(xa), int(l1x), int(nq),
                                          nd.ctypes.data_as(C.POINTER(C.c_int)) if nd is not None else None, _ptr(out),
                                          C.byref(ierr))
        return out, ierr.value

    def variance_device(self, d_x, l1x, nq, d_out, nderiv=None, stream=None):
        """variance with torch CUDA tensors (or raw device pointers); asynchronous on `stream` (None: the handle's
        stream).  Returns ierror."""
        self._check()
        nd = _vec(nderiv, np.int32, self.ndim) if nderiv is not None else None
        ierr = C.c_int(0)
        self.lib.splpak_b200_fit_variance_device(self.h, _dev_ptr(d_x), int(l1x), int(nq),
                                                 nd.ctypes.data_as(C.POINTER(C.c_int)) if nd is not None else None,
                                                 _dev_ptr(d_out), _stream_ptr(stream), C.byref(ierr))
        return ierr.value

    def orthogonal_factor(self, which):
        """Parity-test hook: which = 0 -> per-window triangles (nwindows, 4^ndim, 4^ndim + 1); 1 -> band factor (ncol, b + 2)."""
        self._check()
        n = C.c_int64(0)
        if self.lib.splpak_b200_fit_get_orthogonal_factor(self.h, int(which), None, 0, C.byref(n)) != 0:
            raise SplpakError("no orthogonal factor on this handle")
        out = np.zeros(n.value)
        rc = self.lib.splpak_b200_fit_get_orthogonal_factor(self.h, int(which), _ptr(out), n.value, C.byref(n))
        if rc != 0:
            raise SplpakError(f"get_orthogonal_factor failed: {rc}")
        ncw = 4 ** self.ndim
        return out.reshape(-1, ncw, ncw + 1) if which == 0 else out.reshape(self.ncol, -1)

    def cholesky_factor(self, which, first_col=0, ncols=None):
        """Parity-test hook of the Cholesky factor, after compute (header: fit_get_cholesky_factor).  which = 0 -> band
        columns first_col.. (ncols, lda), row j - first_col = L(j .. j + lda - 1, j), the 64 x 64 diagonal blocks
        excluded from the contract; 1 -> the block inverses L11^-1 of their panels (nblk, 64, 64)."""
        self._check()
        ncols = self.ncol - int(first_col) if ncols is None else int(ncols)
        n = C.c_int64(0)
        rc = self.lib.splpak_b200_fit_get_cholesky_factor(self.h, int(which), int(first_col), ncols, None, 0,
                                                          C.byref(n))
        if rc != 0:
            raise SplpakError(f"get_cholesky_factor failed: {rc}", rc)
        out = np.zeros(n.value)
        rc = self.lib.splpak_b200_fit_get_cholesky_factor(self.h, int(which), int(first_col), ncols, _ptr(out),
                                                          n.value, C.byref(n))
        if rc != 0:
            raise SplpakError(f"get_cholesky_factor failed: {rc}", rc)
        return out.reshape(ncols, -1) if which == 0 else out.reshape(-1, 64, 64)

    def condition_estimate(self):
        """Pivot-ratio LOWER bound of cond(G) from the last Cholesky factor (0.0 when unknown)."""
        self._check()
        v = C.c_double(0.0)
        self.lib.splpak_b200_fit_condition_estimate(self.h, C.byref(v))
        return v.value

    def _check(self):
        if self.h is None:
            raise SplpakError(f"fit handle is not usable (ierror {self.ierror})")

    def add_points(self, x, y, w=None, weighted=None):
        """HOST arrays; x is (n, l1x) C-ordered."""
        self._check()
        xa = np.ascontiguousarray(x, dtype=self.dt)
        if xa.ndim == 1:
            xa = xa.reshape(-1, 1)
        ya = _vec(y, self.dt)
        wa = _vec(w, self.dt) if w is not None else None
        if weighted is None:
            weighted = wa is not None and wa.size > 0 and wa[0] >= 0
        return self.lib.splpak_b200_fit_add_points(self.h, _ptr(xa), xa.shape[1], _ptr(ya),
                                                   _ptr(wa) if wa is not None else None, int(bool(weighted)),
                                                   xa.shape[0])

    def add_points_device(self, d_x, l1x, d_y, d_w, n, weighted=True):
        """torch CUDA tensors / raw device pointers; asynchronous on the handle's stream."""
        self._check()
        return self.lib.splpak_b200_fit_add_points_device(self.h, _dev_ptr(d_x), int(l1x), _dev_ptr(d_y),
                                                          _dev_ptr(d_w), int(bool(weighted and d_w is not None)),
                                                          int(n))

    def partial_buffer(self):
        """(device pointer, count) of the float64 buffer to sum across ranks before compute."""
        self._check()
        p = C.c_void_p()
        n = C.c_int64(0)
        self.lib.splpak_b200_fit_partial_buffer(self.h, C.byref(p), C.byref(n))
        return p.value, n.value

    def partial_tensor(self):
        """The partial buffer as a torch float64 CUDA tensor view (for torch.distributed.all_reduce)."""
        import torch

        ptr, n = self.partial_buffer()

        class _Wrap:
            __cuda_array_interface__ = {"shape": (n,), "typestr": "<f8", "data": (ptr, False), "version": 3}

        return torch.as_tensor(_Wrap(), device=torch.device("cuda", torch.cuda.current_device()))

    def stream(self):
        self._check()
        return self.lib.splpak_b200_fit_stream(self.h)

    def synchronize(self):
        ms = (C.c_double * 7)()
        self.lib.splpak_b200_fit_timings(self.h, ms, 7)

    def compute(self, ncf=None, nwrk=-1):
        """Returns (coef host array, ierror)."""
        self._check()
        ncf = self.ncol if ncf is None else int(ncf)
        coef = np.zeros(max(ncf, 1), dtype=self.dt)
        ierr = C.c_int(0)
        self.lib.splpak_b200_fit_compute(self.h, _ptr(coef), ncf, int(nwrk), C.byref(ierr))
        return coef[:ncf], ierr.value

    def compute_device(self, d_coef, ncf=None, nwrk=-1):
        self._check()
        ncf = self.ncol if ncf is None else int(ncf)
        ierr = C.c_int(0)
        self.lib.splpak_b200_fit_compute_device(self.h, _dev_ptr(d_coef), ncf, int(nwrk), C.byref(ierr))
        return ierr.value

    def refine(self, x, y, w=None, weighted=None, steps=1):
        """Corrected-semi-normal-equations refinement with the same HOST points (after compute).
        Returns (coef, ierror)."""
        self._check()
        xa = np.ascontiguousarray(x, dtype=self.dt)
        if xa.ndim == 1:
            xa = xa.reshape(-1, 1)
        ya = _vec(y, self.dt)
        wa = _vec(w, self.dt) if w is not None else None
        if weighted is None:
            weighted = wa is not None and wa.size > 0 and wa[0] >= 0
        coef = np.zeros(self.ncol, dtype=self.dt)
        ierr = C.c_int(0)
        for _ in range(steps):
            rc = self.lib.splpak_b200_fit_refine_begin(self.h)
            if rc == 0:
                rc = self.lib.splpak_b200_fit_refine_add_points(self.h, _ptr(xa), xa.shape[1], _ptr(ya),
                                                                _ptr(wa) if wa is not None else None,
                                                                int(bool(weighted)), xa.shape[0])
            if rc != 0:
                return coef, rc
            self.lib.splpak_b200_fit_refine_compute(self.h, _ptr(coef), self.ncol, C.byref(ierr))
            if ierr.value != 0:
                break
        return coef, ierr.value

    def refine_device(self, d_x, l1x, d_y, d_w, n, d_coef, weighted=True, allreduce=None):
        """One refinement step with DEVICE points; `allreduce` (optional callable) is applied to the right-hand
        side tensor between the residual pass and the solve (multi-GPU)."""
        self._check()
        rc = self.lib.splpak_b200_fit_refine_begin(self.h)
        if rc != 0:
            return rc
        rc = self.lib.splpak_b200_fit_refine_add_points_device(self.h, _dev_ptr(d_x), int(l1x), _dev_ptr(d_y),
                                                               _dev_ptr(d_w), int(bool(weighted and d_w is not None)),
                                                               int(n))
        if rc != 0:
            return rc
        if allreduce is not None:
            # the collective must be ordered against the handle's private stream: issue it there
            import torch

            with torch.cuda.stream(torch.cuda.ExternalStream(self.stream())):
                allreduce(self.rhs_tensor())
        ierr = C.c_int(0)
        self.lib.splpak_b200_fit_refine_compute_device(self.h, _dev_ptr(d_coef), self.ncol, C.byref(ierr))
        return ierr.value

    def rhs_tensor(self):
        import torch

        p = C.c_void_p()
        n = C.c_int64(0)
        self.lib.splpak_b200_fit_rhs_buffer(self.h, C.byref(p), C.byref(n))
        ptr, cnt = p.value, n.value

        class _Wrap:
            __cuda_array_interface__ = {"shape": (cnt,), "typestr": "<f8", "data": (ptr, False), "version": 3}

        return torch.as_tensor(_Wrap(), device=torch.device("cuda", torch.cuda.current_device()))

    def constraints_fired(self):
        self._check()
        return bool(self.lib.splpak_b200_fit_constraints_fired(self.h))

    def reset(self):
        self._check()
        return self.lib.splpak_b200_fit_reset(self.h)

    def timings(self):
        self._check()
        ms = (C.c_double * 7)()
        self.lib.splpak_b200_fit_timings(self.h, ms, 7)
        keys = ["classify_hist", "bin_scatter", "accumulate", "constraints", "band_expand", "factor", "backsolve"]
        return dict(zip(keys, list(ms)))

    def launch_count(self):
        self._check()
        return int(self.lib.splpak_b200_fit_launch_count(self.h))

    def normal_equations(self):
        """(S[ncol, 4^ndim], g[ncol], cnt[ncol], totlwt, nrows) copied to the host (parity tests)."""
        self._check()
        nst = 4 ** self.ndim
        S = np.zeros(self.ncol * nst)
        g = np.zeros(self.ncol)
        cnt = np.zeros(self.ncol)
        tot = np.zeros(2)
        rc = self.lib.splpak_b200_fit_get_normal_equations(self.h, _ptr(S), _ptr(g), _ptr(cnt), _ptr(tot))
        if rc != 0:
            raise SplpakError(f"get_normal_equations failed: {rc}")
        return S.reshape(self.ncol, nst), g, cnt, tot[0], tot[1]

    def destroy(self):
        if self.h is not None:
            self.lib.splpak_b200_fit_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.destroy()
        except Exception:
            pass


# ---------------------------------------------------------------------------------------------
# splpak_type mirror
# ---------------------------------------------------------------------------------------------
class SplpakType:
    """Mirror of `type(splpak_type)` (src/splpak.F90:45-127): initialize / evaluate / destroy."""

    def __init__(self, *, quiet=False, real32=False):
        self.quiet = quiet
        self.real32 = real32
        self.mdim = 0

    def initialize(self, ndim, xdata, l1xdat, ydata, *rest):
        """Generic `initialize` => splcc | splcw, resolved like the Fortran generic by the presence
        of the extra real array:
            initialize(ndim, xdata, l1xdat, ydata, ndata, xmin, xmax, nodes, xtrap[, ncf, nwrk])         splcc
            initialize(ndim, xdata, l1xdat, ydata, wdata, ndata, xmin, xmax, nodes, xtrap[, ncf, nwrk])  splcw
        Returns (coef, ierror)."""
        if len(rest) >= 1 and np.ndim(rest[0]) >= 1:
            wdata, ndata, xmin, xmax, nodes, xtrap, *tail = rest
        else:
            wdata = None
            ndata, xmin, xmax, nodes, xtrap, *tail = rest
        ncf = tail[0] if len(tail) > 0 else None
        nwrk = tail[1] if len(tail) > 1 else None
        self.mdim = ndim
        return splcw(ndim, xdata, l1xdat, ydata, wdata, ndata, xmin, xmax, nodes, xtrap, ncf, nwrk,
                     quiet=self.quiet, real32=self.real32)

    def evaluate(self, ndim, x, *rest):
        """Generic `evaluate` => splfe | splde, resolved by the integer array:
            evaluate(ndim, x, coef, xmin, xmax, nodes)          splfe
            evaluate(ndim, x, nderiv, coef, xmin, xmax, nodes)  splde
        Returns (value, ierror)."""
        self.mdim = ndim
        if len(rest) == 5:
            nderiv, coef, xmin, xmax, nodes = rest
            return splde(ndim, x, nderiv, coef, xmin, xmax, nodes, quiet=self.quiet, real32=self.real32)
        coef, xmin, xmax, nodes = rest
        return splfe(ndim, x, coef, xmin, xmax, nodes, quiet=self.quiet, real32=self.real32)

    def destroy(self, ndim=None):
        """destroy_splpak (:136-165): the GPU path keeps no per-object state between calls."""
        self.mdim = 0
