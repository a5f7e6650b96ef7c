"""Robust fits (splpak_b200_fit_robust / fit_robust_device): iteratively reweighted Huber and bisquare fits.

The reference is a host IRLS in numpy built independently of the device kernels: the basis rows of every point and the
constraint rows from the oracle (oracle.rows), the dense penalty of test_gpu_smoothing, the exact lower median with
np.partition, the same weight functions, and lstsq on the row-weighted augmented system [w sqrt(u) A; C; sqrt(lam) R^1/2].
Runs with tol = 0 and max_iter = k compare the same iterate."""
import ctypes as C
import threading

import numpy as np
import pytest

import splpak_b200 as sp
from splpak_b200.api import SplpakError
from test_gpu_gcv import rho_of
from test_gpu_smoothing import penalty_dense
from util import coef_tolerance, make_problem

pytestmark = pytest.mark.gpu
MAD_SCALE = 0.6744897501960817
DEFAULT_C = {"huber": 1.345, "bisquare": 4.685}


def add_outliers(y, frac, size, seed):
    """Gross errors of size .. 2 size, random signs, at a random fraction of the points; returns (y, indices)."""
    rng = np.random.default_rng(seed)
    idx = rng.choice(len(y), int(frac * len(y)), replace=False)
    y = y.copy()
    y[idx] += rng.choice([-1.0, 1.0], len(idx)) * rng.uniform(size, 2 * size, len(idx))
    return y, idx


def weights_of(psi, t):
    t = np.abs(t)
    if psi == "huber":
        with np.errstate(divide="ignore"):
            return np.minimum(1.0, 1.0 / t)
    return np.where(t < 1.0, (1.0 - t * t) ** 2, 0.0)


def lower_median(a):
    k = (len(a) + 1) // 2
    return np.partition(a, k - 1)[k - 1]


def host_irls(oracle, ndim, x, y, w, mn, mx, nodes, xtrap, lam, penalty, psi, iters):
    """c^iters of the IRLS with the device's semantics: (coef, sigma, u, M of the last solve)."""
    n = len(y)
    wv = np.ones(n) if w is None else w
    P, _ = oracle.rows(ndim, x, y, None, mn, mx, nodes, 0.0)             # basis row of every point, unweighted
    assert P.shape[0] == n
    ncon = (oracle.rows(ndim, x, y, w, mn, mx, nodes, xtrap)[0].shape[0]
            - oracle.rows(ndim, x, y, w, mn, mx, nodes, 0.0)[0].shape[0]) if xtrap != 0.0 else 0
    Ccon = oracle.rows(ndim, x, y, w, mn, mx, nodes, xtrap)[0][-ncon:] if ncon else np.zeros((0, P.shape[1]))
    Rh = np.zeros((0, P.shape[1]))
    if lam > 0:
        ev, V = np.linalg.eigh(penalty_dense(nodes, mn, mx, penalty))
        Rh = np.sqrt(lam) * (V * np.sqrt(np.maximum(ev, 0.0))) @ V.T

    def solve(rw):
        A = np.vstack([rw[:, None] * P, Ccon, Rh])
        b = np.concatenate([rw * y, np.zeros(len(Ccon) + len(Rh))])
        return np.linalg.lstsq(A, b, rcond=None)[0], A.T @ A

    c, M = solve(wv)
    pos = wv > 0
    sigma, u = 0.0, pos.astype(float)
    for _ in range(iters):
        r = wv * (y - P @ c)
        sigma = lower_median(np.abs(r[pos])) / MAD_SCALE
        u = np.where(pos, weights_of(psi, r / (DEFAULT_C[psi] * sigma)), 0.0)
        c, M = solve(wv * np.sqrt(u))
    return c, sigma, u, M


PARITY_CASES = [
    # ndim, nodes, ndata, xtrap, weighted, hole, lambda factor (x rho), penalty, psi
    (1, [12], 500, 0.0, True, False, 0.0, "curvature", "bisquare"),
    (1, [12], 500, 1.0, False, True, 1e-3, "curvature", "huber"),
    (2, [8, 7], 3000, 0.0, False, False, 0.0, "curvature", "huber"),
    (2, [8, 7], 3000, 1.0, True, True, 1e-2, "thin_plate", "bisquare"),
    (3, [6, 5, 6], 6000, 1.0, True, True, 0.0, "curvature", "bisquare"),
    (3, [6, 5, 6], 6000, 0.0, False, False, 1e-3, "thin_plate", "huber"),
    (4, [4, 4, 5, 4], 4000, 1.0, True, True, 0.0, "curvature", "huber"),
    (4, [4, 5, 4, 4], 4000, 0.0, False, False, 1e-3, "curvature", "bisquare"),
]


def robust_handle(ndim, mn, mx, nodes, xtrap, lam, penalty, real32=False):
    h = sp.FitHandle(ndim, mn, mx, nodes, xtrap, real32=real32)
    assert h.ierror == 0
    if lam > 0:
        assert h.set_smoothing(lam, penalty) == 0
    return h


@pytest.mark.parametrize("ndim,nodes,ndata,xtrap,weighted,hole,lamf,penalty,psi", PARITY_CASES)
def test_iterates_match_host_irls(oracle, ndim, nodes, ndata, xtrap, weighted, hole, lamf, penalty, psi):
    x, y, w, mn, mx = make_problem(ndim, nodes, ndata, seed=5 * ndim + len(PARITY_CASES), weighted=weighted, hole=hole)
    y, _ = add_outliers(y, 0.05, 0.3, seed=ndim)
    wv = w if weighted else None
    lam = 0.0
    if lamf > 0:
        P, _ = oracle.rows(ndim, x, y, wv, mn, mx, nodes, 0.0)
        lam = lamf * rho_of(nodes, mn, mx, penalty, P.T @ P)
    for iters in (1, 2, 5):
        h = robust_handle(ndim, mn, mx, nodes, xtrap, lam, penalty)
        coef, info, ierr = h.robust_fit(x, y, wv, psi=psi, max_iter=iters, tol=0.0, return_weights=True)
        assert ierr == 0, (iters, info)
        assert info["iterations"] == iters and not info["converged"]
        c_ref, sigma_ref, u_ref, M = host_irls(oracle, ndim, x, y, wv, mn, mx, nodes, xtrap, lam, penalty, psi, iters)
        tol, cond = coef_tolerance(M)
        scale = np.abs(c_ref).max()
        err = np.abs(coef - c_ref).max() / scale
        assert err <= (iters + 1) * tol, (iters, err, tol, cond)
        # The intermediate iterates are Cholesky solves at cond(M) (the refinement steps run after the last solve only),
        # so the previous iterate carries |dc| <= (iters + 1) tol |c| and every residual |w P dc|, hence the median, at
        # most max |w| max_i sum_j |P_ij| that much: 1e-12 relative where M is well conditioned, the propagated bound
        # elsewhere.  u (|du/dt| <= 1.6 for both weight functions) follows t = |r| / (c sigma).
        P, _ = oracle.rows(ndim, x, y, None, mn, mx, nodes, 0.0)
        dr = (1.0 if wv is None else wv.max()) * np.abs(P).sum(axis=1).max() * (iters + 1) * tol * scale
        tol_sigma = max(1e-12 * sigma_ref, dr / MAD_SCALE)
        assert abs(info["sigma"] - sigma_ref) <= tol_sigma, (iters, info["sigma"], sigma_ref, tol_sigma)
        tol_u = 1e-10 + 1.6 * (dr + DEFAULT_C[psi] * tol_sigma) / (DEFAULT_C[psi] * sigma_ref)
        assert np.abs(info["u"] - u_ref).max() <= tol_u, (iters, np.abs(info["u"] - u_ref).max(), tol_u)
        pos = (np.ones(len(y)) if wv is None else wv) > 0
        assert info["n_rejected"] == int(((u_ref == 0) & pos).sum())
        assert abs(info["sum_u"] - u_ref.sum()) <= len(y) * tol_u
        h.destroy()


MEDIAN_CASES = ["odd", "even", "ties", "zero_weights", "near_zero"]


@pytest.mark.parametrize("case", MEDIAN_CASES)
def test_first_scale_is_the_exact_lower_median(oracle, monkeypatch, case):
    """sigma of iteration 1 equals, bit for bit, lower_median(|w (y - s(x))|) / 0.6744897501960817 with s from
    eval_batch of the plain fit (deterministic mode: the robust call's c^0 is then the plain fit bit for bit)."""
    monkeypatch.setenv("SPLPAK_B200_DETERMINISTIC", "1")
    ndim, nodes = 2, [7, 6]
    ndata = {"odd": 2001, "even": 2000}.get(case, 1500)
    x, y, w, mn, mx = make_problem(ndim, nodes, ndata, seed=17, weighted=True)
    if case == "ties":
        x = np.vstack([x, x[:500]])                 # duplicated points: identical residuals
        y = np.concatenate([y, y[:500]])
        w = np.concatenate([w, w[:500]])
    if case == "zero_weights":
        w[::7] = 0.0                                # excluded from m
    if case == "near_zero":
        y[: int(0.7 * len(y))] = 1.0                # residuals of a few ulps, exact zeros among them
    plain = sp.FitHandle(ndim, mn, mx, nodes, 0.0)
    assert plain.add_points(x, y, w, weighted=True) == 0
    c0, ierr = plain.compute()
    assert ierr == 0
    s, ierr = sp.eval_batch(ndim, x, c0, mn, mx, nodes)
    assert ierr == 0
    r = np.abs(w * (y - s))
    want = lower_median(r[w > 0]) / MAD_SCALE
    h = robust_handle(ndim, mn, mx, nodes, 0.0, 0.0, "curvature")
    _, info, ierr = h.robust_fit(x, y, w, psi="bisquare", max_iter=1, tol=0.0)
    assert ierr == 0
    assert info["sigma"] == want, (info["sigma"], want)
    if want == 0.0:
        assert info["converged"] and info["iterations"] == 0


def test_zero_mad_stops_converged():
    """Data on the fit: every residual is exactly 0, MAD = 0, the call stops with c^0 and u = 1 where w > 0."""
    ndim, nodes = 2, [6, 6]
    x, _, w, mn, mx = make_problem(ndim, nodes, 800, seed=3, weighted=True)
    w[::5] = 0.0
    y = np.zeros(len(x))
    h = robust_handle(ndim, mn, mx, nodes, 0.0, 0.0, "curvature")
    coef, info, ierr = h.robust_fit(x, y, w, max_iter=10, return_weights=True)
    assert ierr == 0
    assert info["converged"] and info["iterations"] == 0 and info["sigma"] == 0.0
    assert np.array_equal(info["u"], (w > 0).astype(float))
    assert info["sum_u"] == (w > 0).sum() and info["n_rejected"] == 0
    assert np.all(coef == 0.0)


def truth3(x):
    return np.sin(2 * x[:, 0]) * np.cos(1.5 * x[:, 1]) + 0.5 * x[:, 2] ** 2


def test_bisquare_rejects_gross_outliers(oracle):
    ndim, nodes, n, noise = 3, [8, 8, 8], 60000, 0.01
    rng = np.random.default_rng(11)
    x = rng.random((n, ndim))
    clean = truth3(x) + noise * rng.standard_normal(n)
    dirty, idx = add_outliers(clean, 0.10, 50 * noise, seed=12)
    mn, mx = np.zeros(ndim), np.ones(ndim)
    g = np.linspace(0.02, 0.98, 15)
    q = np.stack(np.meshgrid(g, g, g, indexing="ij"), axis=-1).reshape(-1, ndim)

    def rms(coef):
        v, ierr = sp.eval_batch(ndim, q, coef, mn, mx, nodes)
        assert ierr == 0
        return float(np.sqrt(np.mean((v - truth3(q)) ** 2)))

    c_clean, ierr = sp.splcc(ndim, x, ndim, clean, n, mn, mx, nodes, 0.0, quiet=True)
    assert ierr == 0
    c_dirty, ierr = sp.splcc(ndim, x, ndim, dirty, n, mn, mx, nodes, 0.0, quiet=True)
    assert ierr == 0
    h = robust_handle(ndim, mn, mx, nodes, 0.0, 0.0, "curvature")
    coef, info, ierr = h.robust_fit(x, dirty, psi="bisquare", return_weights=True)
    assert ierr == 0 and info["converged"], info
    e_clean, e_dirty, e_rob = rms(c_clean), rms(c_dirty), rms(coef)
    assert e_rob <= 1.5 * e_clean, (e_rob, e_clean)
    assert e_dirty >= 10 * e_clean, (e_dirty, e_clean)
    assert np.all(info["u"][idx] == 0.0)
    assert info["n_rejected"] >= len(idx)


def test_repeatable_and_host_device_agree(monkeypatch):
    """Deterministic mode: repeated calls, and the host and device entries, return the same bits (coef, u, out)."""
    import torch

    monkeypatch.setenv("SPLPAK_B200_DETERMINISTIC", "1")
    ndim, nodes = 3, [7, 6, 7]
    x, y, w, mn, mx = make_problem(ndim, nodes, 20000, seed=23, weighted=True, hole=True)
    y, _ = add_outliers(y, 0.05, 0.3, seed=24)
    runs = []
    for _ in range(2):
        h = robust_handle(ndim, mn, mx, nodes, 1.0, 0.0, "curvature")
        coef, info, ierr = h.robust_fit(x, y, w, psi="huber", max_iter=6, return_weights=True)
        assert ierr == 0
        runs.append((coef, info.pop("u"), info))
        h.destroy()
    for a, b in zip(runs[0], runs[1]):
        assert np.array_equal(a, b) if isinstance(a, np.ndarray) else a == b
    dev = torch.device("cuda", torch.cuda.current_device())
    d_x, d_y, d_w = (torch.from_numpy(np.ascontiguousarray(a)).to(dev) for a in (x, y, w))
    h = robust_handle(ndim, mn, mx, nodes, 1.0, 0.0, "curvature")
    d_c = torch.zeros(h.ncol, dtype=torch.float64, device=dev)
    d_u = torch.zeros(len(y), dtype=torch.float64, device=dev)
    info, ierr = h.robust_fit_device(d_x, ndim, d_y, d_w, len(y), d_c, psi="huber", max_iter=6, d_u=d_u)
    assert ierr == 0
    assert np.array_equal(d_c.cpu().numpy(), runs[0][0])
    assert np.array_equal(d_u.cpu().numpy(), runs[0][1])
    assert info == runs[0][2]


def test_real32_agrees_with_real64():
    ndim, nodes = 2, [9, 8]
    x, y, w, mn, mx = make_problem(ndim, nodes, 20000, seed=31, weighted=True)
    y, _ = add_outliers(y, 0.05, 0.3, seed=32)
    h64 = robust_handle(ndim, mn, mx, nodes, 0.0, 0.0, "curvature")
    c64, i64, e64 = h64.robust_fit(x, y, w, psi="bisquare", max_iter=8)
    h32 = robust_handle(ndim, mn, mx, nodes, 0.0, 0.0, "curvature", real32=True)
    c32, i32, e32 = h32.robust_fit(x.astype(np.float32), y.astype(np.float32), w.astype(np.float32), psi="bisquare",
                                   max_iter=8)
    assert e64 == 0 and e32 == 0
    scale = np.abs(c64).max()
    assert np.abs(c32 - c64).max() <= 1e-3 * scale, np.abs(c32 - c64).max() / scale
    assert abs(i32["sigma"] - i64["sigma"]) <= 1e-3 * i64["sigma"]
    assert abs(i32["n_rejected"] - i64["n_rejected"]) <= 0.01 * len(y)


def _ngpu():
    import torch

    return torch.cuda.device_count() if torch.cuda.is_available() else 0


@pytest.mark.skipif(_ngpu() < 2, reason="needs 2 GPUs on one box")
@pytest.mark.parametrize("deterministic", [False, True])
def test_two_devices_bit_identical_replicas(monkeypatch, deterministic):
    import torch

    if deterministic:
        monkeypatch.setenv("SPLPAK_B200_DETERMINISTIC", "1")
    lib = sp.load()
    ndim, nodes = 2, [9, 8]
    x, y, w, mn, mx = make_problem(ndim, nodes, 30000, seed=41, weighted=True, hole=True)
    y, _ = add_outliers(y, 0.05, 0.3, seed=42)
    devs = (C.c_int * 2)(0, 1)
    comms = (C.c_void_p * 2)()
    assert lib.splpak_b200_comm_init_all(2, devs, comms) == 0
    half = len(x) // 2
    res = [None, None]

    def rank(r):
        # one host thread per device: the call all-reduces (and waits) inside
        torch.cuda.set_device(r)
        lo, hi = (0, half) if r == 0 else (half, len(x))
        h = robust_handle(ndim, mn, mx, nodes, 1.0, 0.0, "curvature")
        dev = torch.device("cuda", r)
        d_x, d_y, d_w = (torch.from_numpy(np.ascontiguousarray(a[lo:hi])).to(dev) for a in (x, y, w))
        d_c = torch.zeros(h.ncol, dtype=torch.float64, device=dev)
        info, ierr = h.robust_fit_device(d_x, ndim, d_y, d_w, hi - lo, d_c, psi="bisquare", max_iter=10,
                                         comm=comms[r])
        res[r] = (d_c.cpu().numpy(), info, ierr)
        h.destroy()

    threads = [threading.Thread(target=rank, args=(r,)) for r in range(2)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    torch.cuda.set_device(0)
    for r in range(2):
        assert lib.splpak_b200_comm_destroy(comms[r]) == 0
    assert res[0][2] == 0 and res[1][2] == 0, (res[0][1:], res[1][1:])
    assert np.array_equal(res[0][0], res[1][0])
    assert res[0][1] == res[1][1]
    one = robust_handle(ndim, mn, mx, nodes, 1.0, 0.0, "curvature")
    c1, info1, ierr = one.robust_fit(x, y, w, psi="bisquare", max_iter=10)
    assert ierr == 0
    assert res[0][1]["iterations"] == info1["iterations"] and res[0][1]["n_rejected"] == info1["n_rejected"]
    assert np.abs(res[0][0] - c1).max() <= 1e-9 * np.abs(c1).max()


def test_refusals():
    ndim, nodes = 2, [6, 6]
    x, y, w, mn, mx = make_problem(ndim, nodes, 500, seed=51, weighted=True)
    lib = sp.load()

    def call(h, **kw):
        a = dict(l1x=ndim, n=len(y), psi=1, tuning=0.0, max_iter=5, tol=1e-6, ncf=h.ncol, nout=6)
        a.update(kw)
        xa, ya, wa = (np.ascontiguousarray(v) for v in (x, y, w))
        coef, out, ierr = np.zeros(h.ncol), np.zeros(6), C.c_int(-1)
        rc = lib.splpak_b200_fit_robust(h.h, C.c_void_p(xa.ctypes.data), a["l1x"], C.c_void_p(ya.ctypes.data),
                                        C.c_void_p(wa.ctypes.data), 1, a["n"], a["psi"], a["tuning"], a["max_iter"],
                                        a["tol"], None, C.c_void_p(coef.ctypes.data), a["ncf"], None,
                                        C.c_void_p(out.ctypes.data), a["nout"], C.byref(ierr))
        assert rc == ierr.value
        return rc

    h = robust_handle(ndim, mn, mx, nodes, 0.0, 0.0, "curvature")
    for kw in (dict(psi=2), dict(psi=-1), dict(tuning=float("nan")), dict(tuning=float("inf")), dict(max_iter=0),
               dict(tol=-1.0), dict(tol=float("nan")), dict(nout=5), dict(l1x=1)):
        assert call(h, **kw) == 203, kw
    assert call(h, ncf=h.ncol - 1) == 104
    assert call(h, n=0) == 105
    assert call(h) == 0
    assert call(h) == 203                                   # used handle
    assert lib.splpak_b200_fit_refine_begin(h.h) == 203     # would walk back to the plain fit
    with pytest.raises(SplpakError):
        h.smoothing_score(0.0)
    assert h.reset() == 0
    assert call(h) == 0                                     # a reset handle is fresh again
    used = robust_handle(ndim, mn, mx, nodes, 0.0, 0.0, "curvature")
    assert used.add_points(x, y, w, weighted=True) == 0
    assert call(used) == 203
    ortho = sp.FitHandle(ndim, mn, mx, nodes, 0.0, solver="orthogonal")
    assert call(ortho) == 203
    with pytest.raises(SplpakError):
        h.robust_fit(x, y, w, psi="cauchy")
    # too few points for the columns: a non-positive pivot, 107
    few = robust_handle(ndim, mn, mx, nodes, 0.0, 0.0, "curvature")
    assert call(few, n=10) == 107


def test_cfg3_scale():
    """cfg3 size: 1e8 device-resident points, 24^3 nodes, 5 % gross outliers -> converged, held-out error at noise level."""
    import torch

    dev = torch.device("cuda", torch.cuda.current_device())
    n, ndim, nodes, noise = 100_000_000, 3, [24, 24, 24], 0.01
    gen = torch.Generator(device=dev)
    gen.manual_seed(7)
    x = torch.rand((n, ndim), dtype=torch.float64, device=dev, generator=gen)

    def f(t):
        return torch.sin(2 * t[:, 0]) * torch.cos(1.5 * t[:, 1]) + 0.5 * t[:, 2] ** 2

    y = f(x) + noise * torch.randn(n, dtype=torch.float64, device=dev, generator=gen)
    bad = torch.rand(n, dtype=torch.float64, device=dev, generator=gen) < 0.05
    y += bad * 50 * noise * torch.sign(torch.randn(n, dtype=torch.float64, device=dev, generator=gen))
    del bad
    mn, mx = np.zeros(ndim), np.ones(ndim)
    h = robust_handle(ndim, mn, mx, nodes, 0.0, 0.0, "curvature")
    d_c = torch.zeros(h.ncol, dtype=torch.float64, device=dev)
    info, ierr = h.robust_fit_device(x, ndim, y, None, n, d_c, psi="bisquare", max_iter=30, tol=1e-6)
    assert ierr == 0 and info["converged"], info
    del x, y
    q = torch.rand((200_000, ndim), dtype=torch.float64, device=dev, generator=gen)
    v = torch.zeros(len(q), dtype=torch.float64, device=dev)
    assert sp.eval_batch_device(ndim, q, ndim, len(q), d_c, mn, mx, nodes, v) == 0
    torch.cuda.synchronize()
    err = float(torch.sqrt(torch.mean((v - f(q)) ** 2)))
    assert err < 0.1 * noise, (err, info)
