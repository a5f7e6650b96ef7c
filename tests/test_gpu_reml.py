"""Choosing lambda by REML (splpak_b200_fit_reml_score / select_smoothing_reml).

References are dense and built from the oracle's rows, independently of the device kernels, as in test_gpu_gcv.py:
M = G0 + C + lambda R, c = M^-1 g0, n = the data rows plus the constraint rows, D_p = |b0 - A0 c|^2 + c^T (C + lambda R) c
(the constraint rows have a zero response), log|M| from numpy.linalg.slogdet, and
V_R = (n - Mp) log(D_p / (n - Mp)) + log|M| - (p - Mp) log lambda."""
import ctypes as C

import numpy as np
import pytest

import splpak_b200 as sp
from splpak_b200.api import SplpakError
from splpak_b200.distributed import fit_sharded
from test_gpu_gcv import SCORE_CASES, dense_system, gcv_handle, half_bandwidth, rho_of
from test_gpu_smoothing import penalty_dense
from util import dense_from_stencil, make_problem

pytestmark = pytest.mark.gpu
EPS = np.finfo(float).eps


def null_dim(ndim, penalty):
    return 2 ** ndim if penalty == "curvature" else ndim + 1


def dense_reml(oracle, ndim, x, y, w, mn, mx, nodes, xtrap, lam, penalty):
    """The dense reference: a dict of V_R, D_p, log|M|, n with M, c, g0 and the solved system's pieces."""
    M, G0, g0, A0, b0 = dense_system(oracle, ndim, x, y, w, mn, mx, nodes, xtrap, lam, penalty)
    ncon = 0
    if xtrap != 0.0:
        ncon = (oracle.rows(ndim, x, y, w, mn, mx, nodes, xtrap)[0].shape[0]
                - oracle.rows(ndim, x, y, w, mn, mx, nodes, 0.0)[0].shape[0])
    n = A0.shape[0] + ncon
    p, mp = M.shape[0], null_dim(ndim, penalty)
    c = np.linalg.solve(M, g0)
    dp = float(((b0 - A0 @ c) ** 2).sum() + c @ (M - G0) @ c)
    sign, logdet = np.linalg.slogdet(M)
    assert sign > 0
    v = (n - mp) * np.log(dp / (n - mp)) + logdet - (p - mp) * np.log(lam)
    return {"reml": v, "dp": dp, "logdet": logdet, "n": n}, M, c, g0


def check_against_dense(got, ref, M, c, g0, mp, constrained):
    """First-order bounds for a backward error |E| <= 100 eps |M| of the factor (and of the assembly):
        |d log|M|| <= 100 eps sum |Sigma_ij M_ij|  (+ the fixed-order sum of p logs: 2 p eps sum |log L_jj|)
        |d D_p|    <= 100 eps (|c|^T |M| |c| + ywy + 2 |c.g| + c^T M c)
    and V_R held to the propagated sum.  Each bound must be small enough to discriminate; V_R is used through its
    differences over lambda, so its bound must be below 1e-2.  Where constraint rows fire, their Gram entries are ~dxin^4
    times the data's and cancel in c^T C c, so |c|^T |C| |c| dominates the componentwise bound: there (the 1-D and 2-D
    cases with a hole at the smaller lambda) the V_R bound reaches 2e-2 and is required to be below 5e-2."""
    Sig = np.linalg.inv(M)
    p = M.shape[0]
    L = np.linalg.cholesky(M)
    tol_logdet = 100 * EPS * np.abs(Sig * M).sum() + 2 * p * EPS * np.abs(np.log(np.diag(L))).sum()
    absc = np.abs(c)
    tol_dp = 100 * EPS * (absc @ np.abs(M) @ absc + got["ywy"] + 2 * abs(c @ g0) + c @ M @ c)
    tol_v = (ref["n"] - mp) * tol_dp / ref["dp"] + tol_logdet + 10 * EPS * abs(ref["reml"])
    msg = (f"cond(M) {np.linalg.cond(M):.2e}, tol logdet {tol_logdet:.2e}, tol dp {tol_dp:.2e} ({tol_dp / ref['dp']:.1e} "
           f"relative), tol V {tol_v:.2e}")
    assert tol_dp < 1e-3 * ref["dp"] and tol_logdet < 1e-6 * max(1.0, abs(ref["logdet"])), msg
    assert tol_v < (5e-2 if constrained else 1e-2), msg
    assert got["n"] == ref["n"], (got["n"], ref["n"])
    assert abs(got["logdet"] - ref["logdet"]) <= tol_logdet, (got, ref, msg)
    assert abs(got["dp"] - ref["dp"]) <= tol_dp, (got, ref, msg)
    assert abs(got["reml"] - ref["reml"]) <= tol_v, (got, ref, msg)


@pytest.mark.parametrize("ndim,nodes,ndata,xtrap,weighted,hole,outside,penalty", SCORE_CASES)
def test_scores_match_dense_reference(oracle, ndim, nodes, ndata, xtrap, weighted, hole, outside, penalty):
    x, y, w, mn, mx = make_problem(ndim, nodes, ndata, seed=ndim * 11 + nodes[0], weighted=weighted, hole=hole,
                                   outside=outside)
    wv = w if weighted else None
    h = gcv_handle(ndim, mn, mx, nodes, xtrap, x, y, wv)
    A0, _ = oracle.rows(ndim, x, y, wv, mn, mx, nodes, 0.0)
    rho = rho_of(nodes, mn, mx, penalty, A0.T @ A0)
    for f in (1e-3, 1e-1):
        lam = f * rho
        ref, M, c, g0 = dense_reml(oracle, ndim, x, y, wv, mn, mx, nodes, xtrap, lam, penalty)
        got = h.reml_score(lam, penalty)
        mp = null_dim(ndim, penalty)
        assert got["phi"] == got["dp"] / (got["n"] - mp)
        check_against_dense(got, ref, M, c, g0, mp, xtrap != 0.0)
    h.destroy()


@pytest.mark.parametrize("ndim,nodes,penalty", [(1, [9], "curvature"), (1, [9], "thin_plate"), (2, [6, 5], "curvature"),
                                                (2, [6, 5], "thin_plate"), (3, [4, 5, 4], "curvature"),
                                                (3, [4, 5, 4], "thin_plate"), (4, [4, 4, 4, 4], "curvature"),
                                                (4, [4, 4, 4, 4], "thin_plate")])
def test_null_space_dimension(ndim, nodes, penalty):
    """The dense R has exactly p - Mp eigenvalues above 1e-10 of the largest."""
    mn, mx = np.zeros(ndim), np.linspace(1.0, 2.0, ndim)
    ev = np.linalg.eigvalsh(penalty_dense(nodes, mn, mx, penalty))
    p = int(np.prod(nodes))
    assert int((ev > 1e-10 * ev.max()).sum()) == p - null_dim(ndim, penalty)


@pytest.mark.parametrize("ndim,nodes,penalty", [(1, [30], "curvature"), (2, [10, 9], "curvature"),
                                                (2, [10, 9], "thin_plate"), (3, [6, 7, 6], "thin_plate")])
def test_analytic_limits(oracle, ndim, nodes, penalty):
    """lambda -> inf: V_R -> (n - Mp) log(D_null / (n - Mp)) + log pdet(R) + log det(Z^T (G0 + C) Z), Z an orthonormal
    null basis of R and D_null the residual of the least-squares fit within the null space; the distance falls like
    1/lambda.  lambda -> 0 along a grid: V_R rises without bound, by about (p - Mp) log 100 per two decades."""
    ncol = int(np.prod(nodes))
    x, y, w, mn, mx = make_problem(ndim, nodes, 40 * ncol, seed=5 + ndim)
    h = gcv_handle(ndim, mn, mx, nodes, 0.0, x, y, w)
    A, b = oracle.rows(ndim, x, y, w, mn, mx, nodes, 0.0)
    keep = np.abs(A).sum(axis=1) > 0
    A, b = A[keep], b[keep]
    n, mp = A.shape[0], null_dim(ndim, penalty)
    R = penalty_dense(nodes, mn, mx, penalty)
    ev, U = np.linalg.eigh(R)
    order = np.argsort(ev)
    Z = U[:, order[:mp]]
    log_pdet = np.log(ev[order[mp:]]).sum()
    AZ = A @ Z
    z = np.linalg.lstsq(AZ, b, rcond=None)[0]
    d_null = float(((b - AZ @ z) ** 2).sum())
    v_inf = (n - mp) * np.log(d_null / (n - mp)) + log_pdet + np.linalg.slogdet(AZ.T @ AZ)[1]
    rho = np.trace(A.T @ A) / np.trace(R)
    e1 = h.reml_score(1e5 * rho, penalty)["reml"] - v_inf
    e2 = h.reml_score(1e6 * rho, penalty)["reml"] - v_inf
    e3 = h.reml_score(1e8 * rho, penalty)["reml"] - v_inf
    assert 7 < e1 / e2 < 13, (e1, e2)
    # at 1e8 rho the 1/lambda law gives 1e-3 e1; the rest (about 2e-3 in the dense reference itself) is the rounding
    # of log|M| with the penalty's entries 1e8 times the data's
    assert abs(e3) < 1e-2 * abs(e1), (e1, e3)
    vs = [h.reml_score(10.0 ** t * rho, penalty)["reml"] for t in (-8, -10, -12, -14)]
    step = (ncol - mp) * np.log(100.0)
    assert all(0.9 * step < b_ - a_ < 1.1 * step for a_, b_ in zip(vs, vs[1:])), (vs, step)
    h.destroy()


def noisy_problem(ndim, nodes, n, sigma, seed):
    rng = np.random.default_rng(seed)
    x = rng.random((n, ndim))
    truth = lambda p: np.sin(4 * p[:, 0]) + (np.cos(3 * p[:, 1]) * p[:, 0] if p.shape[1] > 1 else 0.0)
    y = truth(x) + sigma * rng.standard_normal(n)
    return x, y, truth


@pytest.mark.parametrize("ndim,nodes,penalty", [(1, [40], "curvature"), (2, [12, 11], "thin_plate")])
def test_selection_matches_dense_minimiser(oracle, ndim, nodes, penalty):
    """The selected lambda is within 0.03 decades of the minimiser of the dense V_R on a fine grid; the returned V_R is
    at most every trace row."""
    x, y, _ = noisy_problem(ndim, nodes, 1500 * ndim, 0.1, seed=ndim)
    mn, mx = np.zeros(ndim), np.ones(ndim)
    h = gcv_handle(ndim, mn, mx, nodes, 0.0, x, y, None)
    lam, score, trace = h.select_smoothing(penalty, criterion="reml")
    assert trace.shape[1] == 4 and len(trace) > 10
    ok = np.isfinite(trace[:, 1])
    assert score["reml"] <= trace[ok, 1].min()
    assert np.any(trace[:, 0] == lam)
    row = trace[trace[:, 0] == lam][0]
    assert (row[1], row[2], row[3]) == (score["reml"], score["dp"], score["logdet"])
    h.destroy()
    A, b = oracle.rows(ndim, x, y, None, mn, mx, nodes, 0.0)
    G0, g0, ywy = A.T @ A, A.T @ b, float(b @ b)
    R = penalty_dense(nodes, mn, mx, penalty)
    n, p, mp = A.shape[0], G0.shape[0], null_dim(ndim, penalty)

    def v(t):
        lm = 10.0 ** t
        M = G0 + lm * R
        c = np.linalg.solve(M, g0)
        dp = ywy - 2 * c @ g0 + c @ M @ c
        return (n - mp) * np.log(dp / (n - mp)) + np.linalg.slogdet(M)[1] - (p - mp) * np.log(lm)

    t_sel = np.log10(lam)
    coarse = np.arange(t_sel - 3, t_sel + 3, 0.05)
    t0 = coarse[np.argmin([v(t) for t in coarse])]
    fine = np.arange(t0 - 0.1, t0 + 0.1, 0.002)
    t_min = fine[np.argmin([v(t) for t in fine])]
    assert abs(t_sel - t_min) <= 0.03, (t_sel, t_min)


def test_noise_level_and_sparse_data():
    """2-D, 200,000 points, sigma = 0.1: phi recovers sigma^2 within 5 %.  N ~ 3 ncol noisy samples: the selected fit's
    RMS error against the truth beats the fits at both ends of the search range."""
    nodes = [12, 12]
    rng = np.random.default_rng(123)
    n = 200_000
    x = rng.random((n, 2))
    sigma = 0.1
    y = np.sin(3 * x[:, 0]) * np.cos(2 * x[:, 1]) + sigma * rng.standard_normal(n)
    mn, mx = np.zeros(2), np.ones(2)
    h = gcv_handle(2, mn, mx, nodes, 0.0, x, y, None)
    lam, score, trace = h.select_smoothing("curvature", criterion="reml")
    assert abs(score["phi"] / sigma ** 2 - 1) < 0.05, score
    assert score["n"] == n
    h.destroy()

    nodes = [14, 14]
    ncol = 196
    rng = np.random.default_rng(7)
    x = rng.random((3 * ncol, 2))
    truth = lambda p: np.sin(4 * p[:, 0]) + np.cos(3 * p[:, 1]) * p[:, 0]
    y = truth(x) + 0.2 * rng.standard_normal(len(x))
    h = gcv_handle(2, mn, mx, nodes, 0.0, x, y, None)
    lam, score, trace = h.select_smoothing("thin_plate", criterion="reml")
    g = np.stack(np.meshgrid(np.linspace(0, 1, 41), np.linspace(0, 1, 41)), -1).reshape(-1, 2)
    errs = {}
    for name, l in (("best", lam), ("lo", trace[0, 0]), ("hi", trace[:, 0].max())):
        f = sp.FitHandle(2, mn, mx, nodes, 0.0)
        assert f.set_smoothing(l, "thin_plate") == 0
        assert f.add_points(x, y) == 0
        c, ierr = f.compute()
        assert ierr == 0
        v = sp.eval_batch(2, g, c, mn, mx, nodes)
        v = v[0] if isinstance(v, tuple) else v
        errs[name] = float(np.sqrt(np.mean((v - truth(g)) ** 2)))
        f.destroy()
    h.destroy()
    assert errs["best"] < errs["lo"] and errs["best"] < errs["hi"], errs


def selected_inverse_rc(h):
    n = C.c_int64(0)
    return h.lib.splpak_b200_fit_get_selected_inverse(h.h, None, 0, C.byref(n))


def test_no_selected_inverse_and_the_variance_hazard(monkeypatch):
    """reml_score leaves a factor, not Sigma, in the band storage: get_selected_inverse returns 203 after it, and
    smoothing_score(l1) -> reml_score(l2) -> set_smoothing(l1) -> prepare_variance builds the tables of a fresh handle
    (the reuse check of prepare_variance must not take the factor for Sigma).  prepare_variance after
    select_smoothing_reml scores by GCV once and gives a fresh handle's tables and sigma2."""
    monkeypatch.setenv("SPLPAK_B200_DETERMINISTIC", "1")
    nodes = [9, 8]
    x, y, w, mn, mx = make_problem(2, nodes, 8000, seed=12, hole=True)
    q = make_problem(2, nodes, 500, seed=13, outside=0.1)[0]
    l1, l2 = 1e-3, 3e-2

    def fresh(lam):
        f = gcv_handle(2, mn, mx, nodes, 1.0, x, y, w)
        assert f.set_smoothing(lam, "curvature") == 0
        pv = f.prepare_variance()
        out = [f.variance(q, nderiv=nd)[0] for nd in ([0, 0], [1, 0], [0, 2])]
        f.destroy()
        return pv, out

    h = gcv_handle(2, mn, mx, nodes, 1.0, x, y, w)
    h.smoothing_score(l1, "curvature")
    assert selected_inverse_rc(h) == 0
    h.reml_score(l2, "curvature")
    assert selected_inverse_rc(h) == 203
    with pytest.raises(SplpakError):
        h.selected_inverse()
    assert h.set_smoothing(l1, "curvature") == 0
    pv = h.prepare_variance()
    got = [h.variance(q, nderiv=nd)[0] for nd in ([0, 0], [1, 0], [0, 2])]
    h.destroy()
    pv_ref, want = fresh(l1)
    assert pv == pv_ref
    for a, b in zip(got, want):
        assert np.array_equal(a, b)

    h = gcv_handle(2, mn, mx, nodes, 1.0, x, y, w)
    lam, score, _ = h.select_smoothing("curvature", criterion="reml")
    assert selected_inverse_rc(h) == 203
    n0 = h.launch_count()
    pv = h.prepare_variance()
    assert h.launch_count() > n0 + 1                          # one GCV score, then the table build
    assert pv["sigma2"] == pv["rss"] / (pv["n"] - pv["edf"])
    got = [h.variance(q, nderiv=nd)[0] for nd in ([0, 0], [1, 0], [0, 2])]
    h.destroy()
    pv_ref, want = fresh(lam)
    assert pv == pv_ref
    for a, b in zip(got, want):
        assert np.array_equal(a, b)


def test_no_side_effects(monkeypatch):
    """Deterministic mode: compute after REML scores and a REML selection is bit-identical to a fresh handle's compute
    with the selected lambda; S is untouched; compute and a GCV score launch what they launch without REML calls; the
    GCV selection returns the same lambda, scores and trace whether or not REML calls came before it."""
    monkeypatch.setenv("SPLPAK_B200_DETERMINISTIC", "1")
    nodes = [8, 7, 6]
    x, y, w, mn, mx = make_problem(3, nodes, 30000, seed=17, hole=True)
    h = gcv_handle(3, mn, mx, nodes, 1.0, x, y, w)
    S_before = h.normal_equations()[0].copy()
    for lam in (1e-6, 1e-3, 1.0):
        h.reml_score(lam, "thin_plate")
    lam, score, trace = h.select_smoothing("thin_plate", criterion="reml")
    assert np.array_equal(h.normal_equations()[0], S_before)
    n0 = h.launch_count()
    c1, ierr = h.compute()
    assert ierr == 0
    n_compute = h.launch_count() - n0
    h.destroy()
    f = gcv_handle(3, mn, mx, nodes, 1.0, x, y, w)
    assert f.set_smoothing(lam, "thin_plate") == 0
    n0 = f.launch_count()
    c2, ierr = f.compute()
    assert ierr == 0
    assert f.launch_count() - n0 == n_compute
    f.destroy()
    assert np.array_equal(c1, c2)

    res = {}
    for mode in ("gcv", "reml_first"):
        h = gcv_handle(3, mn, mx, nodes, 1.0, x, y, w)
        if mode == "reml_first":
            h.reml_score(1e-4, "curvature")
            h.select_smoothing("curvature", criterion="reml")
        s = h.smoothing_score(1e-3, "curvature")
        n0 = h.launch_count()                            # a second score: S1 = G0 + C is cached in both modes
        assert h.smoothing_score(1e-3, "curvature") == s
        n_score = h.launch_count() - n0
        sel = h.select_smoothing("curvature")
        res[mode] = (s, n_score, sel[0], sel[1], sel[2].copy(), h.selected_inverse().copy())
        h.destroy()
    a, b = res["gcv"], res["reml_first"]
    assert a[:4] == b[:4]
    assert np.array_equal(a[4], b[4]) and np.array_equal(a[5], b[5])


def test_determinism_ranks_and_fit_sharded(monkeypatch):
    """Repeated scores are bit-identical on one handle and on two handles holding the same buffer; 2 and 3 emulated
    ranks (partial buffers summed and written back) select the same lambda bit for bit; fit_sharded(criterion="reml")
    gives the coefficients of a direct REML selection (deterministic assembly: both handles hold the same sums)."""
    import torch

    ndim, nodes = 2, [8, 8]
    x, y, w, mn, mx = make_problem(ndim, nodes, 6000, seed=44, hole=True)
    h = gcv_handle(ndim, mn, mx, nodes, 1.0, x, y, w)
    a = h.reml_score(1e-3, "thin_plate")
    h.reml_score(1e-1, "thin_plate")
    assert h.reml_score(1e-3, "thin_plate") == a
    h2 = gcv_handle(ndim, mn, mx, nodes, 1.0, x[:10], y[:10], w[:10])
    h.synchronize()
    h2.synchronize()
    h2.partial_tensor().copy_(h.partial_tensor())
    torch.cuda.synchronize()
    assert h2.reml_score(1e-3, "thin_plate") == a
    assert h2.select_smoothing("thin_plate", criterion="reml")[:2] == h.select_smoothing("thin_plate", criterion="reml")[:2]
    h.destroy()
    h2.destroy()
    for nranks in (2, 3):
        parts, total = [], None
        for r in range(nranks):
            lo, hi = r * len(x) // nranks, (r + 1) * len(x) // nranks
            hr = gcv_handle(ndim, mn, mx, nodes, 1.0, x[lo:hi], y[lo:hi], w[lo:hi])
            hr.synchronize()
            t = hr.partial_tensor().clone()
            total = t if total is None else total + t
            parts.append(hr)
        for hr in parts:
            hr.partial_tensor().copy_(total)
        torch.cuda.synchronize()
        res = [(hr.reml_score(1e-3, "thin_plate"), hr.select_smoothing("thin_plate", criterion="reml")[:2])
               for hr in parts]
        for r in res[1:]:
            assert r == res[0]
        # the summed buffer differs from the single handle's in its rounding; (n - Mp) ~ 6,000 times the relative
        # change of D_p moves V_R by ~1e-5
        np.testing.assert_allclose(res[0][0]["reml"], a["reml"], rtol=1e-7)
        for hr in parts:
            hr.destroy()

    monkeypatch.setenv("SPLPAK_B200_DETERMINISTIC", "1")
    hs = sp.FitHandle(ndim, mn, mx, nodes, 1.0)
    assert hs.enable_gcv() == 0
    coef, ierr = fit_sharded(hs, x, y, w, select_smoothing="thin_plate", criterion="reml")
    assert ierr == 0
    hs.destroy()
    hd = gcv_handle(ndim, mn, mx, nodes, 1.0, x, y, w)
    hd.select_smoothing("thin_plate", criterion="reml")
    c2, ierr = hd.compute()
    assert ierr == 0
    hd.destroy()
    assert np.array_equal(coef, c2)


@pytest.mark.parametrize("ndim,nodes,ndata,xtrap,weighted,hole,outside,penalty",
                         [SCORE_CASES[1], SCORE_CASES[3], SCORE_CASES[5], SCORE_CASES[7], SCORE_CASES[8]])
def test_solver_paths_agree(oracle, monkeypatch, ndim, nodes, ndata, xtrap, weighted, hole, outside, penalty):
    """SPLPAK_B200_SOLVER=graph (kernel-per-phase factor) against the dense reference with the bounds of the score test,
    and against the default path."""
    x, y, w, mn, mx = make_problem(ndim, nodes, ndata, seed=ndim * 11 + nodes[0], weighted=weighted, hole=hole,
                                   outside=outside)
    wv = w if weighted else None
    A0, _ = oracle.rows(ndim, x, y, wv, mn, mx, nodes, 0.0)
    lam = 1e-3 * rho_of(nodes, mn, mx, penalty, A0.T @ A0)
    ref, M, c, g0 = dense_reml(oracle, ndim, x, y, wv, mn, mx, nodes, xtrap, lam, penalty)
    got = {}
    for solver in ("persistent", "graph"):
        if solver == "graph":
            monkeypatch.setenv("SPLPAK_B200_SOLVER", "graph")
        else:
            monkeypatch.delenv("SPLPAK_B200_SOLVER", raising=False)
        h = gcv_handle(ndim, mn, mx, nodes, xtrap, x, y, wv)
        got[solver] = h.reml_score(lam, penalty)
        h.destroy()
        check_against_dense(got[solver], ref, M, c, g0, null_dim(ndim, penalty), xtrap != 0.0)


def test_scale_cfg3_logdet_against_banded_cholesky():
    """cfg3 (24^3, xtrap = 1, 1e8 device-resident points): log|M| against scipy's cholesky_banded of the band of
    fit_get_normal_equations after a compute at the same lambda (S + C + lambda R), within 100 eps sum |Sigma_ij M_ij|
    (Sigma's band from the GCV score of the same lambda) plus the summation of the logs."""
    import torch
    from scipy.linalg import cholesky_banded

    nodes = [24, 24, 24]
    n = 100_000_000
    g = torch.Generator(device="cuda").manual_seed(9)
    x = torch.rand((n, 3), dtype=torch.float64, device="cuda", generator=g)
    y = torch.sin(3 * x[:, 0]) + x[:, 1] * x[:, 2] + 0.05 * torch.randn(n, dtype=torch.float64, device="cuda", generator=g)
    w = 0.5 + torch.rand(n, dtype=torch.float64, device="cuda", generator=g)
    mn, mx = np.zeros(3), np.ones(3)
    h = sp.FitHandle(3, mn, mx, nodes, 1.0)
    assert h.enable_gcv() == 0
    assert h.add_points_device(x, 3, y, w, n) == 0
    del x, y, w
    lam = 1e-2
    s = h.reml_score(lam, "curvature")
    assert s["n"] >= n and np.isfinite(s["reml"])
    h.smoothing_score(lam, "curvature")
    Sig = h.selected_inverse()
    assert h.set_smoothing(lam, "curvature") == 0
    c, ierr = h.compute()
    assert ierr == 0
    S = h.normal_equations()[0]
    ncol = h.ncol
    h.destroy()
    torch.cuda.empty_cache()
    bw = half_bandwidth(nodes)
    M = dense_from_stencil(S, nodes)
    ab = np.zeros((bw + 1, ncol))
    for k in range(bw + 1):
        ab[k, : ncol - k] = np.diagonal(M, -k)
    del M
    L = cholesky_banded(ab, lower=True)
    logL = np.log(L[0])
    ref = 2.0 * logL.sum()
    mag = np.abs(Sig[:, 0] * ab[0]).sum()
    for k in range(1, bw + 1):
        mag += 2.0 * np.abs(Sig[: ncol - k, k] * ab[k, : ncol - k]).sum()
    tol = 100 * EPS * mag + 2 * ncol * EPS * np.abs(logL).sum()
    assert tol < 1e-6 * abs(ref)
    assert abs(s["logdet"] - ref) <= tol, (s["logdet"], ref, tol)


def test_scale_cfg4_score():
    nodes = [12, 12, 12, 12]
    n = 4_000_000
    rng = np.random.default_rng(4)
    x = rng.random((n, 4))
    y = np.sin(2 * x[:, 0]) * x[:, 1] + x[:, 2] - x[:, 3] ** 2 + 0.01 * rng.standard_normal(n)
    mn, mx = np.zeros(4), np.ones(4)
    h = gcv_handle(4, mn, mx, nodes, 1.0, x, y, None)
    s = h.reml_score(1e-4, "curvature")
    assert np.isfinite(s["reml"]) and s["dp"] > 0 and s["n"] >= n
    h.destroy()


def test_real32_scores_agree_with_real64():
    """The score path is FP64 in both libraries; the assembly of S and g differs in rounding, so 1e-5 relative, as
    the GCV scores."""
    nodes = [9, 8]
    x, y, w, mn, mx = make_problem(2, nodes, 20000, seed=13, hole=True)
    x, y, w = (a.astype(np.float32) for a in (x, y, w))
    out = []
    for real32 in (False, True):
        h = sp.FitHandle(2, mn, mx, nodes, 1.0, real32=real32)
        assert h.enable_gcv() == 0
        args = (x, y, w) if real32 else (x.astype(np.float64), y.astype(np.float64), w.astype(np.float64))
        assert h.add_points(*args) == 0
        out.append(h.reml_score(1e-3, "curvature"))
        h.destroy()
    for k in out[0]:
        np.testing.assert_allclose(out[1][k], out[0][k], rtol=1e-5, err_msg=k)


def test_refusals(monkeypatch):
    nodes = [6, 6]
    x, y, w, mn, mx = make_problem(2, nodes, 2000, seed=3)
    h = sp.FitHandle(2, mn, mx, nodes, 1.0)
    assert h.add_points(x, y, w) == 0
    with pytest.raises(SplpakError) as e:
        h.reml_score(1e-3)                                        # GCV not enabled
    assert e.value.args[1] == 203
    with pytest.raises(SplpakError) as e:
        h.select_smoothing(criterion="reml")
    assert e.value.args[1] == 203
    h.destroy()
    h = gcv_handle(2, mn, mx, nodes, 1.0, x, y, w)
    for lam in (0.0, -1e-3, float("nan"), float("inf")):
        with pytest.raises(SplpakError) as e:
            h.reml_score(lam)
        assert e.value.args[1] == 203
    with pytest.raises(SplpakError) as e:
        h.reml_score(1e-3, 2)
    assert e.value.args[1] == 203
    out = np.zeros(6)
    ierr = C.c_int(0)
    assert h.lib.splpak_b200_fit_reml_score(h.h, 1e-3, 0, out.ctypes.data_as(C.c_void_p), 5, C.byref(ierr)) == 203
    assert ierr.value == 203
    lam = C.c_double(0.0)
    nt = C.c_int64(0)
    assert h.lib.splpak_b200_fit_select_smoothing_reml(h.h, 0, 0.0, 0.0, C.byref(lam), out.ctypes.data_as(C.c_void_p),
                                                       5, None, 0, C.byref(nt), C.byref(ierr)) == 203
    with pytest.raises(SplpakError) as e:
        h.select_smoothing(lo=1.0, hi=1e-3, criterion="reml")
    assert e.value.args[1] == 203
    with pytest.raises(SplpakError):
        h.select_smoothing(criterion="aic")
    assert h.compute()[1] == 0
    with pytest.raises(SplpakError) as e:
        h.reml_score(1e-3)                                        # finalized
    assert e.value.args[1] == 203
    h.destroy()
    monkeypatch.setenv("SPLPAK_B200_FIT", "orthogonal")
    he = sp.FitHandle(2, mn, mx, nodes, 1.0)
    assert he.solver() == "orthogonal"
    assert he.add_points(x, y, w) == 0
    with pytest.raises(SplpakError) as e:
        he.reml_score(1e-3)                                       # orthogonal solver
    assert e.value.args[1] == 203
    he.destroy()
