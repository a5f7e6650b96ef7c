"""Smoothing fits (splpak_b200_fit_set_smoothing): the streaming Cholesky fit with a roughness penalty lambda * R.

The reference for the coefficients is the dense augmented least-squares problem [A; sqrt(lambda) R^(1/2)] c ~ [b; 0],
built independently of the penalty kernels: A, b from the oracle's rows (constraint rows included when xtrap != 0), R as
the Kronecker sum of 1-D Gram matrices of the oracle's bascmp at 4-point Gauss-Legendre points."""
import ctypes as C

import numpy as np
import pytest

import splpak_b200 as sp
from splpak_b200.api import _ptr
from util import coef_tolerance, dense_from_stencil, make_problem

pytestmark = pytest.mark.gpu
EPS = np.finfo(float).eps
GL_T, GL_W = np.polynomial.legendre.leggauss(4)
_GRAM = {}


def gram_1d(n, lo, hi, k):
    """M^(k)[i][j] = integral over [lo, hi] of phi_i^(k) phi_j^(k), the functions of the reference's index box per cell."""
    key = (n, float(lo), float(hi), k)
    if key not in _GRAM:
        from oracle import Oracle

        o = Oracle()
        dx = (hi - lo) / (n - 1)
        M = np.zeros((n, n))
        for c in range(n - 1):
            box = range(max(c - 1, 0), min(c + 2, n - 1) + 1)
            for t, wq in zip(GL_T, GL_W):
                x = lo + (c + 0.5 + 0.5 * t) * dx
                phi = np.array([o.bascmp([i], [x], [k], [lo], [hi], [n])[1] for i in box])
                M[box.start:box.stop, box.start:box.stop] += 0.5 * dx * wq * np.outer(phi, phi)
        _GRAM[key] = M
    return _GRAM[key]


def penalty_dense(nodes, mn, mx, penalty):
    """R = sum over the penalty's terms of kron_d M_d^(k_d) (dimension 1 fastest in the column index)."""
    ndim = len(nodes)
    terms = [(1.0, [2 if d == t else 0 for d in range(ndim)]) for t in range(ndim)]
    if penalty == "thin_plate":
        terms += [(2.0, [1 if d in (i, j) else 0 for d in range(ndim)]) for i in range(ndim) for j in range(i + 1, ndim)]
    R = 0.0
    for wt, ks in terms:
        K = np.ones((1, 1))
        for d in range(ndim):
            K = np.kron(gram_1d(nodes[d], mn[d], mx[d], ks[d]), K)
        R = R + wt * K
    return R


def smoothed_reference(oracle, ndim, x, y, w, mn, mx, nodes, xtrap, lam, penalty):
    """(c_smooth, c_plain, G + lam R, A) from dense least squares."""
    A, b = oracle.rows(ndim, x, y, w, mn, mx, nodes, xtrap)
    R = penalty_dense(nodes, mn, mx, penalty)
    ev, V = np.linalg.eigh(R)
    Rh = (V * np.sqrt(np.clip(ev, 0.0, None))) @ V.T
    Aa = np.vstack([A, np.sqrt(lam) * Rh])
    ba = np.concatenate([b, np.zeros(R.shape[0])])
    c = np.linalg.lstsq(Aa, ba, rcond=None)[0]
    c0 = np.linalg.lstsq(A, b, rcond=None)[0]
    return c, c0, A.T @ A + lam * R, A


def lam_for(nodes, mn, mx, penalty, G, f=1e-2):
    """lambda at a fixed fraction f of the data Gram scale against the penalty's."""
    R = penalty_dense(nodes, mn, mx, penalty)
    return f * np.abs(np.diag(G)).max() / np.abs(np.diag(R)).max()


def fit(ndim, x, y, w, mn, mx, nodes, xtrap, lam=None, penalty="curvature", refine=0, **kw):
    h = sp.FitHandle(ndim, mn, mx, nodes, xtrap, **kw)
    assert h.ierror == 0
    if lam is not None:
        assert h.set_smoothing(lam, penalty) == 0
    assert h.add_points(x, y, w) == 0
    c, ierr = h.compute()
    if ierr == 0 and refine:
        c, ierr = h.refine(x, y, w, steps=refine)
    return h, c, ierr


@pytest.mark.parametrize("ndim,nodes", [(1, [9]), (2, [6, 5]), (3, [5, 4, 6]), (4, [4, 5, 4, 4])])
@pytest.mark.parametrize("penalty", ["curvature", "thin_plate"])
def test_penalty_matrix(ndim, nodes, penalty):
    """S after a smoothed compute minus S after a plain one is lambda R, entry for entry (xtrap = 0: no constraint rows)."""
    x, y, w, mn, mx = make_problem(ndim, nodes, 3000, seed=5 + ndim, xmin=[-0.5] * ndim, xmax=[1.5 + 0.25 * d for d in range(ndim)])
    hp, _, _ = fit(ndim, x, y, w, mn, mx, nodes, 0.0)
    S0 = hp.normal_equations()[0]
    R = penalty_dense(nodes, mn, mx, penalty)
    lam = 0.37 * np.abs(S0).max() / np.abs(R).max()
    hs, _, ierr = fit(ndim, x, y, w, mn, mx, nodes, 0.0, lam, penalty)
    assert ierr == 0
    S1 = hs.normal_equations()[0]
    D = dense_from_stencil(S1 - S0, nodes)
    tol = 1e-13 * (np.abs(S0).max() + lam * np.abs(R).max())
    np.testing.assert_allclose(D, lam * R, rtol=0, atol=tol)
    hp.destroy()
    hs.destroy()


def test_large_grid_reads_the_tables_from_global_memory(oracle):
    """A 1-D grid of 700 nodes: the tables (67 KB) exceed the shared-memory staging limit of the add and residual kernels,
    which then read them through L1.  S + lambda R, the coefficients and one refinement step against the reference."""
    nodes = [700]
    x, y, w, mn, mx = make_problem(1, nodes, 20000, seed=8)
    A, _ = oracle.rows(1, x, y, w, mn, mx, nodes, 0.0)
    lam = lam_for(nodes, mn, mx, "curvature", A.T @ A)
    ref, ref0, Gl, _ = smoothed_reference(oracle, 1, x, y, w, mn, mx, nodes, 0.0, lam, "curvature")
    hp, _, _ = fit(1, x, y, w, mn, mx, nodes, 0.0)
    S0 = hp.normal_equations()[0]
    hp.destroy()
    h, c, ierr = fit(1, x, y, w, mn, mx, nodes, 0.0, lam, "curvature")
    assert ierr == 0
    R = penalty_dense(nodes, mn, mx, "curvature")
    D = dense_from_stencil(h.normal_equations()[0] - S0, nodes)
    np.testing.assert_allclose(D, lam * R, rtol=0, atol=1e-13 * (np.abs(S0).max() + lam * np.abs(R).max()))
    c1, ierr = h.refine(x, y, w, steps=1)
    h.destroy()
    assert ierr == 0
    tol, cond = coef_tolerance(Gl)
    scale = np.abs(ref).max()
    for got in (c, c1):
        np.testing.assert_allclose(got, ref, rtol=0, atol=tol * scale, err_msg=f"cond {cond:.2e}")
    assert np.abs(ref0 - ref).max() / scale > 100 * tol


SMOOTH_CASES = [
    # ndim, nodes, ndata, xtrap, weighted, hole, outside, penalty
    (1, [10], 200, 0.0, True, False, 0.0, "curvature"),
    (1, [12], 300, 1.0, False, True, 0.1, "thin_plate"),
    (2, [6, 7], 2000, 0.0, True, False, 0.2, "curvature"),
    (2, [9, 8], 3000, 1.0, False, True, 0.0, "thin_plate"),
    (3, [5, 4, 6], 4000, 0.0, True, False, 0.1, "thin_plate"),
    (3, [6, 6, 6], 5000, 1.0, True, True, 0.0, "curvature"),
    (4, [4, 4, 4, 4], 6000, 0.0, True, False, 0.0, "curvature"),
    (4, [5, 4, 5, 4], 8000, 0.5, False, True, 0.0, "thin_plate"),
]


@pytest.mark.parametrize("ndim,nodes,ndata,xtrap,weighted,hole,outside,penalty", SMOOTH_CASES)
def test_coefficients_match_augmented_least_squares(oracle, ndim, nodes, ndata, xtrap, weighted, hole, outside, penalty):
    """Coefficients of the smoothed fit against the dense augmented problem; the penalty visibly moves them.  Where the
    constraint rows fire, two refinement steps bring the fit to eps cond(A) as in the unsmoothed handle path."""
    x, y, w, mn, mx = make_problem(ndim, nodes, ndata, seed=ndim * 11 + nodes[0], weighted=weighted, hole=hole,
                                   outside=outside)
    A, _ = oracle.rows(ndim, x, y, w, mn, mx, nodes, xtrap)
    lam = lam_for(nodes, mn, mx, penalty, A.T @ A)
    ref, ref0, Gl, A = smoothed_reference(oracle, ndim, x, y, w, mn, mx, nodes, xtrap, lam, penalty)
    fired = A.shape[0] > len(x)
    if hole and xtrap != 0:
        assert fired, "constraint rows were expected to fire in this case"
    h, c, ierr = fit(ndim, x, y, w, mn, mx, nodes, xtrap, lam, penalty, refine=2 if fired else 0)
    assert ierr == 0
    h.destroy()
    tol, cond = coef_tolerance(Gl)
    if fired:
        tol = max(1e-10, 10.0 * EPS * np.sqrt(cond))
    scale = np.abs(ref).max()
    err = np.abs(c - ref).max() / scale
    assert err <= tol, f"coef rel err {err:.3e} > {tol:.3e} (cond {cond:.3e})"
    moved = np.abs(ref0 - ref).max() / scale
    assert moved > 100 * tol, f"the penalty moves the solution by only {moved:.3e} (tol {tol:.3e})"


@pytest.mark.parametrize("ndim,nodes,penalty", [(2, [9, 7], "curvature"), (3, [8, 6, 7], "curvature"),
                                                (4, [5, 6, 5, 4], "curvature"), (2, [9, 7], "thin_plate"),
                                                (3, [6, 7, 5], "thin_plate")])
def test_null_space_is_reproduced(ndim, nodes, penalty):
    """Multilinear data under the curvature penalty and affine data under thin plate are not penalised: the spline
    reproduces them, in and outside the box, for lambda over 12 decades of the data Gram scale.  The tolerance is that of
    test_multilinear_reproduction_K1 with cond(G + lambda R), but with the full eps cond: when lambda R dominates, the
    unpenalised component is fixed by G alone under entries ~cond times larger (0.5 eps cond measured at 1e6 x scale)."""
    rng = np.random.default_rng(ndim + len(penalty))
    x = rng.random((20000, ndim))
    a = rng.random(ndim) + 0.5
    b = rng.random(ndim) - 0.5
    if penalty == "curvature":
        f = lambda p: np.prod(a + b * p, axis=-1)
    else:
        f = lambda p: 0.3 + p @ b
    mn, mx = [0.0] * ndim, [1.0] * ndim
    h0 = sp.FitHandle(ndim, mn, mx, nodes, 0.0)
    assert h0.add_points(x, f(x), None) == 0
    S0 = h0.normal_equations()[0]
    h0.destroy()
    R = penalty_dense(nodes, mn, mx, penalty)
    base = np.abs(np.diag(dense_from_stencil(S0, nodes))).max() / np.abs(np.diag(R)).max()
    q = rng.random((500, ndim)) * 1.6 - 0.3
    for rel in (1e-6, 1.0, 1e6):
        lam = rel * base
        h = sp.FitHandle(ndim, mn, mx, nodes, 0.0)
        assert h.set_smoothing(lam, penalty) == 0
        assert h.add_points(x, f(x), None) == 0
        coef, ierr = h.compute()
        S = h.normal_equations()[0]
        h.destroy()
        assert ierr == 0
        cond = np.linalg.cond(dense_from_stencil(S, nodes))
        tol = max(5e-10, EPS * cond)
        v, _ = sp.eval_batch(ndim, q, coef, mn, mx, nodes)
        np.testing.assert_allclose(v, f(q), rtol=0, atol=tol, err_msg=f"lambda {rel:.0e} x scale, cond {cond:.2e}")


def test_hole_without_constraint_rows_is_bridged():
    """The rank-deficient hole problem of test_solver_failures_map_to_107 (xtrap = 0 -> 107) is well posed with
    lambda > 0: y = x is in the penalty's null space, so the fit reproduces it across the hole.  Fewer points than
    columns is no longer an error either."""
    xh = np.concatenate([np.linspace(0, 0.2, 40), np.linspace(0.8, 1, 40)]).reshape(-1, 1)
    for penalty in ("curvature", "thin_plate"):
        h = sp.FitHandle(1, [0.0], [1.0], [20], 0.0)
        assert h.set_smoothing(1e-4, penalty) == 0
        assert h.add_points(xh, xh[:, 0]) == 0
        coef, ierr = h.compute()
        tol = max(5e-10, 0.1 * EPS * np.linalg.cond(dense_from_stencil(h.normal_equations()[0], [20])))
        h.destroy()
        assert ierr == 0
        q = np.linspace(-0.1, 1.1, 121).reshape(-1, 1)
        v, _ = sp.eval_batch(1, q, coef, [0.0], [1.0], [20])
        np.testing.assert_allclose(v, q[:, 0], rtol=0, atol=tol)
    x5 = np.array([[0.1], [0.35], [0.5], [0.62], [0.9]])
    h = sp.FitHandle(1, [0.0], [1.0], [10], 0.0)
    assert h.set_smoothing(1e-3) == 0
    assert h.add_points(x5, 2.0 * x5[:, 0] - 1.0) == 0
    coef, ierr = h.compute()
    tol = max(5e-10, 0.1 * EPS * np.linalg.cond(dense_from_stencil(h.normal_equations()[0], [10])))
    h.destroy()
    assert ierr == 0
    v, _ = sp.eval_batch(1, np.linspace(0, 1, 11).reshape(-1, 1), coef, [0.0], [1.0], [10])
    np.testing.assert_allclose(v, 2.0 * np.linspace(0, 1, 11) - 1.0, rtol=0, atol=tol)


def test_lambda_zero_is_the_unsmoothed_fit(monkeypatch):
    """lambda = 0 launches nothing and changes nothing: coefficients and launch counts bit-identical to a handle without
    set_smoothing (deterministic mode, so that two fits can be compared bit for bit); lambda > 0 adds two launches."""
    monkeypatch.setenv("SPLPAK_B200_DETERMINISTIC", "1")
    x, y, w, mn, mx = make_problem(3, [6, 5, 6], 8000, seed=9, hole=True)
    nodes = [6, 5, 6]
    out = {}
    for mode in ("none", "zero", "positive"):
        h = sp.FitHandle(3, mn, mx, nodes, 1.0)
        if mode == "zero":
            assert h.set_smoothing(0.0, "thin_plate") == 0
        if mode == "positive":
            assert h.set_smoothing(1e-3, "curvature") == 0
        assert h.add_points(x, y, w) == 0
        h.synchronize()
        n0 = h.launch_count()
        c, ierr = h.compute()
        assert ierr == 0
        out[mode] = (c, h.launch_count() - n0)
        h.destroy()
    assert np.array_equal(out["none"][0], out["zero"][0])
    assert out["none"][1] == out["zero"][1]
    assert out["positive"][1] == out["none"][1] + 2
    assert not np.array_equal(out["none"][0], out["positive"][0])


def test_large_lambda_approaches_multilinear_least_squares():
    """lambda -> inf with the curvature penalty: the fit tends to the weighted least-squares fit on the multilinear
    features prod_d (1, x_d), at a distance that falls as 1/lambda."""
    ndim, nodes = 2, [7, 6]
    x, y, w, mn, mx = make_problem(ndim, nodes, 3000, seed=12)
    F = np.stack([np.ones(len(x)), x[:, 0], x[:, 1], x[:, 0] * x[:, 1]], axis=1)
    beta = np.linalg.lstsq(F * w[:, None], y * w, rcond=None)[0]
    q = np.random.default_rng(1).random((400, ndim)) * 1.4 - 0.2
    want = np.stack([np.ones(len(q)), q[:, 0], q[:, 1], q[:, 0] * q[:, 1]], axis=1) @ beta
    h0 = sp.FitHandle(ndim, mn, mx, nodes, 0.0)
    assert h0.add_points(x, y, w) == 0
    S0 = h0.normal_equations()[0]
    h0.destroy()
    base = np.abs(S0).max() / np.abs(penalty_dense(nodes, mn, mx, "curvature")).max()
    errs = []
    lams = (1e3 * base, 1e5 * base)
    for lam in lams:
        h, c, ierr = fit(ndim, x, y, w, mn, mx, nodes, 0.0, lam, "curvature")
        S = h.normal_equations()[0]
        h.destroy()
        assert ierr == 0
        v, _ = sp.eval_batch(ndim, q, c, mn, mx, nodes)
        floor = 10 * EPS * np.linalg.cond(dense_from_stencil(S, nodes)) * np.abs(c).max()
        errs.append((np.abs(v - want).max(), floor))
    assert errs[0][0] < 1e-2, errs
    # 100x the lambda -> ~100x closer (within 3x of the 1/lambda law, or down at the solver's own accuracy)
    assert errs[1][0] <= 3.0 * errs[0][0] * lams[0] / lams[1] + errs[1][1], errs


@pytest.mark.parametrize("ndim,nodes,n,seed,penalty", [(2, [9, 8], 6000, 3, "curvature"), (3, [7, 6, 8], 9000, 4, "thin_plate")])
def test_refinement_keeps_the_penalty(oracle, ndim, nodes, n, seed, penalty):
    """A hole with xtrap = 1 and lambda > 0: after two refinement steps the coefficients match the augmented reference
    at eps sqrt(cond(G + lambda R)) and stay far from the unsmoothed solution."""
    x, y, w, mn, mx = make_problem(ndim, nodes, n, seed=seed, hole=True)
    A, _ = oracle.rows(ndim, x, y, w, mn, mx, nodes, 1.0)
    lam = lam_for(nodes, mn, mx, penalty, A.T @ A)
    ref, ref0, Gl, _ = smoothed_reference(oracle, ndim, x, y, w, mn, mx, nodes, 1.0, lam, penalty)
    h, c0, ierr = fit(ndim, x, y, w, mn, mx, nodes, 1.0, lam, penalty)
    assert ierr == 0 and h.constraints_fired()
    c2, ierr = h.refine(x, y, w, steps=2)
    h.destroy()
    assert ierr == 0
    _, cond = coef_tolerance(Gl)
    tol = max(1e-10, 10.0 * EPS * np.sqrt(cond))
    scale = np.abs(ref).max()
    e0 = np.abs(c0 - ref).max() / scale
    e2 = np.abs(c2 - ref).max() / scale
    assert e2 <= tol, f"refined {e2:.2e} > {tol:.2e}, plain {e0:.2e}"
    assert np.abs(c2 - ref0).max() / scale > 100 * tol


def _refine_step_parts(handles, shards):
    """One refinement residual pass per emulated rank over its own shard; returns the summed right-hand sides."""
    import torch

    total = None
    for h, (x, y, w) in zip(handles, shards):
        assert h.lib.splpak_b200_fit_refine_begin(h.h) == 0
        xa, ya, wa = (np.ascontiguousarray(a) for a in (x, y, w))
        assert h.lib.splpak_b200_fit_refine_add_points(h.h, _ptr(xa), xa.shape[1], _ptr(ya), _ptr(wa), 1, len(xa)) == 0
        h.synchronize()
        t = h.rhs_tensor().clone()
        total = t if total is None else total + t
    torch.cuda.synchronize()
    return total


@pytest.mark.parametrize("nranks", [2, 4])
def test_emulated_ranks_count_the_penalty_once(oracle, nranks):
    """Multi-GPU contract on one device: every rank sets the same lambda, the partial buffers are summed and written back
    into every rank, each rank computes (the penalty is added after the sum, once) and gets bit-identical coefficients
    equal to the single-handle smoothed fit; one refinement step with the summed right-hand side does too."""
    import torch

    ndim, nodes = 2, [8, 8]
    x, y, w, mn, mx = make_problem(ndim, nodes, 6000, seed=44, hole=True)
    A, _ = oracle.rows(ndim, x, y, w, mn, mx, nodes, 1.0)
    lam = lam_for(nodes, mn, mx, "thin_plate", A.T @ A)
    full = sp.FitHandle(ndim, mn, mx, nodes, 1.0)
    assert full.set_smoothing(lam, "thin_plate") == 0
    assert full.add_points(x, y, w) == 0
    c_single, ierr = full.compute()
    assert ierr == 0
    S_full = full.normal_equations()[0]
    parts, shards, total = [], [], None
    for r in range(nranks):
        lo, hi = r * len(x) // nranks, (r + 1) * len(x) // nranks
        hr = sp.FitHandle(ndim, mn, mx, nodes, 1.0)
        assert hr.set_smoothing(lam, "thin_plate") == 0
        assert hr.add_points(x[lo:hi], y[lo:hi], w[lo:hi], weighted=True) == 0
        hr.synchronize()
        t = hr.partial_tensor().clone()
        total = t if total is None else total + t
        parts.append(hr)
        shards.append((x[lo:hi], y[lo:hi], w[lo:hi]))
    for hr in parts:
        hr.partial_tensor().copy_(total)
    torch.cuda.synchronize()
    coefs = []
    for hr in parts:
        c, ierr = hr.compute()
        assert ierr == 0
        coefs.append(c)
    for c in coefs[1:]:
        assert np.array_equal(c, coefs[0]), "the replicas differ"
    tol, cond = coef_tolerance(dense_from_stencil(S_full, nodes))
    scale = np.abs(c_single).max()
    np.testing.assert_allclose(coefs[0], c_single, rtol=0, atol=tol * scale)
    # one refinement step: residual passes per shard, summed right-hand side, re-solve on every rank
    c1_single, ierr = full.refine(x, y, w, steps=1)
    assert ierr == 0
    rhs = _refine_step_parts(parts, shards)
    ref1 = []
    for hr in parts:
        hr.rhs_tensor().copy_(rhs)
        torch.cuda.synchronize()
        c = np.zeros(hr.ncol)
        ie = C.c_int(0)
        hr.lib.splpak_b200_fit_refine_compute(hr.h, _ptr(c), hr.ncol, C.byref(ie))
        assert ie.value == 0
        ref1.append(c)
    for c in ref1[1:]:
        assert np.array_equal(c, ref1[0]), "the replicas differ after refinement"
    np.testing.assert_allclose(ref1[0], c1_single, rtol=0, atol=tol * scale)
    for p in parts:
        p.destroy()
    full.destroy()


@pytest.mark.parametrize("ndim,nodes,ndata", [(3, [9, 8, 10], 6000), (2, [24, 20], 5000), (1, [300], 5000),
                                              (1, [65], 3000), (2, [13, 5], 3000), (3, [5, 5, 5], 5000)])
def test_solver_paths_agree_on_smoothed_systems(oracle, monkeypatch, ndim, nodes, ndata):
    """The persistent kernels and SPLPAK_B200_SOLVER=graph solve the same smoothed system, both at parity with the
    augmented reference."""
    x, y, w, mn, mx = make_problem(ndim, nodes, ndata, seed=ndim + ndata)
    A, _ = oracle.rows(ndim, x, y, w, mn, mx, nodes, 0.0)
    lam = lam_for(nodes, mn, mx, "thin_plate", A.T @ A)
    ref, _, Gl, _ = smoothed_reference(oracle, ndim, x, y, w, mn, mx, nodes, 0.0, lam, "thin_plate")
    tol, cond = coef_tolerance(Gl)
    scale = np.abs(ref).max()
    got = {}
    for mode in ("persistent", "graph"):
        if mode == "graph":
            monkeypatch.setenv("SPLPAK_B200_SOLVER", "graph")
        else:
            monkeypatch.delenv("SPLPAK_B200_SOLVER", raising=False)
        h, c, ierr = fit(ndim, x, y, w, mn, mx, nodes, 0.0, lam, "thin_plate")
        h.destroy()
        assert ierr == 0, mode
        np.testing.assert_allclose(c, ref, rtol=0, atol=tol * scale, err_msg=f"{mode}, cond {cond:.2e}")
        got[mode] = c
    np.testing.assert_allclose(got["persistent"], got["graph"], rtol=0, atol=tol * scale)


def test_deterministic_mode_with_smoothing(monkeypatch):
    monkeypatch.setenv("SPLPAK_B200_DETERMINISTIC", "1")
    x, y, w, mn, mx = make_problem(3, [7, 6, 8], 50_000, seed=71, hole=True, outside=0.05)
    runs = []
    for _ in range(2):
        h, c, ierr = fit(3, x, y, w, mn, mx, [7, 6, 8], 1.0, 2e-3, "thin_plate", refine=1)
        assert ierr == 0
        runs.append((h.normal_equations()[0].copy(), c.copy()))
        h.destroy()
    assert np.array_equal(runs[0][0], runs[1][0])
    assert np.array_equal(runs[0][1], runs[1][1])


def test_streaming_chunks_and_reset_keep_the_setting():
    """Chunked add_points with set_smoothing before or after the points equals one shot; the setting survives reset."""
    nodes = [6, 5, 6]
    x, y, w, mn, mx = make_problem(3, nodes, 9000, seed=33, hole=True)
    h1, one, ierr = fit(3, x, y, w, mn, mx, nodes, 1.0, 5e-3, "curvature")
    assert ierr == 0
    tol, cond = coef_tolerance(dense_from_stencil(h1.normal_equations()[0], nodes))
    scale = np.abs(one).max()
    for when in ("before", "after"):
        h = sp.FitHandle(3, mn, mx, nodes, 1.0)
        if when == "before":
            assert h.set_smoothing(5e-3, "curvature") == 0
        for lo in range(0, len(x), 2500):
            assert h.add_points(x[lo:lo + 2500], y[lo:lo + 2500], w[lo:lo + 2500]) == 0
        if when == "after":
            assert h.set_smoothing(5e-3, "curvature") == 0
        c, ierr = h.compute()
        assert ierr == 0
        np.testing.assert_allclose(c, one, rtol=0, atol=tol * scale, err_msg=f"{when}, cond {cond:.2e}")
        h.destroy()
    assert h1.reset() == 0
    assert h1.add_points(x, y, w) == 0
    again, ierr = h1.compute()
    assert ierr == 0
    np.testing.assert_allclose(again, one, rtol=0, atol=tol * scale)
    h1.destroy()


def test_refusals(monkeypatch):
    nodes = [6, 6]
    x, y, w, mn, mx = make_problem(2, nodes, 2000, seed=3)
    h = sp.FitHandle(2, mn, mx, nodes, 1.0)
    for lam in (-1e-3, float("nan"), float("inf"), -float("inf")):
        assert h.set_smoothing(lam) == 203, lam
    assert h.set_smoothing(1e-3, 2) == 203
    assert h.set_smoothing(1e-3, -1) == 203
    with pytest.raises(sp.SplpakError):
        h.set_smoothing(1e-3, "biharmonic")
    # the handle is still usable and unsmoothed after the refused calls
    assert h.add_points(x, y, w) == 0
    c, ierr = h.compute()
    assert ierr == 0
    plain, ierr = sp.splcw(2, x, 2, y, w, len(x), mn, mx, nodes, 1.0, quiet=True)
    tol, _ = coef_tolerance(dense_from_stencil(h.normal_equations()[0], nodes))
    np.testing.assert_allclose(c, plain, rtol=0, atol=max(tol, 1e-9) * np.abs(plain).max())
    assert h.set_smoothing(1e-3) == 203                       # finalized
    assert h.reset() == 0 and h.set_smoothing(1e-3) == 0      # usable again after reset
    h.destroy()
    # orthogonal solver, both orders
    ho = sp.FitHandle(2, mn, mx, nodes, 1.0, solver="orthogonal")
    assert ho.set_smoothing(1e-3) == 203
    assert ho.set_smoothing(0.0) == 0
    assert ho.add_points(x, y, w) == 0
    assert ho.compute()[1] == 0
    ho.destroy()
    hc = sp.FitHandle(2, mn, mx, nodes, 1.0)
    assert hc.set_smoothing(1e-3, "thin_plate") == 0
    assert hc.lib.splpak_b200_fit_set_solver(hc.h, 1) == 203
    assert hc.solver() == "cholesky"
    assert hc.add_points(x, y, w) == 0
    assert hc.compute()[1] == 0
    hc.destroy()
    monkeypatch.setenv("SPLPAK_B200_FIT", "orthogonal")
    he = sp.FitHandle(2, mn, mx, nodes, 1.0)
    assert he.solver() == "orthogonal"
    assert he.set_smoothing(1e-3) == 203
    assert he.add_points(x, y, w) == 0
    assert he.compute()[1] == 0
    he.destroy()


def test_real32_smoothed_fit(oracle32):
    """REAL32 library: lambda stays a double and the penalty and solve are FP64; a 2-D smoothed fit agrees with the
    real64 one on the float32-rounded inputs to the rounding of the outputs and of the grid spacing."""
    nodes = [6, 6]
    x, y, w, mn, mx = make_problem(2, nodes, 1500, seed=55)
    x32, y32, w32 = (a.astype(np.float32) for a in (x, y, w))
    h32 = sp.FitHandle(2, mn, mx, nodes, 1.0, real32=True)
    assert h32.set_smoothing(3e-3, "thin_plate") == 0
    assert h32.add_points(x32, y32, w32) == 0
    c32, ierr = h32.compute()
    h32.destroy()
    assert ierr == 0 and c32.dtype == np.float32
    h64, c64, ierr = fit(2, *(a.astype(np.float64) for a in (x32, y32, w32)), mn, mx, nodes, 1.0, 3e-3, "thin_plate")
    h64.destroy()
    assert ierr == 0
    np.testing.assert_allclose(c32, c64, rtol=0, atol=100.0 * float(np.finfo(np.float32).eps) * np.abs(c64).max())
