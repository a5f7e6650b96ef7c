"""Generalized cross-validation of smoothing fits (splpak_b200_fit_smoothing_score / select_smoothing) and the band
selected inverse behind it.

References are dense and built from the oracle's rows, independently of the device kernels: G0 = A^T A of the data rows,
C = the constraint rows' Gram, R the penalty (penalty_dense), M = G0 + C + lambda R, Sigma = inv(M),
edf = tr(A M^-1 A^T), RSS from the residuals of the dense solution, V = N RSS / (N - edf)^2."""
import numpy as np
import pytest

import splpak_b200 as sp
from splpak_b200.api import SplpakError
from splpak_b200.distributed import partial_layout
from test_gpu_smoothing import SMOOTH_CASES, penalty_dense
from util import make_problem

pytestmark = pytest.mark.gpu
EPS = np.finfo(float).eps


def dense_system(oracle, ndim, x, y, w, mn, mx, nodes, xtrap, lam, penalty):
    """(M, G0, g0, A0, b0) of the dense reference."""
    A0, b0 = oracle.rows(ndim, x, y, w, mn, mx, nodes, 0.0)
    keep = np.abs(A0).sum(axis=1) > 0
    A0, b0 = A0[keep], b0[keep]
    G0 = A0.T @ A0
    M = G0.copy()
    if xtrap != 0.0:
        Ax, _ = oracle.rows(ndim, x, y, w, mn, mx, nodes, xtrap)
        M = Ax.T @ Ax
    if lam > 0:
        M = M + lam * penalty_dense(nodes, mn, mx, penalty)
    return M, G0, A0.T @ b0, A0, b0


def dense_scores(M, G0, g0, A0, b0, N):
    c = np.linalg.solve(M, g0)
    rss = float(((b0 - A0 @ c) ** 2).sum())
    edf = float(np.trace(np.linalg.solve(M, G0)))
    return {"gcv": N * rss / (N - edf) ** 2, "rss": rss, "edf": edf}


def band_of(Sig, bw):
    n = Sig.shape[0]
    out = np.zeros((n, bw + 1))
    for k in range(bw + 1):
        out[: n - k, k] = np.diagonal(Sig, k)
    return out


def half_bandwidth(nodes):
    b, s = 0, 1
    for n in nodes:
        b += 3 * s
        s *= n
    return min(b, int(np.prod(nodes)) - 1)


def gcv_handle(ndim, mn, mx, nodes, xtrap, x, y, w, **kw):
    h = sp.FitHandle(ndim, mn, mx, nodes, xtrap, **kw)
    assert h.ierror == 0
    assert h.enable_gcv() == 0
    assert h.add_points(x, y, w) == 0
    return h


def rho_of(nodes, mn, mx, penalty, G0):
    return np.trace(G0) / np.trace(penalty_dense(nodes, mn, mx, penalty))


SELINV_CASES = [
    # ndim, nodes, ndata, xtrap, lambda factor (x rho), penalty
    (1, [700], 20000, 0.0, 0.0, "curvature"),
    (1, [700], 3000, 1.0, 1e-4, "thin_plate"),
    (2, [20, 19], 20000, 1.0, 0.0, "curvature"),
    (3, [9, 8, 7], 30000, 0.0, 1e-3, "curvature"),
    (3, [9, 8, 7], 5000, 1.0, 1e-3, "thin_plate"),
    (4, [5, 4, 4, 5], 30000, 1.0, 1e-2, "thin_plate"),
    # odd ncol with more than one panel: the score scratch must keep the X panel 16-byte aligned
    (2, [9, 9], 3000, 1.0, 1e-3, "curvature"),
    (1, [101], 2000, 0.0, 0.0, "curvature"),
    (3, [5, 5, 5], 6000, 1.0, 1e-3, "thin_plate"),
]


@pytest.mark.parametrize("solver", ["persistent", "graph"])
@pytest.mark.parametrize("ndim,nodes,ndata,xtrap,lamf,penalty", SELINV_CASES)
def test_selected_inverse_matches_dense_inverse(oracle, monkeypatch, solver, ndim, nodes, ndata, xtrap, lamf, penalty):
    """Every band entry of Sigma against inv(M), at 100 eps cond(M) max|Sigma| (the forward error of an inverse formed
    from a backward-stable factor)."""
    if solver == "graph":
        monkeypatch.setenv("SPLPAK_B200_SOLVER", "graph")
    else:
        monkeypatch.delenv("SPLPAK_B200_SOLVER", raising=False)
    x, y, w, mn, mx = make_problem(ndim, nodes, ndata, seed=ndim * 7 + nodes[0], hole=xtrap != 0.0)
    A0, _ = oracle.rows(ndim, x, y, w, mn, mx, nodes, 0.0)
    lam = lamf * rho_of(nodes, mn, mx, penalty, A0.T @ A0) if lamf > 0 else 0.0
    M, *_ = dense_system(oracle, ndim, x, y, w, mn, mx, nodes, xtrap, lam, penalty)
    h = gcv_handle(ndim, mn, mx, nodes, xtrap, x, y, w)
    h.smoothing_score(lam, penalty)
    got = h.selected_inverse()
    h.destroy()
    bw = half_bandwidth(nodes)
    assert got.shape == (M.shape[0], bw + 1)
    Sig = np.linalg.inv(M)
    ref = band_of(Sig, bw)
    tol = 100 * EPS * np.linalg.cond(M) * np.abs(Sig).max()
    np.testing.assert_allclose(got, ref, rtol=0, atol=tol)


SCORE_CASES = SMOOTH_CASES + [
    # odd ncol with more than one panel
    (2, [9, 9], 3000, 1.0, True, True, 0.0, "curvature"),
    (3, [5, 5, 5], 4000, 0.0, True, False, 0.0, "thin_plate"),
    (1, [101], 1500, 0.0, False, False, 0.0, "thin_plate"),
]


@pytest.mark.parametrize("ndim,nodes,ndata,xtrap,weighted,hole,outside,penalty", SCORE_CASES)
def test_scores_match_dense_reference(oracle, ndim, nodes, ndata, xtrap, weighted, hole, outside, penalty):
    """V, RSS and edf against the dense reference at two lambdas.  The tolerances are first-order perturbation bounds
    for a backward error E of M with |E| <= 100 eps |M| (the Cholesky factor, the selected inverse and the dense
    reference are all backward stable), not cond(M) bounds:
        |d edf| <= |E| tr(Sigma G0 Sigma) + 100 eps sum |Sigma_ij G0_ij|
        |d RSS| <= 2 |Sigma A^T r| |E| |c| + 100 eps (ywy + 2 |c.g0| + c^T G0 c)   (the second term: the cancellation)
    Each is also required to be below 1e-3 of the quantity, so that the comparison discriminates on every case."""
    x, y, w, mn, mx = make_problem(ndim, nodes, ndata, seed=ndim * 11 + nodes[0], weighted=weighted, hole=hole,
                                   outside=outside)
    h = gcv_handle(ndim, mn, mx, nodes, xtrap, x, y, w if weighted else None)
    A0, _ = oracle.rows(ndim, x, y, w if weighted else None, mn, mx, nodes, 0.0)
    rho = rho_of(nodes, mn, mx, penalty, A0.T @ A0)
    for f in (1e-4, 1e-1):
        lam = f * rho
        M, G0, g0, A, b = dense_system(oracle, ndim, x, y, w if weighted else None, mn, mx, nodes, xtrap, lam, penalty)
        N = A.shape[0]
        ref = dense_scores(M, G0, g0, A, b, N)
        got = h.smoothing_score(lam, penalty)
        assert got["n"] == N
        np.testing.assert_allclose(got["ywy"], float((b ** 2).sum()), rtol=1e-13)
        Sig = np.linalg.inv(M)
        c = Sig @ g0
        r = b - A @ c
        dM = 100 * EPS * np.linalg.norm(M, 2)
        tol_edf = dM * np.trace(Sig @ G0 @ Sig) + 100 * EPS * np.abs(Sig * G0).sum()
        tol_rss = (2 * np.linalg.norm(Sig @ (A.T @ r)) * dM * np.linalg.norm(c)
                   + 100 * EPS * (got["ywy"] + 2 * abs(c @ g0) + c @ G0 @ c))
        msg = f"lambda {lam:.3e}, cond(M) {np.linalg.cond(M):.2e}, tol edf {tol_edf:.2e}, tol rss {tol_rss:.2e}"
        assert tol_edf < 1e-3 * ref["edf"] and tol_rss < 1e-3 * ref["rss"], msg
        assert abs(got["edf"] - ref["edf"]) <= tol_edf, (got, ref, msg)
        assert abs(got["rss"] - ref["rss"]) <= tol_rss, (got, ref, msg)
        # V = N RSS / (N - edf)^2: relative error propagated from the two
        rel_v = tol_rss / ref["rss"] + 2 * tol_edf / (N - ref["edf"])
        np.testing.assert_allclose(got["gcv"], ref["gcv"], rtol=rel_v, err_msg=msg)
    h.destroy()


@pytest.mark.parametrize("ndim,nodes,penalty,null_dim", [(1, [30], "curvature", 2), (2, [10, 9], "curvature", 4),
                                                          (2, [10, 9], "thin_plate", 3),
                                                          (3, [6, 7, 6], "thin_plate", 4)])
def test_analytic_limits(ndim, nodes, penalty, null_dim):
    """lambda = 0 without constraint rows: edf = ncol.  Large lambda: edf -> dim of the penalty's null space (2^ndim for
    curvature, ndim + 1 for thin plate), the distance falling as 1/lambda.  edf strictly decreasing along a grid."""
    ncol = int(np.prod(nodes))
    x, y, w, mn, mx = make_problem(ndim, nodes, 40 * ncol, seed=5 + ndim)
    h = gcv_handle(ndim, mn, mx, nodes, 0.0, x, y, w)
    s0 = h.smoothing_score(0.0, penalty)
    assert abs(s0["edf"] - ncol) <= 1e-8 * ncol
    G = h.normal_equations()[0]
    rho = G.reshape(ncol, -1)[:, 0].sum() / np.trace(penalty_dense(nodes, mn, mx, penalty))
    assert abs(h.smoothing_score(1e8 * rho, penalty)["edf"] - null_dim) < 1e-3
    # (between 1e5 and 1e6: far enough from the eps cond(M) floor that the ratio is the 1/lambda law's)
    e1 = h.smoothing_score(1e5 * rho, penalty)["edf"] - null_dim
    e2 = h.smoothing_score(1e6 * rho, penalty)["edf"] - null_dim
    assert 0 < e2 < e1
    assert 7 < e1 / e2 < 13, (e1, e2)
    edfs = [h.smoothing_score(10.0 ** t * rho, penalty)["edf"] for t in np.arange(-8, 4.5, 1.0)]
    assert all(a > b for a, b in zip(edfs, edfs[1:])), edfs
    h.destroy()


def test_no_side_effects_on_compute(monkeypatch):
    """Deterministic mode: enable_gcv, several scores and a selection, then compute, give coefficients bit-identical to a
    fresh handle with set_smoothing(best) + compute."""
    monkeypatch.setenv("SPLPAK_B200_DETERMINISTIC", "1")
    nodes = [8, 7, 6]
    x, y, w, mn, mx = make_problem(3, nodes, 30000, seed=17, hole=True)
    h = gcv_handle(3, mn, mx, nodes, 1.0, x, y, w)
    S_before = h.normal_equations()[0].copy()
    for lam in (0.0, 1e-6, 1e-3):
        h.smoothing_score(lam, "thin_plate")
    lam, score, trace = h.select_smoothing("thin_plate")
    assert np.array_equal(h.normal_equations()[0], S_before)
    c1, ierr = h.compute()
    assert ierr == 0
    h.destroy()
    f = sp.FitHandle(3, mn, mx, nodes, 1.0)
    assert f.set_smoothing(lam, "thin_plate") == 0
    assert f.add_points(x, y, w) == 0
    c2, ierr = f.compute()
    assert ierr == 0
    f.destroy()
    assert np.array_equal(c1, c2)


def test_without_enable_gcv_nothing_changes():
    """Without enable_gcv: the partial buffer has today's size and add_points + compute today's launch count."""
    nodes = [7, 6]
    x, y, w, mn, mx = make_problem(2, nodes, 5000, seed=2)
    counts = {}
    for mode in ("plain", "gcv"):
        h = sp.FitHandle(2, mn, mx, nodes, 1.0)
        if mode == "gcv":
            assert h.enable_gcv() == 0
        assert h.add_points(x, y, w) == 0
        h.synchronize()
        n_part = h.partial_tensor().numel()
        c, ierr = h.compute()
        assert ierr == 0
        counts[mode] = (n_part, h.launch_count())
        h.destroy()
    _, total = partial_layout(2, nodes)
    assert counts["plain"][0] == total
    assert counts["gcv"][0] == total + 1
    # the ywy kernel and its finish per chunk are the only extra launches
    assert counts["gcv"][1] == counts["plain"][1] + 2


def test_selection_trace_and_noise_level():
    """The returned V is <= every trace row; rows are well formed; RSS / (N - edf) recovers sigma^2 within 5 %."""
    nodes = [12, 12]
    rng = np.random.default_rng(123)
    n = 200_000
    x = rng.random((n, 2))
    sigma = 0.1
    y = np.sin(3 * x[:, 0]) * np.cos(2 * x[:, 1]) + sigma * rng.standard_normal(n)
    mn, mx = np.zeros(2), np.ones(2)
    h = gcv_handle(2, mn, mx, nodes, 0.0, x, y, None)
    lam, score, trace = h.select_smoothing("curvature")
    assert trace.shape[1] == 4 and len(trace) > 10
    assert np.all(trace[:, 0] > 0)
    ok = np.isfinite(trace[:, 1])
    assert score["gcv"] <= trace[ok, 1].min()
    assert np.any(trace[:, 0] == lam)
    assert np.all(trace[ok, 3] > 0) and np.all(trace[ok, 3] <= h.ncol + 1e-6)
    s2 = score["rss"] / (score["n"] - score["edf"])
    assert abs(s2 / sigma ** 2 - 1) < 0.05, s2
    # the selected inverse left behind is the selected lambda's, whichever point the search evaluated last
    sig_sel = h.selected_inverse().copy()
    assert h.smoothing_score(lam, "curvature") == score
    assert np.array_equal(h.selected_inverse(), sig_sel)
    h.destroy()


def test_selection_beats_both_ends_on_sparse_data():
    """N ~ 3 ncol noisy samples: the selected fit's RMS error against the true function on a test grid beats the fits
    at both ends of the search range."""
    nodes = [14, 14]
    ncol = 196
    rng = np.random.default_rng(7)
    x = rng.random((3 * ncol, 2))
    truth = lambda p: np.sin(4 * p[:, 0]) + np.cos(3 * p[:, 1]) * p[:, 0]
    y = truth(x) + 0.2 * rng.standard_normal(len(x))
    mn, mx = np.zeros(2), np.ones(2)
    h = gcv_handle(2, mn, mx, nodes, 0.0, x, y, None)
    lam, score, trace = h.select_smoothing("thin_plate")
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


def test_repeated_scores_bit_identical():
    nodes = [9, 8, 7]
    x, y, w, mn, mx = make_problem(3, nodes, 40000, seed=31, hole=True)
    h = gcv_handle(3, mn, mx, nodes, 1.0, x, y, w)
    a = h.smoothing_score(1e-4, "curvature")
    s_a = h.selected_inverse().copy()
    h.smoothing_score(1e-1, "curvature")
    b = h.smoothing_score(1e-4, "curvature")
    assert a == b
    assert np.array_equal(s_a, h.selected_inverse())
    h.destroy()


@pytest.mark.parametrize("nranks", [2, 3])
def test_emulated_ranks_select_the_same_lambda(nranks):
    """Per-rank handles, partial buffers (ywy included) summed and written back: every rank gets the same scores and the
    same lambda, bit for bit; the summed ywy matches the single handle's."""
    import torch

    ndim, nodes = 2, [8, 8]
    x, y, w, mn, mx = make_problem(ndim, nodes, 6000, seed=44, hole=True)
    full = gcv_handle(ndim, mn, mx, nodes, 1.0, x, y, w)
    s_full = full.smoothing_score(1e-3, "thin_plate")
    full.destroy()
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
    res = [(hr.smoothing_score(1e-3, "thin_plate"), hr.select_smoothing("thin_plate")[:2]) for hr in parts]
    for r in res[1:]:
        assert r == res[0]
    np.testing.assert_allclose(res[0][0]["ywy"], s_full["ywy"], rtol=1e-13)
    np.testing.assert_allclose(res[0][0]["gcv"], s_full["gcv"], rtol=1e-9)
    for hr in parts:
        hr.destroy()


def test_streaming_and_reset():
    """Chunked add_points gives the scores of one shot (to rounding); reset zeroes ywy and keeps the setting."""
    nodes = [10, 9]
    x, y, w, mn, mx = make_problem(2, nodes, 20000, seed=8, hole=True)
    one = gcv_handle(2, mn, mx, nodes, 1.0, x, y, w)
    a = one.smoothing_score(1e-3, "curvature")
    ch = sp.FitHandle(2, mn, mx, nodes, 1.0)
    assert ch.enable_gcv() == 0
    for k in range(0, len(x), 3001):
        assert ch.add_points(x[k:k + 3001], y[k:k + 3001], w[k:k + 3001]) == 0
    b = ch.smoothing_score(1e-3, "curvature")
    for k in a:
        np.testing.assert_allclose(b[k], a[k], rtol=1e-9)
    assert one.reset() == 0
    one.synchronize()
    off, total = partial_layout(2, nodes, gcv=True)
    buf = one.partial_tensor().cpu().numpy()
    assert len(buf) == total and buf[off["ywy"][0]] == 0.0
    assert one.add_points(x, y, w) == 0
    c = one.smoothing_score(1e-3, "curvature")
    for k in a:
        np.testing.assert_allclose(c[k], a[k], rtol=1e-9)
    one.destroy()
    ch.destroy()


def test_refusals(monkeypatch):
    nodes = [6, 6]
    x, y, w, mn, mx = make_problem(2, nodes, 2000, seed=3)
    lib = sp.FitHandle(2, mn, mx, nodes, 1.0).lib
    h = sp.FitHandle(2, mn, mx, nodes, 1.0)
    with pytest.raises(SplpakError):
        h.smoothing_score(1e-3)                                   # GCV not enabled
    assert h.add_points(x, y, w) == 0
    assert h.enable_gcv() == 203                                  # after add_points
    h.destroy()
    h = gcv_handle(2, mn, mx, nodes, 1.0, x, y, w)
    assert lib.splpak_b200_fit_set_solver(h.h, 1) == 203          # orthogonal after enable_gcv
    for lam in (-1e-3, float("nan"), float("inf")):
        with pytest.raises(SplpakError) as e:
            h.smoothing_score(lam)
        assert e.value.args[1] == 203
    with pytest.raises(SplpakError) as e:
        h.smoothing_score(1e-3, 2)
    assert e.value.args[1] == 203
    with pytest.raises(SplpakError) as e:
        h.select_smoothing(lo=1.0, hi=1e-3)
    assert e.value.args[1] == 203
    assert h.compute()[1] == 0
    with pytest.raises(SplpakError) as e:
        h.smoothing_score(1e-3)                                   # finalized
    assert e.value.args[1] == 203
    h.destroy()
    # 107: a singular system (too few points, lambda = 0, no constraint rows)
    h = gcv_handle(2, mn, mx, nodes, 0.0, x[:10], y[:10], w[:10])
    with pytest.raises(SplpakError) as e:
        h.smoothing_score(0.0)
    assert e.value.args[1] == 107
    with pytest.raises(SplpakError) as e:
        h.select_smoothing(lo=1e-30, hi=1e-29)
    assert e.value.args[1] == 107
    h.destroy()
    monkeypatch.setenv("SPLPAK_B200_FIT", "orthogonal")
    he = sp.FitHandle(2, mn, mx, nodes, 1.0)
    assert he.solver() == "orthogonal"
    assert he.enable_gcv() == 203
    he.destroy()


def test_real32_scores_agree_with_real64():
    """REAL32 library on float-rounded inputs: the score path is FP64 in both libraries; what differs is the
    assembly of S and g, which the REAL32 library does not form bit-identically (measured: 4e-7 relative in V on this
    problem), so the scores agree to 1e-5 relative."""
    nodes = [9, 8]
    x, y, w, mn, mx = make_problem(2, nodes, 20000, seed=13, hole=True)
    x, y, w = (a.astype(np.float32) for a in (x, y, w))
    out = []
    for real32 in (False, True):
        h = sp.FitHandle(2, mn, mx, nodes, 1.0, real32=real32)
        assert h.enable_gcv() == 0
        args = (x, y, w) if real32 else (x.astype(np.float64), y.astype(np.float64), w.astype(np.float64))
        assert h.add_points(*args) == 0
        out.append(h.smoothing_score(1e-3, "curvature"))
        h.destroy()
    for k in out[0]:
        np.testing.assert_allclose(out[1][k], out[0][k], rtol=1e-5, err_msg=k)


def test_scale_cfg3_columns_of_sigma():
    """cfg3 grid (24^3, xtrap = 1, 1e7 points): six columns of Sigma against scipy's banded solve of M e_j."""
    from scipy.linalg import solveh_banded

    nodes = [24, 24, 24]
    n = 10_000_000
    rng = np.random.default_rng(3)
    x = rng.random((n, 3))
    y = np.sin(3 * x[:, 0]) + x[:, 1] * x[:, 2] + 0.01 * rng.standard_normal(n)
    mn, mx = np.zeros(3), np.ones(3)
    h = gcv_handle(3, mn, mx, nodes, 1.0, x, y, None)
    lam = 1e-6
    s = h.smoothing_score(lam, "curvature")
    assert 0 < s["edf"] < h.ncol
    Sig = h.selected_inverse()
    # M = G0 + C + lam R from the handle's own system: compute() with the same lambda returns S + C + lam R
    assert h.set_smoothing(lam, "curvature") == 0
    c, ierr = h.compute()
    assert ierr == 0
    S = h.normal_equations()[0]
    h.destroy()
    from util import dense_from_stencil

    ncol = h.ncol
    bw = half_bandwidth(nodes)
    M = dense_from_stencil(S, nodes)
    ab = np.zeros((bw + 1, ncol))
    for k in range(bw + 1):
        ab[k, : ncol - k] = np.diagonal(M, -k)
    cols = [0, ncol // 2, ncol - 1] + list(np.random.default_rng(0).integers(0, ncol, 3))
    for j in cols:
        e = np.zeros(ncol)
        e[j] = 1.0
        ref = solveh_banded(ab, e, lower=True)
        got = np.array([Sig[j, i - j] if i >= j else Sig[i, j - i] for i in range(max(0, j - bw), min(ncol, j + bw + 1))])
        want = ref[max(0, j - bw): min(ncol, j + bw + 1)]
        np.testing.assert_allclose(got, want, rtol=0, atol=1e-8 * np.abs(want).max())


def test_scale_cfg4_score():
    nodes = [12, 12, 12, 12]
    n = 4_000_000
    rng = np.random.default_rng(4)
    x = rng.random((n, 4))
    y = np.sin(2 * x[:, 0]) * x[:, 1] + x[:, 2] - x[:, 3] ** 2 + 0.01 * rng.standard_normal(n)
    mn, mx = np.zeros(4), np.ones(4)
    h = gcv_handle(4, mn, mx, nodes, 1.0, x, y, None)
    s = h.smoothing_score(1e-4, "curvature")
    assert 2 ** 4 < s["edf"] < h.ncol
    assert np.isfinite(s["gcv"])
    h.destroy()
