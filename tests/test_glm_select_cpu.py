"""CPU checks of the host references behind test_gpu_glm_select: the known-scale criteria (UBRE, REML with phi = 1)
against their brute-force definitions, and the host copy of the device's lambda search on small cases."""
import numpy as np
import pytest

from test_gpu_glm_select import criterion, host_search, select_step
from test_gpu_smoothing import penalty_dense


def small_system(seed, n=60, nodes=(8,), weighted=True):
    """A random row-weighted working system on a 1-D grid: A0 = sqrt(W) P with a smooth P, b0 = sqrt(W) z."""
    rng = np.random.default_rng(seed)
    x = np.sort(rng.random(n))
    knots = np.linspace(0.0, 1.0, nodes[0])
    P = np.maximum(0.0, 1.0 - np.abs(x[:, None] - knots[None, :]) * (nodes[0] - 1) / 1.5) ** 2
    rw = rng.uniform(0.5, 2.0, n) if weighted else np.ones(n)
    z = np.sin(3 * x) + 0.3 * rng.standard_normal(n)
    R = penalty_dense(list(nodes), np.zeros(1), np.ones(1), "curvature")
    return dict(A0=rw[:, None] * P, b0=rw * z, Cc=np.zeros((0, nodes[0])), R=R, N=n)


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_ubre_matches_its_definition(seed):
    """U = ||(I - A) b||^2 / N - 1 + 2 tr(A) / N with the influence matrix A = X M^-1 X^T W formed densely."""
    s = small_system(seed)
    for lam in (1e-4, 1e-2, 1.0):
        got, M, _ = criterion("poisson", "prediction", s, lam, 2)
        A = s["A0"] @ np.linalg.solve(M, s["A0"].T)
        r = s["b0"] - A @ s["b0"]
        want = r @ r / s["N"] - 1.0 + 2.0 * np.trace(A) / s["N"]
        assert got == pytest.approx(want, rel=1e-11, abs=1e-13)


@pytest.mark.parametrize("seed", [0, 1])
def test_known_scale_reml_matches_the_restricted_likelihood(seed):
    """With phi = 1, -2 log of the restricted likelihood is, up to lambda-independent constants, the limit tau -> inf of
    -2 log N(b; 0, I + A Sigma_tau A^T) - Mp log tau, where the coefficients have the prior precision lambda R + I/tau
    on the null space of R (tau: its variance there).  Formed densely on the n x n covariance at tau and 2 tau (the
    error is O(1/tau): Richardson extrapolation removes it), against D_p + log|M| - (p - Mp) log lambda."""
    s = small_system(seed, n=40)
    A, b, R = s["A0"], s["b0"], s["R"]
    ev, V = np.linalg.eigh(R)
    null = ev < 1e-9 * ev.max()
    mp = int(null.sum())
    assert mp == 2
    logdet_r = float(np.log(ev[~null]).sum())
    n, p = A.shape

    def brute(lam, tau):
        prec = V @ np.diag(np.where(null, 1.0 / tau, lam * ev)) @ V.T
        cov = np.eye(n) + A @ np.linalg.solve(prec, A.T)
        sign, logdet = np.linalg.slogdet(cov)
        assert sign > 0
        m2ll = n * np.log(2 * np.pi) + logdet + b @ np.linalg.solve(cov, b)
        return m2ll + mp * np.log(1.0 / tau) - n * np.log(2 * np.pi) + logdet_r

    for lam in (1e-3, 1e-1, 10.0):
        got, _, _ = criterion("poisson", "reml", s, lam, mp)
        want = 2.0 * brute(lam, 2e5) - brute(lam, 1e5)
        assert got == pytest.approx(want, rel=1e-8), (lam, got, want)


def test_search_finds_the_minimum_of_a_smooth_function():
    for t0 in (-7.3, -2.0, 0.41, 3.6):
        t, v, n, glo, ghi = host_search(lambda t: (t - t0) ** 2 + 1.0, -10.0, 4.0)
        assert abs(t - t0) <= 0.02 and n > 29 and not glo and not ghi


def test_search_ties_go_to_the_larger_lambda_and_infinite_points_lose():
    t, v, _, glo, ghi = host_search(lambda t: 1.0, -2.0, 2.0)
    assert t == 2.0 and ghi and not glo
    t, v, _, _, _ = host_search(lambda t: np.inf if t < 0.5 else (t - 1.0) ** 2, -2.0, 2.0)
    assert abs(t - 1.0) <= 0.02
    t, v, n, _, _ = host_search(lambda t: np.inf, -1.0, 1.0)
    assert t is None and n > 0


def test_window_search_falls_back_to_the_whole_range():
    """k >= 2 searches lambda_(k-1) +- 1 decade; a best grid point at an end of that window that is not an end of the
    range sends the search over the whole range."""
    f = lambda t: (t + 6.0) ** 2                                  # noqa: E731
    t, _, n = select_step(f, 2, 0.0, -10.0, 4.0)
    assert abs(t + 6.0) <= 0.02 and n > 40
    t, _, n = select_step(f, 2, -6.2, -10.0, 4.0)
    assert abs(t + 6.0) <= 0.02 and n < 25
    # at an end of the range the window is clipped and no fallback happens
    t, _, n = select_step(lambda t: -t, 2, 3.8, -10.0, 4.0)
    assert t == 4.0 and n < 25


def test_search_on_a_working_system_matches_a_dense_grid():
    s = small_system(5, n=80, nodes=(10,))
    for family, crit in (("poisson", "reml"), ("poisson", "prediction"), ("gamma", "reml"), ("gamma", "prediction")):
        score = lambda t: criterion(family, crit, s, 10.0 ** t, 2)[0]   # noqa: E731
        t, v, _, _, _ = host_search(score, -8.0, 4.0)
        grid = np.linspace(-8.0, 4.0, 1201)
        vals = np.array([score(g) for g in grid])
        assert v <= vals.min() + 1e-6 * abs(vals.min()), (family, crit, v, vals.min())
        assert abs(t - grid[np.argmin(vals)]) <= 0.05, (family, crit, t, grid[np.argmin(vals)])


def test_unknown_names_raise_without_a_device():
    from splpak_b200.api import FitHandle, SplpakError

    h = FitHandle.__new__(FitHandle)
    for kw, msg in ((dict(family="probit"), "unknown family"), (dict(criterion="aic"), "unknown criterion"),
                    (dict(penalty="tension"), "unknown penalty")):
        a = dict(family="poisson", criterion="reml", penalty="curvature", lo=None, hi=None)
        a.update(kw)
        with pytest.raises(SplpakError, match=msg):
            h._glm_select_args(a["family"], a["criterion"], a["penalty"], a["lo"], a["hi"])
        with pytest.raises(SplpakError, match=msg):
            h.glm_select(np.zeros((3, 1)), np.zeros(3), **kw)
        with pytest.raises(SplpakError, match=msg):
            h.glm_select_device(0, 1, 0, None, 3, 0, **kw)
