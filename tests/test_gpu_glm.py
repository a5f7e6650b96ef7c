"""GLM fits (splpak_b200_fit_glm / fit_glm_device): penalized IRLS for Poisson, binomial and Gamma responses.

The reference is a host PIRLS in numpy built independently of the device kernels: the basis rows of every point from the
oracle (oracle.rows), the constraint rows of oracle.rows with the first iteration's row weights, the dense penalty of
test_gpu_smoothing, R's links, clamps, start values and unit deviances written out here, glm.fit's halving rule, and
lstsq on the row-weighted augmented system [sqrt(W) P; C; sqrt(lam) R^1/2].  Runs with tol = 0 and max_iter = k compare
the same iterate."""
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
EPS = 2.0 ** -52


class Family:
    """R's poisson(log), binomial(logit) and Gamma(log): make.link clamps, glm.fit's mustart, dev.resids."""

    def __init__(self, name):
        self.name = name

    def valid(self, y):
        if self.name == "poisson":
            return np.isfinite(y) & (y >= 0)
        if self.name == "binomial":
            return (y >= 0) & (y <= 1)
        return np.isfinite(y) & (y > 0)

    def start(self, y, a):
        return {"poisson": y + 0.1, "binomial": (a * y + 0.5) / (a + 1.0), "gamma": y}[self.name]

    def link(self, mu):
        return np.log(mu / (1.0 - mu)) if self.name == "binomial" else np.log(mu)

    def linkinv(self, eta):
        with np.errstate(over="ignore"):
            if self.name == "binomial":
                t = np.where(eta < -30, EPS, np.where(eta > 30, 1.0 / EPS, np.exp(np.clip(eta, -30, 30))))
                return t / (1.0 + t)
            return np.maximum(np.exp(eta), EPS)

    def mu_eta(self, eta):
        with np.errstate(over="ignore"):
            if self.name == "binomial":
                e = np.exp(np.clip(eta, -30, 30))
                return np.where(np.abs(eta) > 30, EPS, e / (1.0 + e) ** 2)
            return np.maximum(np.exp(eta), EPS)

    def var(self, mu):
        return {"poisson": mu, "binomial": mu * (1.0 - mu), "gamma": mu * mu}[self.name]

    def dvar(self, mu):
        return {"poisson": np.ones_like(mu), "binomial": 1.0 - 2.0 * mu, "gamma": 2.0 * mu}[self.name]

    def dev(self, y, mu, a):
        with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
            if self.name == "poisson":
                return 2.0 * a * np.where(y > 0, y * np.log(np.where(y > 0, y, 1.0) / mu) - (y - mu), mu)

            def ylogy(u, m):
                return np.where(u != 0, u * np.log(np.where(u != 0, u, 1.0) / m), 0.0)

            if self.name == "binomial":
                return 2.0 * a * (ylogy(y, mu) + ylogy(1.0 - y, 1.0 - mu))
            return -2.0 * a * (np.log(y / mu) - (y - mu) / mu)


def working(fam, y, wv, o, eta, pos, start=False):
    """mu, mu', V and the working response / row weight; 0 where w <= 0 (y not read there)."""
    a = wv * wv
    ys = np.where(pos, y, 1.0 if fam.name == "gamma" else 0.5)
    if start:
        eta = fam.link(fam.start(ys, a))
        zb = eta - o
    else:
        zb = eta - o
    mu = fam.linkinv(eta)
    mue = fam.mu_eta(eta)
    v = fam.var(mu)
    with np.errstate(invalid="ignore", over="ignore", divide="ignore"):
        z = np.where(pos, zb + (ys - mu) / mue, 0.0)
        rw = np.where(pos, wv * mue / np.sqrt(v), 0.0)
        dev = fam.dev(ys, mu, a)[pos].sum()
        x2 = (a * (ys - mu) ** 2 / v)[pos].sum()
    return z, rw, mu, dev, x2


def host_pirls(oracle, ndim, x, y, w, o, mn, mx, nodes, xtrap, lam, penalty, family, iters, tol=0.0):
    """PIRLS with the device's semantics.  Returns dict(c, dev, x2, mu, halvings, iterations, converged, M, P, trace),
    trace = per iteration (halvings, finite deviance); c is the last iterate with a finite deviance (c^1 at k = 1) and
    "error" is 107 when the halving rule gave up."""
    fam = Family(family)
    n = len(y)
    wv = np.ones(n) if w is None else np.asarray(w, float)
    ov = np.zeros(n) if o is None else np.asarray(o, float)
    pos = wv > 0
    P, _ = oracle.rows(ndim, x, y, None, mn, mx, nodes, 0.0)
    assert P.shape[0] == n
    z, rw, mu, dold, x2 = working(fam, y, wv, ov, None, pos, start=True)
    ncon = 0
    if xtrap != 0.0:
        ncon = (oracle.rows(ndim, x, z, rw, mn, mx, nodes, xtrap)[0].shape[0]
                - oracle.rows(ndim, x, z, rw, mn, mx, nodes, 0.0)[0].shape[0])
    Ccon = oracle.rows(ndim, x, z, rw, mn, mx, nodes, xtrap)[0][-ncon:] if ncon else np.zeros((0, P.shape[1]))
    Rh = np.zeros((0, P.shape[1]))
    if lam > 0:
        ev, V = np.linalg.eigh(penalty_dense(nodes, mn, mx, penalty))
        Rh = np.sqrt(lam) * (V * np.sqrt(np.maximum(ev, 0.0))) @ V.T

    def solve(rw, z):
        A = np.vstack([rw[:, None] * P, Ccon, Rh])
        b = np.concatenate([rw * z, np.zeros(len(Ccon) + len(Rh))])
        return np.linalg.lstsq(A, b, rcond=None)[0], A.T @ A

    res = dict(halvings=0, converged=False, trace=[], error=0, change=0.0)
    c = None
    for k in range(1, iters + 1):
        cprev = c
        c, M = solve(rw, z)
        res["iterations"], res["M"] = k, M
        znew, rwnew, mu, dev, x2 = working(fam, y, wv, ov, P @ c + ov, pos)
        nh = 0
        while not np.isfinite(dev) and k > 1 and nh < 10:
            c = 0.5 * (c + cprev)
            znew, rwnew, mu, dev, x2 = working(fam, y, wv, ov, P @ c + ov, pos)
            nh += 1
        res["halvings"] += nh
        res["trace"].append(nh)
        if not np.isfinite(dev):
            res["error"] = 107
            if k > 1:
                c = cprev
                _, _, mu, dev, x2 = working(fam, y, wv, ov, P @ c + ov, pos)
            break
        z, rw = znew, rwnew
        res["change"] = abs(dev - dold) / (abs(dev) + 0.1)
        dold = dev
        if res["change"] < tol:
            res["converged"] = True
            break
    res.update(c=c, dev=dev, x2=x2, mu=mu, P=P, fam=fam, wv=wv, ov=ov, pos=pos, y=y)
    return res


def glm_data(family, ndim, nodes, ndata, seed, weighted=False, hole=False, offset=False, level=1.0):
    """Seeded responses of each family with log / logit mean level + f(x) (+ o): counts, proportions out of 1..19
    trials (w = sqrt(trials); a single trial when unweighted), Gamma with shape 4."""
    x, f, w, mn, mx = make_problem(ndim, nodes, ndata, seed=seed, weighted=weighted, hole=hole)
    rng = np.random.default_rng(seed + 1000)
    o = 0.3 * rng.standard_normal(len(x)) if offset else None
    eta = level + f + (0.0 if o is None else o)
    if family == "poisson":
        y = rng.poisson(np.exp(eta)).astype(float)
    elif family == "binomial":
        trials = rng.integers(1, 20, len(x)) if weighted else np.ones(len(x), dtype=np.int64)
        y = rng.binomial(trials, 1.0 / (1.0 + np.exp(-(eta - level)))) / trials
        w = np.sqrt(trials.astype(float)) if weighted else None
    else:
        y = rng.gamma(4.0, np.exp(eta) / 4.0)
    return x, y, w, o, mn, mx


def glm_handle(ndim, mn, mx, nodes, xtrap, lam, penalty="curvature", real32=False):
    h = sp.FitHandle(ndim, mn, mx, nodes, xtrap, real32=real32)
    assert h.ierror == 0
    if lam > 0:
        assert h.set_smoothing(lam, penalty) == 0
    return h


def propagated(ref, dc):
    """Bounds of |dD|, |dX^2| and |dmu_i| from a coefficient error of at most dc in every entry: |d eta_i| <=
    sum_j |P_ij| dc (plus 1e-12 (1 + |eta_i|) for the rounding of the two evaluations of s), and dD/deta =
    -2 a (y - mu) mu' / V, dX^2/deta = -a mu' (2 (y - mu) / V + (y - mu)^2 V' / V^2)."""
    fam, pos, a = ref["fam"], ref["pos"], ref["wv"] ** 2
    mu = ref["mu"]
    eta = ref["P"] @ ref["c"] + ref["ov"]
    deta = np.abs(ref["P"]).sum(axis=1) * dc + 1e-12 * (1.0 + np.abs(eta))
    mue, v = fam.mu_eta(eta), fam.var(mu)
    r = np.abs(np.where(pos, ref["y"], 0.0) - mu)
    dD = (2 * a * r * mue / v * deta)[pos].sum()
    dX = (a * mue * (2 * r / v + r * r * np.abs(fam.dvar(mu)) / v ** 2) * deta)[pos].sum()
    return dD, dX, mue * deta


PARITY_CASES = [
    # family, ndim, nodes, ndata, xtrap, weighted, hole, lambda factor (x rho), penalty, offset
    ("poisson", 1, [12], 500, 0.0, True, False, 0.0, "curvature", True),
    ("binomial", 1, [12], 800, 1.0, True, True, 1e-3, "curvature", False),
    ("gamma", 1, [12], 500, 1.0, False, True, 0.0, "curvature", True),
    ("poisson", 2, [8, 7], 3000, 1.0, False, True, 1e-2, "thin_plate", False),
    ("binomial", 2, [8, 7], 3000, 0.0, False, False, 0.0, "curvature", True),
    ("gamma", 2, [8, 7], 3000, 0.0, True, False, 1e-3, "curvature", False),
    ("poisson", 3, [6, 5, 6], 6000, 1.0, True, True, 0.0, "curvature", True),
    ("binomial", 3, [6, 5, 6], 6000, 1.0, True, True, 1e-3, "thin_plate", True),
    ("gamma", 3, [6, 5, 6], 6000, 0.0, False, False, 1e-3, "thin_plate", False),
    ("poisson", 4, [4, 4, 5, 4], 4000, 0.0, False, False, 1e-3, "curvature", False),
    ("binomial", 4, [4, 5, 4, 4], 4000, 0.0, True, False, 0.0, "curvature", False),
    ("gamma", 4, [4, 4, 5, 4], 4000, 1.0, True, True, 0.0, "curvature", True),
]


@pytest.mark.parametrize("family,ndim,nodes,ndata,xtrap,weighted,hole,lamf,penalty,offset", PARITY_CASES)
def test_iterates_match_host_pirls(oracle, family, ndim, nodes, ndata, xtrap, weighted, hole, lamf, penalty, offset):
    x, y, w, o, mn, mx = glm_data(family, ndim, nodes, ndata, seed=7 * ndim + len(family), weighted=weighted,
                                  hole=hole, offset=offset)
    lam = 0.0
    if lamf > 0:
        P, _ = oracle.rows(ndim, x, y, w, mn, mx, nodes, 0.0)
        lam = lamf * rho_of(nodes, mn, mx, penalty, P.T @ P)
    for iters in (1, 2, 5):
        h = glm_handle(ndim, mn, mx, nodes, xtrap, lam, penalty)
        coef, info, ierr = h.glm_fit(x, y, w, family=family, offset=o, max_iter=iters, tol=0.0, return_mu=True)
        assert ierr == 0, (iters, info)
        assert info["iterations"] == iters and not info["converged"] and info["halvings"] == 0
        ref = host_pirls(oracle, ndim, x, y, w, o, mn, mx, nodes, xtrap, lam, penalty, family, iters)
        assert ref["halvings"] == 0 and ref["error"] == 0
        assert info["m"] == int(ref["pos"].sum())
        tol, cond = coef_tolerance(ref["M"])
        scale = np.abs(ref["c"]).max()
        err = np.abs(coef - ref["c"]).max() / scale
        # Every iterate carries the solve's error, and the earlier ones reach the next through z and W: the PIRLS map is
        # Newton's for the canonical links (its derivative vanishes at the solution) and Fisher scoring, a contraction,
        # for Gamma's log link, so each step adds at most one solve's error: (k + 1) tol, as in the robust test.
        assert err <= (iters + 1) * tol, (iters, err, tol, cond)
        dD, dX, dmu = propagated(ref, (iters + 1) * tol * scale)
        assert abs(info["deviance"] - ref["dev"]) <= 1e-11 * abs(ref["dev"]) + dD, (iters, info, ref["dev"], dD)
        assert abs(info["pearson"] - ref["x2"]) <= 1e-11 * abs(ref["x2"]) + dX, (iters, info, ref["x2"], dX)
        assert np.all(np.abs(info["mu"] - ref["mu"]) <= 1e-12 * np.abs(ref["mu"]) + dmu), iters
        h.destroy()


def score_check(ndim, x, y, w, o, mn, mx, nodes, lam, penalty, family, coef):
    """max_i |P^T A r - lam R c|_i / ((|B|^T A |r|)_i + lam (|R| |c|)_i), r = (y - mu) mu' / V, mu from eval_batch."""
    from oracle.cpu_matched import assemble_stencil

    fam = Family(family)
    s, ierr = sp.eval_batch(ndim, x, coef, mn, mx, nodes)
    assert ierr == 0
    eta = s + (0.0 if o is None else o)
    mu = fam.linkinv(eta)
    r = (y - mu) * fam.mu_eta(eta) / fam.var(mu)
    _, g, gabs = assemble_stencil(ndim, x, r, w, mn, mx, nodes, rhs_only=True)
    R = penalty_dense(nodes, mn, mx, penalty)
    lhs, rhs = g, lam * (R @ coef)
    scale = gabs + lam * (np.abs(R) @ np.abs(coef))
    return np.abs(lhs - rhs) / scale, g, scale


@pytest.mark.parametrize("family", ["poisson", "binomial", "gamma"])
def test_stationarity_at_scale(family):
    """Converged 3-D fit of 2^22 points on 12^3 nodes, lambda > 0, xtrap = 0: the penalized score equations
    P^T A ((y - mu) mu' / V) = lambda R c hold entry by entry to 1e-9 of (|B|^T A |r|)_i + lambda (|R| |c|)_i.  The solves
    are accurate to about eps cond(M) ~ 1e-11 relative here, and tol = 1e-13 stops the iteration at its fixed point to
    that level.  One response changed by one count (one trial, one unit) moves one entry by a mu'/V |B_ij| ~ 0.1 .. 1
    against a scale of ~1e4: the check must then fail by at least 100x."""
    ndim, nodes, n = 3, [12, 12, 12], 1 << 22
    x, y, w, o, mn, mx = glm_data(family, ndim, nodes, n, seed=61, weighted=family == "binomial", offset=True)
    lam = 1e-4 * n / 1728.0
    h = glm_handle(ndim, mn, mx, nodes, 0.0, lam)
    coef, info, ierr = h.glm_fit(x, y, w, family=family, offset=o, max_iter=60, tol=1e-13)
    assert ierr == 0 and info["converged"], info
    ratio, g, scale = score_check(ndim, x, y, w, o, mn, mx, nodes, lam, "curvature", family, coef)
    worst = float(ratio.max()) / 1e-9
    # one count at the point with the largest basis value in the entry of largest scale
    y2 = y.copy()
    i = int(np.argmax(np.abs(x - 0.5).sum(axis=1) < 0.05))
    step = {"poisson": 1.0, "binomial": 1.0 / (w[i] ** 2 if w is not None else 1.0), "gamma": 1.0}[family]
    y2[i] = y[i] + step if family != "binomial" or y[i] + step <= 1 else y[i] - step
    ratio2, _, _ = score_check(ndim, x, y2, w, o, mn, mx, nodes, lam, "curvature", family, coef)
    sens = float(ratio2.max()) / 1e-9
    print(f"{family}: iterations {info['iterations']}, worst ratio {worst:.3e}, one count changed {sens:.3e}")
    assert worst <= 1.0, worst
    assert sens >= 100.0, sens


def test_offset_invariance(oracle):
    """c(o + kappa) = c(o) - kappa c1, c1 the coefficients of the constant 1 from an ordinary fit of y = 1: constants
    lie in the spline space and in the null space of the penalty, and mu0 does not depend on the offset."""
    ndim, nodes, lamf = 2, [9, 8], 1e-3
    for family in ("poisson", "binomial", "gamma"):
        x, y, w, o, mn, mx = glm_data(family, ndim, nodes, 20000, seed=71, weighted=True, offset=True)
        P, _ = oracle.rows(ndim, x, y, None, mn, mx, nodes, 0.0)
        lam = lamf * rho_of(nodes, mn, mx, "curvature", P.T @ P)
        plain = glm_handle(ndim, mn, mx, nodes, 0.0, 0.0)
        assert plain.add_points(x, np.ones(len(x))) == 0
        c1, ierr = plain.compute()
        assert ierr == 0
        kappa = 0.75
        runs = []
        for oo in (o, o + kappa):
            h = glm_handle(ndim, mn, mx, nodes, 0.0, lam)
            coef, info, ierr = h.glm_fit(x, y, w, family=family, offset=oo, max_iter=6, tol=0.0, return_mu=True)
            assert ierr == 0
            runs.append((coef, info))
        a = (w if w is not None else np.ones(len(x))) ** 2
        fam = Family(family)
        mu = runs[0][1]["mu"]
        W = a * fam.mu_eta(fam.link(mu)) ** 2 / fam.var(mu)
        tol, cond = coef_tolerance(P.T @ (W[:, None] * P) + lam * penalty_dense(nodes, mn, mx, "curvature"))
        scale = np.abs(runs[0][0]).max()
        err = np.abs(runs[1][0] - (runs[0][0] - kappa * c1)).max() / scale
        assert err <= 2 * 7 * tol, (family, err, tol, cond)
        assert abs(runs[1][1]["deviance"] - runs[0][1]["deviance"]) <= 1e-9 * runs[0][1]["deviance"]


def halving_case():
    """1-D Gamma data whose offset has one spike of -12: the first fit misses the spiked point by a factor of about e^6,
    its working response at iteration 2 is about that large, and the full second step overflows exp (max eta 1.1e4;
    it takes 4 halvings, to max eta 675).  The third step is of order 1e15 in eta: 10 halvings cannot save it."""
    rng = np.random.default_rng(5)
    x = np.sort(rng.random(60))
    y = rng.gamma(4.0, 0.25, 60)
    o = np.zeros(60)
    o[30] = -12.0
    return x, y, o, np.zeros(1), np.ones(1), [10]


def test_step_halving_matches_host(oracle):
    """max_iter = 2: the second step is halved 4 times and accepted.  max_iter = 8: the third step finds no finite
    deviance in 10 halvings, so the call returns 107 with the (halved) second iterate.  With xmax = 1.3 and xtrap = 1
    the nodes past the data get constraint rows; the second step then needs 5 halvings (max eta 780 after 4, 390 after
    5), and the refinement steps must not run: they would move the halved iterate back towards the full step, which
    overflows exp."""
    x, y, o, mn, mx, nodes = halving_case()
    for xmax, xtrap, iters, halvings, err_code, done in ((mx, 0.0, 2, [0, 4], 0, 2), (mx, 0.0, 8, [0, 4, 10], 107, 3),
                                                          (np.array([1.3]), 1.0, 2, [0, 5], 0, 2)):
        ref = host_pirls(oracle, 1, x, y, None, o, mn, xmax, nodes, xtrap, 0.0, "curvature", "gamma", iters)
        assert ref["trace"] == halvings and ref["error"] == err_code
        h = glm_handle(1, mn, xmax, nodes, xtrap, 0.0)
        coef, info, ierr = h.glm_fit(x, y, family="gamma", offset=o, max_iter=iters, tol=0.0)
        assert ierr == err_code, info
        assert h.constraints_fired() == (xtrap != 0.0)
        assert info["iterations"] == done and info["halvings"] == sum(halvings), (info, ref["trace"])
        tol, cond = coef_tolerance(ref["M"])
        scale = np.abs(ref["c"]).max()
        assert np.abs(coef - ref["c"]).max() <= 3 * tol * scale, (np.abs(coef - ref["c"]).max() / scale, tol)
        assert abs(info["deviance"] - ref["dev"]) <= 1e-8 * abs(ref["dev"]), (info, ref["dev"])


def test_no_finite_deviance_at_the_first_iterate(oracle):
    """Offsets alternating 0 and 1600 in every cell: the first fit sits near -800, exp(eta) overflows at half the
    points, and there is no earlier iterate to halve towards: 107 with c^1 in coef."""
    ndim, nodes = 1, [8]
    x = np.linspace(0.01, 0.99, 400)
    y = np.full(400, 2.0)
    o = np.where(np.arange(400) % 2 == 0, 0.0, 1600.0)
    mn, mx = np.zeros(1), np.ones(1)
    ref = host_pirls(oracle, ndim, x, y, None, o, mn, mx, nodes, 0.0, 0.0, "curvature", "poisson", 3)
    assert ref["error"] == 107 and ref["iterations"] == 1
    h = glm_handle(ndim, mn, mx, nodes, 0.0, 0.0)
    coef, info, ierr = h.glm_fit(x, y, family="poisson", offset=o, max_iter=3, tol=0.0)
    assert ierr == 107 and info["iterations"] == 1 and info["halvings"] == 0
    assert not np.isfinite(info["deviance"])
    tol, _ = coef_tolerance(ref["M"])
    assert np.abs(coef - ref["c"]).max() <= 2 * tol * np.abs(ref["c"]).max()


def _truth(q):
    return 0.8 * np.sin(2 * q[:, 0]) * np.cos(1.5 * q[:, 1]) + 0.5 * q[:, 2] ** 2


@pytest.mark.parametrize("family", ["poisson", "binomial"])
def test_truth_recovery(family):
    """Seeded counts with an exposure offset (Poisson) or proportions out of 1..19 trials (binomial), with the
    log-rate / logit a smooth function on [0, 1]^3.  The threshold for the RMS error of the fitted linear predictor at
    random queries q is derived from the two parts of that error.
      bias   the fit tends to the projection of the truth on the spline space in the Fisher metric: the weighted least-
             squares fit c_b = F^-1 B^T W f, F = B^T W B with W the Fisher weights at the truth.  Its RMS error at the
             queries, rms_b, is computed.
      noise  asymptotically c - c_b ~ N(0, F^-1), so the squared RMS of the noise part at the queries is a Gaussian
             quadratic form with mean tr K = se^2 and variance 2 tr K^2, K = B_q F^-1 B_q^T / Q.
    By the triangle inequality for the RMS, rms <= rms_b + sqrt(se^2 + 5 sqrt(2 tr K^2)): five standard deviations of
    the quadratic form."""
    ndim, nodes, n = 3, [8, 8, 8], 200_000
    rng = np.random.default_rng(91)
    x = rng.random((n, ndim))
    mn, mx = np.zeros(ndim), np.ones(ndim)
    f = _truth(x)
    if family == "poisson":
        expo = rng.uniform(0.5, 3.0, n)
        o = np.log(expo)
        y = rng.poisson(np.exp(f + o)).astype(float)
        w = None
        Wt = np.exp(f + o)
    else:
        trials = rng.integers(1, 20, n)
        p = 1.0 / (1.0 + np.exp(-f))
        y = rng.binomial(trials, p) / trials
        o, w = None, np.sqrt(trials.astype(float))
        Wt = trials * p * (1 - p)
    h = glm_handle(ndim, mn, mx, nodes, 0.0, 0.0)
    coef, info, ierr = h.glm_fit(x, y, w, family=family, offset=o)
    assert ierr == 0 and info["converged"], info
    q = rng.uniform(0.05, 0.95, (4000, ndim))
    s, ierr = sp.eval_batch(ndim, q, coef, mn, mx, nodes)
    assert ierr == 0
    rms = float(np.sqrt(np.mean((s - _truth(q)) ** 2)))
    from oracle.cpu_matched import assemble_stencil
    from util import dense_from_stencil

    S, g, _ = assemble_stencil(ndim, x, f, np.sqrt(Wt), mn, mx, nodes)
    F = dense_from_stencil(S.reshape(-1, 4 ** ndim), nodes)
    Finv = np.linalg.inv(F)
    Bq = np.stack([sp.eval_batch(ndim, q, e, mn, mx, nodes)[0] for e in np.eye(len(coef))], axis=1)
    rms_b = float(np.sqrt(np.mean((Bq @ (Finv @ g) - _truth(q)) ** 2)))
    H = Finv @ (Bq.T @ Bq) / len(q)
    se2, var2 = float(np.trace(H)), 2.0 * float(np.trace(H @ H))
    bound = rms_b + np.sqrt(se2 + 5.0 * np.sqrt(var2))
    print(f"{family}: iterations {info['iterations']}, rms {rms:.3e}, bias rms {rms_b:.3e}, se {np.sqrt(se2):.3e}, "
          f"bound {bound:.3e}")
    assert rms <= bound, (rms, rms_b, se2, var2)


def test_repeatable_and_host_device_agree(monkeypatch):
    """Deterministic mode: repeated calls, and the host and device entries, return the same bits (coef, mu, out)."""
    import torch

    monkeypatch.setenv("SPLPAK_B200_DETERMINISTIC", "1")
    ndim, nodes = 3, [7, 6, 7]
    x, y, w, o, mn, mx = glm_data("poisson", ndim, nodes, 20000, seed=23, weighted=True, hole=True, offset=True)
    runs = []
    for _ in range(2):
        h = glm_handle(ndim, mn, mx, nodes, 1.0, 1e-3)
        coef, info, ierr = h.glm_fit(x, y, w, family="poisson", offset=o, return_mu=True)
        assert ierr == 0 and info["converged"]
        runs.append((coef, info.pop("mu"), info))
        h.destroy()
    for a, b in zip(runs[0], runs[1]):
        assert np.array_equal(a, b) if isinstance(a, np.ndarray) else a == b
    dev = torch.device("cuda", torch.cuda.current_device())
    d_x, d_y, d_w, d_o = (torch.from_numpy(np.ascontiguousarray(a)).to(dev) for a in (x, y, w, o))
    h = glm_handle(ndim, mn, mx, nodes, 1.0, 1e-3)
    d_c = torch.zeros(h.ncol, dtype=torch.float64, device=dev)
    d_mu = torch.zeros(len(y), dtype=torch.float64, device=dev)
    info, ierr = h.glm_fit_device(d_x, ndim, d_y, d_w, len(y), d_c, family="poisson", d_offset=d_o, d_mu=d_mu)
    assert ierr == 0
    assert np.array_equal(d_c.cpu().numpy(), runs[0][0])
    assert np.array_equal(d_mu.cpu().numpy(), runs[0][1])
    assert info == runs[0][2]


@pytest.mark.parametrize("family", ["poisson", "binomial", "gamma"])
def test_real32_agrees_with_real64(oracle, family):
    """Eight iterations in both libraries (tol = 0, so both stop at the same iterate; near the solution the PIRLS map
    contracts, so the difference is that of the two fixed points).  The REAL32 library rounds to float, once each, x,
    y, w and o, the evaluation of s, and the z and row weights it hands to its assembly; everything else is FP64.  At
    the solution dz/ds = 0, so a change d_eta of the linear predictor moves z and sqrt(W) only through mu':
    |dz| <= 2 |y - mu| / mu' |d_eta|.  Per point the roundings therefore move z (or, equivalently, the weighted row) by
    at most eps32 t_i, with
        t_i = |z_i| + |y_i| / mu'_i + 2 |y_i - mu_i| / mu'_i (1 + |eta_i| + 2 (N - 1) max|c|),
    where 2 (N - 1) max|c| bounds |ds/dx| on [0, 1] (x rounds by up to eps32).  The coefficients are linear in z:
    dc = G dz with G = M^-1 P^T W, M = P^T W P.  The roundings are independent from point to point, so dc_j has a
    standard deviation of at most sigma_j = eps32 sqrt(sum_i G_ji^2 t_i^2).  The float output adds eps32 max|c|, and
    the test allows 6 sigma.  The deviance moves by at most sum |dD/deta| times the change of eta this implies."""
    ndim, nodes = 2, [9, 8]
    x, y, w, o, mn, mx = glm_data(family, ndim, nodes, 20000, seed=31, weighted=True, offset=True)
    h64 = glm_handle(ndim, mn, mx, nodes, 0.0, 0.0)
    c64, i64, e64 = h64.glm_fit(x, y, w, family=family, offset=o, max_iter=8, tol=0.0)
    h32 = glm_handle(ndim, mn, mx, nodes, 0.0, 0.0, real32=True)
    f32 = [None if a is None else a.astype(np.float32) for a in (x, y, w, o)]
    c32, i32, e32 = h32.glm_fit(f32[0], f32[1], f32[2], family=family, offset=f32[3], max_iter=8, tol=0.0)
    assert e64 == 0 and e32 == 0, (i64, i32)
    fam = Family(family)
    P, _ = oracle.rows(ndim, x, y, None, mn, mx, nodes, 0.0)
    scale = np.abs(c64).max()
    eta = P @ c64 + o
    mu, mue = fam.linkinv(eta), fam.mu_eta(eta)
    a = w ** 2
    W = a * mue ** 2 / fam.var(mu)
    z = eta - o + (y - mu) / mue
    G = np.linalg.solve(P.T @ (W[:, None] * P), P.T * W)
    r = np.abs(y - mu) / mue
    t = np.abs(z) + np.abs(y) / mue + 2 * r * (1 + np.abs(eta) + 2 * (max(nodes) - 1) * scale)
    eps32 = float(np.finfo(np.float32).eps)
    bound = eps32 * scale + 6 * eps32 * np.sqrt(G ** 2 @ t ** 2).max()
    dc = np.abs(c32.astype(float) - c64).max()
    print(f"{family}: REAL32 max|dc| = {dc / scale:.3e} max|c|, {dc / bound:.3e} of the bound")
    assert dc <= bound, (dc / scale, bound / scale)
    deta = np.abs(P).sum(axis=1).max() * dc + eps32 * (1 + np.abs(eta).max() + 2 * (max(nodes) - 1) * scale)
    dD = (2 * a * np.abs(y - mu) * mue / fam.var(mu)).sum() * deta
    assert abs(i32["deviance"] - i64["deviance"]) <= 2 * dD + 1e-6 * i64["deviance"], (i32, i64, dD)


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
    x, y, w, o, mn, mx = glm_data("binomial", ndim, nodes, 30000, seed=41, weighted=True, hole=True, offset=True)
    devs = (C.c_int * 2)(0, 1)
    comms = (C.c_void_p * 2)()
    assert lib.splpak_b200_comm_init_all(2, devs, comms) == 0
    half = len(x) // 2
    res = [None, None]

    def rank(r):
        # one host thread per device: the call all-reduces (and waits) inside
        torch.cuda.set_device(r)
        lo, hi = (0, half) if r == 0 else (half, len(x))
        h = glm_handle(ndim, mn, mx, nodes, 1.0, 0.0)
        dev = torch.device("cuda", r)
        d_x, d_y, d_w, d_o = (torch.from_numpy(np.ascontiguousarray(a[lo:hi])).to(dev) for a in (x, y, w, o))
        d_c = torch.zeros(h.ncol, dtype=torch.float64, device=dev)
        info, ierr = h.glm_fit_device(d_x, ndim, d_y, d_w, hi - lo, d_c, family="binomial", d_offset=d_o,
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
    one = glm_handle(ndim, mn, mx, nodes, 1.0, 0.0)
    c1, info1, ierr = one.glm_fit(x, y, w, family="binomial", offset=o)
    assert ierr == 0
    assert res[0][1]["iterations"] == info1["iterations"] and res[0][1]["m"] == info1["m"]
    assert np.abs(res[0][0] - c1).max() <= 1e-9 * np.abs(c1).max()


BAD_Y = {"poisson": [-1.0, np.nan, np.inf], "binomial": [-0.1, 1.5, np.nan], "gamma": [0.0, -2.0, np.inf]}


def test_refusals():
    ndim, nodes = 2, [6, 6]
    x, y, w, o, mn, mx = glm_data("poisson", ndim, nodes, 500, seed=51, weighted=True, offset=True)
    lib = sp.load()

    def call(h, yy=None, ww=None, **kw):
        a = dict(l1x=ndim, n=len(y), family=0, max_iter=5, tol=1e-8, ncf=h.ncol, nout=7)
        a.update(kw)
        xa, ya, wa, oa = (np.ascontiguousarray(v) for v in (x, y if yy is None else yy, w if ww is None else ww, o))
        coef, out, ierr = np.zeros(h.ncol), np.zeros(7), C.c_int(-1)
        rc = lib.splpak_b200_fit_glm(h.h, C.c_void_p(xa.ctypes.data), a["l1x"], C.c_void_p(ya.ctypes.data),
                                     C.c_void_p(wa.ctypes.data), 1, C.c_void_p(oa.ctypes.data), a["n"], a["family"],
                                     a["max_iter"], a["tol"], None, C.c_void_p(coef.ctypes.data), a["ncf"], None,
                                     C.c_void_p(out.ctypes.data), a["nout"], C.byref(ierr))
        assert rc == ierr.value
        return rc

    h = glm_handle(ndim, mn, mx, nodes, 0.0, 0.0)
    for kw in (dict(family=3), dict(family=-1), dict(max_iter=0), dict(tol=-1.0), dict(tol=float("nan")),
               dict(nout=6), dict(l1x=1)):
        assert call(h, **kw) == 203, kw
    assert call(h, ncf=h.ncol - 1) == 104
    assert call(h, n=0) == 105
    assert call(h, ww=np.zeros(len(y))) == 105                   # m = 0
    assert call(h) == 0
    assert call(h) == 203                                       # used handle
    assert lib.splpak_b200_fit_refine_begin(h.h) == 203
    with pytest.raises(SplpakError):
        h.smoothing_score(0.0)
    assert h.reset() == 0
    assert call(h) == 0                                         # a reset handle is fresh again
    used = glm_handle(ndim, mn, mx, nodes, 0.0, 0.0)
    assert used.add_points(x, y, w, weighted=True) == 0
    assert call(used) == 203
    ortho = sp.FitHandle(ndim, mn, mx, nodes, 0.0, solver="orthogonal")
    assert call(ortho) == 203
    with pytest.raises(SplpakError):
        h.glm_fit(x, y, w, family="probit")
    for short in (dict(y=y[:-1]), dict(w=w[:-1]), dict(offset=o[:-1])):
        a = dict(y=y, w=w, offset=o)
        a.update(short)
        with pytest.raises(SplpakError):
            h.glm_fit(x, a["y"], a["w"], offset=a["offset"])
    # a bad y where w > 0: 203 and the handle stays fresh; where w = 0 it is not read
    ys = {"poisson": y, "binomial": np.clip(y / 10.0, 0, 1), "gamma": y + 0.5}
    for fam, code in (("poisson", 0), ("binomial", 1), ("gamma", 2)):
        for bad in BAD_Y[fam]:
            f = glm_handle(ndim, mn, mx, nodes, 0.0, 0.0)
            yb = ys[fam].copy()
            yb[17] = bad
            assert call(f, yy=yb, family=code) == 203, (fam, bad)
            wz = w.copy()
            wz[17] = 0.0
            assert call(f, yy=yb, ww=wz, family=code) == 0, (fam, bad)
    # too few points for the columns: a non-positive pivot, 107
    few = glm_handle(ndim, mn, mx, nodes, 0.0, 0.0)
    assert call(few, n=10) == 107


def test_cfg3_scale():
    """cfg3 size: 1e8 device-resident Poisson points, 24^3 nodes, xtrap = 1 -> converged at tol = 1e-8, and the
    returned deviance equals, to 1e-10, the deviance recomputed from eval_batch of the returned coefficients."""
    import torch

    dev = torch.device("cuda", torch.cuda.current_device())
    n, ndim, nodes = 100_000_000, 3, [24, 24, 24]
    gen = torch.Generator(device=dev)
    gen.manual_seed(7)
    x = torch.rand((n, ndim), dtype=torch.float64, device=dev, generator=gen)
    rate = torch.exp(1.0 + torch.sin(2 * x[:, 0]) * torch.cos(1.5 * x[:, 1]) + 0.5 * x[:, 2] ** 2)
    y = torch.poisson(rate, generator=gen)
    del rate
    mn, mx = np.zeros(ndim), np.ones(ndim)
    h = glm_handle(ndim, mn, mx, nodes, 1.0, 0.0)
    d_c = torch.zeros(h.ncol, dtype=torch.float64, device=dev)
    info, ierr = h.glm_fit_device(x, ndim, y, None, n, d_c, family="poisson", max_iter=25, tol=1e-8)
    assert ierr == 0 and info["converged"], info
    s = torch.zeros(n, dtype=torch.float64, device=dev)
    assert sp.eval_batch_device(ndim, x, ndim, n, d_c, mn, mx, nodes, s) == 0
    torch.cuda.synchronize()
    mu = torch.clamp(torch.exp(s), min=EPS)
    pos = y > 0
    d = torch.where(pos, y * torch.log(torch.where(pos, y, 1.0) / mu) - (y - mu), mu)
    D = float(2.0 * d.sum())
    print(f"cfg3 poisson: {info}")
    assert abs(info["deviance"] - D) <= 1e-10 * D, (info["deviance"], D)
