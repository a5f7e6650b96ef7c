"""GLM fits with the smoothing parameter chosen on each PIRLS working system (splpak_b200_fit_glm_select[_device]).

The reference is the host PIRLS of test_gpu_glm (oracle rows, R's links and deviances, lstsq on the row-weighted
augmented system) driven by the lambda path the device reports in its trace, and the dense criteria of test_gpu_gcv /
test_gpu_reml on each of its working systems: M = (sqrt(W) P)^T (sqrt(W) P) + C^T C + lambda R with the constraint
rows C of the first working system, g = (sqrt(W) P)^T (sqrt(W) z).  Runs with tol = 0 and max_iter = k compare the
same iterate."""
import ctypes as C
import threading

import numpy as np
import pytest

import splpak_b200 as sp
from splpak_b200.api import SplpakError
from test_gpu_glm import Family, glm_data, propagated, score_check, working
from test_gpu_reml import null_dim
from test_gpu_smoothing import penalty_dense
from test_gpu_variance import basis_rows
from util import coef_tolerance

pytestmark = pytest.mark.gpu
EPS = 2.0 ** -52
CRIT = {"reml": 0, "prediction": 1}


# ---------------------------------------------------------------------------------------------------------------------
# host references (also used by test_glm_select_cpu)
# ---------------------------------------------------------------------------------------------------------------------
def criterion(family, crit, sysk, lam, mp):
    """The device's criterion on one working system (dict A0, b0, Cc, R, N): REML with phi = 1 (Poisson, binomial) or
    profiled (Gamma); UBRE (phi = 1) or GCV (Gamma).  Returns (value, M, c)."""
    A0, b0, Cc, R, N = sysk["A0"], sysk["b0"], sysk["Cc"], sysk["R"], sysk["N"]
    G0 = A0.T @ A0
    M = G0 + Cc.T @ Cc + lam * R
    c = np.linalg.solve(M, A0.T @ b0)
    rss = float(((b0 - A0 @ c) ** 2).sum())
    p = M.shape[0]
    if crit == "reml":
        dp = rss + float(c @ (M - G0) @ c)
        sign, logdet = np.linalg.slogdet(M)
        assert sign > 0
        if family != "gamma":
            return dp + logdet - (p - mp) * np.log(lam), M, c
        n = N + len(Cc)
        return (n - mp) * np.log(dp / (n - mp)) + logdet - (p - mp) * np.log(lam), M, c
    edf = float(np.trace(np.linalg.solve(M, G0)))
    if family != "gamma":
        return rss / N - 1.0 + 2.0 * edf / N, M, c
    return N * rss / (N - edf) ** 2, M, c


def host_search(score, t_lo, t_hi):
    """The device's search over log10 lambda: a grid at 2 points per decade, golden section on the bracket of the best
    grid point to 0.02 decades, ties to the larger lambda, non-finite points as +inf.  Returns (t, value, evaluations,
    best grid point at the low end, at the high end); t is None when no point was finite."""
    best = [None, np.inf]
    count = [0]

    def ev(t):
        count[0] += 1
        v = score(t)
        v = v if np.isfinite(v) else np.inf
        if np.isfinite(v) and (best[0] is None or v < best[1] or (v == best[1] and t > best[0])):
            best[0], best[1] = t, v
        return v

    K = max(int(np.ceil(2.0 * (t_hi - t_lo) - 1e-9)), 0)
    kbest, vbest = 0, np.inf
    for k in range(K + 1):
        t = t_lo + (t_hi - t_lo) * k / K if K > 0 else t_lo
        v = ev(t)
        if k == 0 or v <= vbest:
            vbest, kbest = v, k
    if K > 0:
        def grid_t(k):
            return t_lo + (t_hi - t_lo) * k / K

        a, b = grid_t(max(kbest - 1, 0)), grid_t(min(kbest + 1, K))
        gr = 0.5 * (np.sqrt(5.0) - 1.0)
        c, d = b - gr * (b - a), a + gr * (b - a)
        fc, fd = ev(c), ev(d)
        while b - a > 0.02:
            if fc < fd:
                b, d, fd = d, c, fc
                c = b - gr * (b - a)
                fc = ev(c)
            else:
                a, c, fc = c, d, fd
                d = a + gr * (b - a)
                fd = ev(d)
    return best[0], best[1], count[0], K > 0 and kbest == 0, K > 0 and kbest == K


def select_step(score, k, t_prev, t_lo, t_hi):
    """One selecting iteration: the whole range at k = 1, else log10 lambda_(k-1) +- 1 clipped, and the whole range
    again when the best grid point is an end of the window that is not an end of the range."""
    a, b = (t_lo, t_hi) if k == 1 else (max(t_lo, t_prev - 1.0), min(t_hi, t_prev + 1.0))
    t, v, n, glo, ghi = host_search(score, a, b)
    if k > 1 and ((glo and a > t_lo) or (ghi and b < t_hi)):
        t, v, n2, _, _ = host_search(score, t_lo, t_hi)
        n += n2
    return t, v, n


class HostGlm:
    """Host PIRLS on the oracle's rows with the device's semantics; solve(lam) takes one step with the given lambda."""

    def __init__(self, oracle, ndim, x, y, w, o, mn, mx, nodes, xtrap, penalty, family):
        self.fam = Family(family)
        self.family, self.penalty, self.ndim = family, penalty, ndim
        n = len(y)
        self.y = y
        self.wv = np.ones(n) if w is None else np.asarray(w, float)
        self.ov = np.zeros(n) if o is None else np.asarray(o, float)
        self.pos = self.wv > 0
        self.P, _ = oracle.rows(ndim, x, y, None, mn, mx, nodes, 0.0)
        self.z, self.rw, self.mu, self.dev, self.x2 = working(self.fam, y, self.wv, self.ov, None, self.pos, True)
        ncon = 0
        if xtrap != 0.0:
            ncon = (oracle.rows(ndim, x, self.z, self.rw, mn, mx, nodes, xtrap)[0].shape[0]
                    - oracle.rows(ndim, x, self.z, self.rw, mn, mx, nodes, 0.0)[0].shape[0])
        self.Cc = (oracle.rows(ndim, x, self.z, self.rw, mn, mx, nodes, xtrap)[0][-ncon:] if ncon
                   else np.zeros((0, self.P.shape[1])))
        self.R = penalty_dense(nodes, mn, mx, penalty)
        ev, V = np.linalg.eigh(self.R)
        self.Rh = (V * np.sqrt(np.maximum(ev, 0.0))) @ V.T
        self.N = int((self.rw > 0).sum())
        self.mp = null_dim(ndim, penalty)
        self.c = None
        A0 = self.rw[:, None] * self.P
        self.rho = np.trace(A0.T @ A0) / np.trace(self.R)

    def system(self):
        keep = self.rw > 0
        return dict(A0=(self.rw[:, None] * self.P)[keep], b0=(self.rw * self.z)[keep], Cc=self.Cc, R=self.R, N=self.N)

    def score(self, crit, lam):
        return criterion(self.family, crit, self.system(), lam, self.mp)

    def solve(self, lam):
        """One PIRLS step at lam (no halving: the cases here never need one).  Returns M of the solve."""
        A = np.vstack([self.rw[:, None] * self.P, self.Cc, np.sqrt(lam) * self.Rh])
        b = np.concatenate([self.rw * self.z, np.zeros(len(self.Cc) + len(self.Rh))])
        self.c = np.linalg.lstsq(A, b, rcond=None)[0]
        self.last = self.system()
        self.z, self.rw, self.mu, self.dev, self.x2 = working(self.fam, self.y, self.wv, self.ov,
                                                              self.P @ self.c + self.ov, self.pos)
        return A.T @ A

    def ref(self):
        return dict(fam=self.fam, pos=self.pos, wv=self.wv, mu=self.mu, P=self.P, c=self.c, ov=self.ov, y=self.y)


def select_handle(ndim, mn, mx, nodes, xtrap, real32=False):
    h = sp.FitHandle(ndim, mn, mx, nodes, xtrap, real32=real32)
    assert h.ierror == 0
    return h


# ---------------------------------------------------------------------------------------------------------------------
# 1. every iterate against the host
# ---------------------------------------------------------------------------------------------------------------------
ITERATE_CASES = [
    # family, criterion, ndim, nodes, ndata, xtrap, weighted, hole, penalty, offset
    ("poisson", "reml", 1, [14], 800, 0.0, True, False, "curvature", True),
    ("binomial", "prediction", 1, [14], 1200, 1.0, True, True, "curvature", False),
    ("gamma", "reml", 2, [8, 7], 3000, 1.0, False, True, "thin_plate", False),
    ("poisson", "prediction", 2, [8, 7], 3000, 0.0, True, False, "curvature", True),
    ("binomial", "reml", 3, [6, 5, 6], 6000, 0.0, True, False, "thin_plate", True),
    ("gamma", "prediction", 3, [6, 5, 6], 6000, 1.0, True, True, "curvature", False),
    ("poisson", "reml", 4, [4, 4, 5, 4], 5000, 1.0, False, True, "curvature", False),
    ("gamma", "reml", 1, [14], 800, 0.0, False, False, "curvature", True),
]


@pytest.mark.parametrize("family,crit,ndim,nodes,ndata,xtrap,weighted,hole,penalty,offset", ITERATE_CASES)
def test_iterates_match_host(oracle, family, crit, ndim, nodes, ndata, xtrap, weighted, hole, penalty, offset):
    x, y, w, o, mn, mx = glm_data(family, ndim, nodes, ndata, seed=11 * ndim + len(family), weighted=weighted,
                                  hole=hole, offset=offset)
    h = select_handle(ndim, mn, mx, nodes, xtrap)
    _, full, _, ierr = h.glm_select(x, y, w, family=family, offset=o, criterion=crit, penalty=penalty)
    assert ierr == 0 and full["converged"], full
    last = full["iterations"]
    worst_crit = 0.0
    for iters in sorted({1, 2, last}):
        h = select_handle(ndim, mn, mx, nodes, xtrap)
        coef, info, trace, ierr = h.glm_select(x, y, w, family=family, offset=o, criterion=crit, penalty=penalty,
                                               max_iter=iters, tol=0.0, return_mu=True)
        assert ierr == 0 and info["iterations"] == iters and len(trace) == iters, (iters, info)
        assert info["halvings"] == 0 and not info["converged"]
        host = HostGlm(oracle, ndim, x, y, w, o, mn, mx, nodes, xtrap, penalty, family)
        t_lo, t_hi = np.log10(host.rho * 1e-10), np.log10(host.rho * 1e4)
        t_prev, selecting = None, True
        for k in range(1, iters + 1):
            lam_k, crit_k, nscore = trace[k - 1, :3]
            if selecting:
                assert nscore > 0 and np.isfinite(crit_k)
                want, M, _ = host.score(crit, lam_k)
                tol = max(1e-9 * abs(want), 1e3 * EPS * np.linalg.cond(M) * max(1.0, abs(want)))
                worst_crit = max(worst_crit, abs(crit_k - want) / tol)
                assert abs(crit_k - want) <= tol, (k, crit_k, want, tol)
                t_h, v_h, _ = select_step(lambda t: host.score(crit, 10.0 ** t)[0], k, t_prev, t_lo, t_hi)
                t_d = np.log10(lam_k)
                assert abs(t_d - t_h) <= 0.05 or abs(want - v_h) <= 1e-9 * abs(v_h), (k, t_d, t_h, want, v_h)
                if k > 1 and abs(t_d - t_prev) <= 0.05:
                    selecting = False
                t_prev = t_d
            else:
                assert nscore == 0 and np.isnan(crit_k) and lam_k == trace[k - 2, 0]
            M = host.solve(lam_k)
            assert abs(trace[k - 1, 3] - host.dev) <= 1e-8 * abs(host.dev), (k, trace[k - 1], host.dev)
        ref = host.ref()
        tol, cond = coef_tolerance(M)
        scale = np.abs(ref["c"]).max()
        err = np.abs(coef - ref["c"]).max() / scale
        assert err <= (iters + 1) * tol, (iters, err, tol, cond)
        dD, dX, dmu = propagated(ref, (iters + 1) * tol * scale)
        assert abs(info["deviance"] - host.dev) <= 1e-11 * abs(host.dev) + dD, (iters, info, host.dev, dD)
        assert abs(info["pearson"] - host.x2) <= 1e-11 * abs(host.x2) + dX, (iters, info, host.x2, dX)
        assert np.all(np.abs(info["mu"] - ref["mu"]) <= 1e-12 * np.abs(ref["mu"]) + dmu), iters
        # edf of the last solve's system
        G0 = host.last["A0"].T @ host.last["A0"]
        Ml = G0 + host.Cc.T @ host.Cc + info["lam"] * host.R
        edf = float(np.trace(np.linalg.solve(Ml, G0)))
        assert abs(info["edf"] - edf) <= max(1e-9 * edf, 1e3 * EPS * np.linalg.cond(Ml) * edf), (info["edf"], edf)
        h.destroy()
    print(f"{family} {crit} {ndim}-D: {last} iterations, {full['select_iterations']} selecting, settled "
          f"{full['settled']}, lam {full['lam']:.4e}, edf {full['edf']:.3f}, worst criterion error {worst_crit:.2e} "
          f"of the tolerance")


# ---------------------------------------------------------------------------------------------------------------------
# 2. the fixed point
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("family,crit", [("poisson", "reml"), ("binomial", "prediction"), ("gamma", "reml"),
                                         ("gamma", "prediction")])
def test_settled_fit_is_the_fixed_lambda_fit(family, crit):
    ndim, nodes, n = 3, [9, 9, 9], 1 << 20
    x, y, w, o, mn, mx = glm_data(family, ndim, nodes, n, seed=61, weighted=family == "binomial", offset=True)
    h = select_handle(ndim, mn, mx, nodes, 0.0)
    coef, info, trace, ierr = h.glm_select(x, y, w, family=family, offset=o, criterion=crit, max_iter=60, tol=1e-13)
    assert ierr == 0 and info["converged"] and info["settled"], (info, trace)
    plain = select_handle(ndim, mn, mx, nodes, 0.0)
    assert plain.set_smoothing(info["lam"], "curvature") == 0
    c2, info2, ierr = plain.glm_fit(x, y, w, family=family, offset=o, max_iter=60, tol=1e-13)
    assert ierr == 0 and info2["converged"]
    err = np.abs(coef - c2).max() / np.abs(c2).max()
    assert err <= 1e-8, err
    assert abs(info["deviance"] - info2["deviance"]) <= 1e-9 * info2["deviance"]
    ratio, _, _ = score_check(ndim, x, y, w, o, mn, mx, nodes, info["lam"], "curvature", family, coef)
    print(f"{family} {crit}: lam {info['lam']:.4e}, {info['iterations']} iterations ({info['select_iterations']} "
          f"selecting), coef difference {err:.2e}, score equations {ratio.max() / 1e-9:.2e} of the tolerance")
    assert ratio.max() <= 1e-9


# ---------------------------------------------------------------------------------------------------------------------
# 3. edf, scale and variances
# ---------------------------------------------------------------------------------------------------------------------
def test_variances_leverages_and_queries(oracle, monkeypatch):
    monkeypatch.setenv("SPLPAK_B200_DETERMINISTIC", "1")
    family, ndim, nodes = "gamma", 2, [9, 8]
    x, y, w, o, mn, mx = glm_data(family, ndim, nodes, 4000, seed=5, weighted=True, offset=True)
    h = select_handle(ndim, mn, mx, nodes, 0.0)
    _, info, _, ierr = h.glm_select(x, y, w, family=family, offset=o, criterion="reml")
    assert ierr == 0
    K = info["iterations"]
    runs = []
    for iters in (K - 1, K):
        h = select_handle(ndim, mn, mx, nodes, 0.0)
        coef, info, trace, ierr = h.glm_select(x, y, w, family=family, offset=o, criterion="reml", max_iter=iters,
                                               tol=0.0, variance=iters == K)
        assert ierr == 0
        runs.append((h, coef, info))
    h, coef, info = runs[1]
    cprev = runs[0][1]
    # rw of the last solve: from c^(K-1)
    fam = Family(family)
    s, ierr = sp.eval_batch(ndim, x, cprev, mn, mx, nodes)
    assert ierr == 0
    z, rw, _, _, _ = working(fam, y, w, o, s + o, w > 0)
    q, ierr = h.variance(x)
    assert ierr == 0
    total = float((rw ** 2 * q).sum())
    assert abs(total - info["edf"]) <= 1e-9 * info["edf"], (total, info["edf"])
    # q at random queries against the dense b^T M^-1 b of the final working system
    P, _ = oracle.rows(ndim, x, y, None, mn, mx, nodes, 0.0)
    A0 = rw[:, None] * P
    M = A0.T @ A0 + info["lam"] * penalty_dense(nodes, mn, mx, "curvature")
    Sig = np.linalg.inv(M)
    rng = np.random.default_rng(3)
    qx = rng.uniform(0.0, 1.0, (200, ndim))
    cols, vals = basis_rows(oracle, qx, [0] * ndim, mn, mx, nodes)
    got, ierr = h.variance(qx)
    assert ierr == 0
    for i in range(len(qx)):
        b = np.zeros(M.shape[0])
        np.add.at(b, cols[i], vals[i])
        ref = b @ Sig @ b
        assert abs(got[i] - ref) <= 1e-9 * ref + 1e3 * EPS * np.linalg.cond(M) * ref, (i, got[i], ref)
    # phi-hat of the Gamma fit: Pearson's X^2 / (m - edf)
    assert info["scale"] == pytest.approx(info["pearson"] / (info["m"] - info["edf"]), rel=1e-15)
    with pytest.raises(SplpakError):
        h.cholesky_factor(0, 0, 1)                              # Sigma has overwritten the factor


def _truth_1d(u):
    return 1.0 + np.sin(2 * np.pi * u) * np.exp(-u)


def test_coverage_of_poisson_intervals():
    """Ten seeded 1-D Poisson replicates: the mean across-the-function coverage of eta-hat +- 1.96 sqrt(phi q) (Wood's
    Bayesian intervals: their average coverage over the function is close to nominal)."""
    nodes, n = [30], 2000
    mn, mx = np.zeros(1), np.ones(1)
    g = np.linspace(0.01, 0.99, 400)
    covs = {}
    for crit in ("reml", "prediction"):
        cov = []
        for rep in range(10):
            rng = np.random.default_rng(100 + rep)
            x = rng.random(n)
            y = rng.poisson(np.exp(_truth_1d(x))).astype(float)
            h = select_handle(1, mn, mx, nodes, 0.0)
            coef, info, _, ierr = h.glm_select(x, y, criterion=crit, variance=True)
            assert ierr == 0 and info["converged"], info
            s, ierr = sp.eval_batch(1, g, coef, mn, mx, nodes)
            q, ierr2 = h.variance(g)
            assert ierr == 0 and ierr2 == 0
            half = 1.96 * np.sqrt(info["scale"] * q)
            cov.append(float(np.mean(np.abs(s - _truth_1d(g)) <= half)))
        covs[crit] = cov
        print(f"{crit}: coverage per replicate {np.round(cov, 3).tolist()}, mean {np.mean(cov):.3f}")
    for crit, cov in covs.items():
        assert 0.88 <= np.mean(cov) <= 0.99, (crit, cov)


# ---------------------------------------------------------------------------------------------------------------------
# 4. recovery against a fixed-lambda sweep
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("family", ["poisson", "binomial", "gamma"])
def test_recovery_against_a_lambda_sweep(oracle, family):
    ndim, nodes, n = 2, [14, 14], 6000
    rng = np.random.default_rng(17)
    x = rng.random((n, ndim))
    mn, mx = np.zeros(ndim), np.ones(ndim)

    def truth(u):
        return 0.8 * np.sin(3 * u[:, 0]) * np.cos(2 * u[:, 1]) + 0.5 * u[:, 1]

    f = truth(x)
    w = None
    if family == "poisson":
        y = rng.poisson(np.exp(1.0 + f)).astype(float)
        f = f + 1.0
    elif family == "binomial":
        trials = rng.integers(1, 10, n)
        y = rng.binomial(trials, 1.0 / (1.0 + np.exp(-f))) / trials
        w = np.sqrt(trials.astype(float))
    else:
        y = rng.gamma(3.0, np.exp(f) / 3.0)
    gq = np.stack(np.meshgrid(np.linspace(0.02, 0.98, 60), np.linspace(0.02, 0.98, 60)), -1).reshape(-1, 2)
    ft = truth(gq) + (1.0 if family == "poisson" else 0.0)

    def mse(coef):
        s, ierr = sp.eval_batch(ndim, gq, coef, mn, mx, nodes)
        assert ierr == 0
        return float(np.mean((s - ft) ** 2))

    host = HostGlm(oracle, ndim, x, y, w, None, mn, mx, nodes, 0.0, "curvature", family)
    sweep = []
    for t in np.arange(-10.0, 4.0 + 1e-9, 0.5):
        h = select_handle(ndim, mn, mx, nodes, 0.0)
        assert h.set_smoothing(host.rho * 10.0 ** t, "curvature") == 0
        coef, info, ierr = h.glm_fit(x, y, w, family=family)
        sweep.append(mse(coef) if ierr == 0 else np.inf)
    out = {}
    for crit in ("reml", "prediction"):
        h = select_handle(ndim, mn, mx, nodes, 0.0)
        coef, info, _, ierr = h.glm_select(x, y, w, family=family, criterion=crit)
        assert ierr == 0 and info["converged"], info
        out[crit] = mse(coef)
    best = min(sweep)
    print(f"{family}: selected MSE {out}, sweep best {best:.3e}, ends {sweep[0]:.3e} / {sweep[-1]:.3e}")
    for crit, m in out.items():
        assert m <= 1.5 * best and m < sweep[0] and m < sweep[-1], (crit, m, best, sweep[0], sweep[-1])


# ---------------------------------------------------------------------------------------------------------------------
# 5. determinism, ranks, REAL32
# ---------------------------------------------------------------------------------------------------------------------
def test_repeatable_and_host_device_agree(monkeypatch):
    import torch

    monkeypatch.setenv("SPLPAK_B200_DETERMINISTIC", "1")
    ndim, nodes = 3, [7, 6, 7]
    x, y, w, o, mn, mx = glm_data("poisson", ndim, nodes, 20000, seed=23, weighted=True, hole=True, offset=True)
    for crit in ("reml", "prediction"):
        runs = []
        for _ in range(2):
            h = select_handle(ndim, mn, mx, nodes, 1.0)
            coef, info, trace, ierr = h.glm_select(x, y, w, offset=o, criterion=crit, return_mu=True)
            assert ierr == 0 and info["converged"]
            runs.append((coef, info.pop("mu"), info, trace))
            h.destroy()
        for a, b in zip(runs[0], runs[1]):
            assert np.array_equal(a, b, equal_nan=True) if isinstance(a, np.ndarray) else a == b
        dev = torch.device("cuda", torch.cuda.current_device())
        d_x, d_y, d_w, d_o = (torch.from_numpy(np.ascontiguousarray(a)).to(dev) for a in (x, y, w, o))
        h = select_handle(ndim, mn, mx, nodes, 1.0)
        d_c = torch.zeros(h.ncol, dtype=torch.float64, device=dev)
        d_mu = torch.zeros(len(y), dtype=torch.float64, device=dev)
        info, trace, ierr = h.glm_select_device(d_x, ndim, d_y, d_w, len(y), d_c, d_offset=d_o, criterion=crit,
                                                d_mu=d_mu)
        assert ierr == 0
        assert np.array_equal(d_c.cpu().numpy(), runs[0][0])
        assert np.array_equal(d_mu.cpu().numpy(), runs[0][1])
        assert info == runs[0][2]
        assert np.array_equal(trace, runs[0][3], equal_nan=True)


@pytest.mark.parametrize("family", ["poisson", "binomial", "gamma"])
def test_real32_settles_near_real64(family):
    ndim, nodes = 2, [9, 8]
    x, y, w, o, mn, mx = glm_data(family, ndim, nodes, 20000, seed=31, weighted=True, offset=True)
    h64 = select_handle(ndim, mn, mx, nodes, 0.0)
    _, i64, _, e64 = h64.glm_select(x, y, w, family=family, offset=o)
    h32 = select_handle(ndim, mn, mx, nodes, 0.0, real32=True)
    f32 = [None if a is None else a.astype(np.float32) for a in (x, y, w, o)]
    _, i32, _, e32 = h32.glm_select(f32[0], f32[1], f32[2], family=family, offset=f32[3])
    assert e64 == 0 and e32 == 0 and i64["settled"] and i32["settled"], (i64, i32)
    d = abs(np.log10(i32["lam"]) - np.log10(i64["lam"]))
    print(f"{family}: REAL64 lam {i64['lam']:.4e}, REAL32 lam {i32['lam']:.4e}, {d:.4f} decades")
    assert d <= 0.1


def _ngpu():
    import torch

    return torch.cuda.device_count() if torch.cuda.is_available() else 0


@pytest.mark.skipif(_ngpu() < 2, reason="needs 2 GPUs on one box")
def test_two_devices_bit_identical_replicas():
    import torch

    lib = sp.load()
    ndim, nodes = 2, [9, 8]
    x, y, w, o, mn, mx = glm_data("binomial", ndim, nodes, 30000, seed=41, weighted=True, hole=True, offset=True)
    devs = (C.c_int * 2)(0, 1)
    comms = (C.c_void_p * 2)()
    assert lib.splpak_b200_comm_init_all(2, devs, comms) == 0
    half = len(x) // 2
    res = [None, None]

    def rank(r):
        torch.cuda.set_device(r)
        lo, hi = (0, half) if r == 0 else (half, len(x))
        h = select_handle(ndim, mn, mx, nodes, 1.0)
        dev = torch.device("cuda", r)
        d_x, d_y, d_w, d_o = (torch.from_numpy(np.ascontiguousarray(a[lo:hi])).to(dev) for a in (x, y, w, o))
        d_c = torch.zeros(h.ncol, dtype=torch.float64, device=dev)
        info, trace, ierr = h.glm_select_device(d_x, ndim, d_y, d_w, hi - lo, d_c, family="binomial", d_offset=d_o,
                                                criterion="prediction", comm=comms[r])
        res[r] = (d_c.cpu().numpy(), info, trace, ierr)
        h.destroy()

    threads = [threading.Thread(target=rank, args=(r,)) for r in range(2)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    torch.cuda.set_device(0)
    for r in range(2):
        assert lib.splpak_b200_comm_destroy(comms[r]) == 0
    assert res[0][3] == 0 and res[1][3] == 0
    assert np.array_equal(res[0][0], res[1][0])
    assert res[0][1] == res[1][1]
    assert np.array_equal(res[0][2], res[1][2], equal_nan=True)


# ---------------------------------------------------------------------------------------------------------------------
# 6. refusals
# ---------------------------------------------------------------------------------------------------------------------
def test_refusals():
    ndim, nodes = 2, [6, 6]
    x, y, w, o, mn, mx = glm_data("poisson", ndim, nodes, 500, seed=51, weighted=True, offset=True)
    lib = sp.load()

    def call(h, yy=None, **kw):
        a = dict(l1x=ndim, n=len(y), family=0, criterion=0, penalty=0, lo=0.0, hi=0.0, max_select=10, max_iter=5,
                 tol=1e-8, ncf=h.ncol, nout=13, trace_cap=8)
        a.update(kw)
        xa, ya, wa, oa = (np.ascontiguousarray(v) for v in (x, y if yy is None else yy, w, o))
        coef, out, tr, nt, ierr = np.zeros(h.ncol), np.zeros(13), np.zeros(40), C.c_int64(-1), C.c_int(-1)
        rc = lib.splpak_b200_fit_glm_select(h.h, C.c_void_p(xa.ctypes.data), a["l1x"], C.c_void_p(ya.ctypes.data),
                                            C.c_void_p(wa.ctypes.data), 1, C.c_void_p(oa.ctypes.data), a["n"],
                                            a["family"], a["criterion"], a["penalty"], a["lo"], a["hi"],
                                            a["max_select"], 0, a["max_iter"], a["tol"], None,
                                            C.c_void_p(coef.ctypes.data), a["ncf"], None, C.c_void_p(out.ctypes.data),
                                            a["nout"], C.c_void_p(tr.ctypes.data), a["trace_cap"], C.byref(nt),
                                            C.byref(ierr))
        assert rc == ierr.value
        return rc

    h = select_handle(ndim, mn, mx, nodes, 0.0)
    inf, nan = float("inf"), float("nan")
    for kw in (dict(criterion=2), dict(criterion=-1), dict(penalty=2), dict(lo=nan), dict(hi=inf), dict(lo=-inf),
               dict(lo=2.0, hi=1.0), dict(max_select=0), dict(trace_cap=-1), dict(nout=12), dict(family=3),
               dict(max_iter=0), dict(tol=-1.0), dict(l1x=1)):
        assert call(h, **kw) == 203, kw
    assert call(h, ncf=h.ncol - 1) == 104
    assert call(h, n=0) == 105
    yb = y.copy()
    yb[3] = -1.0
    assert call(h, yy=yb) == 203                                # the domain check: the handle stays fresh
    assert call(h, lo=-1.0, hi=5.0) == 0                        # one bound <= 0: the default range
    assert call(h) == 203                                       # used handle
    assert lib.splpak_b200_fit_get_cholesky_factor(h.h, 0, 0, 1, None, 0, C.byref(C.c_int64(0))) == 203
    assert h.reset() == 0
    assert call(h, criterion=1, penalty=1, lo=1e-3, hi=1e3) == 0
    ortho = sp.FitHandle(ndim, mn, mx, nodes, 0.0, solver="orthogonal")
    assert call(ortho) == 203
    for bad in (dict(family="probit"), dict(criterion="gcv"), dict(penalty="tension")):
        with pytest.raises(SplpakError):
            h.glm_select(x, y, w, **bad)


# ---------------------------------------------------------------------------------------------------------------------
# 7. scale
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("crit", ["reml", "prediction"])
def test_cfg3_scale(crit):
    """cfg3 size: 1e8 device-resident Poisson points, 24^3 nodes, xtrap = 1: converged and settled, Mp < edf < ncol,
    and the returned deviance equals the one recomputed from eval_batch of the returned coefficients."""
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
    h = select_handle(ndim, mn, mx, nodes, 1.0)
    d_c = torch.zeros(h.ncol, dtype=torch.float64, device=dev)
    info, trace, ierr = h.glm_select_device(x, ndim, y, None, n, d_c, family="poisson", criterion=crit)
    print(f"cfg3 poisson {crit}: {info}\n{trace}")
    assert ierr == 0 and info["converged"] and info["settled"], info
    assert null_dim(ndim, "curvature") < info["edf"] < h.ncol
    s = torch.zeros(n, dtype=torch.float64, device=dev)
    assert sp.eval_batch_device(ndim, x, ndim, n, d_c, mn, mx, nodes, s) == 0
    torch.cuda.synchronize()
    mu = torch.clamp(torch.exp(s), min=EPS)
    pos = y > 0
    d = torch.where(pos, y * torch.log(torch.where(pos, y, 1.0) / mu) - (y - mu), mu)
    D = float(2.0 * d.sum())
    assert abs(info["deviance"] - D) <= 1e-10 * D, (info["deviance"], D)
