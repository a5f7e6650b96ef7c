"""Pointwise posterior variances of smoothing fits (splpak_b200_fit_prepare_variance / _fit_variance[_device]).

q_k(x) = b_k(x)^T Sigma b_k(x) with b_k(x) the row of basis values (or of their nderiv derivatives) at x, built on the
host from oracle.bascmp, and Sigma = inv(M):
  * against the device's own Sigma (selected_inverse, band entries only): isolates the tables and the contraction,
    |q - ref| <= 64 eps |b|^T |Sigma| |b|;
  * end to end against the dense inverse: |q - b^T inv(M) b| <= 100 eps |z|^T |M| |z| + 64 eps |b|^T |Sigma| |b|,
    z = inv(M) b (the first-order bound for a backward error of 100 eps |M|, as in test_gpu_gcv.py)."""
import ctypes
import itertools

import numpy as np
import pytest

import splpak_b200 as sp
from splpak_b200.api import SplpakError
from splpak_b200.distributed import fit_sharded
from test_gpu_gcv import SELINV_CASES, dense_system, gcv_handle, rho_of
from util import make_problem

pytestmark = pytest.mark.gpu
EPS = np.finfo(float).eps


def basis_rows(oracle, q, nderiv, mn, mx, nodes):
    """(cols (nq, 4^ndim), vals (nq, 4^ndim)): the window nodes of every query and bascmp's value there (0 outside
    the reference's index box, as splde sums it)."""
    ndim = len(nodes)
    q = np.atleast_2d(q)
    nq = len(q)
    cols = np.zeros((nq, 4 ** ndim), dtype=np.int64)
    vals = np.zeros((nq, 4 ** ndim))
    strides = np.cumprod([1] + list(nodes[:-1]))
    for i in range(nq):
        ws, box = [], []
        for d in range(ndim):
            dx = (mx[d] - mn[d]) / (nodes[d] - 1)
            t = (q[i, d] - mn[d]) * (1.0 / dx)
            it = int(np.trunc(t)) if np.isfinite(t) else 0
            it = min(max(it, -4), nodes[d] + 4)
            ws.append(min(max(it - 1, 0), nodes[d] - 4))
            box.append((min(max(it - 1, 0), nodes[d] - 2), max(min(it + 2, nodes[d] - 1), 1)))
        for k, off in enumerate(itertools.product(range(4), repeat=ndim)):
            ib = [ws[d] + off[ndim - 1 - d] for d in range(ndim)]       # dimension 1 fastest
            cols[i, k] = int(np.dot(ib, strides))
            if all(box[d][0] <= ib[d] <= box[d][1] for d in range(ndim)):
                vals[i, k] = oracle.bascmp(ib, q[i], nderiv, mn, mx, nodes)[1]
    return cols, vals


def band_block(Sig, cols):
    """The dense 4^ndim x 4^ndim block Sigma(cols, cols) from the band rows Sig[i, k] = Sigma(i, i + k)."""
    r = np.minimum.outer(cols, cols)
    c = np.abs(np.subtract.outer(cols, cols))
    return Sig[r, c]


def band_reference(Sig, cols, vals):
    """(b^T Sigma b, |b|^T |Sigma| |b|) per query."""
    ref, mag = np.zeros(len(cols)), np.zeros(len(cols))
    for i in range(len(cols)):
        B = band_block(Sig, cols[i])
        ref[i] = vals[i] @ B @ vals[i]
        mag[i] = np.abs(vals[i]) @ np.abs(B) @ np.abs(vals[i])
    return ref, mag


def query_set(ndim, nodes, mn, mx, rng, n_random=24):
    """Interior and edge windows, points on nodes, points several cells outside the box."""
    dx = (np.asarray(mx) - np.asarray(mn)) / (np.asarray(nodes) - 1)
    pts = [mn + rng.random((n_random, ndim)) * (mx - mn)]
    pts.append(mn + rng.random((6, ndim)) * dx * 1.5)                                    # low edge windows
    pts.append(mx - rng.random((6, ndim)) * dx * 1.5)                                    # high edge windows
    pts.append(mn + rng.integers(0, np.asarray(nodes), size=(6, ndim)) * dx)             # on nodes
    out = mn + rng.random((8, ndim)) * (mx - mn)
    out[:, 0] = np.where(np.arange(8) % 2 == 0, mn[0] - 3.5 * dx[0], mx[0] + 4.2 * dx[0])  # several cells outside
    pts.append(out)
    return np.concatenate(pts)


def prepared(ndim, nodes, ndata, xtrap, lamf, penalty, seed, **kw):
    x, y, w, mn, mx = make_problem(ndim, nodes, ndata, seed=seed, hole=xtrap != 0.0)
    h = gcv_handle(ndim, mn, mx, nodes, xtrap, x, y, w, **kw)
    lam = 0.0
    if lamf > 0:
        G = h.normal_equations()[0].reshape(h.ncol, -1)[:, 0]
        from test_gpu_smoothing import penalty_dense
        lam = lamf * G.sum() / np.trace(penalty_dense(nodes, mn, mx, penalty))
        assert h.set_smoothing(lam, penalty) == 0
    score = h.prepare_variance()
    return h, score, lam, (x, y, w, mn, mx)


KERNEL_CASES = [(1, [9]), (2, [7, 6]), (3, [6, 5, 7]), (4, [5, 4, 4, 5])]


@pytest.mark.parametrize("ndim,nodes", KERNEL_CASES)
def test_kernel_matches_band_quadratic_form(oracle, ndim, nodes):
    """Every nderiv combination 0..2 per dimension, interior / edge / node / exterior queries, against b^T Sigma b with
    the device's own Sigma; a NaN coordinate gives NaN."""
    h, score, lam, (x, y, w, mn, mx) = prepared(ndim, nodes, 4000 * ndim, 1.0, 1e-3, "thin_plate", seed=ndim)
    Sig = h.selected_inverse()
    rng = np.random.default_rng(100 + ndim)
    q = query_set(ndim, nodes, mn, mx, rng, n_random=24 if ndim < 4 else 6)
    combos = list(itertools.product(range(3), repeat=ndim))
    for nd in combos:
        cols, vals = basis_rows(oracle, q, list(nd), mn, mx, nodes)
        ref, mag = band_reference(Sig, cols, vals)
        got, ierr = h.variance(q, nderiv=list(nd))
        assert ierr == 0
        err = np.abs(got - ref)
        assert np.all(err <= 64 * EPS * mag), (nd, err.max(), (err / np.maximum(mag, 1e-300)).max() / EPS)
    qn = q[:4].copy()
    qn[1, 0] = np.nan
    qn[3, ndim - 1] = np.nan
    got, ierr = h.variance(qn)
    assert ierr == 0 and np.isnan(got[1]) and np.isnan(got[3]) and np.isfinite(got[0]) and np.isfinite(got[2])
    h.destroy()


@pytest.mark.parametrize("solver", ["persistent", "graph"])
@pytest.mark.parametrize("ndim,nodes,ndata,xtrap,lamf,penalty", SELINV_CASES)
def test_end_to_end_vs_dense_inverse(oracle, monkeypatch, solver, ndim, nodes, ndata, xtrap, lamf, penalty):
    if solver == "graph":
        monkeypatch.setenv("SPLPAK_B200_SOLVER", "graph")
    else:
        monkeypatch.delenv("SPLPAK_B200_SOLVER", raising=False)
    x, y, w, mn, mx = make_problem(ndim, nodes, ndata, seed=ndim * 7 + nodes[0], hole=xtrap != 0.0)
    A0, _ = oracle.rows(ndim, x, y, w, mn, mx, nodes, 0.0)
    lam = lamf * rho_of(nodes, mn, mx, penalty, A0.T @ A0) if lamf > 0 else 0.0
    M, *_ = dense_system(oracle, ndim, x, y, w, mn, mx, nodes, xtrap, lam, penalty)
    h = gcv_handle(ndim, mn, mx, nodes, xtrap, x, y, w)
    assert h.set_smoothing(lam, penalty) == 0
    h.prepare_variance()
    Sig = h.selected_inverse()
    # The componentwise bound resolves 1e-3 of q only while M is moderately conditioned.  In the 1-D case with a data
    # hole of 420 nodes held by constraint rows alone (cond(M) > 1e10), the rows' mixed-sign stencils make
    # |z|^T |M| |z| exceed z^T M z by ~1e16 in the hole, and the Cholesky backward error is not componentwise in |M|
    # there.  That case is held to the forward error of Sigma that test_gpu_gcv.py accepts for the selected inverse,
    # 100 eps cond(M) max|Sigma| per entry, i.e. 100 eps cond(M) max|Sigma| (sum |b|)^2 for q.
    condM = np.linalg.cond(M)
    discriminating = condM < 1e10
    sig_max = np.abs(np.linalg.inv(M)).max()
    rng = np.random.default_rng(7)
    q = query_set(ndim, nodes, mn, mx, rng, n_random=16)
    for nd in ([0] * ndim, [2] + [0] * (ndim - 1), [1] * ndim):
        cols, vals = basis_rows(oracle, q, nd, mn, mx, nodes)
        _, mag = band_reference(Sig, cols, vals)
        got, ierr = h.variance(q, nderiv=nd)
        assert ierr == 0
        for i in range(len(q)):
            b = np.zeros(M.shape[0])
            np.add.at(b, cols[i], vals[i])
            if not b.any():
                assert got[i] == 0.0
                continue
            z = np.linalg.solve(M, b)
            ref = b @ z
            tol = 100 * EPS * (np.abs(z) @ np.abs(M) @ np.abs(z)) + 64 * EPS * mag[i]
            if discriminating:
                assert tol < 1e-3 * ref, (nd, i, tol, ref, condM)
            else:
                tol = max(tol, 100 * EPS * condM * sig_max * np.abs(b).sum() ** 2)
            assert abs(got[i] - ref) <= tol, (nd, i, got[i], ref, tol)
    h.destroy()


def leverage_sum(h, x, w):
    qv, ierr = h.variance(x)
    assert ierr == 0
    w2 = np.ones(len(x)) if w is None else w ** 2
    return float((w2 * qv).sum()), qv


LEVERAGE_CASES = [
    # ndim, nodes, ndata, xtrap, lambda factor, penalty
    (1, [60], 3000, 0.0, 0.0, "curvature"),
    (1, [40], 1500, 1.0, 1e-4, "thin_plate"),
    (2, [10, 9], 3000, 1.0, 0.0, "curvature"),
    (3, [6, 6, 5], 3000, 0.0, 1e-3, "curvature"),
    (3, [6, 5, 5], 2500, 1.0, 1e-3, "thin_plate"),
    (4, [5, 4, 4, 5], 1200, 1.0, 1e-2, "thin_plate"),
]


@pytest.mark.parametrize("ndim,nodes,ndata,xtrap,lamf,penalty", LEVERAGE_CASES)
def test_leverages_sum_to_edf(oracle, ndim, nodes, ndata, xtrap, lamf, penalty):
    """sum_i w_i^2 q_0(x_i) = edf, within the sum of the per-point bounds 64 eps w_i^2 |b|^T |Sigma| |b| (plus the
    summation of the sum itself)."""
    h, score, lam, (x, y, w, mn, mx) = prepared(ndim, nodes, ndata, xtrap, lamf, penalty, seed=ndim * 7 + nodes[0])
    Sig = h.selected_inverse()
    total, qv = leverage_sum(h, x, w)
    cols, vals = basis_rows(oracle, x, [0] * ndim, mn, mx, nodes)
    _, mag = band_reference(Sig, cols, vals)
    tol = 64 * EPS * float((w ** 2 * mag).sum()) + len(x) * EPS * total
    assert abs(total - score["edf"]) <= tol, (total, score["edf"], tol)
    h.destroy()


def test_leverages_sum_to_edf_cfg3_1e8_points(oracle):
    """cfg3 (24^3, xtrap = 1) with 1e8 device-resident points, where no dense reference exists.  The per-point bound
    64 eps w^2 |b|^T |Sigma| |b| is taken as 64 eps w^2 q times twice the largest ratio |b|^T |Sigma| |b| / q over 300
    sampled data points."""
    import torch

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
    h.select_smoothing("curvature")
    score = h.prepare_variance()
    out = torch.empty(n, dtype=torch.float64, device="cuda")
    assert h.variance_device(x, 3, n, out) == 0
    h.synchronize()
    total = float((w * w * out).sum())
    idx = torch.randint(0, n, (300,), device="cuda", generator=g)
    xs, qs = x[idx].cpu().numpy(), out[idx].cpu().numpy()
    cols, vals = basis_rows(oracle, xs, [0, 0, 0], mn, mx, nodes)
    _, mag = band_reference(h.selected_inverse(), cols, vals)
    ratio = float((mag / qs).max())
    tol = 64 * EPS * 2 * ratio * total + n * EPS * total       # the second term: the summation of the sum itself
    assert 0 < score["edf"] < h.ncol
    assert abs(total - score["edf"]) <= tol, (total, score["edf"], tol)
    h.destroy()


def test_scaling_is_the_sampling_variance():
    """lambda = 0, xtrap = 0, weights: sigma2 q_0(x) is the exact sampling variance of s(x) when Var(y_i) = sigma^2 / w_i^2.
    400 seeded noisy fits of one 1-D problem: the sample variance of s at 50 queries against sigma^2 q_0 within 5 standard
    errors of a chi-square with 399 degrees of freedom; the mean sigma2 within 5 % of sigma^2."""
    rng = np.random.default_rng(2024)
    nodes = [16]
    n = 1500
    x = rng.random((n, 1))
    w = 0.5 + rng.random(n)
    f = np.sin(4 * x[:, 0])
    sigma = 0.2
    mn, mx = np.zeros(1), np.ones(1)
    xq = np.linspace(-0.1, 1.1, 50).reshape(-1, 1)
    h = sp.FitHandle(1, mn, mx, nodes, 0.0)
    assert h.enable_gcv() == 0
    vals, s2s, q0 = [], [], None
    for k in range(400):
        assert h.reset() == 0
        y = f + sigma / w * rng.standard_normal(n)
        assert h.add_points(x, y, w) == 0
        s2s.append(h.prepare_variance()["sigma2"])
        c, ierr = h.compute()
        assert ierr == 0
        qk, ierr = h.variance(xq)
        assert ierr == 0
        if q0 is None:
            q0 = qk
        np.testing.assert_allclose(qk, q0, rtol=1e-10)   # same x and w: the same tables up to the assembly's rounding
        vals.append(sp.eval_batch(1, xq, c, mn, mx, nodes)[0])
    h.destroy()
    ratio = np.var(np.array(vals), axis=0, ddof=1) / (sigma ** 2 * q0)
    assert np.all(np.abs(ratio - 1) <= 5 * np.sqrt(2 / 399)), ratio
    assert abs(np.mean(s2s) / sigma ** 2 - 1) < 0.05, np.mean(s2s)


def test_handle_flow(monkeypatch):
    nodes = [9, 8]
    x, y, w, mn, mx = make_problem(2, nodes, 8000, seed=12, hole=True)
    q = make_problem(2, nodes, 500, seed=13)[0]
    h = gcv_handle(2, mn, mx, nodes, 1.0, x, y, w)
    lam, score, _ = h.select_smoothing("curvature")
    n0 = h.launch_count()
    pv = h.prepare_variance()
    assert h.launch_count() == n0 + 1                     # the table build only: no second score
    for k in ("gcv", "rss", "edf", "n", "ywy"):
        assert pv[k] == score[k]
    assert pv["sigma2"] == pv["rss"] / (pv["n"] - pv["edf"])
    q1, ierr = h.variance(q)
    assert ierr == 0
    c, ierr = h.compute()
    assert ierr == 0
    assert np.array_equal(h.variance(q)[0], q1)           # survives compute
    h.refine(x, y, w, steps=1)
    assert np.array_equal(h.variance(q)[0], q1)           # and refinement
    assert h.reset() == 0
    assert h.variance(q)[1] == 203                        # reset invalidates
    h.destroy()
    # add_points and another lambda invalidate; the same lambda does not
    h = gcv_handle(2, mn, mx, nodes, 1.0, x, y, w)
    assert h.set_smoothing(1e-3, "curvature") == 0
    h.prepare_variance()
    assert h.set_smoothing(1e-3, "curvature") == 0
    assert h.variance(q)[1] == 0
    assert h.set_smoothing(2e-3, "curvature") == 0
    assert h.variance(q)[1] == 203
    h.prepare_variance()
    assert h.add_points(x[:100], y[:100], w[:100]) == 0
    assert h.variance(q)[1] == 203
    h.destroy()
    # deterministic mode: compute after prepare_variance is bit-identical to compute without it; launch counts of a
    # handle that never calls it are those of a plain GCV handle
    monkeypatch.setenv("SPLPAK_B200_DETERMINISTIC", "1")
    res = {}
    for mode in ("plain", "var"):
        h = gcv_handle(2, mn, mx, nodes, 1.0, x, y, w)
        assert h.set_smoothing(1e-3, "thin_plate") == 0
        if mode == "var":
            h.prepare_variance()
        n1 = h.launch_count()
        c, ierr = h.compute()
        assert ierr == 0
        res[mode] = (c, h.launch_count() - n1, h.partial_tensor().numel())
        h.destroy()
    assert np.array_equal(res["plain"][0], res["var"][0])
    assert res["plain"][1:] == res["var"][1:]


def test_determinism_and_emulated_ranks():
    import torch

    ndim, nodes = 3, [8, 7, 6]
    x, y, w, mn, mx = make_problem(ndim, nodes, 30000, seed=21, hole=True)
    qh = make_problem(ndim, nodes, 100000, seed=22, outside=0.1)[0]
    d_q = torch.from_numpy(qh).cuda()
    parts, total = [], None
    for r in range(3):
        lo, hi = r * len(x) // 3, (r + 1) * len(x) // 3
        hr = gcv_handle(ndim, mn, mx, nodes, 1.0, x[lo:hi], y[lo:hi], w[lo:hi])
        hr.synchronize()
        t = hr.partial_tensor().clone()
        total = t if total is None else total + t
        parts.append(hr)
    outs = []
    for hr in parts:
        hr.partial_tensor().copy_(total)
        torch.cuda.synchronize()
        hr.select_smoothing("thin_plate")
        hr.prepare_variance()
        o = torch.empty(len(qh), dtype=torch.float64, device="cuda")
        for _ in range(2):
            o2 = torch.empty_like(o)
            assert hr.variance_device(d_q, ndim, len(qh), o2, nderiv=[0, 1, 2]) == 0
            hr.synchronize()
            if _ == 0:
                o = o2
            else:
                assert torch.equal(o, o2)                  # repeated calls bit-identical
        outs.append(o)
    for o in outs[1:]:
        assert torch.equal(o, outs[0])                     # every rank the same tables
    for hr in parts:
        hr.destroy()

    # fit_sharded in one process: the variances of the handle it prepared equal a direct handle's (deterministic
    # assembly, so both handles hold the same sums)
    import os
    os.environ["SPLPAK_B200_DETERMINISTIC"] = "1"
    try:
        hs, hd = fit_sharded_pair(ndim, mn, mx, nodes, x, y, w)
    finally:
        del os.environ["SPLPAK_B200_DETERMINISTIC"]
    assert np.array_equal(hs.variance(qh)[0], hd.variance(qh)[0])
    hs.destroy()
    hd.destroy()


def fit_sharded_pair(ndim, mn, mx, nodes, x, y, w):
    hs = sp.FitHandle(ndim, mn, mx, nodes, 1.0)
    assert hs.enable_gcv() == 0
    coef, ierr = fit_sharded(hs, x, y, w, select_smoothing="thin_plate", prepare_variance=True)
    assert ierr == 0
    hd = gcv_handle(ndim, mn, mx, nodes, 1.0, x, y, w)
    hd.select_smoothing("thin_plate")
    hd.prepare_variance()
    return hs, hd


def test_scale_cfg4_spot_check(oracle):
    """cfg4 (12^4): one prepare, 1e6 device queries, 64 of them against b^T Sigma b with the device's Sigma."""
    import torch

    nodes = [12, 12, 12, 12]
    n = 4_000_000
    g = torch.Generator(device="cuda").manual_seed(4)
    x = torch.rand((n, 4), dtype=torch.float64, device="cuda", generator=g)
    y = torch.sin(2 * x[:, 0]) * x[:, 1] + x[:, 2] - x[:, 3] ** 2 + 0.01 * torch.randn(n, dtype=torch.float64,
                                                                                        device="cuda", generator=g)
    mn, mx = np.zeros(4), np.ones(4)
    h = sp.FitHandle(4, mn, mx, nodes, 1.0)
    assert h.enable_gcv() == 0
    assert h.add_points_device(x, 4, y, None, n, weighted=False) == 0
    assert h.set_smoothing(1e-4, "curvature") == 0
    h.prepare_variance()
    Sig = h.selected_inverse()
    nq = 1_000_000
    q = torch.rand((nq, 4), dtype=torch.float64, device="cuda", generator=g) * 1.2 - 0.1
    out = torch.empty(nq, dtype=torch.float64, device="cuda")
    assert h.variance_device(q, 4, nq, out, nderiv=[1, 0, 2, 0]) == 0
    h.synchronize()
    idx = np.random.default_rng(0).integers(0, nq, 64)
    qh = q.cpu().numpy()[idx]
    cols, vals = basis_rows(oracle, qh, [1, 0, 2, 0], mn, mx, nodes)
    ref, mag = band_reference(Sig, cols, vals)
    got = out.cpu().numpy()[idx]
    assert np.all(np.abs(got - ref) <= 64 * EPS * mag)
    h.destroy()


def test_64bit_query_index():
    """1-D, nq > 2^31 device queries: the entries past 2^31 equal the host path's values at the same points."""
    import torch

    nodes = [40]
    x, y, w, mn, mx = make_problem(1, nodes, 5000, seed=1)
    h = gcv_handle(1, mn, mx, nodes, 0.0, x, y, w)
    assert h.set_smoothing(1e-6, "curvature") == 0
    h.prepare_variance()
    nq = (1 << 31) + 4099
    d_x = torch.linspace(-0.2, 1.2, nq, dtype=torch.float64, device="cuda")
    d_out = torch.full((nq,), -1.0, dtype=torch.float64, device="cuda")
    assert h.variance_device(d_x, 1, nq, d_out) == 0
    h.synchronize()
    idx = np.concatenate([np.arange(0, 8), np.arange(nq - 5000, nq), (1 << 31) + np.arange(-4, 4)])
    ti = torch.from_numpy(idx).cuda()
    want, ierr = h.variance(d_x[ti].cpu().numpy().reshape(-1, 1))
    assert ierr == 0
    assert np.array_equal(d_out[ti].cpu().numpy(), want)
    assert float(d_out.min()) >= 0.0
    del d_x, d_out
    torch.cuda.empty_cache()
    h.destroy()


def test_real32_agrees_with_real64():
    nodes = [9, 8]
    x, y, w, mn, mx = make_problem(2, nodes, 20000, seed=13, hole=True)
    x, y, w = (a.astype(np.float32) for a in (x, y, w))
    q = make_problem(2, nodes, 2000, seed=14, outside=0.1)[0].astype(np.float32)
    out = []
    for real32 in (False, True):
        h = sp.FitHandle(2, mn, mx, nodes, 1.0, real32=real32)
        assert h.enable_gcv() == 0
        dt = np.float32 if real32 else np.float64
        assert h.add_points(x.astype(dt), y.astype(dt), w.astype(dt)) == 0
        assert h.set_smoothing(1e-3, "curvature") == 0
        h.prepare_variance()
        v, ierr = h.variance(q.astype(dt), nderiv=[1, 0])
        assert ierr == 0
        assert v.dtype == dt
        out.append(v.astype(np.float64))
        h.destroy()
    # the assembly of the REAL32 library differs at ~1e-7 relative (test_gpu_gcv.py), the output is rounded to float
    np.testing.assert_allclose(out[1], out[0], rtol=1e-5)


def test_refusals(monkeypatch):
    nodes = [6, 6]
    x, y, w, mn, mx = make_problem(2, nodes, 2000, seed=3)
    q = x[:10]
    h = sp.FitHandle(2, mn, mx, nodes, 1.0)
    assert h.add_points(x, y, w) == 0
    with pytest.raises(SplpakError) as e:
        h.prepare_variance()                                      # GCV not enabled
    assert e.value.args[1] == 203
    assert h.variance(q)[1] == 203
    h.destroy()
    h = gcv_handle(2, mn, mx, nodes, 1.0, x, y, w)
    assert h.variance(q)[1] == 203                                # no tables yet
    out = np.zeros(6)
    assert h.lib.splpak_b200_fit_prepare_variance(h.h, out.ctypes.data_as(ctypes.c_void_p), 5, None) == 203
    h.prepare_variance()
    assert h.variance(q, nderiv=[0, 3])[1] == 104
    assert h.variance(q, nderiv=[-1, 0])[1] == 104
    assert h.variance(q[:0])[1] == 0                             # nq = 0: no-op
    assert h.compute()[1] == 0
    with pytest.raises(SplpakError) as e:
        h.prepare_variance()                                      # finalized
    assert e.value.args[1] == 203
    assert h.variance(q)[1] == 0                                  # the tables stay usable
    h.destroy()
    monkeypatch.setenv("SPLPAK_B200_FIT", "orthogonal")
    he = sp.FitHandle(2, mn, mx, nodes, 1.0)
    assert he.solver() == "orthogonal"
    assert he.add_points(x, y, w) == 0
    with pytest.raises(SplpakError) as e:
        he.prepare_variance()
    assert e.value.args[1] == 203
    he.destroy()
