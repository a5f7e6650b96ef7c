"""Shared helpers for the parity tests (test infrastructure)."""
import numpy as np


def make_problem(ndim, nodes, ndata, seed=0, weighted=True, hole=False, outside=0.0, xmin=None, xmax=None):
    """Seeded scattered data on [xmin, xmax]^ndim (optionally with a data hole so constraint rows fire,
    and a fraction `outside` of points beyond the grid to exercise extrapolation / the :899 quirk)."""
    rng = np.random.default_rng(seed)
    xmin = np.zeros(ndim) if xmin is None else np.asarray(xmin, float)
    xmax = np.ones(ndim) if xmax is None else np.asarray(xmax, float)
    u = rng.random((ndata, ndim))
    if outside > 0:
        nout = int(ndata * outside)
        u[:nout] = u[:nout] * 1.6 - 0.3
    if hole:
        c = 0.5
        r = np.sqrt(((u - c) ** 2).sum(axis=1))
        keep = r > 0.3
        u = u[keep]
    x = xmin + u * (xmax - xmin)
    f = np.ones(len(x))
    for d in range(ndim):
        f = f * np.sin(2.0 * u[:, d] + 0.3 * d) + 0.1 * u[:, d]
    y = f + 0.01 * rng.standard_normal(len(x))
    w = rng.random(len(x)) + 0.5 if weighted else None
    return x, y, w, xmin, xmax


def dense_from_stencil(S, nodes):
    """Expand the orthant-stencil storage S[node, 4^ndim] into the dense symmetric Gram matrix."""
    nodes = [int(n) for n in nodes]
    ndim = len(nodes)
    ncol = int(np.prod(nodes))
    idx = np.arange(ncol)
    multi = []
    k = idx.copy()
    for d in range(ndim):
        multi.append(k % nodes[d])
        k = k // nodes[d]
    multi = np.stack(multi, axis=1)            # (ncol, ndim), dimension 1 fastest
    G = np.zeros((ncol, ncol))
    strides = np.cumprod([1] + nodes[:-1])
    for i in range(ncol):
        delta = np.abs(multi - multi[i])        # (ncol, ndim)
        ok = (delta <= 3).all(axis=1)
        mn = np.minimum(multi, multi[i])
        node = (mn * strides).sum(axis=1)
        sten = (delta * (4 ** np.arange(ndim))).sum(axis=1)
        G[i, ok] = S[node[ok], sten[ok]]
    return G


def stencil_scale(diag, nodes):
    """sqrt(G_ii G_jj) for every entry S[node, sten] of the orthant-stencil storage (i = node, j = node + delta), 0
    where j is off the grid.  By Cauchy-Schwarz it bounds the sum of |terms| of G_ij, so tau times it bounds the
    rounding error of that entry summed in any order."""
    nodes = [int(n) for n in nodes]
    ndim = len(nodes)
    ncol = int(np.prod(nodes))
    strides = np.cumprod([1] + nodes[:-1])
    k = np.arange(ncol)
    multi = []
    for d in range(ndim):
        multi.append(k % nodes[d])
        k = k // nodes[d]
    multi = np.stack(multi, axis=1)
    out = np.zeros((ncol, 4 ** ndim))
    for sten in range(4 ** ndim):
        jm = multi + np.array([(sten >> (2 * d)) & 3 for d in range(ndim)])
        ok = (jm < np.array(nodes)).all(axis=1)
        j = (jm[ok] * strides).sum(axis=1)
        out[ok, sten] = np.sqrt(np.abs(diag[ok] * diag[j]))
    return out


def worst_ratio(got, want, tol):
    """max |got - want| / tol; an entry with tol 0 must match exactly (inf otherwise)."""
    err = np.abs(np.asarray(got) - np.asarray(want))
    with np.errstate(divide="ignore", invalid="ignore"):
        r = np.where(err == 0, 0.0, err / tol)
    return float(r.max()) if r.size else 0.0


def coef_tolerance(G, base=1e-10):
    """max(1e-10, 10 * eps * cond(G)): the north star's "~1e-10 relative, scaled by the system's condition
    estimate".  (SURVEY 8c guessed 0.1*eps*cond from a QR-vs-Cholesky comparison; two runs of THIS
    solver that differ only in the order of the atomic flushes -- a few eps relative in G -- were
    measured to differ by up to 3.2*eps*cond in the coefficients, so the constant is 10.  Fitted VALUES
    are compared separately at a far tighter tolerance: they are well conditioned.)"""
    try:
        cond = np.linalg.cond(G)
    except Exception:
        cond = 1e16
    return max(base, 10.0 * np.finfo(float).eps * cond), cond
