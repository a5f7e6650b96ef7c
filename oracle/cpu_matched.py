"""'Algorithm-matched' CPU baseline (BASELINE.md section 3, optional second CPU row) -- TEST / BENCH INFRASTRUCTURE.

The reference pushes a dense ncol-wide row per point through a streaming QR (~2 ncol^2 flops per point); the GPU
path assembles the sparse normal equations (4^ndim nonzeros per row) and solves them with a band Cholesky.  To
separate the ALGORITHMIC gain from the hardware gain, this module runs the GPU path's algorithm on the host with
numpy / BLAS / LAPACK on all cores the BLAS uses:

    window-sorted points -> per-window P^T W^2 P (BLAS dsyrk-like matmul of the (m x 4^ndim) basis block)
    -> lower band storage -> scipy.linalg.cholesky_banded + cho_solve_banded (LAPACK dpbtrf / dpbtrs)

Value-only basis arithmetic is oracle/numpy_model.window_weights_numpy (same formulas as bascmp).  No derivative
constraint rows (the benchmark's cfg3 has none firing).  Only bench.py's CPU leg and tests/ import this.
"""
from __future__ import annotations

import time

import numpy as np

from .numpy_model import window_weights_numpy


def assemble_banded(ndim, x, y, w, xmin, xmax, nodes):
    """Returns (ab, g, seconds): lower band storage ab[i-j, j] of G = B^T W^2 B and g = B^T W^2 y."""
    nodes = [int(v) for v in nodes]
    n = int(np.prod(nodes))
    strides = [int(np.prod(nodes[:d])) for d in range(ndim)]
    bw = min(n - 1, 3 * sum(strides))
    t0 = time.perf_counter()
    ws, b = [], []
    for d in range(ndim):
        s, v = window_weights_numpy(np.ascontiguousarray(x[:, d]), float(xmin[d]), float(xmax[d]), nodes[d])
        ws.append(s)
        b.append(v)
    # window id and the point order sorted by it
    wid = np.zeros(len(y), dtype=np.int64)
    mult = 1
    for d in range(ndim):
        wid += ws[d] * mult
        mult *= nodes[d] - 3
    order = np.argsort(wid, kind="stable")
    wid_s = wid[order]
    starts = np.flatnonzero(np.r_[True, wid_s[1:] != wid_s[:-1]])
    ends = np.r_[starts[1:], len(wid_s)]
    # basis block of every point: P[p, (k_ndim..k_1)] = prod_d b_d[k_d], dimension 1 fastest
    P = np.ones((len(y), 1))
    for d in range(ndim):
        P = (b[d].T[:, :, None] * P[:, None, :]).reshape(len(y), -1)      # new dim is the slower index
    if w is not None:
        P = P * w[:, None]
        ry = w * y
    else:
        ry = y
    P = P[order]
    ry = ry[order]
    local = np.array([sum(((idx >> (2 * d)) & 3) * strides[d] for d in range(ndim)) for idx in range(4 ** ndim)],
                     dtype=np.int64)
    li, lj = np.meshgrid(local, local, indexing="ij")
    low = li >= lj
    off_i, off_j = (li - lj)[low], lj[low]
    ab = np.zeros((bw + 1, n))
    g = np.zeros(n)
    flat = ab.reshape(-1)
    for s, e in zip(starts, ends):
        Pw = P[s:e]
        base = 0
        wv = int(wid_s[s])
        for d in range(ndim):
            base += (wv % (nodes[d] - 3)) * strides[d]
            wv //= nodes[d] - 3
        blk = Pw.T @ Pw
        np.add.at(flat, off_i * n + (off_j + base), blk[low])
        np.add.at(g, local + base, Pw.T @ ry[s:e])
    return ab, g, time.perf_counter() - t0


# ------------------------------------------------------------------------------------------------------------------
# Float64 host reference of the GPU's assembled normal equations in its own orthant-stencil layout (tests only):
# S[node, sum_d delta_d 4^d] = G[i, j] with node = the per-dimension min of (i, j) and delta_d = |i_d - j_d|
# (tests/util.dense_from_stencil).  No band storage, so it runs at sizes where a band matrix does not fit in memory.
# ------------------------------------------------------------------------------------------------------------------
_PAIRS = [(m, dl) for m in range(4) for dl in range(4 - m)]      # (local min node, |delta|) of one dimension


def _grid(ndim, nodes):
    nodes = [int(v) for v in nodes[:ndim]]
    strides = [int(np.prod(nodes[:d])) for d in range(ndim)]
    return nodes, strides, int(np.prod(nodes))


def _stencil_table(ndim, nodes, strides):
    """Flat S index (node offset * 4^ndim + stencil) of every entry of the per-window tensor, entries ordered
    (pair_{ndim-1}, ..., pair_0) in C order."""
    tab = np.zeros(1, dtype=np.int64)
    for d in reversed(range(ndim)):
        dt = np.array([m * strides[d] * 4 ** ndim + dl * 4 ** d for m, dl in _PAIRS], dtype=np.int64)
        tab = (tab[:, None] + dt[None, :]).reshape(-1)
    return tab


def _point_terms(ndim, x, w, xmin, xmax, nodes, strides):
    """Per point: window id, first node of the window, the two Kronecker halves L (dimensions ndim-1..h) and
    R = w^2 (dimensions h-1..0) of the 10^ndim stencil products, and the 4^ndim basis products P."""
    n = len(x)
    wid = np.zeros(n, dtype=np.int64)
    base = np.zeros(n, dtype=np.int64)
    mult = 1
    s, b = [], []
    for d in range(ndim):
        # the window's nodes outside bascmp's box [ibmn, ibmx] (:822-829) have zero value there: no masking needed
        ws, bd = window_weights_numpy(np.ascontiguousarray(x[:, d], dtype=np.float64), float(xmin[d]),
                                      float(xmax[d]), nodes[d])
        wid += ws * mult
        base += ws * strides[d]
        mult *= nodes[d] - 3
        s.append(np.stack([bd[m] * bd[m + dl] for m, dl in _PAIRS], axis=1))
        b.append(bd.T)
    h = (ndim + 1) // 2
    L = np.ones((n, 1))
    for d in reversed(range(h, ndim)):
        L = (L[:, :, None] * s[d][:, None, :]).reshape(n, -1)
    w2 = np.ones(n) if w is None else np.asarray(w, dtype=np.float64) ** 2
    R = w2[:, None]
    for d in reversed(range(h)):
        R = (R[:, :, None] * s[d][:, None, :]).reshape(n, -1)
    P = np.ones((n, 1))
    for d in reversed(range(ndim)):
        P = (P[:, :, None] * b[d][:, None, :]).reshape(n, -1)
    return wid, base, L, R, P, w2


def _local_offsets(ndim, strides):
    loff = np.zeros(1, dtype=np.int64)
    for d in reversed(range(ndim)):
        loff = (loff[:, None] + np.arange(4, dtype=np.int64)[None, :] * strides[d]).reshape(-1)
    return loff


def assemble_stencil(ndim, x, y, w, xmin, xmax, nodes, chunk_elems=1 << 25, rhs_only=False):
    """Data rows only, float64: (S[ncol, 4^ndim], g = B^T W^2 y, gabs = |B|^T W^2 |y|).  w None: unweighted;
    rhs_only: S is None (the right-hand side of a refinement step).
    Points are sorted by window once and then processed in chunks of that order (memory bounded by chunk_elems
    doubles per array); each window's block is one GEMM L^T R."""
    nodes, strides, ncol = _grid(ndim, nodes)
    nsten = 4 ** ndim
    x = np.asarray(x)
    n = len(x)
    tab = _stencil_table(ndim, nodes, strides)
    loff = _local_offsets(ndim, strides)
    wid = np.zeros(n, dtype=np.int64)
    mult = 1
    for d in range(ndim):                      # window start as in window_weights_numpy
        dxin = 1.0 / ((float(xmax[d]) - float(xmin[d])) / float(nodes[d] - 1))
        it = np.trunc(dxin * (np.asarray(x[:, d], dtype=np.float64) - float(xmin[d]))).astype(np.int64)
        wid += np.clip(it - 1, 0, nodes[d] - 4) * mult
        mult *= nodes[d] - 3
    order = np.argsort(wid, kind="stable")
    del wid
    S = np.zeros(ncol * nsten)
    g = np.zeros(ncol)
    gabs = np.zeros(ncol)
    width = 10 ** ((ndim + 1) // 2) + 10 ** (ndim // 2) + 3 * nsten
    step = max(1024, chunk_elems // width)
    for lo in range(0, n, step):
        sel = order[lo:lo + step]
        yc = np.asarray(y, dtype=np.float64)[sel]
        wid, base, L, R, P, w2 = _point_terms(ndim, x[sel], None if w is None else np.asarray(w)[sel], xmin, xmax,
                                              nodes, strides)
        starts = np.flatnonzero(np.r_[True, wid[1:] != wid[:-1]])
        ends = np.r_[starts[1:], len(wid)]
        if not rhs_only:
            for s, e in zip(starts, ends):
                S[base[s] * nsten + tab] += (L[s:e].T @ R[s:e]).reshape(-1)
        cols = (base[:, None] + loff[None, :]).reshape(-1)
        g += np.bincount(cols, weights=(P * (w2 * yc)[:, None]).reshape(-1), minlength=ncol)
        gabs += np.bincount(cols, weights=(np.abs(P) * (w2 * np.abs(yc))[:, None]).reshape(-1), minlength=ncol)
    return None if rhs_only else S.reshape(ncol, nsten), g, gabs


def nearest_node_histogram(ndim, x, w, xmin, xmax, nodes):
    """splcw :885-907 vectorised: (cnt[ncol], totlwt, nrows).  cnt[node] = sum of the weights of the nonzero-weight
    points whose rounded position is that node, with int() truncation toward zero and the bare `cycle` of :899 (a
    dimension whose index is out of range is left out of the address); nrows = the number of nonzero-weight points."""
    nodes, _, ncol = _grid(ndim, nodes)
    x = np.asarray(x)
    bump = np.ones(len(x)) if w is None else np.asarray(w, dtype=np.float64)
    keep = bump != 0.0
    iin = np.zeros(len(x), dtype=np.int64)
    for d in reversed(range(ndim)):
        inmx = nodes[d] - 1
        dxin = 1.0 / ((float(xmax[d]) - float(xmin[d])) / float(inmx))
        t = dxin * (np.asarray(x[:, d], dtype=np.float64) - float(xmin[d])) + 0.5
        ini = np.trunc(np.clip(t, -4.0, inmx + 4.0)).astype(np.int64)
        ok = (ini >= 0) & (ini <= inmx)
        iin = np.where(ok, (inmx + 1) * iin + ini, iin)
    cnt = np.bincount(iin[keep], weights=bump[keep], minlength=ncol)
    return cnt, float(bump[keep].sum()), int(keep.sum())


def point_contribution(ndim, xp, yp, wp, xmin, xmax, nodes):
    """What one point adds: (flat S indices, values), (g indices, values), (nearest node, weight); wp None: 1."""
    nodes, strides, _ = _grid(ndim, nodes)
    xp = np.asarray(xp, dtype=np.float64).reshape(1, ndim)
    w = None if wp is None else np.array([float(wp)])
    _, base, L, R, P, w2 = _point_terms(ndim, xp, w, xmin, xmax, nodes, strides)
    s_idx = base[0] * 4 ** ndim + _stencil_table(ndim, nodes, strides)
    g_idx = base[0] + _local_offsets(ndim, strides)
    cnt, _, _ = nearest_node_histogram(ndim, xp, w, xmin, xmax, nodes)
    node = int(np.flatnonzero(cnt)[0]) if cnt.any() else 0
    return (s_idx, (L.T @ R).reshape(-1)), (g_idx, P[0] * w2[0] * float(yp)), (node, 1.0 if wp is None else float(wp))


def solve_banded(ab, g):
    """Returns (coef, seconds) through LAPACK's band Cholesky."""
    from scipy.linalg import cho_solve_banded, cholesky_banded

    t0 = time.perf_counter()
    c = cholesky_banded(ab, lower=True, overwrite_ab=False, check_finite=False)
    coef = cho_solve_banded((c, True), g, check_finite=False)
    return coef, time.perf_counter() - t0


def fit(ndim, x, y, w, xmin, xmax, nodes):
    ab, g, t_asm = assemble_banded(ndim, x, y, w, xmin, xmax, nodes)
    coef, t_solve = solve_banded(ab, g)
    return coef, t_asm, t_solve
