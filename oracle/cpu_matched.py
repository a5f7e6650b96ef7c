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


# ------------------------------------------------------------------------------------------------------------------
# Host references of the band Cholesky factor (tests only).  The device keeps G = L L^T in lower band storage with
# leading dimension lda = (b + 65) rounded up to even, panels of 64 columns, and the block inverses L11^-1 of the panels
# in a workspace; FitHandle.cholesky_factor reads both back: band row j = L(j .. j + lda - 1, j), blocks (nblk, 64, 64).
# ------------------------------------------------------------------------------------------------------------------
NB = 64


def band_lda(bw):
    return (int(bw) + NB + 1) & ~1


def half_bandwidth(ndim, nodes):
    nodes, strides, ncol = _grid(ndim, nodes)
    return min(ncol - 1, 3 * sum(strides))


def _lsb_exponent(a):
    """Smallest exponent e such that every nonzero entry of a is an integer multiple of 2^e."""
    v = np.abs(np.asarray(a, dtype=np.float64).reshape(-1))
    v = v[v != 0]
    if v.size == 0:
        return 0
    m, e = np.frexp(v)
    mi = (m * 2.0 ** 53).astype(np.int64)
    return int((e.astype(np.int64) - 53 + np.log2(mi & -mi).astype(np.int64)).min())


def _sum_is_exact(bound, unit_exp):
    """bound: the float64 sum of |terms| of a family of sums whose terms are integer multiples of 2^unit_exp.  Every
    partial sum is then exact in binary64 iff the exact bound is below 2^(53 + unit_exp).  The float64 sum of
    non-negative terms decides that exactly: rounding is monotone, so it stays below 2^(53 + unit_exp) exactly when all
    its partial sums are below it, and then none of them was rounded."""
    return float(np.max(bound, initial=0.0)) < 2.0 ** (53 + unit_exp)


def _tribonacci_inverse(m):
    """t[k] = the k-th subdiagonal of (I - N)^-1, N with unit entries on subdiagonals 1 and 3 (t[k] ~ 1.4656^k)."""
    t = np.zeros(max(int(m), 4))
    t[0] = 1.0
    for k in range(1, len(t)):
        t[k] = t[k - 1] + (t[k - 3] if k >= 3 else 0.0)
    return t


def kron_exact_system(ndim, nodes, scale_exp=0, zero=None, seed=0, check=True):
    """A system whose band Cholesky factorization and solve are exact in binary64 in any summation order.

    M = 2^s (M_ndim x ... x M_1) (dimension 1 fastest, the library's column order), M_d = L_d L_d^T,
    L_d = D_d (I - N_d), N_d with unit entries on subdiagonals 1 and 3 (half bandwidth 3: M fits the orthant-stencil
    storage, whose entries depend only on the per-dimension unordered pairs, as a Kronecker product's do), D_d = 2^(i mod 2)
    per node so that neighbouring pivots differ.  Then chol(M) = 2^(s/2) (x) L_d, the block inverses are the diagonal
    blocks of 2^(-s/2) (x) (I - N_d)^-1 D_d^-1, and for integer c*, g = M c* is exact.  s must be even.
    zero = (d, i): D_d[i] = 0, so every row of M whose node has index i in dimension d vanishes and the first of them
    is a zero pivot (no factor is returned then).
    check: assert that every value lies within 2^+-1020 and that every product sum the device forms -- the panel GEMM
    A21 L11^-T, the trailing update, the blocked inversion, y1 = L11^-1 g1, the right-hand side updates and the
    back-substitution, with |c| <= 2 -- stays below 2^53 units of its terms' smallest power of two.
    Returns dict(part: the partial-buffer image [S | g | cnt | totlwt | nrows], L: scipy CSC factor, linv: (nblk, 64,
    64) with the last block padded with the identity, c: c*, delta: a second integer vector and r = M delta (a
    refinement step's right-hand side), g, M (CSC), bw, lda, ncol)."""
    import scipy.sparse as sps

    from splpak_b200.distributed import partial_layout

    assert scale_exp % 2 == 0
    nodes, strides, ncol = _grid(ndim, nodes)
    Ds, Ls, Ms, tabs = [], [], [], []
    for d in range(ndim):
        nd = nodes[d]
        D = 2.0 ** (np.arange(nd) % 2)
        if zero is not None and zero[0] == d:
            D[zero[1]] = 0.0
        Ld = np.diag(D) - np.diag(D[1:], -1) - np.diag(D[3:], -3)
        Md = Ld @ Ld.T
        tab = np.zeros((nd, 4))
        for dl in range(4):
            tab[:nd - dl, dl] = np.diagonal(Md, -dl)
        Ds.append(D)
        Ls.append(sps.csc_matrix(Ld))
        Ms.append(sps.csc_matrix(Md))
        tabs.append(tab)
    S = tabs[0]
    L = Ls[0]
    M = Ms[0]
    for d in range(1, ndim):
        S = (tabs[d][:, None, :, None] * S[None, :, None, :]).reshape(tabs[d].shape[0] * S.shape[0], -1)
        L = sps.kron(Ls[d], L, format="csc")
        M = sps.kron(Ms[d], M, format="csc")
    S = S * 2.0 ** scale_exp
    M = (M * 2.0 ** scale_exp).tocsc()
    L = (L * 2.0 ** (scale_exp // 2)).tocsc()
    rng = np.random.default_rng(seed)
    c = rng.integers(-2, 3, ncol).astype(np.float64)
    delta = rng.integers(-2, 3, ncol).astype(np.float64)
    g = M @ c
    off, total = partial_layout(ndim, nodes)
    part = np.zeros(total)
    part[off["S"][0]:off["S"][1]] = S.reshape(-1)
    part[off["g"][0]:off["g"][1]] = g
    part[off["cnt"][0]:off["cnt"][1]] = 1.0
    part[off["totlwt"][0]] = part[off["nrows"][0]] = float(ncol)
    bw = half_bandwidth(ndim, nodes)
    out = dict(part=part, c=c, delta=delta, r=M @ delta, g=g, bw=bw, lda=band_lda(bw), ncol=ncol, M=M)
    if zero is not None:
        return out
    # block inverses: X[a, b] = 2^(-s/2) prod_d t[a_d - b_d] / D_d[b_d], zero unless a >= b in every dimension (and then
    # every a_d - b_d < 64, since sum_d (a_d - b_d) stride_d = a - b < 64)
    nblk = (ncol + NB - 1) // NB
    t = _tribonacci_inverse(NB)
    idx = np.minimum(np.arange(nblk * NB).reshape(nblk, NB), ncol - 1)
    X = np.full((nblk, NB, NB), 2.0 ** (-(scale_exp // 2)))
    k = idx.copy()
    for d in range(ndim):
        i_d = k % nodes[d]
        k = k // nodes[d]
        diff = i_d[:, :, None] - i_d[:, None, :]
        X *= np.where(diff >= 0, t[np.clip(diff, 0, NB - 1)], 0.0) / Ds[d][i_d][:, None, :]
    nb_last = ncol - (nblk - 1) * NB
    if nb_last < NB:
        X[-1, nb_last:, :] = 0.0
        X[-1, :, nb_last:] = 0.0
        X[-1, nb_last:, nb_last:] = np.eye(NB - nb_last)
    out.update(L=L, linv=X)
    if check:
        _assert_exact(M, L, X, g, (c, delta), ncol)
    return out


def _assert_exact(M, L, X, g, cs, ncol):
    """The bounds of kron_exact_system's check, each a sum of |terms| of the products the device forms, with the
    actual values of their factors."""
    Ma, La = abs(M), abs(L)
    for name, v in (("M", M.data), ("L", L.data), ("L11^-1", X[X != 0]), ("g", g[g != 0])):
        v = np.abs(v)
        assert v.max(initial=1.0) < 2.0 ** 1020 and v.min(initial=1.0) > 2.0 ** -1020, name
    nblk = X.shape[0]
    X = X.copy()
    nb_last = ncol - (nblk - 1) * NB
    X[-1, nb_last:, nb_last:] = 0.0                       # the identity padding: 1 x 1 products, exact at any scale
    eM, eL, eX = _lsb_exponent(M.data), _lsb_exponent(L.data), _lsb_exponent(X)
    assert _sum_is_exact((Ma + La @ La.T).data, min(eM, 2 * eL)), "trailing update"
    A21 = abs(sps_tril_blocks_off(M))                      # A21 = L21 L11^T: the entries of M below the diagonal blocks
    Xa = np.abs(X)
    for kb in range(nblk):
        j0, j1 = kb * NB, min(ncol, kb * NB + NB)
        nb = j1 - j0
        L11 = np.zeros((NB, NB))
        L11[:nb, :nb] = L[j0:j1, j0:j1].toarray()
        L11a = np.abs(L11)
        # blocked inversion: the 8 x 8 diagonal blocks, then X21 = -X22 (L21 X11) at block sizes 8, 16, 32
        for b0 in range(0, NB, 8):
            assert _sum_is_exact(L11a[b0:b0 + 8, b0:b0 + 8] @ Xa[kb, b0:b0 + 8, b0:b0 + 8], eL + eX), f"inversion, {kb}"
        for sz in (8, 16, 32):
            for q in range(NB // (2 * sz)):
                rb, cb = (2 * q + 1) * sz, 2 * q * sz
                T = L11a[rb:rb + sz, cb:cb + sz] @ Xa[kb, cb:cb + sz, cb:cb + sz]
                assert _sum_is_exact(T, eL + eX), f"inversion, panel {kb}"
                assert _sum_is_exact(Xa[kb, rb:rb + sz, rb:rb + sz] @ np.abs(L11[rb:rb + sz, cb:cb + sz] @
                                                                              X[kb, cb:cb + sz, cb:cb + sz]),
                                     2 * eX + eL), f"inversion, panel {kb}"
        if j1 < ncol:
            assert _sum_is_exact(A21[j1:, j0:j1] @ Xa[kb, :nb, :nb].T, 2 * eL + eX), f"panel GEMM, panel {kb}"
    for c in cs:
        assert _sum_is_exact(Ma @ np.abs(c), eM), "g = M c"
        y = L.T @ c
        assert _sum_is_exact(np.abs(M @ c) + La @ np.abs(y), min(eM, 2 * eL)), "right-hand side updates g - L y"
        assert _sum_is_exact(La.T @ np.abs(c), eL), "back-substitution updates y - L^T c"
        for kb in range(nblk):
            j0, j1 = kb * NB, min(ncol, kb * NB + NB)
            L11 = L[j0:j1, j0:j1]
            Xk = Xa[kb, :j1 - j0, :j1 - j0]
            assert _sum_is_exact(Xk @ np.abs(L11 @ y[j0:j1]), eX + 2 * eL), f"y1 = L11^-1 g1, panel {kb}"
            assert _sum_is_exact(Xk.T @ np.abs(L11.T @ c[j0:j1]), eX + eL), f"c1 = L11^-T y1, panel {kb}"


def sps_tril_blocks_off(M):
    """The entries of a sparse lower-or-full matrix that lie below the 64 x 64 diagonal blocks (CSC)."""
    C = M.tocoo()
    keep = (C.row // NB) > (C.col // NB)
    import scipy.sparse as sps

    return sps.csc_matrix((C.data[keep], (C.row[keep], C.col[keep])), shape=M.shape)


def band_image(L, lda, first_col=0, ncols=None):
    """A lower-triangular (sparse or dense) matrix in FitHandle.cholesky_factor's layout: row j - first_col =
    L(j .. j + lda - 1, j), zero past the matrix."""
    import scipy.sparse as sps

    L = sps.csc_matrix(L)
    n = L.shape[0]
    ncols = n - first_col if ncols is None else ncols
    out = np.zeros((ncols, lda))
    sub = L[:, first_col:first_col + ncols].tocoo()
    r = sub.row - (sub.col + first_col)
    keep = (r >= 0) & (r < lda)
    out[sub.col[keep], r[keep]] = sub.data[keep]
    return out


def diagonal_block_mask(lda, n, first_col=0, ncols=None):
    """True on the entries of the band image that lie in a 64 x 64 diagonal block (not part of the factor's
    contract)."""
    ncols = n - first_col if ncols is None else ncols
    j = np.arange(first_col, first_col + ncols)[:, None]
    i = j + np.arange(lda)[None, :]
    return (i < (j // NB) * NB + NB) & (i < n)


def band_from_stencil(S, nodes, lda):
    """The stencil storage S[ncol, 4^ndim] as a band image (ncol, lda): row j = G(j .. j + lda - 1, j)."""
    nodes = [int(v) for v in nodes]
    ndim = len(nodes)
    ncol = int(np.prod(nodes))
    strides = [int(np.prod(nodes[:d])) for d in range(ndim)]
    j = np.arange(ncol)
    jd = [(j // strides[d]) % nodes[d] for d in range(ndim)]
    out = np.zeros((ncol, lda))
    for combo in np.ndindex(*([7] * ndim)):
        dd = [c - 3 for c in combo]
        off = sum(dd[d] * strides[d] for d in range(ndim))
        if off < 0 or off >= lda:
            continue
        ok = np.ones(ncol, dtype=bool)
        node = np.zeros(ncol, dtype=np.int64)
        sten = 0
        for d in range(ndim):
            idd = jd[d] + dd[d]
            ok &= (idd >= 0) & (idd < nodes[d])
            node += np.where(dd[d] < 0, idd, jd[d]) * strides[d]
            sten += abs(dd[d]) * 4 ** d
        out[j[ok], off] = S[node[ok], sten]
    return out


def _band_view(img, lda, bw, r0, r1, c0, c1):
    """Dense A[r0:r1, c0:c1] of a band image (row j = A(j .. j + lda - 1, j)), entries with i - j outside 0..bw zero."""
    if r1 <= r0 or c1 <= c0:
        return np.zeros((max(r1 - r0, 0), max(c1 - c0, 0)))
    flat = img.reshape(-1)
    v = np.lib.stride_tricks.as_strided(flat[r0 + c0 * (lda - 1):], shape=(r1 - r0, c1 - c0),
                                        strides=(8, 8 * (lda - 1)), writeable=False)
    off = np.arange(r0, r1)[:, None] - np.arange(c0, c1)[None, :]
    return np.where((off >= 0) & (off <= bw), v, 0.0)


# Constant of the replay bounds.  With u = 2^-53 and b the half bandwidth, in the device's arithmetic:
#   * A^(k) = M - sum_{earlier panels} L L^T has at most b + 1 terms per entry, so the device's A^(k) and the host's
#     A_hat differ by at most 2 gamma_{b+1} B, B = |M| + |L_prev||L_prev^T|;
#   * L21 = A21 X^T is a 64-term DMMA dot product per entry: gamma_64 |A21||X|^T, and |A_hat_ij| <= d_i d_j
#     (d_i^2 = A_hat_ii, A_hat positive semidefinite up to the above); forming A_hat21 X^T on the host adds as much again:
#     |L21 - A_hat21 X^T| <= (2 gamma_{b+1} + 2 gamma_64)(B + d d^T)|X|^T <= 2.1 (b + 64) u (B21 + d d^T)|X|^T;
#   * X is checked through X A_hat11 X^T - I.  The square-root-free Cholesky gives L11 L11^T = A11 + F with
#     |F| <= gamma_65 |L11||L11^T| <= gamma_65 d d^T (Cauchy-Schwarz on the rows of L11); the reciprocal (seed + one
#     cubic step) and d^-1/2 (seed + two Goldschmidt steps) add a few u to each pivot, inside gamma_65; the blocked
#     inversion leaves X L11 = I + E, |E| <= gamma_64 |X||L11| <= gamma_64 (|X| d) 1^T <= gamma_64 (|X| d)(|X| d)^T,
#     since X L11 = I makes every (|X| d)_i >= 1.  X A11 X^T - I = E + E^T + E E^T - X F X^T, plus the difference of
#     A11 and A_hat11 (2 gamma_{b+1} |X| B |X|^T):  <= (2 gamma_64 + gamma_65 + 2 gamma_{b+1}) |X|(B11 + d d^T)|X|^T.
# Both come to less than 3.1 (b + 64) u to first order; c = 4 leaves room for the second-order terms.
REPLAY_C = 4.0


def _ratio(err, tol):
    with np.errstate(divide="ignore", invalid="ignore"):
        r = np.where(err == 0, 0.0, err / tol)
    return float(r.max()) if r.size else 0.0


def replay_panels(Mimg, Limg, linv, bw, panels, drop=None):
    """Stepwise replay of the factor from the device's OWN earlier columns: for every panel k in `panels`,
        A_hat = M[., J_k] - L[., C] L[J_k, C]^T,   C = the columns before J_k,
    in float64, and the checks
        |L21 - A_hat21 X_k^T|      <= c (b + 64) u (B21 + d d^T) |X_k|^T
        |X_k A_hat11 X_k^T - I|    <= c (b + 64) u |X_k| (B11 + d d^T) |X_k|^T        (in long double)
    with X_k the stored block inverse, B = |M| + |L_prev||L_prev^T| over the same entries and d_i = sqrt(A_hat_ii) (the
    diagonal of the step-k Schur complement).  Every bound is local: a wrong entry shows at its panel, whatever
    cond(G).  Mimg, Limg: band images (ncol, lda) of G and of the device's factor (diagonal blocks unused); linv:
    (nblk, 64, 64).  drop = (p, row_lo, row_hi): leave panel p's contribution out of those rows of A_hat (the tests'
    sensitivity check).  Returns [(k, ratio L21, ratio X)]."""
    n, lda = Limg.shape
    u = 2.0 ** -53
    tau = REPLAY_C * (bw + NB) * u
    out = []
    for k in panels:
        j0 = k * NB
        nb = min(NB, n - j0)
        r0 = j0 + nb
        m = min(n - r0, bw)
        R1 = r0 + m
        c0 = max(0, j0 - bw)
        LR = _band_view(Limg, lda, bw, j0, R1, c0, j0)               # L[R, C], R = J then the rows below
        MR = _band_view(Mimg, lda, bw, j0, R1, j0, r0)
        LJ = LR[:nb]
        sub = LR @ LJ.T
        if drop is not None:
            p, lo, hi = drop
            pc0, pc1 = max(p * NB, c0) - c0, min(p * NB + NB, j0) - c0
            lo, hi = max(lo, j0) - j0, min(hi, R1) - j0
            if pc1 > pc0 and hi > lo:
                sub[lo:hi] -= LR[lo:hi, pc0:pc1] @ LJ[:, pc0:pc1].T
        Ah = MR - sub
        B = np.abs(MR) + np.abs(LR) @ np.abs(LJ).T
        # symmetric diagonal block: upper triangle from the lower one
        tri = np.tril(np.ones((nb, nb), dtype=bool), -1)
        A11 = np.where(tri.T, Ah[:nb].T, Ah[:nb])
        B11 = np.where(tri.T, B[:nb].T, B[:nb])
        diag = Mimg[j0:R1, 0] - np.einsum("ij,ij->i", LR, LR)
        d = np.sqrt(np.maximum(diag, 0.0))
        X = linv[k, :nb, :nb]
        Xa = np.abs(X)
        rl = 0.0
        if m > 0:
            L21 = _band_view(Limg, lda, lda - 1, r0, R1, j0, r0)
            want = Ah[nb:] @ X.T
            tol = tau * ((B[nb:] + np.outer(d[nb:], d[:nb])) @ Xa.T)
            rl = _ratio(np.abs(L21 - want), tol)
        Xl = X.astype(np.longdouble)
        res = Xl @ A11.astype(np.longdouble) @ Xl.T - np.eye(nb, dtype=np.longdouble)
        tol = tau * (Xa @ (B11 + np.outer(d[:nb], d[:nb])) @ Xa.T)
        rx = _ratio(np.abs(res).astype(np.float64), tol)
        out.append((k, rl, rx))
    return out


def _dropped(Mimg, Limg, bw, k, drop):
    """max |L[rows, C_p] L[J_k, C_p]^T|_ij / sqrt(M_ii M_jj): how much leaving panel p out of those rows of panel k's
    replay changes, relative to the scale of the entries (and so of the replay's bound)."""
    n, lda = Limg.shape
    p, lo, hi = drop
    j0, j1, hi = k * NB, min(n, k * NB + NB), min(hi, n)
    J = _band_view(Limg, lda, bw, j0, j1, p * NB, p * NB + NB)
    R = _band_view(Limg, lda, bw, lo, hi, p * NB, p * NB + NB)
    dm = np.sqrt(np.abs(Mimg[:, 0]))
    with np.errstate(divide="ignore", invalid="ignore"):
        rel = np.abs(R @ J.T) / np.outer(dm[lo:hi], dm[j0:j1])
    return float(np.nan_to_num(rel, posinf=0.0).max(initial=0.0))


def sensitivity_drops(Mimg, Limg, bw):
    """(panel k, drop) pairs for replay_panels: an earlier panel p's contribution left out of (a) a column-0 tile
    (ti, 0), ti >= 1, of update p, replayed at panel p + 1; (b) a rest tile (T - 1, tj), tj >= 1, of its last tile row,
    replayed at panel p + 1 + tj; (c) the diagonal block of panel p + 1.  For each kind, the tile whose left-out product
    is largest relative to sqrt(M_ii M_jj).  The factor of a banded system decays away from the couplings of M (on a
    341 x 6 grid the entries 64..192 below the diagonal are ~1e-19 of the others), so some tiles only ever receive
    products below rounding; a kind whose largest left-out product stays below 1000 x the replay's relative bound
    c (b + 64) u is left out of the result.  (a) and (b) need a window of more than one tile row (b > 64)."""
    least = 1e3 * REPLAY_C * (bw + NB) * 2.0 ** -53
    n = Limg.shape[0]
    nblk = (n + NB - 1) // NB
    cands = {"diagonal": [], "column-0 tile": [], "last-row rest tile": []}
    step = max(1, nblk // 16)                     # a spread of panels is enough to find a large one
    for p in range(0, max(0, nblk - 2), step):
        r0 = p * NB + NB
        m = min(n - r0, bw)
        T = (m + NB - 1) // NB
        cands["diagonal"].append((p + 1, (p, r0, r0 + NB)))
        for t in range(1, T):
            cands["column-0 tile"].append((p + 1, (p, r0 + NB * t, min(r0 + NB * t + NB, r0 + m))))
            if p + 1 + t < nblk:
                cands["last-row rest tile"].append((p + 1 + t, (p, r0 + NB * (T - 1), r0 + m)))
    out = {}
    for name, lst in cands.items():
        if lst:
            size, best = max(((_dropped(Mimg, Limg, bw, *c), c) for c in lst), key=lambda t: t[0])
            if size > least:
                out[name] = best
    return out


def inverse_lower_longdouble(L11):
    """L11^-1 of a lower-triangular block by forward substitution in long double, rounded to float64 once."""
    n = L11.shape[0]
    A = L11.astype(np.longdouble)
    X = np.zeros((n, n), dtype=np.longdouble)
    for i in range(n):
        rhs = -(A[i, :i] @ X[:i])
        rhs[i] += 1.0
        X[i] = rhs / A[i, i]
    return X.astype(np.float64)
