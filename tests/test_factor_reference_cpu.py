"""The host references of the band Cholesky factor (oracle/cpu_matched.py), without a GPU.

  * kron_exact_system: L L^T == M and numpy's Cholesky == (x) L_d bit for bit, the stencil storage expands to M (through
    tests/util.dense_from_stencil and through band_from_stencil), the block inverses times the diagonal blocks are I
    exactly, g == M c* exactly; 1-D to 4-D at every scale 2^s the GPU tests use.
  * replay_panels fed with LAPACK's band factor (dpbtrf through scipy) and correctly rounded block inverses: the worst
    ratio stays <= 1 on assembled spline systems up to cond > 1e12, and rises above 100 when one earlier panel's
    contribution is left out of a column-0 tile, a rest tile of the last tile row, or a diagonal block.
"""
import numpy as np
import pytest
import scipy.linalg as sl

from oracle import cpu_matched as cm
from splpak_b200.distributed import partial_layout
from util import dense_from_stencil, make_problem

SCALES = (-900, -600, 0, 600, 900)


@pytest.mark.parametrize("ndim,nodes", [(1, [65]), (1, [200]), (2, [7, 5]), (2, [21, 9]), (3, [7, 5, 6]),
                                        (3, [4, 4, 4]), (4, [4, 4, 4, 4])])
@pytest.mark.parametrize("scale", SCALES)
def test_kron_exact_system(ndim, nodes, scale):
    sy = cm.kron_exact_system(ndim, nodes, scale)
    n, lda, bw = sy["ncol"], sy["lda"], sy["bw"]
    L, M = sy["L"].toarray(), sy["M"].toarray()
    assert np.array_equal(L @ L.T, M)
    assert np.array_equal(np.linalg.cholesky(M), L)
    assert np.array_equal(M @ sy["c"], sy["g"]) and np.array_equal(M @ sy["delta"], sy["r"])
    off, total = partial_layout(ndim, nodes)
    assert sy["part"].size == total
    S = sy["part"][off["S"][0]:off["S"][1]].reshape(n, -1)
    assert np.array_equal(dense_from_stencil(S, nodes), M)
    assert np.array_equal(sy["part"][off["g"][0]:off["g"][1]], sy["g"])
    assert sy["part"][off["nrows"][0]] >= n
    assert np.array_equal(cm.band_from_stencil(S, nodes, lda), cm.band_image(np.tril(M), lda))
    X = sy["linv"]
    assert X.shape == ((n + 63) // 64, 64, 64)
    for kb in range(X.shape[0]):
        j0, j1 = 64 * kb, min(n, 64 * kb + 64)
        assert np.array_equal(X[kb, :j1 - j0, :j1 - j0] @ L[j0:j1, j0:j1], np.eye(j1 - j0))
    # neighbouring pivots differ, so a route that used the wrong pivot's reciprocal cannot pass
    assert len(np.unique(np.abs(np.diagonal(L)))) > 1
    # the band image: L on and below the diagonal, zero past row n and past the half bandwidth
    img = cm.band_image(sy["L"], lda)
    j = np.arange(n)[:, None]
    r = np.arange(lda)[None, :]
    assert not img[(j + r >= n) | (r > bw)].any()
    assert np.array_equal(img[:, 0], np.diagonal(L))


def test_kron_exact_system_zero_pivot():
    sy = cm.kron_exact_system(2, [341, 6], 0, zero=(1, 3))
    M = sy["M"].tocsc()
    first = int(np.flatnonzero(M.diagonal() == 0)[0])
    assert first == 1023 and M[:, first].nnz == 0
    assert "L" not in sy


def _band(M, bw):
    n = M.shape[0]
    ab = np.zeros((bw + 1, n))
    for k in range(bw + 1):
        ab[k, :n - k] = np.diagonal(M, -k)
    return ab


def _lapack_factor(M, bw):
    """LAPACK's band Cholesky as a band image, with the block inverses of its panels correctly rounded."""
    n = M.shape[0]
    cb = sl.cholesky_banded(_band(M, bw), lower=True)
    lda = cm.band_lda(bw)
    img = np.zeros((n, lda))
    img[:, :bw + 1] = cb.T
    nblk = (n + 63) // 64
    X = np.tile(np.eye(64), (nblk, 1, 1))
    for kb in range(nblk):
        j0, j1 = 64 * kb, min(n, 64 * kb + 64)
        L11 = cm._band_view(img, lda, bw, j0, j1, j0, j1)
        X[kb, :j1 - j0, :j1 - j0] = cm.inverse_lower_longdouble(L11)
    return img, X


CASES = {
    # name: (ndim, nodes, points, decades of weight spread; < 0: weight 10^spread on the half x_1 < 0.5)
    "1-D b = 3": (1, [150], 600, 0),
    "2-D 21 x 9, b = 66": (2, [21, 9], 4000, 0),
    "2-D 30 x 12, b = 93": (2, [30, 12], 20000, 5),
    "2-D 42 x 7, b = 129": (2, [42, 7], 6000, 3),
    "3-D 6 x 6 x 8, b = 129": (3, [6, 6, 8], 8000, 6),
    "2-D 24 x 10, cond > 1e12": (2, [24, 10], 6000, -7),
    # fill 64..192 below the diagonal is ~1e-19 of the entries: only column-0 tiles near the band edge see products
    "2-D 341 x 6, b = 1026": (2, [341, 6], 60000, 0),
}


@pytest.mark.parametrize("name", list(CASES))
def test_replay_of_lapack_factor(name):
    ndim, nodes, npts, spread = CASES[name]
    x, y, _, xmin, xmax = make_problem(ndim, nodes, npts, seed=3)
    if spread >= 0:
        w = 10.0 ** (-spread * np.random.default_rng(4).random(len(y)))
    else:
        w = np.where(x[:, 0] < 0.5, 10.0 ** spread, 1.0)
    S, _, _ = cm.assemble_stencil(ndim, x, y, w, xmin, xmax, nodes)
    M = dense_from_stencil(S, nodes)
    n, bw = M.shape[0], cm.half_bandwidth(ndim, nodes)
    cond = np.linalg.cond(M)
    if "cond" in name:
        assert cond > 1e12
    lda = cm.band_lda(bw)
    Mimg = cm.band_from_stencil(S, nodes, lda)
    Limg, X = _lapack_factor(M, bw)
    res = cm.replay_panels(Mimg, Limg, X, bw, range(X.shape[0]))
    worst = max(max(r[1], r[2]) for r in res)
    print(f"\n{name}: cond {cond:.1e}, worst replay ratio {worst:.2e}", end="")
    assert worst <= 1.0
    drops = cm.sensitivity_drops(Mimg, Limg, bw)
    assert len(drops) == (3 if bw > 64 else 1)
    for what, (k, drop) in drops.items():
        (_, rl, rx), = cm.replay_panels(Mimg, Limg, X, bw, [k], drop=drop)
        print(f"; {what} left out: {max(rl, rx):.1e}", end="")
        assert max(rl, rx) >= 100.0, what
