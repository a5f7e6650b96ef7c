"""The host reference of the assembled normal equations (oracle/cpu_matched.assemble_stencil, nearest_node_histogram,
point_contribution) against the oracle's least-squares rows: S against A^T A, g against A^T r, cnt against the scalar
restatement of the histogram loop, at the positions where binning goes wrong -- points on nodes, on faces and at
xmax, at half-node positions and one ulp either side, just below xmin (the truncation toward zero) and far outside --
with zero weights and negative weights after the first.  tests/test_gpu_assembly_routes.py compares the GPU with this
reference at sizes the oracle cannot run."""
import numpy as np
import pytest

from oracle.cpu_matched import assemble_stencil, nearest_node_histogram, point_contribution
from oracle.numpy_model import SplpakModel
from util import dense_from_stencil, stencil_scale, worst_ratio

TAU = 1e-13


def edge_points(ndim, nodes, xmin, xmax, n, rng):
    """n random points, then rows of each kind of edge position in every coordinate."""
    nodes = np.asarray(nodes)
    dx = (xmax - xmin) / (nodes - 1)
    u = rng.random((n, ndim))
    x = xmin + u * (xmax - xmin) * 1.2 - 0.1 * (xmax - xmin)
    k = rng.integers(0, nodes, size=(n, ndim))
    on_node = xmin + k * dx
    half = xmin + (np.minimum(k, nodes - 2) + 0.5) * dx
    kinds = [
        on_node,
        np.where(rng.random((n, ndim)) < 0.5, xmin, xmax),                   # box faces and corners
        np.broadcast_to(xmax, (n, ndim)),                                    # exactly xmax
        half, np.nextafter(half, -np.inf), np.nextafter(half, np.inf),
        np.nextafter(on_node, -np.inf), np.nextafter(on_node, np.inf),
        xmin - rng.random((n, ndim)) * dx,                                   # (xmin - dx, xmin]: int() truncates to 0
        np.where(rng.random((n, ndim)) < 0.5, xmin - 7.3 * dx, xmax + 11.9 * dx),
    ]
    for kind in kinds:
        mix = rng.random((n, ndim)) < 0.6                                    # mix edge and random coordinates
        x = np.concatenate([x, np.where(mix, kind, x[:n])])
    return x


CASES = [
    # ndim, nodes, xmin, xmax
    (1, [4], [0.0], [1.0]),
    (1, [13], [-2.0], [3.5]),
    (2, [4, 6], [0.0, -1.0], [1.0, 2.0]),
    (2, [7, 5], [0.1, 0.0], [0.7, 3.0]),
    (3, [4, 5, 6], [0.0, 0.0, 0.0], [1.0, 1.0, 1.0]),
    (3, [6, 4, 5], [-1.0, 0.5, 2.0], [1.0, 0.9, 7.0]),
    (4, [4, 5, 4, 4], [0.0] * 4, [1.0] * 4),
    (4, [5, 4, 4, 6], [0.0, -0.3, 1.0, 0.0], [1.0, 0.3, 2.0, 2.0]),
]


def _data(ndim, nodes, xmin, xmax, seed, weights):
    rng = np.random.default_rng(seed)
    x = edge_points(ndim, nodes, np.asarray(xmin), np.asarray(xmax), 60, rng)
    y = np.sin(3.0 * x).sum(axis=1) + 0.1 * rng.standard_normal(len(x))
    if weights == "unweighted":
        return x, y, None
    w = rng.random(len(x)) + 0.5
    w[rng.random(len(x)) < 0.1] = 0.0
    if weights == "negative":
        w[1:][rng.random(len(x) - 1) < 0.3] *= -1.0                        # the first weight decides: weighted
    w[0] = 0.75
    return x, y, w


@pytest.mark.parametrize("weights", ["unweighted", "weighted", "negative"])
@pytest.mark.parametrize("ndim,nodes,xmin,xmax", CASES)
def test_reference_matches_oracle_rows(oracle, ndim, nodes, xmin, xmax, weights):
    x, y, w = _data(ndim, nodes, xmin, xmax, 100 * ndim + nodes[0], weights)
    A, r = oracle.rows(ndim, x, y, w, xmin, xmax, nodes, 0.0)
    Gref, gref = A.T @ A, A.T @ r
    S, g, gabs = assemble_stencil(ndim, x, y, w, xmin, xmax, nodes, chunk_elems=1 << 12)   # several chunks
    G = dense_from_stencil(S, nodes)
    d = np.diag(Gref)
    assert worst_ratio(G, Gref, TAU * np.sqrt(np.outer(d, d))) <= 1.0
    gtol = TAU * (np.abs(A).T @ np.abs(r))
    assert worst_ratio(g, gref, gtol) <= 1.0
    np.testing.assert_allclose(gabs, np.abs(A).T @ np.abs(r), rtol=1e-13, atol=0)
    # stencil entries whose partner node is off the grid stay zero
    assert not S[stencil_scale(S[:, 0], nodes) == 0].any()
    cnt, totlwt, nrows = nearest_node_histogram(ndim, x, w, xmin, xmax, nodes)
    work, tot = SplpakModel().histogram(ndim, x, [-1.0] if w is None else w, xmin, xmax, nodes)
    assert nrows == A.shape[0]
    if w is None:
        assert np.array_equal(cnt, work) and totlwt == tot == len(x)
    else:
        cabs, _, _ = nearest_node_histogram(ndim, x, np.abs(w), xmin, xmax, nodes)
        assert worst_ratio(cnt, work, TAU * cabs) <= 1.0
        assert abs(totlwt - tot) <= TAU * np.abs(w).sum()
        # the same points land on the same nodes (no cancellation between signed weights can hide a move)
        wabs, _ = SplpakModel().histogram(ndim, x, np.abs(w), xmin, xmax, nodes)
        assert worst_ratio(cabs, np.asarray(wabs), TAU * cabs) <= 1.0


@pytest.mark.parametrize("ndim,nodes,xmin,xmax", CASES[::2])
def test_point_contribution_is_the_difference(ndim, nodes, xmin, xmax):
    """Removing one point from the data changes the reference by exactly point_contribution (up to rounding)."""
    x, y, w = _data(ndim, nodes, xmin, xmax, 7 + ndim, "negative")
    S, g, gabs = assemble_stencil(ndim, x, y, w, xmin, xmax, nodes)
    cnt, _, _ = nearest_node_histogram(ndim, x, w, xmin, xmax, nodes)
    scale = stencil_scale(S[:, 0], nodes)
    for p in (3, len(x) - 1, len(x) // 2 + 1):                       # an interior, a far-outside, an edge point
        keep = np.arange(len(x)) != p
        S1, g1, _ = assemble_stencil(ndim, x[keep], y[keep], w[keep], xmin, xmax, nodes)
        cnt1, _, _ = nearest_node_histogram(ndim, x[keep], w[keep], xmin, xmax, nodes)
        (si, sv), (gi, gv), (node, wp) = point_contribution(ndim, x[p], y[p], w[p], xmin, xmax, nodes)
        Sd = S.reshape(-1).copy()
        Sd[si] -= sv
        assert worst_ratio(Sd, S1.reshape(-1), 1e-13 * scale.reshape(-1)) <= 1.0
        gd = g.copy()
        np.add.at(gd, gi, -gv)
        assert worst_ratio(gd, g1, 1e-13 * gabs) <= 1.0
        cd = cnt.copy()
        cd[node] -= wp
        np.testing.assert_allclose(cd, cnt1, rtol=0, atol=1e-13 * np.abs(w).sum())
