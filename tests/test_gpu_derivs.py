"""Derivative sets (splpak_b200_eval_derivs): every partial derivative up to total order 1 or 2 of each query in one
pass.  Component k must be bit-identical to splpak_b200_eval with the nderiv that component names."""
import ctypes as C

import numpy as np
import pytest

import splpak_b200 as sp
from test_gpu_eval import CASES


@pytest.fixture(params=["default", "exact"], autouse=True)
def basis_mode(request, monkeypatch):
    """Default dispatch (uniform phantom-node form of the basis for large batches whose extended table fits in shared
    memory) and SPLPAK_B200_BASIS=exact (bascmp's node-by-node formulas everywhere)."""
    if request.param == "exact":
        monkeypatch.setenv("SPLPAK_B200_BASIS", "exact")
    else:
        monkeypatch.delenv("SPLPAK_B200_BASIS", raising=False)
    return request.param


def _components(ndim, order):
    """nderiv of every output column, in the documented order."""
    comps = [[0] * ndim]
    for d in range(ndim):
        comps.append([int(e == d) for e in range(ndim)])
    if order == 2:
        for i in range(ndim):
            for j in range(i, ndim):
                nd = [0] * ndim
                nd[i] += 1
                nd[j] += 1
                comps.append(nd)
    return comps


def _queries(rng, ndim, nq, mn, mx):
    """Inside and outside the grid, exact node / boundary hits, and NaN coordinates."""
    q = mn + (rng.random((nq, ndim)) * 1.5 - 0.25) * (mx - mn)
    q[0] = mn
    q[1] = mx
    q[2] = mn + (mx - mn) * 0.5
    q[3, 0] = np.nan
    q[4] = np.nan
    return q


def _per_component(ndim, q, coef, mn, mx, nodes, order, real32=False):
    cols = []
    for nd in _components(ndim, order):
        v, ierr = sp.eval_batch(ndim, q, coef, mn, mx, nodes, nderiv=nd, real32=real32)
        assert ierr == 0
        cols.append(v)
    return np.stack(cols, axis=1)


def _tol(coef, ndim, oracle, q, mn, mx, nodes):
    """Reordering roundoff of the 4^ndim-term sum, per query (as for the single-component path): 50 eps sum |c Phi|,
    plus 4 eps sum(nodes) for the uniform form, which does not repeat the reference's rounding of the node positions."""
    eps = np.finfo(float).eps
    floor = 64 * eps * np.abs(coef).max() * 6.0 ** ndim
    bound, _ = oracle.evaluate_batch(ndim, q, np.abs(coef), mn, mx, nodes)
    return np.maximum(floor, (128 + 4 * int(np.sum(nodes))) * eps * np.abs(bound))


def _grid_problem(seed, ndim, nodes):
    rng = np.random.default_rng(seed)
    coef = rng.standard_normal(int(np.prod(nodes)))
    mn = -rng.random(ndim)
    mx = 1.0 + rng.random(ndim)
    return rng, coef, mn, mx


@pytest.mark.gpu
@pytest.mark.parametrize("order", [1, 2])
@pytest.mark.parametrize("ndim,nodes", CASES)
def test_components_match_eval_batch_and_oracle(oracle, ndim, nodes, order):
    rng, coef, mn, mx = _grid_problem(31 * ndim + nodes[0], ndim, nodes)
    q = _queries(rng, ndim, 4000, mn, mx)
    got, ierr = sp.eval_derivs(ndim, q, coef, mn, mx, nodes, order=order)
    assert ierr == 0 and got.shape == (4000, len(_components(ndim, order))) and got.dtype == np.float64
    want = _per_component(ndim, q, coef, mn, mx, nodes, order)
    for k, nd in enumerate(_components(ndim, order)):
        assert np.array_equal(got[:, k], want[:, k], equal_nan=True), (nd, np.nanmax(np.abs(got[:, k] - want[:, k])))
    # against the reference's scalar splde loop (finite queries), with the tolerance of test_splde_all_derivative_orders
    fin = np.isfinite(q).all(axis=1)
    tol = _tol(coef, ndim, oracle, q[fin], mn, mx, nodes)
    dxin = (np.array(nodes) - 1) / (mx - mn)
    for k, nd in enumerate(_components(ndim, order)):
        ref, ie = oracle.evaluate_batch(ndim, q[fin], coef, mn, mx, nodes, nderiv=nd)
        assert ie == 0
        scale = np.prod((3.0 * dxin) ** np.array(nd))
        assert (np.abs(got[fin, k] - ref) <= tol * scale).all(), (nd, np.abs(got[fin, k] - ref).max())


def _ordered(rng, kind, ndim, nq, mn, mx):
    """random: scattered; raster: the points of a tensor grid, dimension 1 fastest (coherent runs); mixed: both halves."""
    if kind == "random":
        return mn + (rng.random((nq, ndim)) * 1.2 - 0.1) * (mx - mn)
    n1 = int(np.ceil(nq ** (1.0 / ndim)))
    axes = [np.linspace(mn[d] - 0.05, mx[d] + 0.05, n1) for d in range(ndim)]
    mesh = np.meshgrid(*axes, indexing="ij")
    raster = np.stack([m.transpose(*reversed(range(ndim))).ravel() for m in mesh], axis=1)[:nq]
    if kind == "raster":
        return np.ascontiguousarray(raster)
    half = nq // 2
    return np.concatenate([raster[:half], _ordered(rng, "random", ndim, nq - half, mn, mx)])


@pytest.mark.gpu
@pytest.mark.parametrize("order", [1, 2])
@pytest.mark.parametrize("ndim,nodes", [(2, [64, 64]), (3, [24, 24, 24]), (4, [12, 12, 12, 12])])
def test_large_batches_every_kernel_route(monkeypatch, ndim, nodes, order):
    """>= 2^18 queries: order probe + regrouping / plain kernel (default), and each kernel forced."""
    rng, coef, mn, mx = _grid_problem(7 * ndim, ndim, nodes)
    nq = (1 << 18) + 4321
    for kind in ("random", "raster", "mixed"):
        q = _ordered(rng, kind, ndim, nq, mn, mx)
        want = _per_component(ndim, q, coef, mn, mx, nodes, order)
        outs = []
        for mode in (None, "plain", "regroup"):
            if mode is None:
                monkeypatch.delenv("SPLPAK_B200_EVAL", raising=False)
            else:
                monkeypatch.setenv("SPLPAK_B200_EVAL", mode)
            got, ierr = sp.eval_derivs(ndim, q, coef, mn, mx, nodes, order=order)
            assert ierr == 0
            outs.append(got)
        monkeypatch.delenv("SPLPAK_B200_EVAL", raising=False)
        for mode, got in zip(("default", "plain", "regroup"), outs):
            assert np.array_equal(got, want), (kind, mode, np.abs(got - want).max())


@pytest.mark.gpu
def test_device_variant_on_a_stream():
    import torch

    rng, coef, mn, mx = _grid_problem(3, 3, [9, 8, 7])
    nodes = [9, 8, 7]
    q = _queries(rng, 3, 50000, mn, mx)
    want = _per_component(3, q, coef, mn, mx, nodes, 2)
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        d_x = torch.tensor(q, device="cuda")
        d_c = torch.tensor(coef, device="cuda")
        d_out = torch.full((len(q), want.shape[1]), -7.0, dtype=torch.float64, device="cuda")
    assert sp.eval_derivs_device(3, d_x, 3, len(q), d_c, mn, mx, nodes, d_out, order=2, stream=s) == 0
    s.synchronize()
    assert np.array_equal(d_out.cpu().numpy(), want)


@pytest.mark.gpu
def test_strided_x_odd_ncol_large_table_and_single_query():
    # l1x > ndim and odd ncol (5 x 7)
    rng = np.random.default_rng(6)
    nodes = [5, 7]
    coef = rng.standard_normal(35)
    q = np.full((600, 4), 99.0)
    q[:, :2] = rng.random((600, 2)) * 1.2 - 0.1
    got, ierr = sp.eval_derivs(2, q, coef, [0, 0], [1, 1], nodes, order=2)
    assert ierr == 0 and np.array_equal(got, _per_component(2, q, coef, [0, 0], [1, 1], nodes, 2))
    # a table larger than shared memory (2-D 200 x 200 = 320 KB): coefficients gathered from L2
    nodes = [200, 200]
    coef = rng.standard_normal(40000)
    q = rng.random((3000, 2)) * 1.2 - 0.1
    got, ierr = sp.eval_derivs(2, q, coef, [0, 0], [1, 1], nodes, order=2)
    assert ierr == 0 and np.array_equal(got, _per_component(2, q, coef, [0, 0], [1, 1], nodes, 2))
    # one query: the latency path
    nodes = [6, 5, 7]
    coef = rng.standard_normal(210)
    q = np.array([[0.3, 0.71, 0.05]])
    got, ierr = sp.eval_derivs(3, q, coef, [0, 0, 0], [1, 1, 1], nodes, order=2)
    assert ierr == 0 and got.shape == (1, 10)
    assert np.array_equal(got, _per_component(3, q, coef, [0, 0, 0], [1, 1, 1], nodes, 2))


@pytest.mark.gpu
def test_chunked_host_path(basis_mode):
    """More queries than one staging chunk (2^22): the double-buffered pipeline with ncomp outputs per query."""
    if basis_mode == "exact":
        pytest.skip("the staging does not depend on the basis form")
    rng = np.random.default_rng(9)
    nodes = [24, 24, 24]
    coef = rng.standard_normal(24 ** 3)
    nq = (1 << 22) * 2 + 12345
    q = rng.random((nq, 3))
    got, ierr = sp.eval_derivs(3, q, coef, [0, 0, 0], [1, 1, 1], nodes, order=1)
    assert ierr == 0 and got.shape == (nq, 4)
    assert np.array_equal(got, _per_component(3, q, coef, [0, 0, 0], [1, 1, 1], nodes, 1))


@pytest.mark.gpu
@pytest.mark.parametrize("ndim,nodes", [(2, [8, 9]), (3, [24, 24, 24]), (4, [5, 4, 6, 5])])
def test_real32_library(monkeypatch, ndim, nodes):
    """Float I/O, float64 arithmetic (as splde of the REAL32 library).  The value column equals eval_batch of the
    float64-internal path (SPLPAK_B200_R32=f64); splfe proper runs in float."""
    rng = np.random.default_rng(40 + ndim)
    coef = rng.standard_normal(int(np.prod(nodes))).astype(np.float32)
    mn, mx = np.zeros(ndim), np.ones(ndim)
    q = _queries(rng, ndim, 3000, mn, mx).astype(np.float32)
    got, ierr = sp.eval_derivs(ndim, q, coef, mn, mx, nodes, order=2, real32=True)
    assert ierr == 0 and got.dtype == np.float32
    comps = _components(ndim, 2)
    for k, nd in enumerate(comps[1:], start=1):
        v, ierr = sp.eval_batch(ndim, q, coef, mn, mx, nodes, nderiv=nd, real32=True)
        assert ierr == 0 and np.array_equal(got[:, k], v), nd
    monkeypatch.setenv("SPLPAK_B200_R32", "f64")
    v, ierr = sp.eval_batch(ndim, q, coef, mn, mx, nodes, real32=True)
    assert ierr == 0 and np.array_equal(got[:, 0], v)


@pytest.mark.gpu
def test_one_fused_pass():
    """One derivative-set call launches what one single-component call launches."""
    rng, coef, mn, mx = _grid_problem(12, 3, [24, 24, 24])
    q = rng.random((1 << 19, 3))
    for order in (1, 2):
        sp.eval_derivs(3, q, coef, mn, mx, [24] * 3, order=order)
        sp.eval_batch(3, q, coef, mn, mx, [24] * 3)
        n0 = sp.total_launches()
        sp.eval_derivs(3, q, coef, mn, mx, [24] * 3, order=order)
        n1 = sp.total_launches()
        sp.eval_batch(3, q, coef, mn, mx, [24] * 3, nderiv=[1, 0, 0])
        n2 = sp.total_launches()
        assert n1 - n0 == n2 - n1 and n1 > n0


@pytest.mark.parametrize("real32", [False, True])
def test_argument_errors(real32):
    """No device needed: 101..103 in the reference's order, then 104 for an order other than 1 or 2, before anything
    is written."""
    lib = sp.load(real32)
    dt = np.float32 if real32 else np.float64
    rp, ip = C.POINTER(lib._real), C.POINTER(C.c_int)

    def call(ndim, nodes, xmin, xmax, order):
        x = np.full((3, max(ndim, 1)), 0.5, dtype=dt)
        coef = np.ones(1000, dtype=dt)
        out = np.full(64, np.nan, dtype=dt)
        mn = np.asarray(xmin, dtype=dt)
        mx = np.asarray(xmax, dtype=dt)
        no = np.asarray(nodes, dtype=np.int32)
        ierr = C.c_int(-1)
        rc = lib.splpak_b200_eval_derivs(ndim, x.ctypes.data, x.shape[1], 3, order, coef.ctypes.data,
                                         mn.ctypes.data_as(rp), mx.ctypes.data_as(rp), no.ctypes.data_as(ip),
                                         out.ctypes.data, C.byref(ierr))
        assert rc == ierr.value
        assert np.isnan(out).all()
        return rc

    for order in (0, 3, -1):
        assert call(2, [5, 6], [0, 0], [1, 1], order) == 104
    assert call(0, [5], [0], [1], 3) == 101
    assert call(5, [5] * 5, [0] * 5, [1] * 5, 1) == 101
    assert call(2, [5, 3], [0, 0], [1, 1], 3) == 102
    assert call(2, [5, 6], [0, 1], [1, 1], 0) == 103
    assert call(2, [3, 6], [0, 1], [1, 1], 1) == 102
    assert sp.eval_derivs(1, [[0.5]], np.ones(10), [0.0], [1.0], [10], order=3, real32=real32)[1] == 104
    assert sp.derivs_ncomp(3, 1) == 4 and sp.derivs_ncomp(3, 2) == 10 and sp.derivs_ncomp(4, 2) == 15

