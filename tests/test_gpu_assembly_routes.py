"""The assembled normal equations, entry by entry, against the float64 host reference (oracle/cpu_matched.py) on every
assembly route, at the sizes where the routes are chosen:

  * two-level partition (spl_part1/2_kernel) against the per-point scatter (spl_perm_kernel): 3-D / 4-D cell path,
    chunks of >= 2^21 points, 2048 <= cells <= 48 * 2048; bucket shifts 6, 9 and 11 (clamped span);
  * work items that split a cell (> 4096 points) or a window (> CH points), cells of more than 100 segments;
  * classify histograms in shared memory with the node counts, in shared memory alone, and in global memory;
  * the deterministic segment sort with 1, 2, 3 and 4 radix passes; host staging across 2^22-point chunks;
  * scratch regrowth inside one handle; strided x; the rhs_only re-assembly of a refinement step.

Tolerances: |S - S_ref|_ij <= TAU sqrt(G_ii G_jj) (Cauchy-Schwarz bounds the sum of |terms| of any entry by that, so
it bounds the rounding error of any summation order), |g - g_ref|_i <= TAU (|B|^T W^2 |y|)_i, the node histogram
exact for unit weights and within count * wmax * 2^-34 otherwise (every weight is rounded to within half a quantum
wmax 2^-bits, bits >= 34 for chunks of <= 2^27 points), the row count exact.  Every case also checks that the
comparison fails by at least 100x when one point -- of the busiest cell, and of an exterior cell -- is taken out of
the reference, so a lost, doubled or misplaced point cannot pass.

The two-level route adds exactly one counted launch per chunk, so launch_count() minus that of the same data under
SPLPAK_B200_BINNING=atomic is the number of chunks that took it.  Run with -s to see the error-to-tolerance ratios.
"""
import time

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")
import splpak_b200 as sp  # noqa: E402
from oracle.cpu_matched import assemble_stencil, nearest_node_histogram, point_contribution  # noqa: E402
from splpak_b200 import synth  # noqa: E402
from util import stencil_scale, worst_ratio  # noqa: E402

TAU = 1e-12
CNT_QUANTUM = 2.0 ** -34
ENV_KEYS = ("SPLPAK_B200_ASSEMBLY", "SPLPAK_B200_DETERMINISTIC", "SPLPAK_B200_CURSOR_STRIDE", "SPLPAK_B200_BINNING",
            "SPLPAK_B200_GLOBAL_HIST")
ATOMIC = {"SPLPAK_B200_BINNING": "atomic"}
DET = {"SPLPAK_B200_DETERMINISTIC": "1"}
SECONDS = {"reference": 0.0, "gpu": 0.0}
REPORT = []


def _uniform(ndim, nodes, n, seed, weighted=True, on_node=0.01, zero=0.01):
    """x uniform on [-0.1, 1.1]^ndim around the box [0, 1]^ndim (exterior cells on every side), a fraction of the
    coordinates exactly on nodes, a fraction of zero weights."""
    rng = np.random.default_rng(seed)
    x = rng.random((n, ndim)) * 1.2 - 0.1
    for d in range(ndim):
        snap = rng.random(n) < on_node
        k = rng.integers(0, nodes[d], snap.sum())
        x[snap, d] = k * (1.0 / (nodes[d] - 1))
    y = np.sin(3.0 * x).sum(axis=1) + 0.05 * rng.standard_normal(n)
    w = None
    if weighted:
        w = 0.5 + rng.random(n)
        w[rng.random(n) < zero] = 0.0
        w[0] = 1.0
    return dict(ndim=ndim, nodes=list(nodes), x=x, y=y, w=w, xmin=[0.0] * ndim, xmax=[1.0] * ndim)


def _skewed(seed):
    """3-D 12^3, 2^22 + 2^21 + 5 points (two host chunks), 40 % of them in 3 cells: more than 200 work items in each."""
    d = _uniform(3, [12] * 3, (1 << 22) + (1 << 21) + 5, seed)
    rng = np.random.default_rng(seed + 1)
    n, dx = len(d["y"]), 1.0 / 11
    cells = np.array([[1, 1, 1], [6, 6, 6], [0, 5, 12]])           # cell j covers [(j - 1) dx, j dx)
    pick = np.flatnonzero(rng.random(n) < 0.4)
    c = cells[rng.integers(0, 3, len(pick))]
    d["x"][pick] = (c - 1 + rng.random((len(pick), 3))) * dx
    d["y"] = np.sin(3.0 * d["x"]).sum(axis=1) + 0.05 * rng.standard_normal(n)
    return d


def _cfg3():
    x, y, w = synth.points_numpy(3, 1 << 22)
    return dict(ndim=3, nodes=[24] * 3, x=x, y=y, w=w, xmin=[0.0] * 3, xmax=[1.0] * 3)


DATA = {
    "3d12": lambda: _uniform(3, [12] * 3, (1 << 21) + 37, 1),
    "3d11": lambda: _uniform(3, [11] * 3, (1 << 21) + 37, 2),
    "3d24_cfg3": _cfg3,
    "3d45": lambda: _uniform(3, [45] * 3, 1 << 21, 4),
    "3d12_skew": lambda: _skewed(5),
    "4d6": lambda: _uniform(4, [6] * 4, (1 << 21) + 11, 6),
    "4d16": lambda: _uniform(4, [16] * 4, 1 << 21, 7),
    "4d17": lambda: _uniform(4, [17] * 4, 1 << 21, 8),
    "4d5": lambda: _uniform(4, [5] * 4, 1 << 21, 9),
    "2d8": lambda: _uniform(2, [8, 8], 1 << 21, 10),
    "2d64": lambda: _uniform(2, [64, 64], (1 << 22) + (1 << 21) + 5, 11, weighted=False),
    "1d50_big": lambda: _uniform(1, [50], (1 << 24) + 1, 12, weighted=False),
    "1d50_200": lambda: _uniform(1, [50], 200, 13),
    "1d50_60000": lambda: _uniform(1, [50], 60000, 14),
    "1d50_4M": lambda: _uniform(1, [50], 1 << 22, 15),
    "3d12_grow": lambda: _uniform(3, [12] * 3, 1_000_000 + 3_000_000 + 1000, 16),
}
_REF = {}


def _cell_keys(d):
    """Cell of every point as the moment path bins it: nodes + 1 cells per dimension, 0 and nodes the exterior."""
    key = np.zeros(len(d["y"]), dtype=np.int64)
    ext = np.zeros(len(d["y"]), dtype=bool)
    for k in reversed(range(d["ndim"])):
        nod = d["nodes"][k]
        t = (1.0 / ((d["xmax"][k] - d["xmin"][k]) / (nod - 1))) * (d["x"][:, k] - d["xmin"][k])
        c = np.where(t < 0.0, 0, np.minimum(np.trunc(np.clip(t, 0.0, nod)), nod - 1) + 1).astype(np.int64)
        key = key * (nod + 1) + c
        ext |= (c == 0) | (c == nod)
    return key, ext


def _probes(d):
    """A nonzero-weight point of the busiest cell and one of an exterior cell (of the emptiest cell if none)."""
    key, ext = _cell_keys(d)
    live = np.ones(len(key), dtype=bool) if d["w"] is None else d["w"] != 0
    counts = np.bincount(key[live])
    busy = int(np.flatnonzero(live & (key == counts.argmax()))[0])
    outside = np.flatnonzero(live & ext)
    if len(outside):
        return [busy, int(outside[len(outside) // 2])]
    sparse = np.where(counts > 0, counts, counts.max() + 1).argmin()
    return [busy, int(np.flatnonzero(live & (key == sparse))[0])]


def reference(name):
    """The data set and its host reference, computed once per module."""
    if name not in _REF:
        d = DATA[name]()
        t0 = time.perf_counter()
        args = (d["ndim"], d["x"])
        d["S"], d["g"], d["gabs"] = assemble_stencil(*args, d["y"], d["w"], d["xmin"], d["xmax"], d["nodes"])
        d["cnt"], d["totlwt"], d["nrows"] = nearest_node_histogram(*args, d["w"], d["xmin"], d["xmax"], d["nodes"])
        if d["w"] is None:
            d["cnt_tol"], d["tot_tol"] = np.zeros_like(d["cnt"]), 0.0
        else:
            live = (d["w"] != 0).astype(np.float64)
            count = nearest_node_histogram(*args, live, d["xmin"], d["xmax"], d["nodes"])[0]
            wmax = float(np.abs(d["w"]).max())
            d["cnt_tol"], d["tot_tol"] = count * wmax * CNT_QUANTUM, d["nrows"] * wmax * CNT_QUANTUM
        d["scale"] = stencil_scale(d["S"][:, 0], d["nodes"])
        d["probes"] = _probes(d)
        SECONDS["reference"] += time.perf_counter() - t0
        _REF[name] = d
    return _REF[name]


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    print("\nassembly routes: worst error / tolerance, and the smallest ratio with one point taken out of the reference")
    for line in REPORT:
        print("  " + line)
    print(f"host reference {SECONDS['reference']:.1f} s, GPU runs {SECONDS['gpu']:.1f} s")
    _REF.clear()


def _set_env(monkeypatch, env):
    for k in ENV_KEYS:
        monkeypatch.delenv(k, raising=False)
    for k, v in env.items():
        monkeypatch.setenv(k, v)


def _run(monkeypatch, d, env, xtrap=1.0, device=False, l1x=None, pieces=None):
    """normal_equations() and launch_count() of one handle fed the data set under `env` (set before the handle is
    created: ASSEMBLY, DETERMINISTIC and CURSOR_STRIDE are read at scratch init)."""
    _set_env(monkeypatch, env)
    t0 = time.perf_counter()
    h = sp.FitHandle(d["ndim"], d["xmin"], d["xmax"], d["nodes"], xtrap)
    assert h.ierror == 0
    x, y, w, n = d["x"], d["y"], d["w"], len(d["y"])
    if device:
        l1x = l1x or d["ndim"]
        dx = torch.full((n, l1x), float("nan"), dtype=torch.float64, device="cuda")     # padding must never be read
        dx[:, :d["ndim"]] = torch.from_numpy(x).cuda()
        dy = torch.from_numpy(y).cuda()
        dw = None if w is None else torch.from_numpy(w).cuda()
        torch.cuda.synchronize()
        assert h.add_points_device(dx, l1x, dy, dw, n, dw is not None) == 0
    else:
        for sl in pieces or [slice(None)]:
            assert h.add_points(x[sl], y[sl], None if w is None else w[sl]) == 0
    ne = h.normal_equations()
    launches = h.launch_count()
    h.destroy()
    SECONDS["gpu"] += time.perf_counter() - t0
    _set_env(monkeypatch, {})
    return ne, launches


def _ratios(d, ne, xtrap, S_ref=None, g_ref=None, cnt_ref=None):
    S, g, cnt, totlwt, nrows = ne
    r = max(worst_ratio(S, d["S"] if S_ref is None else S_ref, TAU * d["scale"]),
            worst_ratio(g, d["g"] if g_ref is None else g_ref, TAU * d["gabs"]))
    if xtrap != 0:
        r = max(r, worst_ratio(cnt, d["cnt"] if cnt_ref is None else cnt_ref, d["cnt_tol"]))
    return r


def _sensitivity(d, ne, xtrap):
    """Smallest error / tolerance over the probes when the probe point is removed from the reference."""
    out = []
    for p in d["probes"]:
        (si, sv), (gi, gv), (node, wp) = point_contribution(d["ndim"], d["x"][p], d["y"][p],
                                                            None if d["w"] is None else d["w"][p],
                                                            d["xmin"], d["xmax"], d["nodes"])
        S1 = d["S"].copy().reshape(-1)
        S1[si] -= sv
        g1 = d["g"].copy()
        np.add.at(g1, gi, -gv)
        c1 = d["cnt"].copy()
        c1[node] -= wp
        out.append(_ratios(d, ne, xtrap, S1.reshape(d["S"].shape), g1, c1))
    return min(out)


def _check(name, label, d, ne, xtrap=1.0):
    S, g, cnt, totlwt, nrows = ne
    assert nrows == d["nrows"], f"{name} {label}: {nrows} rows, expected {d['nrows']}"
    if xtrap != 0:
        assert abs(totlwt - d["totlwt"]) <= d["tot_tol"], f"{name} {label}: totlwt {totlwt} vs {d['totlwt']}"
    r = _ratios(d, ne, xtrap)
    sens = _sensitivity(d, ne, xtrap)
    REPORT.append(f"{name:11s} {label:34s} {r:9.2e}  one point out: {sens:9.2e}")
    print(REPORT[-1], flush=True)
    assert r <= 1.0, f"{name} {label}: error {r:.2e} x the tolerance"
    assert sens >= 100.0, f"{name} {label}: one point less moves the comparison by only {sens:.1f} x the tolerance"


def _two_level(monkeypatch, name, d, env, chunks, **kw):
    """Run under env and under env + BINNING=atomic, check both, and that `chunks` chunks took the two-level route."""
    ne, lc = _run(monkeypatch, d, env, **kw)
    _check(name, "+".join(f"{k[12:]}={v}" for k, v in env.items()) or "default", d, ne, kw.get("xtrap", 1.0))
    ne_a, lc_a = _run(monkeypatch, d, {**env, **ATOMIC}, **kw)
    _check(name, "+".join(f"{k[12:]}={v}" for k, v in {**env, **ATOMIC}.items()), d, ne_a, kw.get("xtrap", 1.0))
    assert lc - lc_a == chunks, f"{name}: {lc - lc_a} two-level chunks, expected {chunks}"
    return lc


def test_3d_12_two_level_shift6_and_switches(monkeypatch):
    """2197 cells: two-level partition with shift 6; the global classify histogram, packed cursors, deterministic mode
    (on the two-level route too) and the direct accumulation on the same data."""
    d = reference("3d12")
    lc = _two_level(monkeypatch, "3d12", d, {}, 1)
    for env in ({"SPLPAK_B200_GLOBAL_HIST": "1"}, {"SPLPAK_B200_CURSOR_STRIDE": "1"}):
        ne, lc_env = _run(monkeypatch, d, env)
        _check("3d12", "+".join(f"{k[12:]}={v}" for k, v in env.items()), d, ne)
        assert lc_env == lc                                        # still the two-level route
    _two_level(monkeypatch, "3d12", d, DET, 1)
    ne, _ = _run(monkeypatch, d, {"SPLPAK_B200_ASSEMBLY": "direct"})
    _check("3d12", "ASSEMBLY=direct", d, ne)


def test_3d_11_per_point_scatter(monkeypatch):
    """1728 cells, just below the two-level threshold: spl_perm_kernel."""
    _two_level(monkeypatch, "3d11", reference("3d11"), {}, 0)


def test_3d_24_cfg3_shape(monkeypatch):
    """The benchmark's cfg3 grid and points: 15625 cells, shift 9; classify with both histograms in shared memory, and
    with the window histogram alone (GLOBAL_HIST)."""
    d = reference("3d24_cfg3")
    lc = _two_level(monkeypatch, "3d24_cfg3", d, {}, 1)
    ne, lc_g = _run(monkeypatch, d, {"SPLPAK_B200_GLOBAL_HIST": "1"})
    _check("3d24_cfg3", "GLOBAL_HIST=1", d, ne)
    assert lc_g == lc


def test_3d_45_shift11_global_classify(monkeypatch):
    """97336 cells: shift 11, span clamped to 2048, 48 buckets, the classify histogram in global memory."""
    _two_level(monkeypatch, "3d45", reference("3d45"), {}, 1)


def test_3d_12_skewed_cells_two_host_chunks(monkeypatch):
    """40 % of 6.3e6 points in 3 cells: two host chunks, both two-level, cells of > 200 work items; deterministic mode
    (whole-cell work items, 3-pass segment sort) on the same data."""
    d = reference("3d12_skew")
    _two_level(monkeypatch, "3d12_skew", d, {}, 2)
    _two_level(monkeypatch, "3d12_skew", d, DET, 2)


@pytest.mark.parametrize("name,chunks", [("4d6", 1), ("4d16", 1), ("4d17", 0)])
def test_4d_partition_routes(monkeypatch, name, chunks):
    """4-D cell path: 2401 cells (shift 6), 83521 cells (shift 11), 104976 cells (above the two-level limit)."""
    _two_level(monkeypatch, name, reference(name), {}, chunks)


def test_4d_5_direct_multi_item_windows(monkeypatch):
    """ASSEMBLY=direct in 4-D: 16 windows of ~131k points, each split into many work items."""
    d = reference("4d5")
    ne, _ = _run(monkeypatch, d, {"SPLPAK_B200_ASSEMBLY": "direct"})
    _check("4d5", "ASSEMBLY=direct", d, ne)


@pytest.mark.parametrize("name", ["2d8", "2d64"])
def test_2d_windows(monkeypatch, name):
    """2-D 8x8: windows of ~84k points; 64x64 (the cfg2 grid), unweighted, across two host chunks."""
    d = reference(name)
    ne, _ = _run(monkeypatch, d, {})
    _check(name, "default", d, ne)


@pytest.mark.parametrize("name,device", [("1d50_200", False), ("1d50_60000", False), ("1d50_4M", False),
                                         ("1d50_big", True)])
def test_1d_deterministic_segment_sort(monkeypatch, name, device):
    """Deterministic mode in 1-D: 1, 2, 3 and (2^24 + 1 points on the device path) 4 radix passes."""
    d = reference(name)
    ne, _ = _run(monkeypatch, d, DET, device=device)
    _check(name, "DETERMINISTIC=1" + (" device" if device else ""), d, ne)
    if name == "1d50_big":
        ne, _ = _run(monkeypatch, d, {}, device=True)
        _check(name, "default device", d, ne)


def test_3d_12_scratch_regrowth(monkeypatch):
    """One handle fed 1e6 (per-point scatter), 3e6 (scratch regrowth, two-level) and 1000 points."""
    d = reference("3d12_grow")
    pieces = [slice(0, 1_000_000), slice(1_000_000, 4_000_000), slice(4_000_000, None)]
    ne, lc = _run(monkeypatch, d, {}, pieces=pieces)
    _check("3d12_grow", "1e6 + 3e6 + 1000", d, ne)
    ne, lc_a = _run(monkeypatch, d, ATOMIC, pieces=pieces)
    _check("3d12_grow", "1e6 + 3e6 + 1000 BINNING=atomic", d, ne)
    assert lc - lc_a == 1


def test_3d_12_strided_device_points(monkeypatch):
    """Device points with l1x = ndim + 2 (NaN padding)."""
    d = reference("3d12")
    ne, _ = _run(monkeypatch, d, {}, device=True, l1x=5)
    _check("3d12", "device l1x=5", d, ne)


def check_refine_rhs(name, label, d, c, rhs, oracle):
    """The rhs_only re-assembly of a refinement step (xtrap = 0: no constraint rows in g) against B^T W^2 (y - B c)
    on the host with the GPU's coefficients c; the residual's own rounding is relative to |y| and |B c|, so the
    tolerance adds TAU |B|^T W^2 |y| to TAU |B|^T W^2 |r|."""
    t0 = time.perf_counter()
    s, ierr = oracle.evaluate_batch(3, d["x"], c, d["xmin"], d["xmax"], d["nodes"])
    assert ierr == 0
    r = d["y"] - s
    _, g_ref, gabs_r = assemble_stencil(3, d["x"], r, d["w"], d["xmin"], d["xmax"], d["nodes"], rhs_only=True)
    SECONDS["reference"] += time.perf_counter() - t0
    tol = TAU * (gabs_r + d["gabs"])
    err = worst_ratio(rhs, g_ref, tol)
    sens = []
    for p in d["probes"]:
        _, (gi, gv), _ = point_contribution(3, d["x"][p], r[p], d["w"][p], d["xmin"], d["xmax"], d["nodes"])
        g1 = g_ref.copy()
        np.add.at(g1, gi, -gv)
        sens.append(worst_ratio(rhs, g1, tol))
    REPORT.append(f"{name:11s} {label:34s} {err:9.2e}  one point out: {min(sens):9.2e}")
    print(REPORT[-1], flush=True)
    assert err <= 1.0
    assert min(sens) >= 100.0


@pytest.mark.parametrize("name", ["3d12", "3d12_skew"])
def test_refinement_rhs_reassembly(monkeypatch, oracle, name):
    """The rhs_only re-assembly of a refinement step with device points (check_refine_rhs)."""
    d = reference(name)
    _set_env(monkeypatch, {})
    t0 = time.perf_counter()
    n = len(d["y"])
    dx, dy, dw = (torch.from_numpy(a).cuda() for a in (d["x"], d["y"], d["w"]))
    torch.cuda.synchronize()
    h = sp.FitHandle(3, d["xmin"], d["xmax"], d["nodes"], 0.0)
    assert h.add_points_device(dx, 3, dy, dw, n, True) == 0
    dcoef = torch.zeros(h.ncol, dtype=torch.float64, device="cuda")
    assert h.compute_device(dcoef) == 0
    c = dcoef.cpu().numpy()
    snap = []
    assert h.refine_device(dx, 3, dy, dw, n, dcoef, weighted=True, allreduce=lambda t: snap.append(t.clone())) == 0
    torch.cuda.synchronize()
    rhs = snap[0].cpu().numpy()
    h.destroy()
    SECONDS["gpu"] += time.perf_counter() - t0
    check_refine_rhs(name, "refine rhs_only", d, c, rhs, oracle)
