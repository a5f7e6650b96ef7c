"""The band Cholesky factor, entry by entry, on every solver route (FitHandle.cholesky_factor against
oracle/cpu_matched.py), at the shapes where spl_solve_launch changes route.  With T = ceil(b / 64) tile rows and P SMs:
the data-flow kernel while T + T(T-1)/2 fits in the grid with one helper per rest tile (to T = 16 on 148 SMs), with
multi-tile helper lists beyond; the per-phase graph once T(T-1)/2 > 4 (P - T) (from T = 32); the diagonal CTA alone
at T = 1.  SPLPAK_B200_SOLVER=barrier / graph, SPLPAK_B200_KBLOCK and SPLPAK_B200_SYRK select the others.

  * Exact family (kron_exact_system, injected through partial_tensor): every route reproduces the off-diagonal blocks
    of L, the block inverses and c = c* bit for bit, leaves zeros past row n and past the half bandwidth, and a
    refinement step with the right-hand side r* = M delta* returns c* + delta* exactly.  Also after a non-positive pivot
    (107, then the valid system on the same handle), on reused handles and with the REAL32 library.
  * Assembled systems: the stepwise replay of every panel from the device's own earlier columns stays within its bound
    (ratio <= 1), and leaving one earlier panel's contribution out of one tile makes it fail by >= 100x.
Run with -s to see the ratios.
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")
import splpak_b200 as sp  # noqa: E402
from oracle import cpu_matched as cm  # noqa: E402
from util import make_problem  # noqa: E402

ROUTE_ENV = ("SPLPAK_B200_SOLVER", "SPLPAK_B200_KBLOCK", "SPLPAK_B200_SYRK", "SPLPAK_B200_GRAPHPRIO",
             "SPLPAK_B200_DETERMINISTIC")
ROUTES = {
    "default": {},
    "barrier": {"SPLPAK_B200_SOLVER": "barrier"},
    "graph KB8": {"SPLPAK_B200_SOLVER": "graph"},
    "graph KB1 syrk256": {"SPLPAK_B200_SOLVER": "graph", "SPLPAK_B200_KBLOCK": "1", "SPLPAK_B200_SYRK": "256"},
    "graph KB1 syrk128": {"SPLPAK_B200_SOLVER": "graph", "SPLPAK_B200_KBLOCK": "1", "SPLPAK_B200_SYRK": "128"},
    "graph KB3": {"SPLPAK_B200_SOLVER": "graph", "SPLPAK_B200_KBLOCK": "3"},
    "graph no priorities": {"SPLPAK_B200_SOLVER": "graph", "SPLPAK_B200_GRAPHPRIO": "0"},
}
SHAPES = {
    "1-D 64": [64], "1-D 65": [65], "1-D 4097": [4097], "3-D 4x4x4": [4, 4, 4], "2-D 20x9": [20, 9],
    "2-D 21x9": [21, 9], "2-D 42x7": [42, 7], "4-D 4^4": [4, 4, 4, 4], "3-D 12x12x6": [12, 12, 6],
    "2-D 340x6": [340, 6], "2-D 341x6": [341, 6], "3-D 24^3": [24, 24, 24], "2-D 660x4": [660, 4],
    "2-D 661x4": [661, 4],
}
SCALES = (-900, -600, 0, 600, 900)
ALL_SCALES = ("2-D 341x6", "3-D 24^3")
CASES = [(s, r, sc) for i, s in enumerate(SHAPES) for r in ROUTES
         for sc in (SCALES if s in ALL_SCALES else (SCALES[i % 5],))]
SLICE = 2048              # columns per hook read
REPORT = []


@pytest.fixture(autouse=True)
def _clean_env(monkeypatch):
    for k in ROUTE_ENV:
        monkeypatch.delenv(k, raising=False)
    yield


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    if REPORT:
        print("\n".join(["", "route | case | worst ratio | one panel left out"] + REPORT))


_SYSTEMS = {}


def _system(nodes, scale, zero=None):
    key = (tuple(nodes), scale, zero)
    if key not in _SYSTEMS:
        if len(_SYSTEMS) > 6:
            _SYSTEMS.clear()
        _SYSTEMS[key] = cm.kron_exact_system(len(nodes), nodes, scale, zero=zero)
    return _SYSTEMS[key]


def _route(bw, env, nsm):
    """The factor driver spl_solve_launch picks: 'dataflow', 'barrier' or 'graph'."""
    T = (bw + 63) // 64
    if env.get("SPLPAK_B200_SOLVER") == "graph" or nsm - T <= 0 or T * (T - 1) // 2 > 4 * (nsm - T):
        return "graph"
    if env.get("SPLPAK_B200_SOLVER") == "barrier":
        return "barrier"
    return "dataflow" if T == 1 or min(T + T * (T - 1) // 2, nsm) >= T + 1 else "barrier"


def _set(monkeypatch, env):
    for k, v in env.items():
        monkeypatch.setenv(k, v)


def _inject(h, part):
    t = h.partial_tensor()
    t.copy_(torch.from_numpy(part).to(t.device))
    torch.cuda.synchronize()


def _handle(nodes, real32=False):
    nd = len(nodes)
    return sp.FitHandle(nd, np.zeros(nd), np.ones(nd), nodes, 0.0, real32=real32)


def _check_exact(h, sy, tag):
    """Off-diagonal blocks of L (and the zeros past n and b) and the block inverses, bit for bit, in column slices."""
    n, lda = sy["ncol"], sy["lda"]
    for c0 in range(0, n, SLICE):
        nc = min(SLICE, n - c0)
        got = h.cholesky_factor(0, c0, nc)
        want = cm.band_image(sy["L"], lda, c0, nc)
        keep = ~cm.diagonal_block_mask(lda, n, c0, nc)
        bad = np.argwhere(keep & (got != want))
        assert bad.size == 0, (f"{tag}: L differs at {len(bad)} entries, first (row, col) = "
                               f"{[(int(c0 + j + r), int(c0 + j)) for j, r in bad[:5]]}")
    X = h.cholesky_factor(1)
    bad = np.argwhere(X != sy["linv"])
    assert bad.size == 0, f"{tag}: L11^-1 differs at {len(bad)} entries, first (panel, row, col) = {bad[:5].tolist()}"


def _compute_exact(h, sy, tag, capfd=None):
    before = h.launch_count()
    c, ierr = h.compute()
    launches = h.launch_count() - before
    assert ierr == 0, f"{tag}: ierror {ierr}"
    assert np.array_equal(c, sy["c"].astype(c.dtype)), f"{tag}: c differs at {np.flatnonzero(c != sy['c'])[:8]}"
    _check_exact(h, sy, tag)
    if capfd is not None:
        err = capfd.readouterr().err
        assert "cooperative launch" not in err and "graph capture" not in err, err
    return launches


def _refine_exact(h, sy, tag):
    d_coef = torch.zeros(sy["ncol"], dtype=torch.float64, device="cuda")
    r = torch.from_numpy(sy["r"]).cuda()
    ierr = h.refine_device(None, h.ndim, None, None, 0, d_coef, allreduce=lambda rhs: rhs.copy_(r))
    assert ierr == 0, f"{tag}: refinement ierror {ierr}"
    got = d_coef.cpu().numpy()
    assert np.array_equal(got, sy["c"] + sy["delta"]), f"{tag}: refined c differs at {np.flatnonzero(got != sy['c'] + sy['delta'])[:8]}"
    _check_exact(h, sy, tag + ", after refinement")


@pytest.mark.parametrize("shape,route,scale", CASES)
def test_exact_family(shape, route, scale, monkeypatch, capfd):
    nodes = SHAPES[shape]
    env = ROUTES[route]
    _set(monkeypatch, env)
    sy = _system(nodes, scale)
    h = _handle(nodes)
    _inject(h, sy["part"])
    tag = f"{route}, {shape}, 2^{scale}"
    launches = _compute_exact(h, sy, tag, capfd)
    nblk = (sy["ncol"] + 63) // 64
    kind = _route(sy["bw"], env, torch.cuda.get_device_properties(0).multi_processor_count)
    if kind != "graph":
        assert launches == 4, f"{tag}: {launches} launches for a persistent factor (expand, factor, back, pivot range)"
    elif nblk > 1:
        assert launches > 4, f"{tag}: {launches} launches for the per-phase graph"
    _refine_exact(h, sy, tag)
    h.destroy()
    REPORT.append(f"{route} ({kind}) | exact {shape}, 2^{scale} | exact | -")


PIVOT_CASES = {"1-D 65": (0, 64), "2-D 341x6": (1, 3), "3-D 24^3": (2, 12)}


@pytest.mark.parametrize("shape", list(PIVOT_CASES))
@pytest.mark.parametrize("route", list(ROUTES))
def test_zero_pivot_then_valid_system(shape, route, monkeypatch):
    nodes = SHAPES[shape]
    _set(monkeypatch, ROUTES[route])
    bad = _system(nodes, 0, zero=PIVOT_CASES[shape])
    h = _handle(nodes)
    _inject(h, bad["part"])
    _, ierr = h.compute()
    assert ierr == 107
    with pytest.raises(sp.SplpakError):
        h.cholesky_factor(1)
    assert h.reset() == 0
    sy = _system(nodes, 600)
    _inject(h, sy["part"])
    _compute_exact(h, sy, f"{route}, {shape} after a zero pivot")
    h.destroy()


def test_handle_reuse(monkeypatch):
    nodes = SHAPES["2-D 341x6"]
    a, b = _system(nodes, 0), _system(nodes, -600)
    h = _handle(nodes)
    _inject(h, a["part"])
    _compute_exact(h, a, "first compute")
    assert h.reset() == 0
    _inject(h, b["part"])
    _compute_exact(h, b, "second compute, another scale")
    # the per-phase graph: captured once, replayed with new data, rebuilt when the blocking changes
    monkeypatch.setenv("SPLPAK_B200_SOLVER", "graph")
    for kb in ("8", "8", "3", "1"):
        monkeypatch.setenv("SPLPAK_B200_KBLOCK", kb)
        sy = a if kb == "3" else b
        assert h.reset() == 0
        _inject(h, sy["part"])
        _compute_exact(h, sy, f"graph, KBLOCK {kb}")
    # two handles of different shapes, alternately
    nodes2 = SHAPES["2-D 42x7"]
    c = _system(nodes2, 900)
    h2 = _handle(nodes2)
    for step in range(2):
        for hh, sy in ((h, a), (h2, c)):
            assert hh.reset() == 0
            _inject(hh, sy["part"])
            _compute_exact(hh, sy, f"alternating handles, step {step}")
    h.destroy()
    h2.destroy()


def test_hook_refusals():
    nodes = SHAPES["2-D 21x9"]
    sy = _system(nodes, 0)
    h = _handle(nodes)
    _inject(h, sy["part"])
    with pytest.raises(sp.SplpakError):
        h.cholesky_factor(0)                    # no factor yet
    _compute_exact(h, sy, "hook refusals")
    for args in ((0, sy["ncol"] - 1, 2), (0, -1, 1), (2, 0, 1)):
        with pytest.raises(sp.SplpakError):
            h.cholesky_factor(*args)
    assert h.reset() == 0
    with pytest.raises(sp.SplpakError):
        h.cholesky_factor(1)                    # reset: no factor
    h.destroy()


def test_real32_library():
    nodes = SHAPES["2-D 341x6"]
    sy = _system(nodes, 900)
    h = _handle(nodes, real32=True)
    _inject(h, sy["part"])
    _compute_exact(h, sy, "REAL32")
    h.destroy()


# ---- assembled systems: stepwise replay ----
def _assembled(name):
    if name == "2-D 21x9, weighted, hole, xtrap 0.37":
        return dict(nodes=[21, 9], xtrap=0.37, data=make_problem(2, [21, 9], 30000, seed=1, hole=True))
    if name == "3-D 12x12x6, curvature lambda":
        return dict(nodes=[12, 12, 6], xtrap=0.0, lam=1e-4, data=make_problem(3, [12, 12, 6], 200000, seed=2))
    if name == "2-D 341x6":
        return dict(nodes=[341, 6], xtrap=0.0, data=make_problem(2, [341, 6], 400000, seed=3))
    if name == "2-D 24x10, cond > 1e12":
        x, y, w, xmin, xmax = make_problem(2, [24, 10], 20000, seed=4)
        return dict(nodes=[24, 10], xtrap=0.0, cond=True,
                    data=(x, y, np.where(x[:, 0] < 0.5, 1e-7, 1.0), xmin, xmax))
    if name == "3-D 24^3":
        return dict(nodes=[24, 24, 24], xtrap=0.0, data=make_problem(3, [24] * 3, 1 << 21, seed=5))
    raise KeyError(name)


ASSEMBLED = ["2-D 21x9, weighted, hole, xtrap 0.37", "3-D 12x12x6, curvature lambda", "2-D 341x6",
             "2-D 24x10, cond > 1e12", "3-D 24^3"]
ASM_ROUTES = {"default": {}, "barrier": ROUTES["barrier"], "graph KB8": ROUTES["graph KB8"],
              "deterministic": {"SPLPAK_B200_DETERMINISTIC": "1"}}


@pytest.mark.parametrize("name", ASSEMBLED)
@pytest.mark.parametrize("route", list(ASM_ROUTES))
def test_replay_of_assembled_system(name, route, monkeypatch):
    _set(monkeypatch, ASM_ROUTES[route])
    case = _assembled(name)
    nodes = case["nodes"]
    x, y, w, xmin, xmax = case["data"]
    h = sp.FitHandle(len(nodes), xmin, xmax, nodes, case["xtrap"])
    if case.get("lam"):
        assert h.set_smoothing(case["lam"]) == 0
    assert h.add_points(x, y, w) == 0
    _, ierr = h.compute()
    assert ierr == 0
    if case["xtrap"]:
        assert h.constraints_fired()
    S = h.normal_equations()[0]                 # after compute: constraint rows and penalty included
    n = S.shape[0]
    bw = cm.half_bandwidth(len(nodes), nodes)
    lda = cm.band_lda(bw)
    Mimg = cm.band_from_stencil(S, nodes, lda)
    Limg = h.cholesky_factor(0)
    X = h.cholesky_factor(1)
    h.destroy()
    if case.get("cond"):
        Md = np.zeros((n, n))
        for j in range(n):
            Md[j:min(n, j + bw + 1), j] = Mimg[j, :min(bw + 1, n - j)]
        Md = np.tril(Md) + np.tril(Md, -1).T
        assert np.linalg.cond(Md) > 1e12
    nblk = X.shape[0]
    res = cm.replay_panels(Mimg, Limg, X, bw, range(nblk))
    k, rl, rx = max(res, key=lambda r: max(r[1], r[2]))
    worst = max(rl, rx)
    drops = cm.sensitivity_drops(Mimg, Limg, bw)
    assert len(drops) == (3 if bw > 64 else 1), sorted(drops)
    least = min(max(cm.replay_panels(Mimg, Limg, X, bw, [kk], drop=d)[0][1:]) for kk, d in drops.values())
    REPORT.append(f"{route} | {name} | {worst:.2e} (panel {k}) | {least:.1e}")
    assert worst <= 1.0, f"{route}, {name}: panel {k}: L21 ratio {rl:.3g}, L11^-1 ratio {rx:.3g}"
    assert least >= 100.0
