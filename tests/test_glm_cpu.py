"""CPU checks of the GLM fit: the refusal that needs no device, and the host PIRLS reference of test_gpu_glm on the cases
the GPU tests build on (the step-halving and no-finite-deviance cases, and stationarity of a converged fit)."""
import numpy as np
import pytest

from test_gpu_glm import Family, glm_data, halving_case, host_pirls
from test_gpu_smoothing import penalty_dense


def test_unknown_family_raises_without_a_device():
    from splpak_b200.api import FitHandle, SplpakError

    h = FitHandle.__new__(FitHandle)
    for call in (lambda: h.glm_fit(np.zeros((3, 1)), np.zeros(3), family="probit"),
                 lambda: h.glm_fit_device(0, 1, 0, None, 3, 0, family="negative_binomial"),
                 lambda: h._family_code("inverse_gaussian")):
        with pytest.raises(SplpakError, match="unknown family"):
            call()
    assert [h._family_code(f) for f in ("poisson", "binomial", "gamma")] == [0, 1, 2]


def test_reference_halving_case_halves(oracle):
    x, y, o, mn, mx, nodes = halving_case()
    ref = host_pirls(oracle, 1, x, y, None, o, mn, mx, nodes, 0.0, 0.0, "curvature", "gamma", 8)
    assert ref["trace"] == [0, 4, 10] and ref["error"] == 107 and ref["iterations"] == 3


def test_reference_first_iterate_without_finite_deviance(oracle):
    x = np.linspace(0.01, 0.99, 400)
    o = np.where(np.arange(400) % 2 == 0, 0.0, 1600.0)
    ref = host_pirls(oracle, 1, x, np.full(400, 2.0), None, o, np.zeros(1), np.ones(1), [8], 0.0, 0.0, "curvature",
                     "poisson", 3)
    assert ref["error"] == 107 and ref["iterations"] == 1 and not np.isfinite(ref["dev"])


@pytest.mark.parametrize("family", ["poisson", "binomial", "gamma"])
def test_reference_converges_to_the_penalized_score_equations(oracle, family):
    """The reference's fixed point satisfies P^T A ((y - mu) mu' / V) = lam R c: its working response and weights are
    the PIRLS ones, whatever the start."""
    ndim, nodes = 2, [7, 6]
    x, y, w, o, mn, mx = glm_data(family, ndim, nodes, 3000, seed=3, weighted=True, offset=True)
    lam = 0.5
    ref = host_pirls(oracle, ndim, x, y, w, o, mn, mx, nodes, 0.0, lam, "curvature", family, 60, tol=1e-14)
    assert ref["converged"], ref["change"]
    fam = Family(family)
    eta = ref["P"] @ ref["c"] + ref["ov"]
    mu = fam.linkinv(eta)
    r = (y - mu) * fam.mu_eta(eta) / fam.var(mu)
    a = ref["wv"] ** 2
    R = penalty_dense(nodes, mn, mx, "curvature")
    lhs, rhs = ref["P"].T @ (a * r), lam * R @ ref["c"]
    scale = np.abs(ref["P"]).T @ (a * np.abs(r)) + lam * np.abs(R) @ np.abs(ref["c"])
    assert np.max(np.abs(lhs - rhs) / scale) <= 1e-9
