"""CPU checks of the REML additions: the criterion-name check that needs no device."""
import pytest


def test_fit_handle_refuses_unknown_criteria_without_a_device():
    from splpak_b200.api import FitHandle, SplpakError

    h = FitHandle.__new__(FitHandle)
    for name in ("aic", "REML", "ml", None):
        with pytest.raises(SplpakError):
            h.select_smoothing("curvature", criterion=name)
    assert h._criterion_is_reml("reml") and not h._criterion_is_reml("gcv")
