"""CPU checks of the GCV additions: the partial-buffer layout with the ywy slot and the refusals that need no device."""
import numpy as np
import pytest

from splpak_b200.distributed import partial_layout


def test_partial_layout_gcv_adds_ywy_at_the_end():
    off, n = partial_layout(3, [24, 24, 24])
    offg, ng = partial_layout(3, [24, 24, 24], gcv=True)
    assert ng == n + 1
    assert offg["ywy"] == (n, n + 1)
    assert {k: v for k, v in offg.items() if k != "ywy"} == off
    assert "ywy" not in off


def test_fit_handle_refuses_unknown_penalty_names_without_a_device():
    from splpak_b200.api import FitHandle, SplpakError

    h = FitHandle.__new__(FitHandle)
    with pytest.raises(SplpakError):
        h._penalty_code("wiggly")
    assert h._penalty_code("thin_plate") == 1 and h._penalty_code(0) == 0
