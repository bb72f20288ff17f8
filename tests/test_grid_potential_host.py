"""Host side of the batched grid potential: its workspace stays bounded whatever the number of (dataset, chain)
pairs, and ``GridLikelihood.loglik_sum_batched`` refuses bad shapes before it touches a device."""
import pytest
import torch


def test_workspace_stays_below_two_gib():
    from sbi_for_diffusion_models_b200 import _native
    L = _native.lib()
    for q in (4.0, 64.0):
        for D, C in ((1, 16_000), (125, 128), (16_000, 1)):
            n = L.ddm_grid_loglik_sum_batched_workspace_floats(D, 50, C, q)
            assert 0 < n * 4 <= 2 * 2**30, (q, D, C, n)
        # tables for a chunk of theta at a time: the size stops growing with D * C
        assert (L.ddm_grid_loglik_sum_batched_workspace_floats(1, 50, 16_000, q)
                - L.ddm_grid_loglik_sum_batched_workspace_floats(1, 50, 8_000, q)) < 2**20
    assert L.ddm_grid_loglik_sum_batched_workspace_floats(0, 50, 128, 4.0) == 0
    assert L.ddm_grid_loglik_sum_batched_workspace_floats(1, 50, 128, 65.0) == 0


@pytest.mark.parametrize("bad", ["theta_2d", "theta_cols", "x_d", "x_cols", "pulses_d", "pulses_t", "pulses_short"])
def test_shape_refusals(bad):
    from sbi_for_diffusion_models_b200.likelihood import GridLikelihood
    D, C, T = 2, 3, 4
    theta, x, pl = torch.ones(D, C, 5), torch.ones(D, T, 2), torch.ones(D, T, 80)
    if bad == "theta_2d":
        theta = torch.ones(C, 5)
    elif bad == "theta_cols":
        theta = torch.ones(D, C, 4)
    elif bad == "x_d":
        x = torch.ones(D + 1, T, 2)
    elif bad == "x_cols":
        x = torch.ones(D, T, 3)
    elif bad == "pulses_d":
        pl = torch.ones(D + 1, T, 80)
    elif bad == "pulses_t":
        pl = torch.ones(D, T + 1, 80)
    elif bad == "pulses_short":
        pl = torch.ones(D, T, 79)
    with pytest.raises(ValueError):
        GridLikelihood().loglik_sum_batched(theta, x, pl)
