"""Workspace sizes of the tensor-core MNLE entry points, from their size queries (no device needed).

The reverse-mode potential gradient carves only the buffers its passes read or write, so its largest admitted call
(8e6 rows) fits a 180 GB B200.  Training, tc64 potential and sampler keep their layouts: the figures below pin their
sizes."""
import pytest

from sbi_for_diffusion_models_b200 import _native
from sbi_for_diffusion_models_b200.build import build_native


@pytest.fixture(scope="module")
def L():
    build_native()
    return _native.lib()


@pytest.mark.parametrize("K", [3, 8])
def test_gradient_workspace_at_the_row_limit_fits_a_b200(L, K):
    n = L.mnle_loglik_grad_tc_workspace_floats(K, 50, 160_000)      # 8e6 rows, the most one call admits
    assert 0 < n * 4 < 64 * 2**30, n * 4 / 2**30


TC64 = {(50, 160_000): 7312741056, (50, 1024): 47537856, (1, 1): 800320, (65, 7): 1204160}
SAMPLE = {(4000, 2000): 7304741056, (1, 1): 800256, (1000, 3): 3492864}
TRAIN = {3: {1: 1754775, 127: 2754594, 4096: 42024804, 8325: 81793572},
         8: {1: 1755422, 127: 2755886, 4096: 42029966, 8325: 81798734}}


@pytest.mark.parametrize("K", [3, 8])
def test_other_workspaces_keep_their_sizes(L, K):
    for (T, C), want in TC64.items():
        assert L.mnle_loglik_tc64_workspace_floats(K, T, C) == want, (T, C)
    for (B, S), want in SAMPLE.items():
        assert L.mnle_sample_tc_workspace_floats(K, B, S) == want, (B, S)
    for R, want in TRAIN[K].items():
        # these are the sizes of the layout without padding between buffers; every buffer starts on a 256-byte boundary,
        # which moves the last one (the partial sums of grad^2) by up to 252 bytes: up to 1 KiB more, never less
        got = L.mnle_train_workspace_floats(K, R)
        assert want <= got < want + 256, (R, got, want)
