"""Host side of the ragged-session potential (no GPU): trial offsets from session lengths, the split of a
request into launches at session boundaries, and the refusals raised before anything is launched."""
import numpy as np
import pytest
import torch

from sbi_for_diffusion_models_b200.mnle_net import session_offsets, split_sessions


def test_offsets_from_lengths():
    want = np.array([0, 50, 57, 58, 58, 188, 252], np.int64)
    for lengths in ([50, 7, 1, 0, 130, 64], (50, 7, 1, 0, 130, 64), np.array([50, 7, 1, 0, 130, 64], np.int32),
                    torch.tensor([50, 7, 1, 0, 130, 64]), torch.tensor([50, 7, 1, 0, 130, 64], dtype=torch.int32)):
        off = session_offsets(lengths)
        assert off.dtype == np.int64 and np.array_equal(off, want)
    assert np.array_equal(session_offsets([]), [0])
    assert np.array_equal(session_offsets([0, 0, 0]), [0, 0, 0, 0])
    assert np.array_equal(session_offsets(torch.empty(0, dtype=torch.int64)), [0])


@pytest.mark.parametrize("bad", [[3, -1, 2], [1.5, 2], torch.tensor([3.0, 2.0]), torch.tensor([[3, 2]]), [[3, 2]],
                                 torch.tensor([3, -2])])
def test_bad_lengths_are_refused(bad):
    with pytest.raises(ValueError):
        session_offsets(bad)


def test_split_at_session_boundaries():
    off = session_offsets([50, 7, 1, 0, 130, 64])
    assert split_sessions(off, 524_280, 2**31 - 1) == [(0, 6)]
    chunks = split_sessions(off, 140, 2**31 - 1)
    assert chunks == [(0, 4), (4, 5), (5, 6)]
    # every chunk within the limit, consecutive, covering all sessions
    assert chunks[0][0] == 0 and chunks[-1][1] == 6 and all(a[1] == b[0] for a, b in zip(chunks, chunks[1:]))
    assert all(off[d1] - off[d0] <= 140 for d0, d1 in chunks)
    assert split_sessions(off, 140, 2) == [(0, 2), (2, 4), (4, 5), (5, 6)]
    assert split_sessions(off, 130, 2**31 - 1) == [(0, 4), (4, 5), (5, 6)]     # a session exactly at the limit fits
    assert split_sessions(session_offsets([0, 0, 0]), 1, 2**31 - 1) == [(0, 3)]
    assert split_sessions(session_offsets([]), 10, 10) == []


def test_a_session_over_the_limit_is_refused():
    with pytest.raises(ValueError, match="session 4 has 130 trials"):
        split_sessions(session_offsets([50, 7, 1, 0, 130, 64]), 129, 2**31 - 1)
