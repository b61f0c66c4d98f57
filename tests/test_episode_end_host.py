"""Host side of the episode-end outputs (no GPU needed): decoding the terminal observations of a step that ended no
episode, and the info keys a batched step reports with and without episode_end_info."""
import numpy as np
import pytest
import torch

from test_obs_hits_format import encode_hits
from test_gpu_parity import C2_DESC, _compiled
from gym_novel_gridworlds_b200.runtime import LazyInfo, obs_to_vector


@pytest.mark.parametrize('fmt', ['i32', 'u8', 'hits'])
def test_obs_to_vector_of_no_rows(fmt):
    """info['terminal_observation'][done] is empty on a step where no episode ended; decoding it gives an empty vector
    batch, from a NumPy selection (strides (0, 0)) and from a tensor alike."""
    cc = _compiled(C2_DESC)
    row = {'i32': cc.obs_dim, 'u8': 84, 'hits': 44}[fmt]
    dtype = np.int32 if fmt == 'i32' else np.uint8
    rows = np.zeros((5, row), dtype)
    none = np.zeros(5, bool)
    got = obs_to_vector(rows[none], [cc], fmt)
    assert isinstance(got, np.ndarray) and got.shape == (0, cc.obs_dim) and got.dtype == np.int32
    got = obs_to_vector(torch.from_numpy(rows)[torch.from_numpy(none)], [cc], fmt)
    assert isinstance(got, torch.Tensor) and tuple(got.shape) == (0, cc.obs_dim)
    got = obs_to_vector(rows[none], [cc, cc], fmt, cfg_ids=np.zeros(0, np.int64))
    assert got.shape == (0, cc.obs_dim)


def test_obs_to_vector_of_selected_hits_rows():
    """a selection of some rows decodes like the rows it selects"""
    cc = _compiled(C2_DESC)
    vec = np.zeros((6, cc.obs_dim), np.int32)
    vec[:, 3] = np.arange(6)
    vec[:, -1] = 7
    rows = encode_hits(vec, cc.c)
    sel = np.array([True, False, True, False, False, True])
    assert np.array_equal(obs_to_vector(rows[sel], [cc], 'hits'), vec[sel])


def test_lazy_info_episode_end_keys():
    result, cost = np.zeros(3, bool), np.zeros(3, np.float32)
    plain = LazyInfo(result, cost)
    assert 'TimeLimit.truncated' not in plain and 'terminal_observation' not in plain.keys()
    assert plain.get('TimeLimit.truncated') is None and plain.get('result') is result
    with pytest.raises(KeyError):
        plain['terminal_observation']
    trunc, rows = np.array([True, False, False]), np.arange(6).reshape(3, 2)
    calls = []

    def fetch():
        calls.append(1)
        return trunc, rows

    info = LazyInfo(result, cost, episode_end=fetch)
    assert calls == [] and 'TimeLimit.truncated' in info and 'terminal_observation' in info.keys()
    assert info['TimeLimit.truncated'] is trunc and info.get('terminal_observation') is rows and calls == [1]
    assert LazyInfo(result, cost, episode_end=(trunc, rows))['terminal_observation'] is rows
