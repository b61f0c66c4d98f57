"""NGW_OBS_HITS rows (include/ngw.h) against the unmodified reference's own observations (no GPU needed): every lidar
observation of the golden traces is encoded into a hits row by the small encoder below, and runtime.obs_to_vector must
give the reference's vector back.  The traces cover 5, 8 and 16 beams and many item sets, so this pins down both the
format (at most one nonzero entry per beam) and the decoder."""
import numpy as np
import pytest
import torch

import golden_util
import scenarios
from gym_novel_gridworlds_b200.compiler import compile_chain
from gym_novel_gridworlds_b200.runtime import obs_to_vector

LIDAR_TRACES = [n for n in golden_util.names() if any(s[0] == 'lidar' for s in golden_util.get(n)['meta']['chain'])]


def hits_row_bytes(c):
    return ((2 * c.n_beams + 3) & ~3) + 4 * c.n_inv_obs


def encode_hits(vec, c, row_bytes=None):
    """The reference's vectors [n, L*B + I_obs] -> hits rows uint8 [n, row_bytes]: (item, range) per beam, zero
    padding to 4 bytes, int32 inventory tail.  Raises if a beam has more than one nonzero entry."""
    vec = np.asarray(vec, dtype=np.int64)
    n, L, B, ni = vec.shape[0], c.n_lidar_items, c.n_beams, c.n_inv_obs
    rows = np.zeros((n, hits_row_bytes(c) if row_bytes is None else row_bytes), np.uint8)
    blocks = vec[:, :L * B].reshape(n, B, L)
    nz = blocks != 0
    assert (nz.sum(axis=2) <= 1).all(), "a beam with more than one nonzero entry"
    item = np.where(nz.any(axis=2), nz.argmax(axis=2) + 1, 0)
    rng = blocks.max(axis=2)
    assert (rng >= 0).all() and (rng <= 255).all()
    rows[:, 0:2 * B:2] = item
    rows[:, 1:2 * B:2] = rng
    off = (2 * B + 3) & ~3
    rows[:, off:off + 4 * ni] = vec[:, L * B:L * B + ni].astype('<i4').view(np.uint8).reshape(n, 4 * ni)
    return rows


def _compiled(meta):
    return compile_chain(scenarios.build_chain(scenarios.b200_namespace(), meta))


def test_golden_traces_cover_the_beam_counts():
    beams = {dict((s[0], s) for s in golden_util.get(n)['meta']['chain'])['lidar'][1] for n in LIDAR_TRACES}
    assert {5, 8, 16} <= beams


@pytest.mark.parametrize('name', LIDAR_TRACES)
def test_hits_rows_carry_the_reference_vector(name):
    g = golden_util.get(name)
    cc = _compiled(g['meta'])
    c = cc.c
    vecs = [g['obs'].reshape(-1, g['obs'].shape[-1])]
    if g['reset_obs'].shape[-1] == cc.obs_dim:
        vecs.append(g['reset_obs'])
    vec = np.concatenate([v.astype(np.int32) for v in vecs])
    assert vec.shape[1] == cc.obs_dim == c.n_lidar_items * c.n_beams + c.n_inv_obs
    rows = encode_hits(vec, c)
    assert rows.shape[1] == ((2 * c.n_beams + 3) & ~3) + 4 * c.n_inv_obs
    out = obs_to_vector(rows, cc, 'hits')
    assert isinstance(out, np.ndarray) and out.dtype == np.int32
    assert np.array_equal(out, vec)
    # the same rows as a (CPU) tensor, and the other two layouts, decode to the same vector
    assert torch.equal(obs_to_vector(torch.from_numpy(rows), [cc], 'hits'), torch.from_numpy(vec))
    assert np.array_equal(obs_to_vector(vec, cc, 'i32'), vec)
    nl, off = c.n_lidar_items * c.n_beams, (c.n_lidar_items * c.n_beams + 3) & ~3
    u8 = np.zeros((vec.shape[0], off + 4 * c.n_inv_obs), np.uint8)
    u8[:, :nl] = vec[:, :nl]
    u8[:, off:] = vec[:, nl:].astype('<i4').view(np.uint8)
    assert np.array_equal(obs_to_vector(u8, cc, 'u8'), vec)


def test_mixed_configs_decode_with_each_envs_own_config():
    """Rows of a mixed batch are as wide as the widest config's; each env is read with its own config's L, B, I_obs."""
    picks = {}
    for n in LIDAR_TRACES:
        b = dict((s[0], s) for s in golden_util.get(n)['meta']['chain'])['lidar'][1]
        picks.setdefault(b, n)
    names = [picks[b] for b in sorted(picks)]
    compiled = [_compiled(golden_util.get(n)['meta']) for n in names]
    width_vec = max(cc.obs_dim for cc in compiled)
    width_row = max(hits_row_bytes(cc.c) for cc in compiled)
    rows, vecs, ids = [], [], []
    for k, (n, cc) in enumerate(zip(names, compiled)):
        v = golden_util.get(n)['obs'][:, :8].reshape(-1, cc.obs_dim).astype(np.int32)
        rows.append(encode_hits(v, cc.c, width_row))
        vecs.append(np.pad(v, ((0, 0), (0, width_vec - cc.obs_dim))))
        ids.append(np.full(v.shape[0], k))
    perm = np.random.RandomState(0).permutation(sum(len(i) for i in ids))
    rows, vecs, ids = np.concatenate(rows)[perm], np.concatenate(vecs)[perm], np.concatenate(ids)[perm]
    assert np.array_equal(obs_to_vector(rows, compiled, 'hits', ids), vecs)
    assert torch.equal(obs_to_vector(torch.from_numpy(rows), compiled, 'hits', torch.from_numpy(ids)),
                       torch.from_numpy(vecs))


def test_unknown_format_is_rejected():
    cc = _compiled(golden_util.get(LIDAR_TRACES[0])['meta'])
    with pytest.raises(ValueError):
        obs_to_vector(np.zeros((1, 4), np.uint8), cc, 'u16')
