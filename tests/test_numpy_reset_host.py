"""Host side of the numpy reset stream (no GPU): the seeding the device restates, the global-stream round trip of a
one-env reset, and the option's plumbing through the env constructor."""
import ctypes as C

import numpy as np
import pytest

import gym_novel_gridworlds_b200 as g
from gym_novel_gridworlds_b200 import capi
from gym_novel_gridworlds_b200.capi import ConfigC
from gym_novel_gridworlds_b200.compiler import compile_chain
from gym_novel_gridworlds_b200.runtime import global_stream_reset
from oracle import oracle_lib


@pytest.mark.parametrize('seed', [0, 1, 5489, 123456789, 2 ** 32 - 1])
def test_init_genrand_is_np_random_seed(seed):
    """mt_seed_kernel and ngo_mt_seed run the same recurrence; it is numpy's RandomState.seed for every seed it takes."""
    mt = oracle_lib.MT(seed)
    raw = np.frombuffer(mt.buf.raw, np.uint8)
    _, key, pos, _, _ = np.random.RandomState(seed).get_state()
    assert np.array_equal(raw[:624 * 4].view(np.uint32), key)
    assert int(raw[624 * 4:624 * 4 + 4].view(np.int32)[0]) == pos == 624


class _OracleHandle(object):
    """Stands in for a one-env numpy-stream BatchHandle: the state calls and the reset run on the oracle."""

    def __init__(self, cc):
        self.cc = cc
        self.cfg = ConfigC()
        C.memmove(C.byref(self.cfg), C.byref(cc.c), C.sizeof(ConfigC))
        self.mt = C.create_string_buffer(oracle_lib.lib().ngo_sizeof_mt())
        ms = cc.map_size
        self.map = np.zeros(ms * ms, np.int8)
        self.pose = np.zeros(4, np.uint8)
        self.inv = np.zeros(cc.n_items, np.int32)
        self.loads = 0

    def load_rng_state(self, key, pos, first=0):
        assert np.asarray(key).shape == (1, 624) and np.asarray(pos).shape == (1,) and first == 0
        raw = np.zeros(len(self.mt.raw), np.uint8)
        raw[:624 * 4] = np.asarray(key, np.uint32).reshape(-1).view(np.uint8)
        raw[624 * 4:624 * 4 + 4] = np.asarray(pos, np.int32).view(np.uint8)
        C.memmove(self.mt, raw.ctypes.data, len(raw))
        self.loads += 1

    def reset(self, want_obs=True):
        L = oracle_lib.lib()
        rc = L.ngo_reset_legacy(C.byref(self.cfg), self.cc.map_size, self.mt, self.map.ctypes.data, self.pose.ctypes.data,
                                self.inv.ctypes.data, 1, 0, self.cc.c.n_reset_ops)
        assert rc == 0

    def rng_state(self, first=0, count=None):
        raw = np.frombuffer(self.mt.raw, np.uint8)
        return raw[:624 * 4].view(np.uint32).reshape(1, 624).copy(), raw[624 * 4:624 * 4 + 4].view(np.int32).copy()


def test_global_stream_reset_advances_np_random_and_keeps_the_cached_gaussian():
    env = g.LidarInFront(g.make('NovelGridworld-Pogostick-v1', reset_rng='numpy'), num_beams=8)
    cc = compile_chain(env)
    np.random.seed(31)
    np.random.standard_normal()                      # leaves a cached Gaussian in the global state
    before = np.random.get_state()
    assert before[3] == 1
    fake = _OracleHandle(cc)
    global_stream_reset(fake, want_obs=False)
    after = np.random.get_state()
    k, p = fake.rng_state()
    assert fake.loads == 1 and after[2] == int(p[0]) and np.array_equal(after[1], k[0])
    assert after[2] != before[2] or not np.array_equal(after[1], before[1])
    assert after[3] == before[3] and after[4] == before[4]
    # the map the oracle drew from the same global state, and the stream after it
    mt = oracle_lib.MT(0)
    raw = np.zeros(len(mt.buf.raw), np.uint8)
    raw[:624 * 4] = np.asarray(before[1], np.uint32).view(np.uint8)
    raw[624 * 4:624 * 4 + 4] = np.array([before[2]], np.int32).view(np.uint8)
    C.memmove(mt.buf, raw.ctypes.data, len(raw))
    m = np.zeros_like(fake.map); pose = np.zeros(4, np.uint8); inv = np.zeros_like(fake.inv)
    oracle_lib.lib().ngo_reset_legacy(C.byref(fake.cfg), cc.map_size, mt.buf, m.ctypes.data, pose.ctypes.data,
                                      inv.ctypes.data, 1, 0, cc.c.n_reset_ops)
    assert np.array_equal(m, fake.map) and np.array_equal(pose, fake.pose)


def test_reset_rng_option_of_the_env_constructor():
    with pytest.raises(ValueError, match="reset_rng"):
        g.make('NovelGridworld-Pogostick-v1', reset_rng='mt19937')
    env = g.make('NovelGridworld-Bow-v1', reset_rng='numpy', num_envs=8)
    assert env.unwrapped.reset_rng == 'numpy'
    assert env.seed(40) == [40] and env.unwrapped.reset_rng == 'numpy' and env.unwrapped.rng_seed == 40
    assert g.make('NovelGridworld-Bow-v1').unwrapped.reset_rng == 'philox'
    # a batched numpy-stream env skips the construction-time reset of add_new_items, as the Philox stream does
    g.inject_novelty(g.LidarInFront(env, num_beams=8), 'axe', 'medium', 'wooden', '')


def test_binding_declares_the_rng_calls():
    assert capi.ABI_VERSION == 13 and (capi.RNG_PHILOX, capi.RNG_NUMPY) == (0, 1)
    for name in ('ngw_set_reset_rng', 'ngw_load_rng_state', 'ngw_export_rng_state'):
        assert name in capi.EXPORTS
