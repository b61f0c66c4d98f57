"""ctypes binding of oracle/libngw_oracle.so.  TEST INFRASTRUCTURE ONLY (see ngw_oracle.c header):
imported by tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs."""
import ctypes as C
import os
import subprocess

import numpy as np

from gym_novel_gridworlds_b200.capi import ConfigC

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = os.path.join(_HERE, 'libngw_oracle.so')
_lib = None


def build(force=False):
    src = os.path.join(_HERE, 'ngw_oracle.c')
    hdr = os.path.join(_HERE, '..', 'include', 'ngw.h')
    stale = (not os.path.exists(_LIB)) or any(
        os.path.exists(p) and os.path.getmtime(p) > os.path.getmtime(_LIB) for p in (src, hdr))
    if force or stale:
        subprocess.check_call(['make', '-C', _HERE, '-B', 'libngw_oracle.so'], stdout=subprocess.DEVNULL)
    return _LIB


def lib():
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(_LIB)
        assert L.ngo_sizeof_config() == C.sizeof(ConfigC), \
            "ngw_config layout mismatch: C %d vs ctypes %d" % (L.ngo_sizeof_config(), C.sizeof(ConfigC))
        L.ngo_beam_offset.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int)]
        L.ngo_mt_seed.argtypes = [C.c_void_p, C.c_uint32]
        L.ngo_mt_next.argtypes = [C.c_void_p]
        L.ngo_mt_next.restype = C.c_uint32
        L.ngo_randint.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32]
        L.ngo_randint.restype = C.c_uint32
        L.ngo_shuffle_i32.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
        L.ngo_reset_legacy.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                       C.c_int, C.c_int, C.c_int]
        L.ngo_observe.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.ngo_step.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32,
                               C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.ngo_step_batch.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p,
                                     C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                     C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]
        L.ngo_rollout.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p,
                                  C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p,
                                  C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
        L.ngo_reset_batch.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int64, C.c_uint32, C.c_void_p, C.c_void_p,
                                      C.c_void_p, C.c_int, C.c_void_p]
        L.ngo_philox4x32_10.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        L.ngo_philox_below.argtypes = [C.c_uint64, C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint32, C.c_int64, C.c_void_p,
                                       C.c_void_p]
        L.ngo_policy_draw.argtypes = [C.c_uint64, C.c_uint64, C.c_uint32, C.c_uint32, C.c_void_p]
        L.ngo_policy_draw.restype = C.c_int32
        L.ngo_reset_philox.argtypes = [C.c_void_p, C.c_int, C.c_uint64, C.c_uint64, C.c_uint32, C.c_uint32, C.c_void_p,
                                       C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]
        L.ngo_reset_philox_batch.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int64, C.c_uint64, C.c_uint64,
                                             C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                             C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int]
        L.ngo_policy_draw_batch.argtypes = [C.c_uint64, C.c_uint64, C.c_int64, C.c_void_p, C.c_uint32, C.c_int,
                                            C.c_void_p, C.c_void_p, C.c_int]
        _lib = L
    return _lib


def _p(a):
    return None if a is None else a.ctypes.data


class MT(object):
    """Legacy np.random.RandomState stream (MT19937) as restated in ngw_oracle.c."""

    def __init__(self, seed):
        self.buf = C.create_string_buffer(lib().ngo_sizeof_mt())
        lib().ngo_mt_seed(self.buf, seed)

    def next_u32(self):
        return lib().ngo_mt_next(self.buf)

    def randint(self, low, high):
        return lib().ngo_randint(self.buf, low, high)

    def shuffle(self, arr):
        a = np.ascontiguousarray(arr, dtype=np.int32)
        lib().ngo_shuffle_i32(self.buf, a.ctypes.data, len(a))
        return a


_U64 = 2 ** 64 - 1
# counters of ngo_reset_philox (ngw_oracle.c): what the restated resets did, summed over the envs
RESET_EVENTS = ('fallback', 'place_fail', 'treetap_fail', 'subset', 'all_win', 'list', 'arrival')


def philox4x32_10(ctr, key):
    """One block of the device's Philox4x32-10 as restated in ngw_oracle.c: 4 uint32 words."""
    c = np.ascontiguousarray(ctr, np.uint32)
    k = np.ascontiguousarray(key, np.uint32)
    out = np.zeros(4, np.uint32)
    lib().ngo_philox4x32_10(c.ctypes.data, k.ctypes.data, out.ctypes.data)
    return out


def philox_below(seed, gid, episode, stream, n, count):
    """The first `count` values of the device generator's below(n) on one stream, and the words they consumed."""
    out = np.zeros(count, np.uint32)
    used = C.c_uint32()
    lib().ngo_philox_below(int(seed) & _U64, int(gid) & _U64, int(episode) & 0xFFFFFFFF, stream, n, count, out.ctypes.data,
                           C.byref(used))
    return out, used.value


def policy_draw(seed, gid, t, n):
    """(action, branch) of the device's random policy at step t of env gid: branch 0 = plain draw, 1 = inside Lemire's
    threshold test but kept, 2 = rejected and continued on stream 0xFFE."""
    br = C.c_int()
    a = lib().ngo_policy_draw(int(seed) & _U64, int(gid) & _U64, int(t), int(n), C.byref(br))
    return int(a), br.value


def policy_draws(seed, first_gid, n_actions, n_steps, t0=0, n_threads=8):
    """(actions int32 [n_steps, n], branch uint8 [n_steps, n]) of the device's random policy for envs first_gid + i."""
    na = np.ascontiguousarray(n_actions, np.int32)
    out = np.zeros((n_steps, na.size), np.int32)
    br = np.zeros((n_steps, na.size), np.uint8)
    lib().ngo_policy_draw_batch(int(seed) & _U64, int(first_gid) & _U64, na.size, na.ctypes.data, int(t0), int(n_steps),
                                out.ctypes.data, br.ctypes.data, n_threads)
    return out, br


class OracleBatch(object):
    """A batch of oracle envs sharing one map_size; state lives in NumPy arrays laid out like the GPU SoA."""

    def __init__(self, compiled, n_envs, cfg_id=None):
        self.compiled = list(compiled)
        self.ms = self.compiled[0].map_size
        assert all(c.map_size == self.ms for c in self.compiled)
        self.cfgs = (ConfigC * len(self.compiled))()
        for i, cc in enumerate(self.compiled):
            C.memmove(C.byref(self.cfgs, i * C.sizeof(ConfigC)), C.byref(cc.c), C.sizeof(ConfigC))
        self.n = int(n_envs)
        self.inv_stride = max(cc.n_items for cc in self.compiled)
        self.obs_dim = max(cc.obs_dim for cc in self.compiled)
        self.cfg_id = np.zeros(self.n, np.uint8) if cfg_id is None else np.ascontiguousarray(cfg_id, np.uint8)
        self.map = np.zeros((self.n, self.ms * self.ms), np.int8)
        self.pose = np.zeros((self.n, 4), np.uint8)
        self.inv = np.zeros((self.n, self.inv_stride), np.int32)
        self.err = np.zeros(self.n, np.uint32)
        self.msg = np.zeros(self.n, np.uint16)       # info['message'] codes of the last step (enum ngw_msg | arg << 5)

    def reset_legacy(self, seed0):
        """env i <- reference reset under np.random.seed(seed0 + i)."""
        lib().ngo_reset_batch(self.cfgs, _p(self.cfg_id), self.ms, self.n, seed0, _p(self.map), _p(self.pose),
                              _p(self.inv), self.inv_stride, _p(self.err))
        return self.err.copy()

    def reset_one(self, i, seed, with_obs=True):
        """Reference reset of env i under np.random.seed(seed); returns the reset observation taken where the
        reference takes it (after cfg.reset_obs_after_ops ops) or None when there is no lidar."""
        cfg_ptr = C.byref(self.cfgs, int(self.cfg_id[i]) * C.sizeof(ConfigC))
        cc = self.compiled[int(self.cfg_id[i])]
        mt = MT(seed)
        self.inv[i] = 0
        m, p, v = self.map[i], self.pose[i], self.inv[i]
        k = cc.c.reset_obs_after_ops
        rc = lib().ngo_reset_legacy(cfg_ptr, self.ms, mt.buf, _p(m), _p(p), _p(v), 1, 0, k)
        obs = None
        if with_obs and cc.obs_dim:
            obs = np.zeros(self.obs_dim, np.int32)
            lib().ngo_observe(cfg_ptr, self.ms, _p(m), _p(p), _p(v), _p(obs))
        rc |= lib().ngo_reset_legacy(cfg_ptr, self.ms, mt.buf, _p(m), _p(p), _p(v), 0, k, cc.c.n_reset_ops)
        return rc, obs

    def reset_philox(self, seed, first_gid, episode, key_mask=0xFFFFFFFF, k_obs=None, mask=None, want_obs=True,
                     n_threads=8):
        """Resets with the DEVICE's generator (ngw_oracle.c, last section): env i (where mask, default all) is reset at
        gid first_gid + i and episode word episode (scalar or [n]; the word the reset uses and stores, i.e. the env's
        previous episode + 1).  Returns (flags uint32 [n]: the reset's PLACEMENT bit, 0 for envs not reset; observation
        int32 [n, obs_dim] taken after k_obs ops (scalar or [n]; None = each config's reset_obs_after_ops), or None;
        event counters, a dict over RESET_EVENTS)."""
        ep = np.ascontiguousarray(np.broadcast_to(np.asarray(episode, np.uint64) & 0xFFFFFFFF, (self.n,)), np.uint32)
        ko = None if k_obs is None else np.ascontiguousarray(np.broadcast_to(k_obs, (self.n,)), np.int32)
        mk = None if mask is None else np.ascontiguousarray(mask, np.uint8)
        flags = np.zeros(self.n, np.uint32)
        obs = np.zeros((self.n, self.obs_dim), np.int32) if (want_obs and self.obs_dim) else None
        counters = np.zeros(8, np.int64)
        lib().ngo_reset_philox_batch(self.cfgs, _p(self.cfg_id), self.ms, self.n, int(seed) & _U64, int(first_gid) & _U64,
                                     _p(ep), int(key_mask) & 0xFFFFFFFF, _p(mk), _p(ko), _p(self.map), _p(self.pose),
                                     _p(self.inv), self.inv_stride, _p(obs), self.obs_dim, _p(flags), _p(counters),
                                     n_threads)
        return flags, obs, dict(zip(RESET_EVENTS, counters.tolist()))

    def observe(self):
        obs = np.zeros((self.n, max(self.obs_dim, 1)), np.int32)
        for i in range(self.n):
            cfg_ptr = C.byref(self.cfgs, int(self.cfg_id[i]) * C.sizeof(ConfigC))
            lib().ngo_observe(cfg_ptr, self.ms, _p(self.map[i]), _p(self.pose[i]), _p(self.inv[i]), _p(obs[i]))
        return obs[:, :self.obs_dim]

    def step(self, actions, n_threads=1, want_obs=True):
        actions = np.ascontiguousarray(actions, np.int32)
        obs = np.zeros((self.n, self.obs_dim), np.int32) if (want_obs and self.obs_dim) else None
        reward = np.zeros(self.n, np.float32)
        done = np.zeros(self.n, np.uint8)
        cost = np.zeros(self.n, np.float32)
        result = np.zeros(self.n, np.uint8)
        lib().ngo_step_batch(self.cfgs, _p(self.cfg_id), self.ms, self.n, _p(self.map), _p(self.pose), _p(self.inv),
                             self.inv_stride, _p(actions), _p(obs), self.obs_dim, _p(reward), _p(done), _p(cost),
                             _p(result), _p(self.err), n_threads, _p(self.msg))
        return obs, reward, done, cost, result

    def rollout(self, action_sets, n_steps, n_threads=1):
        """n_steps steps of every env without a per-step barrier (CPU-baseline driver); step s uses
        action_sets[s % len(action_sets)].  Returns the outputs of the last step."""
        acts = np.ascontiguousarray(action_sets, np.int32).reshape(-1, self.n)
        obs = np.zeros((self.n, max(self.obs_dim, 1)), np.int32)
        reward = np.zeros(self.n, np.float32)
        done = np.zeros(self.n, np.uint8)
        cost = np.zeros(self.n, np.float32)
        result = np.zeros(self.n, np.uint8)
        lib().ngo_rollout(self.cfgs, _p(self.cfg_id), self.ms, self.n, _p(self.map), _p(self.pose), _p(self.inv),
                          self.inv_stride, _p(acts), acts.shape[0], int(n_steps), _p(obs) if self.obs_dim else None,
                          self.obs_dim, _p(reward), _p(done), _p(cost), _p(result), _p(self.err), n_threads)
        return obs[:, :self.obs_dim], reward, done, cost, result
