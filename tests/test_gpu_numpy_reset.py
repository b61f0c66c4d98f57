"""The numpy reset stream (ngw_set_reset_rng(NGW_RNG_NUMPY)): every regeneration path of the device draws the reference's
own legacy np.random (MT19937) stream, so the maps are the reference's bit for bit.  Checked against the reference's
stored resets (tests/golden), against the oracle's restatement of the reference's reset carrying one MT19937 state across
consecutive episodes (ngo_reset_legacy), and against numpy itself."""
import ctypes as C

import numpy as np
import pytest
import torch

import golden_util
import scenarios
from gym_novel_gridworlds_b200 import capi
from gym_novel_gridworlds_b200 import opcodes as oc
from gym_novel_gridworlds_b200.capi import ConfigC
from gym_novel_gridworlds_b200.compiler import compile_chain
from gym_novel_gridworlds_b200.runtime import BatchHandle
from oracle import oracle_lib
from oracle.oracle_lib import OracleBatch

pytestmark = pytest.mark.gpu
MT_WORDS = 624


def _compiled(desc):
    return compile_chain(scenarios.build_chain(scenarios.b200_namespace(), desc))


def _np_state(seed):
    """(key uint32 [624], pos) of np.random.RandomState(seed)."""
    _, key, pos, _, _ = np.random.RandomState(seed).get_state()
    return np.asarray(key, np.uint32), int(pos)


class OracleStream(object):
    """Oracle twins of a batch: env i carries its own legacy np.random state across resets (ngo_mt: key[624], pos)."""

    def __init__(self, compiled, n, cfg_id=None, keys=None, pos=None):
        self.ob = OracleBatch(compiled, n, cfg_id)
        self.size = oracle_lib.lib().ngo_sizeof_mt()
        self.mt = [C.create_string_buffer(self.size) for _ in range(n)]
        if keys is not None:
            for i in range(n):
                self.set_state(i, keys[i], pos[i])

    def set_state(self, i, key, pos):
        raw = np.zeros(self.size, np.uint8)
        raw[:MT_WORDS * 4] = np.asarray(key, np.uint32).view(np.uint8)
        raw[MT_WORDS * 4:MT_WORDS * 4 + 4] = np.array([pos], np.int32).view(np.uint8)
        C.memmove(self.mt[i], raw.ctypes.data, self.size)

    def state(self, i):
        raw = np.frombuffer(self.mt[i].raw, np.uint8)
        return raw[:MT_WORDS * 4].view(np.uint32).copy(), int(raw[MT_WORDS * 4:MT_WORDS * 4 + 4].view(np.int32)[0])

    def states(self):
        st = [self.state(i) for i in range(self.ob.n)]
        return np.stack([k for k, _ in st]), np.array([p for _, p in st], np.int32)

    def reset(self, i, k_obs=None):
        """The reference reset of env i from its state; a part that fails ends the program.  Returns (rc, observation
        taken after k_obs ops (default: the config's reset_obs_after_ops) or None)."""
        L = oracle_lib.lib()
        ob = self.ob
        cc = ob.compiled[int(ob.cfg_id[i])]
        cfg = C.byref(ob.cfgs, int(ob.cfg_id[i]) * C.sizeof(ConfigC))
        k = cc.c.reset_obs_after_ops if k_obs is None else k_obs
        ob.inv[i] = 0
        m, p, v = ob.map[i], ob.pose[i], ob.inv[i]
        rc = L.ngo_reset_legacy(cfg, ob.ms, self.mt[i], m.ctypes.data, p.ctypes.data, v.ctypes.data, 1, 0, k)
        obs = None
        if cc.obs_dim:
            obs = np.zeros(max(ob.obs_dim, 1), np.int32)
            L.ngo_observe(cfg, ob.ms, m.ctypes.data, p.ctypes.data, v.ctypes.data, obs.ctypes.data)
            obs = obs[:cc.obs_dim]
        if rc == 0:
            rc = L.ngo_reset_legacy(cfg, ob.ms, self.mt[i], m.ctypes.data, p.ctypes.data, v.ctypes.data, 0, k,
                                    cc.c.n_reset_ops)
        return rc, obs


def _numpy_handle(compiled, n, seed=0, first_env_gid=0, cfg_id=None, **kw):
    return BatchHandle(compiled, n, seed=seed, first_env_gid=first_env_gid, cfg_id=cfg_id, reset_rng='numpy', **kw)


def _assert_state(h, ors, where, idx=None):
    """map, pose, inventory and (key, pos) of the handle equal the oracle twins' (envs idx, default all)."""
    ob = ors.ob
    idx = np.arange(ob.n) if idx is None else np.asarray(idx)
    w = ob.inv.shape[1]
    assert np.array_equal(h.map.cpu().numpy().reshape(h.n, -1)[idx], ob.map[idx]), where + ": map"
    assert np.array_equal(h.pose.cpu().numpy()[idx], ob.pose[idx]), where + ": pose"
    assert np.array_equal(h.inventory.cpu().numpy()[idx, :w], ob.inv[idx]), where + ": inventory"
    key, pos = h.rng_state()
    okey, opos = ors.states()
    assert np.array_equal(pos[idx], opos[idx]), where + ": pos"
    assert np.array_equal(key[idx], okey[idx]), where + ": key"


# ---------------------------------------------------------------------------------------------- 1. reference fixtures
def test_every_reference_reset_of_the_golden_traces_from_its_seed():
    """Every scenario of traces.npz, every episode: a numpy-stream handle given np.random.RandomState(ep_seed)'s state
    resets to the reference's stored state and reset observation, and leaves the oracle's stream position."""
    for name in golden_util.names():
        g = golden_util.get(name)
        cc = _compiled(g['meta'])
        seeds = g['meta']['seeds']
        n_items = g['reset_inv'].shape[1]
        h = _numpy_handle([cc], len(seeds))
        st = [_np_state(s) for s in seeds]
        keys, pos = np.stack([k for k, _ in st]), np.array([p for _, p in st], np.int32)
        h.load_rng_state(keys, pos)
        obs = h.reset(want_obs=True)
        ors = OracleStream([cc], len(seeds), keys=keys, pos=pos)
        for ep in range(len(seeds)):
            rc, _ = ors.reset(ep)
            assert rc == 0, name
        where = name
        assert not h.error_flags.cpu().numpy().any(), where
        assert np.array_equal(h.map.cpu().numpy().reshape(len(seeds), -1), g['reset_map']), where
        assert np.array_equal(h.pose.cpu().numpy(), g['reset_pose']), where
        assert np.array_equal(h.inventory.cpu().numpy()[:, :n_items], g['reset_inv']), where
        if g['meta']['reset_kind'] == 'lidar':
            assert np.array_equal(obs.cpu().numpy()[:, :cc.obs_dim], g['reset_obs'].astype(np.int32)), where
        _assert_state(h, ors, where)
        h.close()


def test_seeding_on_the_device_is_np_random_seed():
    """ngw_set_reset_rng seeds env e as np.random.seed(seed + first_env_gid + e), up to the largest seed numpy takes."""
    cc = _compiled(golden_util.get('pogo_limit_lidar')['meta'])
    for seed, gid0, n in ((0, 0, 37), (12345, 1000, 70), (2 ** 32 - 40, 7, 33)):
        h = _numpy_handle([cc], n, seed=seed, first_env_gid=gid0)
        key, pos = h.rng_state()
        for e in (0, 1, n // 2, n - 1):
            k, p = _np_state(seed + gid0 + e)
            assert pos[e] == p and np.array_equal(key[e], k), (seed, gid0, e)
        h.close()


# ---------------------------------------------------------------------------------------------- 2. hashed long traces
def _reset_hash(h, n_items_of, idx_of):
    m, p, v = h.map.cpu().numpy().reshape(h.n, -1), h.pose.cpu().numpy(), h.inventory.cpu().numpy()
    out = np.zeros(h.n, np.uint64)
    for idx, n_items in zip(idx_of, n_items_of):
        z = np.zeros(len(idx))
        out[idx] = golden_util.trace_hash(np.zeros((len(idx), 0)), z, z, z, z, v[idx, :n_items], p[idx], m[idx])
    return out


@pytest.mark.skipif(not golden_util.long_names(), reason="tests/golden/long_traces.npz is missing")
@pytest.mark.parametrize('case', ['C2', 'C3', 'C4', 'C5'])
def test_long_reference_traces_from_seeds_alone(case):
    """Every reset of the hashed long traces generated on the device from its seed (C4: one mixed batch, env j -> novelty
    j mod 4, states loaded from RandomState(seed0_k + episode)); then the unperturbed (even) episodes replayed from those
    device-generated states, with no state injected, every step's hash compared."""
    names = ['C4_0', 'C4_1', 'C4_2', 'C4_3'] if case == 'C4' else [case]
    gs = [golden_util.long_get(nm) for nm in names]
    compiled = [_compiled(g['meta']) for g in gs]
    E, T = gs[0]['actions'].shape
    k = len(names)
    n = E * k
    cfg = (np.arange(n) % k).astype(np.int32)
    if k == 1:
        h = _numpy_handle(compiled, n, seed=gs[0]['meta']['seed0'])
    else:
        h = _numpy_handle(compiled, n, cfg_id=cfg)
        st = [_np_state(gs[j % k]['meta']['seed0'] + j // k) for j in range(n)]
        h.load_rng_state(np.stack([s[0] for s in st]), np.array([s[1] for s in st], np.int32))
    h.reset(want_obs=False)
    idx_of = [np.nonzero(cfg == j)[0] for j in range(k)]
    n_items_of = [g['init_inv'].shape[1] for g in gs]
    got = _reset_hash(h, n_items_of, idx_of)
    for j, g in enumerate(gs):
        assert np.array_equal(got[idx_of[j]], g['reset_hash']), "%s: %d resets differ" % (
            names[j], int((got[idx_of[j]] != g['reset_hash']).sum()))
    assert not h.error_flags.cpu().numpy().any()
    actions = np.zeros((n, T), np.int32)
    hashes = np.zeros((n, T), np.uint64)
    for j, g in enumerate(gs):
        actions[j::k] = g['actions']
        hashes[j::k] = g['hash']
    even = [idx[(idx // k) % 2 == 0] for idx in idx_of]          # episode index of env idx is idx // k
    acts = torch.from_numpy(actions.T.copy()).cuda()
    for t in range(T):
        obs, rew, done, cost, res = h.step(acts[t])
        o, r, d, c, s = (x.cpu().numpy() for x in (obs, rew, done, cost, res))
        m, p, v = h.map.cpu().numpy().reshape(n, -1), h.pose.cpu().numpy(), h.inventory.cpu().numpy()
        for idx, cc, n_items in zip(even, compiled, n_items_of):
            hh = golden_util.trace_hash(o[idx, :cc.obs_dim], r[idx], d[idx], s[idx], c[idx], v[idx, :n_items], p[idx],
                                        m[idx])
            bad = hh != hashes[idx, t]
            assert not bad.any(), "%s step %d: %d envs differ from the reference" % (case, t, int(bad.sum()))
    h.close()


# ---------------------------------------------------------------------------------------------- 3. continuing streams
# chains whose resets exercise every op: plain placement, Q3 split + fences, v0 TREETAP, replace, 40x40 shuffles
STREAM_CHAINS = ['pogo_limit_lidar', 'bow_C3_axe_medium_fence_hard', 'pogo0_lidar', 'pogo_A_replaceitem_hard_log',
                 'pogo_B_additem_medium', 'pogo_ms40_additem_hard']
EPISODES = 6


def _stream_case(name, n, desc=None):
    cc = _compiled(golden_util.get(name)['meta'] if desc is None else desc)
    seed = 1000 + 37 * len(name)
    h = _numpy_handle([cc], n, seed=seed)
    st = [_np_state(seed + e) for e in range(n)]
    ors = OracleStream([cc], n, keys=np.stack([s[0] for s in st]), pos=np.array([s[1] for s in st], np.int32))
    return cc, h, ors


def _oracle_reset_all(ors, mask=None, k_obs=None):
    obs = []
    for i in range(ors.ob.n):
        if mask is None or mask[i]:
            rc, o = ors.reset(i, k_obs)
            assert rc == 0
            obs.append(o)
        else:
            obs.append(None)
    return obs


@pytest.mark.parametrize('name', STREAM_CHAINS)
def test_masked_resets_continue_the_stream(name):
    n = 45
    cc, h, ors = _stream_case(name, n)
    rng = np.random.RandomState(5)
    for ep in range(EPISODES):
        mask = (rng.rand(n) < 0.6).astype(np.uint8) if ep else np.ones(n, np.uint8)
        obs = h.reset(mask=mask).cpu().numpy() if cc.obs_dim else h.reset(mask=mask, want_obs=False)
        oobs = _oracle_reset_all(ors, mask)
        _assert_state(h, ors, "%s episode %d" % (name, ep))
        if cc.obs_dim:
            for i in np.nonzero(mask)[0]:
                assert np.array_equal(obs[i, :cc.obs_dim], oobs[i]), "%s episode %d env %d" % (name, ep, i)
    h.close()


def _one_step_path(h, path, acts):
    if path == 'step':
        return h.step(acts, auto_reset=True, max_episode_steps=1)
    if path == 'step_many':
        from gym_novel_gridworlds_b200.runtime import step_many
        return step_many([h], [acts], auto_reset=True, max_episode_steps=1)[0]
    out = h.step_host(acts.cpu().numpy(), auto_reset=True, max_episode_steps=1)
    return tuple(torch.as_tensor(np.asarray(x)) for x in out)


def _valid_actions(cc, rng, shape):
    return torch.from_numpy(rng.choice(np.asarray(cc.external_ids), size=shape).astype(np.int32)).cuda()


def _oracle_follow(h, ors, ep_before, k_obs=None):
    """The oracle resets each env as often as the device did (episode counter delta); returns (resets [n], the reset
    observations per env)."""
    resets = (h.episode.cpu().numpy().astype(np.int64) - ep_before.astype(np.int64))
    obs = [[ors.reset(i, k_obs) for _ in range(int(resets[i]))] for i in range(len(resets))]
    assert all(rc == 0 for per in obs for rc, _ in per)
    return resets, [[o for _, o in per] for per in obs]


@pytest.mark.parametrize('path', ['step', 'step_many', 'host'])
@pytest.mark.parametrize('name', ['pogo_limit_lidar', 'bow_C3_axe_medium_fence_hard', 'pogo0_lidar'])
def test_auto_resets_of_the_one_step_paths_continue_the_stream(name, path):
    """max_episode_steps=1: every step ends every episode, so each step's queued auto-reset regenerates every env; the
    observation of the step is the new episode's reset observation (taken after reset_obs_after_ops ops)."""
    n = 70
    cc, h, ors = _stream_case(name, n)
    h.reset(want_obs=False)
    _oracle_reset_all(ors)
    rng = np.random.RandomState(9)
    for t in range(EPISODES):
        acts = _valid_actions(cc, rng, n)
        ep = h.episode.cpu().numpy().copy()
        obs = _one_step_path(h, path, acts)[0]
        torch.cuda.synchronize()
        resets, oobs = _oracle_follow(h, ors, ep)
        assert (resets == 1).all(), "%s %s step %d: every env ends its episode" % (name, path, t)
        _assert_state(h, ors, "%s %s step %d" % (name, path, t))
        o = obs.cpu().numpy() if isinstance(obs, torch.Tensor) else np.asarray(obs)
        for i in range(n):
            assert np.array_equal(o[i, :cc.obs_dim], oobs[i][0]), "%s %s step %d env %d" % (name, path, t, i)
    assert not h.error_flags.cpu().numpy().any()
    h.close()


def _policy(cc, n_pa=6, seed=3):
    rng = np.random.RandomState(seed)
    w = torch.from_numpy(rng.randint(-3, 4, size=(cc.obs_dim, n_pa)).astype(np.int32)).cuda()
    b = torch.from_numpy(rng.randint(-3, 4, size=n_pa).astype(np.int32)).cuda()
    return w, b


@pytest.mark.parametrize('record', [False, True])
@pytest.mark.parametrize('mode', ['given', 'random', 'policy'])
@pytest.mark.parametrize('name', ['pogo_limit_lidar', 'bow_C3_axe_medium_fence_hard', 'pogo_ms40_additem_hard'])
def test_rollout_resets_continue_the_stream(name, mode, record):
    """The in-kernel regeneration of both rollout kernels (10x10: lane pairs, 40x40: the fallback kernel): K steps with
    max_episode_steps=1 regenerate every env K times; the state, the stream and every recorded observation (taken after
    ALL reset ops) equal the oracle's, and a one-step twin ends in the same state."""
    n, K = 40, EPISODES
    cc, h, ors = _stream_case(name, n)
    _, twin, _ = _stream_case(name, n)
    h.reset(want_obs=False)
    twin.reset(want_obs=False)
    _oracle_reset_all(ors)
    rng = np.random.RandomState(4)
    acts = _valid_actions(cc, rng, (K, n))
    rec = h.rollout_record(K) if record else None
    kw = dict(auto_reset=True, max_episode_steps=1, record=rec, record_actions=True)
    ep = h.episode.cpu().numpy().copy()
    if mode == 'given':
        out = h.rollout(K, actions=acts, **kw)
    elif mode == 'random':
        out = h.rollout(K, policy_seed=77, **kw)
    else:
        w, b = _policy(cc)
        out = h.rollout(K, policy=(w, b), **kw)
    torch.cuda.synchronize()
    taken = out[-2] if record else out[-1]
    resets, recorded = _oracle_follow(h, ors, ep, k_obs=cc.c.n_reset_ops)
    # max_episode_steps=1: an env regenerates after every step it took a valid action in (an invalid one — the random
    # policy draws over [0, n_actions) — leaves the env and its episode untouched)
    valid = np.array([cc.c.actions[a].op != oc.OP_INVALID for a in range(cc.c.n_actions)])
    assert np.array_equal(resets, valid[taken.cpu().numpy()].sum(axis=0)), resets
    if mode != 'random':
        assert (resets == K).all(), resets
    _assert_state(h, ors, "%s %s rollout" % (name, mode))
    if record and cc.obs_dim:
        robs = rec.obs.cpu().numpy()
        for i in np.nonzero(resets == K)[0]:                 # an env regenerated at every step: record t = reset t
            for t in range(K):
                assert np.array_equal(robs[t, i, :cc.obs_dim], recorded[i][t]), "%s %s record step %d env %d" % (
                    name, mode, t, i)
    for t in range(K):                                    # the one-step twin takes the actions the rollout took
        twin.step(taken[t].contiguous(), auto_reset=True, max_episode_steps=1)
    torch.cuda.synchronize()
    assert torch.equal(twin.map, h.map) and torch.equal(twin.pose, h.pose) and torch.equal(twin.inventory, h.inventory)
    tk, tp = twin.rng_state()
    hk, hp = h.rng_state()
    assert np.array_equal(tk, hk) and np.array_equal(tp, hp)
    h.close()
    twin.close()


@pytest.mark.parametrize('nov', [None, ['novelty', 'additem', 'hard', 'spring', '']])
def test_largest_grid_resets_auto_resets_and_rollouts(nov):
    """64x64, the largest map_size: the candidate lists take ngw_reset's and the queued auto-reset's shared memory past
    48 KB per CTA, and the fallback rollout kernel's plan grows by one list."""
    desc = {'env': scenarios.POGO, 'map_size': 64,
            'chain': [['limit', scenarios.C2_SET], ['lidar', 8]] + ([nov] if nov else [])}
    n = 36
    cc, h, ors = _stream_case('ms64', n, desc)
    obs = h.reset().cpu().numpy()
    oobs = _oracle_reset_all(ors)
    _assert_state(h, ors, "ms64 reset")
    for i in range(n):
        assert np.array_equal(obs[i, :cc.obs_dim], oobs[i]), "ms64 reset env %d" % i
    rng = np.random.RandomState(6)
    ep = h.episode.cpu().numpy().copy()
    obs = h.step(_valid_actions(cc, rng, n), auto_reset=True, max_episode_steps=1)[0].cpu().numpy()
    resets, oobs = _oracle_follow(h, ors, ep)
    assert (resets == 1).all()
    _assert_state(h, ors, "ms64 auto-reset step")
    for i in range(n):
        assert np.array_equal(obs[i, :cc.obs_dim], oobs[i][0]), "ms64 auto-reset env %d" % i
    ep = h.episode.cpu().numpy().copy()
    h.rollout(2, actions=_valid_actions(cc, rng, (2, n)), auto_reset=True, max_episode_steps=1)
    torch.cuda.synchronize()
    resets, _ = _oracle_follow(h, ors, ep, k_obs=cc.c.n_reset_ops)
    assert (resets == 2).all()
    _assert_state(h, ors, "ms64 rollout")
    assert not h.error_flags.cpu().numpy().any()
    h.close()


# ---------------------------------------------------------------------------------------------- 5. edge cases
def test_placement_failure_matches_the_oracle_flag_and_stream_position():
    """A crowded AxeHard-iron chain on a small grid: the resets that run out of cells fail exactly where the oracle's do,
    with the same stream position afterwards, and skip the rest of their program."""
    desc = {'env': scenarios.POGO, 'map_size': 9, 'chain': [['lidar', 8], ['novelty', 'axe', 'hard', 'iron', 'true']]}
    cc = _compiled(desc)
    n = 256
    h = _numpy_handle([cc], n, seed=40)
    st = [_np_state(40 + e) for e in range(n)]
    ors = OracleStream([cc], n, keys=np.stack([s[0] for s in st]), pos=np.array([s[1] for s in st], np.int32))
    for ep in range(3):
        h.reset(want_obs=False)
        rcs = np.array([ors.reset(i)[0] for i in range(n)], np.uint32)
        flags = h.error_flags.cpu().numpy().astype(np.uint32)
        assert np.array_equal(flags & 2, rcs & 2), ep
        ok = np.nonzero(rcs == 0)[0]
        _assert_state(h, ors, "episode %d" % ep, idx=ok)
        key, pos = h.rng_state()
        okey, opos = ors.states()
        assert np.array_equal(pos, opos) and np.array_equal(key, okey), ep
    assert (rcs != 0).any() and (rcs == 0).any(), "the chain should fail some resets and not others"
    h.close()


def test_sharding_by_first_env_gid_generates_the_same_episodes():
    cc = _compiled(golden_util.get('bow_C3_axe_medium_fence_hard')['meta'])
    one = _numpy_handle([cc], 96, seed=300)
    a = _numpy_handle([cc], 40, seed=300)
    b = _numpy_handle([cc], 56, seed=300, first_env_gid=40)
    acts = _valid_actions(cc, np.random.RandomState(2), (5, 96))
    for hh in (one, a, b):
        hh.reset()
    for t in range(5):
        one.step(acts[t].contiguous(), auto_reset=True, max_episode_steps=2)
        a.step(acts[t, :40].contiguous(), auto_reset=True, max_episode_steps=2)
        b.step(acts[t, 40:].contiguous(), auto_reset=True, max_episode_steps=2)
    torch.cuda.synchronize()
    assert torch.equal(one.map, torch.cat([a.map, b.map])) and torch.equal(one.pose, torch.cat([a.pose, b.pose]))
    k1, p1 = one.rng_state()
    ka, pa = a.rng_state()
    kb, pb = b.rng_state()
    assert np.array_equal(k1, np.concatenate([ka, kb])) and np.array_equal(p1, np.concatenate([pa, pb]))
    for hh in (one, a, b):
        hh.close()


def test_captured_rotation_of_numpy_handles_with_auto_reset_equals_eager_twins():
    """Three numpy-stream handles stepped in rotation with auto-reset inside one CUDA graph (parallel branches, queued
    resets drawing from each handle's own states), replayed, against eager twins."""
    cc = _compiled(golden_util.get('pogo_limit_lidar')['meta'])
    n, R, T = 32 * 90 + 5, 3, 4
    hs = [_numpy_handle([cc], n, seed=500 + 1000 * k) for k in range(R)]
    tw = [_numpy_handle([cc], n, seed=500 + 1000 * k) for k in range(R)]
    rng = np.random.RandomState(8)
    acts = [_valid_actions(cc, rng, n) for _ in range(T)]
    for hh in hs + tw:
        hh.reset()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        with torch.cuda.graph(g, stream=s):
            for t in range(T):
                for hh in hs:
                    hh.step(acts[t], auto_reset=True, max_episode_steps=3)
    torch.cuda.synchronize()
    for rep in range(2):
        g.replay()
        for t in range(T):
            for hh in tw:
                hh.step(acts[t], auto_reset=True, max_episode_steps=3)
                torch.cuda.synchronize()
    torch.cuda.synchronize()
    for a, b in zip(hs, tw):
        assert torch.equal(a.map, b.map) and torch.equal(a.pose, b.pose) and torch.equal(a.inventory, b.inventory)
        assert torch.equal(a.obs, b.obs) and torch.equal(a.episode, b.episode)
        ka, pa = a.rng_state()
        kb, pb = b.rng_state()
        assert np.array_equal(ka, kb) and np.array_equal(pa, pb)
        assert int(a.episode.min().item()) >= 2
    for hh in hs + tw:
        hh.close()


def test_switching_between_philox_and_numpy_and_back():
    """The episode counter runs on through numpy-stream resets; Philox resets afterwards are what a Philox-only handle
    produces at the same episode, and the numpy reset in between is the oracle's."""
    cc = _compiled(golden_util.get('pogo_limit_lidar')['meta'])
    n = 50
    h = BatchHandle([cc], n, seed=21)
    ref = BatchHandle([cc], n, seed=21)
    h.reset(); ref.reset()
    h.set_reset_rng('numpy')
    h.reset(); ref.reset()
    ors = OracleStream([cc], n, keys=np.stack([_np_state(21 + e)[0] for e in range(n)]),
                       pos=np.full(n, MT_WORDS, np.int32))
    _oracle_reset_all(ors)
    _assert_state(h, ors, "numpy reset")
    h.set_reset_rng('philox')
    with pytest.raises(RuntimeError, match="no np.random states"):
        h.rng_state()
    h.reset(); ref.reset()
    torch.cuda.synchronize()
    assert torch.equal(h.map, ref.map) and torch.equal(h.pose, ref.pose) and torch.equal(h.episode, ref.episode)
    h.close(); ref.close()


def test_error_paths_enqueue_nothing():
    cc = _compiled(golden_util.get('pogo_limit_lidar')['meta'])
    n = 40
    h = _numpy_handle([cc], n, seed=9)
    h.reset()
    torch.cuda.synchronize()
    key0, pos0 = h.rng_state()
    map0 = h.map.clone()
    lib, hp, s = h.lib, h._h, h._stream()
    count0 = h.launch_count()
    dk = torch.zeros((n, MT_WORDS), dtype=torch.int32, device='cuda')
    dp = torch.full((n,), 5, dtype=torch.int32, device='cuda')
    p = C.c_void_p
    assert lib.ngw_set_reset_rng(hp, 7, s) != 0
    dp[3] = 625
    assert lib.ngw_load_rng_state(hp, p(dk.data_ptr()), p(dp.data_ptr()), 0, n, s) != 0
    assert b"outside [0, 624]" in lib.ngw_last_error()
    dp[3] = -1
    assert lib.ngw_load_rng_state(hp, p(dk.data_ptr()), p(dp.data_ptr()), 0, n, s) != 0
    dp[3] = 5
    assert lib.ngw_load_rng_state(hp, p(dk.data_ptr()), p(dp.data_ptr()), 1, n, s) != 0
    assert lib.ngw_export_rng_state(hp, p(dk.data_ptr()), p(dp.data_ptr()), -1, 2, s) != 0
    assert lib.ngw_export_rng_state(hp, p(dk.data_ptr()), p(dp.data_ptr()), 0, n + 1, s) != 0
    torch.cuda.synchronize()
    assert h.launch_count() == count0
    key1, pos1 = h.rng_state()
    assert np.array_equal(key0, key1) and np.array_equal(pos0, pos1) and torch.equal(map0, h.map)
    # seeds numpy does not take: nothing is allocated or seeded, the Philox handle stays as it was
    big = BatchHandle([cc], n, seed=2 ** 32 - n + 1)
    c0 = big.launch_count()
    with pytest.raises(RuntimeError, match="below 2\\^32"):
        big.set_reset_rng('numpy')
    assert big.launch_count() == c0 and big.reset_rng == 'philox'
    with pytest.raises(RuntimeError, match="no np.random states"):
        big.rng_state()
    assert lib.ngw_load_rng_state(big._h, p(dk.data_ptr()), p(dp.data_ptr()), 0, n, s) != 0
    ok = BatchHandle([cc], n, seed=2 ** 32 - n)             # the largest batch that still fits
    ok.set_reset_rng('numpy')
    k, q = ok.rng_state(n - 1, 1)
    assert np.array_equal(k[0], _np_state(2 ** 32 - 1)[0])
    for hh in (h, big, ok):
        hh.close()


# ---------------------------------------------------------------------------------------------- 4. against numpy itself
def _oracle_after(cc, state, n_ops=None):
    """(map, pose, inventory, (key, pos)) of the reference reset of `cc` from np.random state `state`."""
    ors = OracleStream([cc], 1, keys=[np.asarray(state[1], np.uint32)], pos=[int(state[2])])
    rc, _ = ors.reset(0)
    return rc, ors.ob.map[0].copy(), ors.ob.pose[0].copy(), ors.state(0)


NUMPY_CHAINS = [
    ('plain', {'env': scenarios.POGO, 'map_size': 10, 'chain': [['limit', scenarios.C2_SET], ['lidar', 8]]}),
    ('crate', {'env': scenarios.POGO, 'map_size': 10, 'chain': [['lidar', 8], ['novelty', 'crate', 'hard', '', '']]}),
    ('remapaction', {'env': scenarios.POGO, 'map_size': 10,
                     'chain': [['lidar', 8], ['novelty', 'remapaction', 'hard', '', '']]}),
    ('axe_medium', {'env': scenarios.POGO, 'map_size': 10,
                    'chain': [['lidar', 8], ['novelty', 'axe', 'medium', 'wooden', '']]}),
    ('axetobreak_medium', {'env': scenarios.BOW, 'map_size': 10,
                           'chain': [['lidar', 8], ['novelty', 'axetobreak', 'medium', 'wooden', '']]}),
]


def _build_numpy_env(ns, desc, seed):
    """np.random.seed(seed); env = make(...); wrappers — construction-time draws included, no re-seeding between."""
    np.random.seed(seed)
    env = ns['make'](desc['env'], **({'reset_rng': 'numpy'} if ns is not None and ns.get('_b200') else {}))
    if desc.get('map_size', 10) != 10:
        env.map_size = desc['map_size']
    for step in desc['chain']:
        if step[0] == 'limit':
            env = ns['LimitActions'](env, set(step[1]))
        elif step[0] == 'lidar':
            env = ns['LidarInFront'](env, num_beams=step[1])
        else:
            env = ns['inject_novelty'](env, step[1], step[2], step[3], step[4])
    return env


def _b200_ns():
    ns = dict(scenarios.b200_namespace())
    ns['_b200'] = True
    return ns


@pytest.mark.parametrize('case', [c for c, _ in NUMPY_CHAINS])
def test_single_env_reset_follows_the_global_np_random(case):
    """num_envs == 1 on the numpy stream: after np.random.seed(s), make and wrappers, reset() gives the oracle's map from
    the global state and leaves np.random.get_state() where the oracle's reset leaves it; the next np.random.randint
    returns what it returns after the reference's reset.  AxeMedium / AxetoBreakMedium run the base env's reset at
    construction (add_new_items); that consumes the same draws the reference's does."""
    desc = dict(NUMPY_CHAINS)[case]
    for seed in (0, 11, 2024):
        if case in ('axe_medium', 'axetobreak_medium'):
            # the construction-time reset of the base env with its tables as add_new_items leaves them
            np.random.seed(seed)
            env = _build_numpy_env(_b200_ns(), {'env': desc['env'], 'chain': desc['chain'][:-1]}, seed)
            before = np.random.get_state()
            env = _build_numpy_env(_b200_ns(), desc, seed)
            after_build = np.random.get_state()
            rc, _, _, (k, p) = _oracle_after(compile_chain(env.unwrapped), before)
            assert rc == 0 and after_build[2] == p and np.array_equal(np.asarray(after_build[1], np.uint32), k), seed
        else:
            env = _build_numpy_env(_b200_ns(), desc, seed)
        state = np.random.get_state()
        env.reset()
        rc, m, pose, (k, p) = _oracle_after(compile_chain(env), state)
        assert rc == 0
        base = env.unwrapped
        assert np.array_equal(np.asarray(base.map, np.int8).reshape(-1), m), (case, seed)
        assert tuple(base.agent_location) == (int(pose[0]), int(pose[1])) and base.agent_facing_id == int(pose[2])
        now = np.random.get_state()
        assert now[2] == p and np.array_equal(np.asarray(now[1], np.uint32), k), (case, seed)
        expect = np.random.RandomState()
        expect.set_state(('MT19937', k, p, state[3], state[4]))
        assert np.random.randint(0, 10 ** 6) == expect.randint(0, 10 ** 6)
        env.close()


@pytest.mark.skipif(scenarios.reference_root() is None, reason="the reference package is not available here")
@pytest.mark.parametrize('case', [c for c, _ in NUMPY_CHAINS])
def test_single_env_reset_equals_the_unmodified_reference_in_process(case):
    desc = dict(NUMPY_CHAINS)[case]
    ref_ns = scenarios.reference_namespace()
    for seed in (3, 77):
        ref = _build_numpy_env(ref_ns, desc, seed)
        ref.reset()
        ref_map = np.array(ref.unwrapped.map, np.int64)
        ref_state = np.random.get_state()
        ours = _build_numpy_env(_b200_ns(), desc, seed)
        ours.reset()
        assert np.array_equal(np.asarray(ours.unwrapped.map, np.int64), ref_map), (case, seed)
        st = np.random.get_state()
        assert st[2] == ref_state[2] and np.array_equal(st[1], ref_state[1]), (case, seed)
        ours.close()
