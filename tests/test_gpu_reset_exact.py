"""The device's map generator and random policy bit for bit against their CPU restatement (oracle/ngw_oracle.c, last
section; run on the B200 box: pytest -m gpu).  Every case predicts the whole state from the seed alone — map, pose,
inventory, episode word, episode length, error flags — and the observation rows in the handle's layout, on every entry
point that regenerates an env: ngw_reset (one launch, or the three-launch split when the observation is taken between
the ops), the queued auto-reset behind every one-step kernel shape, ngw_step_many and ngw_step_host, and the in-place
resets of both rollout kernels.  The GPU state is never loaded into the CPU twin.  Counters straddle 2^32 (env ids)
and wrap (episode words), and both words of every seed are non-zero."""
import os

import numpy as np
import pytest
import torch

import golden_util
import scenarios
from gym_novel_gridworlds_b200.runtime import BatchHandle, StepGroup
from oracle.oracle_lib import OracleBatch, policy_draw, policy_draws
from test_gpu_kernel_routing import ROUTES, _inputs
from test_gpu_messages_stats import ROLLOUT_CASES
from test_gpu_parity import C2_DESC, _c4_descs, _compiled, rollout_case_inputs
from test_obs_hits_format import encode_hits
from test_philox_restatement import LEMIRE_ACCEPT, LEMIRE_REJECT, overfilled

pytestmark = pytest.mark.gpu

SEED = 0x9E3779B97F4A7C15
POLICY_SEED = 0x5DEECE66D2545F49  # the seed LEMIRE_* were found for
T = 3                             # max_episode_steps of the one-step cases
EPISODES = np.array([0x7FFFFFFE, 0x7FFFFFFF, 0x80000000, 0xFFFFFFFE, 0xFFFFFFFF], np.uint32)   # episode words before a reset


def _meta(name):
    return golden_util.get(name)['meta']


def _additem64():
    return _compiled({'env': scenarios.POGO, 'map_size': 64, 'chain': [['limit', scenarios.C2_SET], ['lidar', 8],
                                                                        ['novelty', 'additem', 'hard', 'spring', '']]})


# case -> (compiled configs, n, cfg_id, events that must occur)
def reset_case(case):
    one = {'C2': C2_DESC, 'Bow-v1': {'env': scenarios.BOW, 'map_size': 10, 'chain': [['lidar', 8]]},
           'no-lidar': {'env': scenarios.POGO, 'map_size': 10, 'chain': []}}
    if case in one:
        return [_compiled(one[case])], 2048, None, ()
    if case == 'c4-mixed':
        n = 32 * 40 + 5
        return [_compiled(d) for d in _c4_descs()], n, (np.arange(n) % 4).astype(np.uint8), ('list',)
    if case == 'additem-64':
        return [_additem64()], 48, None, ('list',)
    if case == 'axe-crowded':
        return [_compiled(_meta('pogo_A_axe_hard_iron_inc'))], 20000, None, ('place_fail',)
    if case == 'overfilled':
        return [overfilled(_compiled(_meta('pogo_A_axe_hard_iron_inc')))], 131072, None, ('place_fail', 'fallback')
    cc = _compiled(_meta(case))
    whole = ('pogo_A_fence_hard', 'bow0_C_firewall_hard')     # 90-100 % of a handful of candidates: the bin wins whole
    must = () if case == 'pogo0_lidar' else ('all_win',) if case in whole else ('list',)
    return [cc], 256 if cc.map_size > 20 else 2048, None, must


RESET_CASES = ['C2', 'Bow-v1', 'pogo0_lidar', 'pogo_A_fence_hard', 'pogo_A_additem_hard', 'pogo_A_replaceitem_medium_log',
               'pogo_A_crate_hard', 'bow0_C_firewall_hard', 'pogo_ms40_additem_hard', 'additem-64', 'axe-crowded',
               'overfilled', 'c4-mixed', 'no-lidar']


def _handle(compiled, n, cfg_id=None, seed=SEED, first_gid=None, fmt='i32', key_mask=None):
    if key_mask is not None:
        os.environ['NGW_DEBUG_KEY_MASK'] = hex(key_mask)
    try:
        h = BatchHandle(compiled, n, seed=seed, first_env_gid=(1 << 32) - n // 2 if first_gid is None else first_gid,
                        cfg_id=None if cfg_id is None else np.asarray(cfg_id).astype(np.int32), obs_format=fmt)
    finally:
        os.environ.pop('NGW_DEBUG_KEY_MASK', None)
    return h


def _u32(t):
    return t.cpu().numpy().view(np.uint32)


def _rows(h, vec, cfg_id):
    """The oracle's observation vectors -> the rows the handle must hold (layout and zero padding included)."""
    n, width = h.n, h.obs.shape[1]
    if h.obs_format == 'i32':
        out = np.zeros((n, width), np.int32)
        out[:, :vec.shape[1]] = vec
        return out
    out = np.zeros((n, width), np.uint8)
    ids = np.zeros(n, np.int64) if cfg_id is None else np.asarray(cfg_id, np.int64)
    for k, cc in enumerate(h.compiled):
        sel = ids == k
        c = cc.c
        if not sel.any() or c.n_beams == 0:
            continue
        if h.obs_format == 'hits':
            out[sel, :h.obs_row_bytes] = encode_hits(vec[sel, :cc.obs_dim], c, h.obs_row_bytes)
        else:
            lb, ni = c.n_lidar_items * c.n_beams, c.n_inv_obs
            off = (lb + 3) & ~3
            out[sel, :lb] = vec[sel, :lb]
            out[sel, off:off + 4 * ni] = vec[sel, lb:lb + ni].astype('<i4').view(np.uint8).reshape(-1, 4 * ni)
    return out


class Twin(object):
    """The CPU prediction of one handle from its seed: oracle steps and restated resets."""

    def __init__(self, h, compiled, cfg_id=None, key_mask=0xFFFFFFFF, policy_seed=0):
        self.h, self.n, self.cfg_id = h, h.n, cfg_id
        self.ob = OracleBatch(compiled, h.n, cfg_id=cfg_id)
        assert self.ob.inv_stride == h.inv_stride and self.ob.obs_dim == h.obs_dim
        self.seed, self.first_gid = SEED, (1 << 32) - h.n // 2
        self.key_mask = key_mask
        self.episode = np.zeros(self.n, np.uint32)
        self.ep_len = np.zeros(self.n, np.int32)
        self.err = np.zeros(self.n, np.uint32)
        self.obs = np.zeros((self.n, h.obs_dim), np.int32)
        ids = np.zeros(self.n, np.int64) if cfg_id is None else np.asarray(cfg_id, np.int64)
        self.n_act = np.array([cc.c.n_actions for cc in compiled])[ids]
        self.events = dict.fromkeys(('resets', 'truncations', 'split'), 0)

    def preset(self, rng, err_bits=0):
        """Episode words near 2^31 and 2^32 - 1, and (err_bits) stale error bits, on the handle and the twin alike."""
        self.episode = rng.choice(EPISODES, self.n)
        self.h.episode.copy_(torch.from_numpy(self.episode.view(np.int32)).cuda())
        if err_bits:
            self.err = np.where(rng.rand(self.n) < 0.5, err_bits, 0).astype(np.uint32)
            self.h.error_flags.copy_(torch.from_numpy(self.err.view(np.int32)).cuda())

    def _regenerate(self, sel, k_obs, want_obs):
        ep = self.episode + np.uint32(1)
        flags, obs, ev = self.ob.reset_philox(self.seed, self.first_gid, ep, self.key_mask, k_obs, sel, want_obs)
        for k, v in ev.items():
            self.events[k] = self.events.get(k, 0) + v
        self.episode = np.where(sel, ep, self.episode)
        self.events['resets'] += int(sel.sum())
        return flags, obs

    def reset(self, mask=None, want_obs=True):
        """ngw_reset: the reset ASSIGNS the env's error flags and zeroes ep_len."""
        sel = np.ones(self.n, bool) if mask is None else np.asarray(mask, bool)
        flags, obs = self._regenerate(sel, None, want_obs)
        self.err = np.where(sel, flags, self.err)
        self.ep_len[sel] = 0
        if obs is not None:
            self.obs[sel] = obs[sel]
            self.events['split'] += int(sum(cc.c.reset_obs_after_ops < cc.c.n_reset_ops for cc in self.ob.compiled))
        return obs

    def step(self, a, limit, k_obs=None, want_obs=True):
        """One valid step with auto-reset and truncation at `limit`; finished envs are regenerated and OR their flags."""
        obs, rew, term, cost, res = self.ob.step(a, n_threads=8, want_obs=want_obs)
        term = term.astype(bool)
        length = self.ep_len + 1
        fin = term | (length >= limit)
        self.ep_len = np.where(fin, 0, length).astype(np.int32)
        self.events['truncations'] += int((fin & ~term).sum())
        if fin.any():
            flags, robs = self._regenerate(fin, k_obs, want_obs and self.h.obs_dim > 0)
            self.err |= flags
            if robs is not None:
                obs[fin] = robs[fin]
        if obs is not None:
            self.obs = obs
        return rew, fin.astype(np.uint8), cost, res

    def actions(self, rng):
        return (rng.randint(0, 1 << 30, size=self.n) % self.n_act).astype(np.int32)

    def check(self, where, obs_rows=None):
        h, n = self.h, self.n
        m, p, v = h.export_state()
        assert np.array_equal(m.reshape(n, -1).cpu().numpy(), self.ob.map), "%s: map, %d envs differ" % (
            where, int((m.reshape(n, -1).cpu().numpy() != self.ob.map).any(1).sum()))
        assert np.array_equal(p.cpu().numpy(), self.ob.pose), where + ": pose"
        assert np.array_equal(v.cpu().numpy(), self.ob.inv), where + ": inventory"
        assert np.array_equal(_u32(h.episode), self.episode), where + ": episode"
        assert np.array_equal(h.ep_len.cpu().numpy(), self.ep_len), where + ": ep_len"
        assert np.array_equal(_u32(h.error_flags), self.err), where + ": error flags"
        if h.obs_dim:
            got = h.obs.cpu().numpy() if obs_rows is None else np.asarray(obs_rows)
            assert np.array_equal(got, _rows(h, self.obs, self.cfg_id)), where + ": observation rows"


def _reset_round(h, twin, rng, where, obs=True):
    """ngw_reset of all envs, then of a random mask (the other envs keep every byte, observation rows included)."""
    twin.reset(want_obs=obs)
    h.reset(want_obs=obs)
    twin.check(where + " all")
    mask = rng.rand(h.n) < 0.4
    twin.reset(mask, want_obs=obs)
    h.reset(mask=torch.from_numpy(mask.astype(np.uint8)).cuda(), want_obs=obs)
    twin.check(where + " masked")


@pytest.mark.parametrize('case', RESET_CASES)
def test_ngw_reset_equals_the_restatement(case):
    """ngw_reset with and without an observation, all envs and masked; i32 rows everywhere, u8 and hits rows on C2, a
    split config and the mixed batch.  Stale error bits are cleared: ngw_reset assigns the flags."""
    compiled, n, cfg_id, must = reset_case(case)
    rng = np.random.RandomState(RESET_CASES.index(case))
    for fmt in ('i32', 'u8', 'hits') if case in ('C2', 'pogo_A_fence_hard', 'c4-mixed') else ('i32',):
        h = _handle(compiled, n, cfg_id, fmt=fmt)
        twin = Twin(h, compiled, cfg_id)
        twin.preset(rng, err_bits=0x100)
        for obs in (True, False):
            _reset_round(h, twin, rng, "%s %s obs=%s" % (case, fmt, obs), obs)
        for ev in must:
            assert twin.events[ev] > 0, (ev, twin.events)
        if any(cc.c.reset_obs_after_ops < cc.c.n_reset_ops for cc in compiled):
            assert twin.events['split'] > 0
        h.close()


def test_split_reset_keeps_the_placement_flag_of_the_ops_after_the_observation():
    """pogo0_lidar with ONE tree log and the observation taken before TREETAP: ngw_reset runs the op in its third launch
    (phase 1), where it must fail, and that launch must keep the PLACEMENT flag; the queued auto-reset ORs it in too."""
    cc = _compiled(_meta('pogo0_lidar'))
    log = cc.item_names.index('tree_log')
    cc.c.place_qty[list(cc.c.place_item[:cc.c.n_place]).index(log)] = 1
    cc.c.reset_obs_after_ops = 0
    n = 512
    h = _handle([cc], n)
    twin = Twin(h, [cc])
    rng = np.random.RandomState(3)
    twin.preset(rng, err_bits=0x100)
    _reset_round(h, twin, rng, "one log")
    assert (twin.err == 2).all() and twin.events['treetap_fail'] > 0 and twin.events['split'] > 0
    twin.preset(rng, err_bits=0x100)
    for t in range(T):
        a = twin.actions(rng)
        twin.step(a, T)
        h.step(torch.from_numpy(a).cuda(), auto_reset=True, max_episode_steps=T)
        twin.check("one log, step %d" % t)
    assert set(np.unique(twin.err)) == {2, 0x102}


def _run_steps(hs, twins, rng, steps, where, how='step'):
    for t in range(steps):
        acts = [tw.actions(rng) for tw in twins]
        want = [tw.step(a, T) for tw, a in zip(twins, acts)]
        if how == 'many':
            StepGroup(hs).step([torch.from_numpy(a).cuda() for a in acts], auto_reset=True, max_episode_steps=T)
        for k, (h, tw, a, w) in enumerate(zip(hs, twins, acts, want)):
            rows = None
            if how == 'host':
                out = h.step_host(a, auto_reset=True, max_episode_steps=T)
                rows, got = out[0], out[1:]
            else:
                if how == 'step':
                    h.step(torch.from_numpy(a).cuda(), auto_reset=True, max_episode_steps=T)
                got = [x.cpu().numpy() for x in (h.reward, h.done, h.step_cost, h.result)]
            tw.check("%s handle %d step %d" % (where, k, t), rows)
            assert np.array_equal(got[0], w[0]) and np.array_equal(got[1], w[1]) and np.array_equal(got[3], w[3])
            np.testing.assert_allclose(got[2], w[2], rtol=1e-6)
    for tw in twins:
        assert tw.events['resets'] > tw.n and tw.events['truncations'] > 0, tw.events


def _stepping(compiled, n, cfg_id, rng, key_mask=None):
    h = _handle(compiled, n, cfg_id, key_mask=key_mask)
    twin = Twin(h, compiled, cfg_id, key_mask=0xFFFFFFFF if key_mask is None else key_mask)
    twin.preset(rng, err_bits=0x100)
    twin.reset()
    h.reset()
    twin.check("initial reset")
    twin.preset(rng, err_bits=0x100)            # the auto-resets wrap the episode word and OR into stale bits
    return h, twin


@pytest.mark.parametrize('case', sorted(ROUTES))
def test_one_step_auto_reset_equals_the_restatement(case):
    """Every one-step kernel shape with auto-reset and truncation: each finished env is regenerated by reset_list_kernel
    at episode + 1, its observation row taken after reset_obs_after_ops ops."""
    compiled, n, cfg_id = _inputs(case)
    rng = np.random.RandomState(5)
    h, twin = _stepping(compiled, n, cfg_id, rng)
    _run_steps([h], [twin], rng, 2 * T + 1, case)


def test_step_many_and_host_path_auto_reset_equal_the_restatement():
    """ngw_step_many over two handles of different kernels (C2 on the warp-per-tile kernel, map 40 AddItem), and
    ngw_step_host."""
    rng = np.random.RandomState(6)
    specs = [([_compiled(C2_DESC)], 32 * 37 + 5, None), ([_compiled(_meta('pogo_ms40_additem_hard'))], 32 * 3 + 5, None)]
    pairs = [_stepping(c, n, i, rng) for c, n, i in specs]
    _run_steps([p[0] for p in pairs], [p[1] for p in pairs], rng, 2 * T + 1, 'step_many', how='many')
    compiled, n, cfg_id = [_compiled(d) for d in _c4_descs()], 32 * 9 + 3, (np.arange(32 * 9 + 3) % 4).astype(np.uint8)
    h, twin = _stepping(compiled, n, cfg_id, rng)
    _run_steps([h], [twin], rng, 2 * T + 1, 'step_host', how='host')


@pytest.mark.parametrize('key_mask', [0x3, 0x0])
def test_tied_keys_follow_the_restated_order(key_mask):
    """NGW_DEBUG_KEY_MASK keeps 2 key bits or none: boundary ties of more than 32 candidates are decided by arrival
    order (with mask 0 every key is equal, so the winners are the first in arrival order), smaller ties by cell index.
    ngw_reset (all, masked, split) and the queued auto-reset.  (The rollouts' in-place resets keep every key bit.)"""
    rng = np.random.RandomState(key_mask + 11)
    for compiled, n, cfg_id in (([_compiled(_meta('pogo_ms40_additem_hard'))], 32 * 4 + 5, None),
                                ([_compiled(_meta('pogo_A_fence_hard'))], 1024, None),
                                ([_compiled(d) for d in _c4_descs()], 32 * 20 + 5, (np.arange(32 * 20 + 5) % 4).astype(np.uint8))):
        h = _handle(compiled, n, cfg_id, key_mask=key_mask)
        twin = Twin(h, compiled, cfg_id, key_mask=key_mask)
        twin.preset(rng)
        _reset_round(h, twin, rng, "mask %#x" % key_mask)
        h.reset(); twin.reset()
        _run_steps([h], [twin], rng, T + 1, "mask %#x" % key_mask)
        if compiled[0].map_size == 40:
            assert twin.events['arrival'] > 0, twin.events
        if len(compiled) > 1:                   # ~58 air cells of a 10x10 grid: 2 key bits leave ~15 per key, a list
            assert twin.events['list' if key_mask else 'arrival'] > 0, twin.events


def _rollout_case(compiled, n, cfg_id, first_gid, K, mode, rng, limit=5):
    """One K-step rollout with auto-reset and truncation against a CPU rollout of restated draws (random policy) or the
    given actions, oracle steps and restated resets (after all ops, as the rollouts regenerate in place)."""
    h = _handle(compiled, n, cfg_id, first_gid=first_gid)
    twin = Twin(h, compiled, cfg_id)
    twin.first_gid = first_gid
    twin.preset(rng)
    twin.reset()
    h.reset()
    twin.preset(rng, err_bits=0x100)
    if mode == 'random':
        acts, branch = policy_draws(POLICY_SEED, first_gid, twin.n_act, K)
        out = h.rollout(K, None, policy_seed=POLICY_SEED, auto_reset=True, max_episode_steps=limit, record_actions=True)
        assert np.array_equal(out[-1].cpu().numpy(), acts), "actions_out"
    else:
        acts, branch = np.stack([twin.actions(rng) for _ in range(K)]), None
        out = h.rollout(K, torch.from_numpy(acts).cuda(), auto_reset=True, max_episode_steps=limit)
    rew = np.zeros(n, np.float32)
    cost = np.zeros(n, np.float32)
    dones = np.zeros(n, np.int32)
    for t in range(K):
        r, d, c, res = twin.step(acts[t], limit, k_obs=8, want_obs=False)
        rew += r; cost += c; dones += d
    if h.obs_dim:
        twin.obs = twin.ob.observe()
    twin.check("rollout %s" % mode, out[0].cpu().numpy() if h.obs_dim else None)
    assert np.array_equal(out[1].cpu().numpy(), rew) and np.array_equal(out[3].cpu().numpy(), dones)
    assert np.array_equal(out[4].cpu().numpy(), d) and np.array_equal(out[5].cpu().numpy(), res)
    np.testing.assert_allclose(out[2].cpu().numpy(), cost, rtol=1e-5)
    assert twin.events['resets'] > n and twin.events['truncations'] > 0, twin.events
    h.close()
    return acts, branch


@pytest.mark.parametrize('mode', ['random', 'given'])
@pytest.mark.parametrize('case', ROLLOUT_CASES)
def test_rollouts_equal_the_restatement(case, mode):
    """Both rollout kernels (lane-pair kernel up to 32x32, one warp per tile on 40x40 grids and 16 beams)."""
    compiled, n, cfg_id = rollout_case_inputs(case)
    _rollout_case(compiled, n, None if cfg_id is None else cfg_id.astype(np.uint8), (1 << 32) - n // 2, 12, mode,
                  np.random.RandomState(len(case)))


@pytest.mark.parametrize('kernel', ['rollout2', 'rollout'])
@pytest.mark.parametrize('which', ['reject', 'accept'])
def test_random_policy_lemire_branch_on_the_device(kernel, which):
    """A batch holding the env id whose draw at step t enters Lemire's threshold test (rejected and continued on stream
    0xFFE, or kept), run past t on the lane-pair kernel (C2, 10x10) and the one-warp-per-tile kernel (C2's actions on 40x40)."""
    seed, gid, t = LEMIRE_REJECT if which == 'reject' else LEMIRE_ACCEPT
    assert seed == POLICY_SEED
    desc = C2_DESC if kernel == 'rollout2' else dict(C2_DESC, map_size=40)
    n, e = 32 * 3 + 5, 37
    acts, branch = _rollout_case([_compiled(desc)], n, None, gid - e, t + 3, 'random', np.random.RandomState(t))
    assert branch[t, e] == (2 if which == 'reject' else 1) and acts[t, e] == policy_draw(seed, gid, t, 10)[0]
