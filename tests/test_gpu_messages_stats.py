"""info['message'] codes (ngw_set_message_buffer) and the episode statistics (ngw_stats) against the C oracle (run on the
B200 box: pytest -m gpu).  The oracle's codes are pinned to the reference's strings by tests/test_oracle_messages.py; here
every one-step kernel shape, the host path, ngw_step_many and both rollout kernels are compared with it, with invalid
action ids, envs that hold the goal item, auto-reset and truncation in every batch, and the calls that must leave the
message buffer and the counters alone are checked."""
import ctypes as C

import numpy as np
import pytest
import torch

import golden_util
import scenarios
from gym_novel_gridworlds_b200 import capi
from gym_novel_gridworlds_b200.runtime import BatchHandle, StepGroup, decode_message
from oracle.oracle_lib import OracleBatch
from test_gpu_episode_end import C5, _oracle_inputs
from test_gpu_kernel_routing import ROUTES, _inputs
from test_gpu_parity import C2_DESC, _c4_descs, _compiled, many_config_inputs, rollout_case_inputs

pytestmark = pytest.mark.gpu

STEPS, EPISODES, SUCCESSES, REWARD_SUM, COST_SUM, RESETS, INVALID, RESERVED = range(8)
EXACT = [STEPS, EPISODES, SUCCESSES, REWARD_SUM, RESETS, INVALID, RESERVED]
SENTINEL = 0x5A5A                 # kind 26: no code; fills the message buffer before a call, lanes nobody wrote keep it
T = 3                             # max_episode_steps of the auto-reset cases
WARP0_KINDS = {9, 10, 11}         # MISSING / NEED_TABLE / CRAFTED: crafts, stepped by warp 0 of a tile group
WARP1_KINDS = {1, 2, 7}           # BLOCK_IN_PATH / CANNOT_BREAK / NO_TAP: moves and block-in-front actions, warp 1


def _handle(compiled, n, cfg_id=None, seed=0):
    h = BatchHandle(compiled, n, seed=seed, cfg_id=None if cfg_id is None else np.asarray(cfg_id).astype(np.int32))
    h.enable_messages()
    return h


def _codes(h):
    return h.msg.cpu().numpy().view(np.uint16)


def _stats(h):
    """The counters since the last call (ngw_stats with reset_after)."""
    return h.stats(reset=True).cpu().numpy().copy()


class Mirror(object):
    """The oracle twin of one handle.  prepare() gives ~2 % of the envs the goal item (so that any valid action on them is
    a success), copies the handle's state into the oracle and draws actions with ~3 % invalid ids; expect() steps the oracle
    and returns the message codes and the counters the handle's step must produce."""

    def __init__(self, h, compiled, cfg_id=None):
        self.h, self.n = h, h.n
        self.ob = OracleBatch(compiled, h.n, cfg_id=cfg_id)
        assert self.ob.inv_stride == h.inv_stride
        ids = np.zeros(h.n, np.int64) if cfg_id is None else np.asarray(cfg_id, np.int64)
        self.n_act = np.array([cc.c.n_actions for cc in compiled])[ids]
        self.goal = np.array([cc.c.id_goal for cc in compiled])[ids]
        self.total = np.zeros(8)
        self.kinds = set()
        self.truncated = 0

    def give_goal(self, rng):
        won = rng.choice(self.n, max(1, self.n // 50), replace=False)
        self.h.inventory[torch.from_numpy(won).cuda(), torch.from_numpy(self.goal[won]).cuda()] = 1
        return won

    def load(self):
        m, p, v = self.h.export_state()
        self.ob.map[:] = m.reshape(self.n, -1).cpu().numpy()
        self.ob.pose[:] = p.cpu().numpy()
        self.ob.inv[:] = v.cpu().numpy()

    def actions(self, rng, invalid=True):
        a = (rng.randint(0, 1 << 30, size=self.n) % self.n_act).astype(np.int32)
        if invalid:                                           # negative ids and ids >= the env's n_actions
            bad = rng.choice(self.n, max(2, 3 * self.n // 100), replace=False)
            lo, hi = bad[::2], bad[1::2]
            a[lo] = -1 - rng.randint(0, 1000, size=lo.size)
            a[hi] = self.n_act[hi] + rng.randint(0, 1000, size=hi.size)
        return a

    def prepare(self, rng):
        self.h.msg.fill_(SENTINEL)
        self.give_goal(rng)
        self.load()
        self.ep_len = self.h.ep_len.cpu().numpy()
        return self.actions(rng)

    def expect(self, a, limit=0, auto_reset=True):
        """(codes, counters) of one oracle step; limit = max_episode_steps (0: none), ep_len from prepare()."""
        ob = self.ob
        ob.err[:] = 0
        _, rew, term, cost, _ = ob.step(a, n_threads=8, want_obs=False)
        invalid = (ob.err & 1) != 0
        valid = ~invalid
        term = term.astype(bool)
        done = term | (valid & (self.ep_len + 1 >= limit)) if limit > 0 else term
        st = np.zeros(8)
        st[STEPS] = valid.sum()
        st[EPISODES] = done.sum()
        st[SUCCESSES] = (valid & (ob.inv[np.arange(self.n), self.goal] >= 1)).sum()
        st[REWARD_SUM] = rew.astype(np.float64).sum()
        st[COST_SUM] = cost.astype(np.float64).sum()
        st[RESETS] = done.sum() if auto_reset else 0
        st[INVALID] = invalid.sum()
        self.total += st
        self.truncated += int((done & ~term).sum())
        self.kinds |= set(int(k) for k in np.unique(ob.msg & 31))
        return ob.msg.copy(), st

    def check(self, where, a, limit=T, auto_reset=True):
        """The handle's codes and counters after the step it took with actions `a`."""
        codes, st = self.expect(a, limit, auto_reset)
        got = _codes(self.h)
        assert np.array_equal(got, codes), "%s: %d of %d codes differ, e.g. env %d: %#x vs %#x" % (
            where, int((got != codes).sum()), self.n, *_first_diff(got, codes))
        _same_stats(where, _stats(self.h), st)

    def assert_bites(self, both_warps=False):
        assert self.total[SUCCESSES] > 0 and self.total[INVALID] > 0, self.total
        assert self.total[RESETS] > 0 and self.truncated > 0, (self.total, self.truncated)
        if both_warps:
            assert self.kinds & WARP0_KINDS and self.kinds & WARP1_KINDS, sorted(self.kinds)


def _first_diff(got, want):
    i = int(np.nonzero(got != want)[0][0])
    return i, int(got[i]), int(want[i])


def _same_stats(where, got, want):
    """Counts and the reward sum exactly; the cost sum to float rounding (the kernels add float partials per warp and CTA)."""
    assert np.array_equal(got[EXACT], want[EXACT]), "%s: %s vs %s" % (where, got.tolist(), want.tolist())
    np.testing.assert_allclose(got[COST_SUM], want[COST_SUM], rtol=1e-5, err_msg=where)


def _step_inputs(case):
    if case.startswith('configs-'):                     # NC = 16 inline configs (6) and the global table (20)
        return many_config_inputs(int(case.split('-')[1]))
    return _oracle_inputs(case)                         # ROUTES, the FireWall chain and C5 (map 40)


@pytest.mark.parametrize('case', sorted(ROUTES) + ['firewall', 'C5', 'configs-6', 'configs-20'])
def test_step_messages_and_stats_against_the_oracle(case):
    """Every one-step kernel shape (full and partial tiles, several tiles per CTA, several waves, mixed configs): at every
    step the message codes equal the oracle's on every env, and the counters ngw_stats returns equal a count made from the
    oracle's outputs: steps and invalid lanes, episodes = terminated | truncated on valid lanes, successes, reward and
    cost sums, resets."""
    compiled, n, cfg_id = _step_inputs(case)
    h = _handle(compiled, n, cfg_id, seed=31)
    h.reset()
    mirror = Mirror(h, compiled, cfg_id)
    rng = np.random.RandomState(41)
    for t in range(8):
        a = mirror.prepare(rng)
        h.step(torch.from_numpy(a).cuda(), auto_reset=True, max_episode_steps=T)
        mirror.check("%s step %d" % (case, t), a)
    mirror.assert_bites(both_warps=case[:2] in ('G2', 'G4'))


@pytest.mark.parametrize('case', ['warp-3', 'G2-multi'])
def test_host_path_messages_and_stats_against_the_oracle(case):
    """ngw_step_host and ngw_step_host_begin / _end write the same codes and counters as the oracle's."""
    compiled, n, cfg_id = _inputs(case)
    hosts = [_handle(compiled, n, cfg_id, seed=5) for _ in range(2)]
    mirrors = [Mirror(h, compiled, cfg_id) for h in hosts]
    for h in hosts:
        h.reset()
    rng = np.random.RandomState(6)
    for t in range(7):
        for k, (h, mirror) in enumerate(zip(hosts, mirrors)):
            a = mirror.prepare(rng)
            if k == 0:
                h.step_host(a, auto_reset=True, max_episode_steps=T)
            else:
                h.step_host_begin(a, auto_reset=True, max_episode_steps=T)
                h.step_host_end()
            mirror.check("%s %s step %d" % (case, ('step_host', 'begin/end')[k], t), a)
    for mirror in mirrors:
        mirror.assert_bites()


ROLLOUT_CASES = ['pogo_ms23', 'c4_mixed', 'pogo_ms40', 'bow12_16beams']    # rollout2_kernel x 2, rollout_kernel x 2


@pytest.mark.parametrize('case', ROLLOUT_CASES)
def test_rollout_messages_and_stats_against_the_oracle(case):
    """A K-step rollout with the device's random policy, its actions recorded and replayed through the oracle: the final
    codes are the oracle's last-step codes, the counters the sum of the oracle's per-step counts.  ~2 % of the envs hold
    the goal item, so every one of their steps is a success and ends an episode."""
    compiled, n, cfg_id = rollout_case_inputs(case)
    h = _handle(compiled, n, cfg_id, seed=12)
    h.reset()
    mirror = Mirror(h, compiled, cfg_id)
    rng = np.random.RandomState(13)
    K = 12
    for rnd, kw in enumerate([dict(policy_seed=7)] + ([dict(policy=_policy(h, compiled, rng))] if case == 'pogo_ms23' else [])):
        mirror.give_goal(rng)
        mirror.load()
        h.msg.fill_(SENTINEL)
        taken = h.rollout(K, record_actions=True, **kw)[-1].cpu().numpy()
        want = np.zeros(8)
        for t in range(K):
            codes, st = mirror.expect(taken[t], limit=0, auto_reset=False)
            want += st
        where = "%s %s" % (case, 'closed loop' if 'policy' in kw else 'random policy')
        got = _codes(h)
        assert np.array_equal(got, codes), "%s: %d codes differ, e.g. env %d: %#x vs %#x" % (
            where, int((got != codes).sum()), *_first_diff(got, codes))
        _same_stats(where, _stats(h), want)
        assert want[SUCCESSES] > 0 and want[EPISODES] > 0, want
        m, p, v = h.export_state()
        assert np.array_equal(m.reshape(n, -1).cpu().numpy(), mirror.ob.map) and np.array_equal(v.cpu().numpy(), mirror.ob.inv)


def _policy(h, compiled, rng):
    A = max(cc.c.n_actions for cc in compiled)
    assert A <= 16
    return (rng.randint(-9, 10, size=(h.obs_dim, A)).astype(np.int32), rng.randint(-30, 31, size=A).astype(np.int32))


@pytest.mark.parametrize('case', ROLLOUT_CASES)
def test_rollout_with_auto_reset_equals_the_sum_of_one_step_counters(case):
    """Given actions with invalid ids, auto-reset and truncation inside one rollout: the counters equal the sum of what a
    one-step twin (tied to the oracle by the tests above) counts step by step, and the final codes are the twin's."""
    compiled, n, cfg_id = rollout_case_inputs(case)
    roll, twin = _handle(compiled, n, cfg_id, seed=8), _handle(compiled, n, cfg_id, seed=8)
    mirror = Mirror(roll, compiled, cfg_id)
    rng = np.random.RandomState(9)
    won = rng.choice(n, max(1, n // 50), replace=False)
    for h in (roll, twin):
        h.reset()
        h.inventory[torch.from_numpy(won).cuda(), torch.from_numpy(mirror.goal[won]).cuda()] = 1
    K = 10
    acts = torch.from_numpy(np.stack([mirror.actions(rng) for _ in range(K)])).cuda()
    roll.msg.fill_(SENTINEL)
    roll.rollout(K, acts, auto_reset=True, max_episode_steps=T)
    want = np.zeros(8)
    for t in range(K):
        twin.step(acts[t], auto_reset=True, max_episode_steps=T)
        want += _stats(twin)
    assert np.array_equal(_codes(roll), _codes(twin)), case
    _same_stats(case, _stats(roll), want)
    assert want[SUCCESSES] > 0 and want[INVALID] > 0 and want[RESETS] > 0 and want[EPISODES] == want[RESETS], want
    assert torch.equal(roll.episode, twin.episode) and torch.equal(roll.ep_len, twin.ep_len)


def test_step_group_messages_stats_and_overlap():
    """ngw_step_many over handles that take different kernels, each with its own message buffer: the launches overlap as
    before and every handle's codes and counters equal its oracle's.  Two handles that share one message buffer are never
    overlapped: the buffer is in the launch's write set."""
    specs = [([_compiled(C2_DESC)], 32 * 70 + 3, None),
             ([_compiled(golden_util.get(C5)['meta'])], 32 * 6 + 1, None),
             ([_compiled({'env': scenarios.BOW, 'map_size': 12, 'chain': [['lidar', 16]]})], 300, None),
             ([_compiled(d) for d in _c4_descs()], 32 * 40 + 5, (np.arange(32 * 40 + 5) % 4).astype(np.int32))]
    hs = [_handle(compiled, n, cfg_id, seed=300 + k) for k, (compiled, n, cfg_id) in enumerate(specs)]
    mirrors = [Mirror(h, compiled, cfg_id) for h, (compiled, n, cfg_id) in zip(hs, specs)]
    for h in hs:
        h.reset()
    group = StepGroup(hs)
    rng = np.random.RandomState(10)
    c0 = sum(h.concurrent_launch_count() for h in hs)
    rounds = 7
    for rnd in range(rounds):
        acts = [torch.from_numpy(m.prepare(rng)).cuda() for m in mirrors]
        group.step(acts, auto_reset=True, max_episode_steps=T)
        for k, m in enumerate(mirrors):
            m.check("round %d handle %d" % (rnd, k), acts[k].cpu().numpy())
    assert sum(h.concurrent_launch_count() for h in hs) - c0 == rounds * (len(hs) - 1)
    for m in mirrors:
        m.assert_bites()

    A, B = hs[0], hs[2]
    a = [torch.zeros(h.n, dtype=torch.int32, device='cuda') for h in (A, B)]
    pair = StepGroup([A, B])
    for shared in (False, True):
        if shared:
            capi.check(B.lib, B.lib.ngw_set_message_buffer(B._h, C.c_void_p(A.msg.data_ptr())))
        c0 = A.concurrent_launch_count() + B.concurrent_launch_count()
        pair.step(a)
        assert A.concurrent_launch_count() + B.concurrent_launch_count() - c0 == (0 if shared else 1), shared
    B.enable_messages()


def test_calls_that_leave_the_message_buffer_and_the_counters_alone():
    """ngw_observe, ngw_reset (all envs and masked), ngw_load_state, ngw_export_state and ngw_stats write no message code
    and count nothing; after enable_messages(False) neither a step nor a rollout touches the tensor that was enabled."""
    cc = _compiled(C2_DESC)
    n = 32 * 40 + 9
    h = _handle([cc], n, seed=8)

    def quiet_calls():
        h.msg.fill_(SENTINEL)
        h.reset()
        h.observe()
        h.reset(mask=(torch.arange(n, device='cuda') % 3 == 0))
        h.load_state(*h.export_state())
        h.observe()
        first = h.stats().cpu().numpy().copy()
        torch.cuda.synchronize()
        assert (_codes(h) == SENTINEL).all()
        assert not first.any() and not _stats(h).any()

    quiet_calls()
    a = torch.from_numpy(np.random.RandomState(1).randint(0, cc.c.n_actions, size=n).astype(np.int32)).cuda()
    h.step(a, auto_reset=True, max_episode_steps=2)
    st = _stats(h)
    assert st[STEPS] == n and not (_codes(h) == SENTINEL).any()
    quiet_calls()                                                # counters were zeroed by the read above; still zero

    old = h.msg
    old.fill_(SENTINEL)
    h.enable_messages(False)
    assert h.msg is None
    h.step(a, auto_reset=True, max_episode_steps=2)
    h.rollout(4, policy_seed=3, auto_reset=True, max_episode_steps=2)
    torch.cuda.synchronize()
    assert (old.cpu().numpy().view(np.uint16) == SENTINEL).all()
    h.enable_messages().fill_(SENTINEL)
    h.step(a)
    assert not (_codes(h) == SENTINEL).any() and (old.cpu().numpy().view(np.uint16) == SENTINEL).all()


@pytest.mark.parametrize('path', ['device', 'numpy'])
def test_gym_api_messages_equal_the_oracle(path):
    """make(..., num_envs=n, messages=True): info['message'] holds the reference's strings of the oracle's codes, on the
    device path (CUDA actions) and on the host-buffer path (NumPy actions)."""
    import gym_novel_gridworlds_b200 as gym
    n = 1000
    env = gym.make('NovelGridworld-Pogostick-v1', num_envs=n, seed=7, auto_reset=True, max_episode_steps=5, messages=True)
    env = gym.LidarInFront(gym.LimitActions(env, set(scenarios.C2_SET)))
    env.reset()
    rt = env.unwrapped._runtime
    h, cc = rt.handle, rt.compiled
    mirror = Mirror(h, [cc])
    rng = np.random.RandomState(2)
    kinds = set()
    for t in range(12):
        mirror.load()
        a = mirror.actions(rng, invalid=False)
        mirror.ob.step(a, n_threads=8, want_obs=False)
        codes = mirror.ob.msg.copy()
        _, _, _, info = env.step(torch.from_numpy(a).cuda() if path == 'device' else a)
        got = info['message']
        assert got is not None, "%s step %d: no messages" % (path, t)
        assert list(got) == [decode_message(c, cc) for c in codes], "%s step %d" % (path, t)
        kinds |= set(int(k) for k in np.unique(codes & 31))
    assert len(kinds - {0}) >= 3, sorted(kinds)
