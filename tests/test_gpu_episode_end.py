"""Episode-end outputs of the one-step calls (ngw_set_episode_end_buffers; run on the B200 box: pytest -m gpu):
truncated flags (gym's TimeLimit rule) and the last observation of every auto-reset env, against the C oracle on every
one-step kernel shape, and on every path that writes them or must leave them alone."""
import ctypes as C
import json

import numpy as np
import pytest
import torch

import golden_util
import scenarios
from gym_novel_gridworlds_b200 import capi
from gym_novel_gridworlds_b200.runtime import BatchHandle, StepGroup, obs_to_vector
from oracle.oracle_lib import OracleBatch
from test_gpu_kernel_routing import ROUTES, _inputs
from test_gpu_parity import C2_DESC, _compiled

pytestmark = pytest.mark.gpu

SENTINEL = 0xA5                                  # fills final_obs / truncated before a step: rows nobody wrote keep it
FIREWALL = 'pogo_A_firewall_hard'                # FireWall kills the agent next to a fire wall: natural terminations
C5 = 'pogo_ms40_additem_hard'


def _handle(compiled, n, cfg_id=None, seed=0, fmt='i32', episode_end=True):
    h = BatchHandle(compiled, n, seed=seed, cfg_id=None if cfg_id is None else np.asarray(cfg_id).astype(np.int32),
                    obs_format=fmt)
    if episode_end:
        h.enable_episode_end()
    return h


def _n_act(compiled, n, cfg_id):
    ids = np.zeros(n, np.int64) if cfg_id is None else np.asarray(cfg_id, np.int64)
    return np.array([cc.c.n_actions for cc in compiled])[ids]


def _fill(h):
    h.truncated.fill_(SENTINEL)
    h.final_obs.view(torch.uint8).fill_(SENTINEL)


def _oracle_inputs(case):
    if case == 'firewall':
        return [_compiled(golden_util.get(FIREWALL)['meta'])], 32 * 60 + 7, None
    if case == 'C5':
        return [_compiled(golden_util.get(C5)['meta'])], 32 * 12 + 5, None
    return _inputs(case)


ORACLE_CASES = [(c, 'i32') for c in sorted(ROUTES) + ['firewall', 'C5']] + \
               [(c, f) for c in ('warp-3', 'G4-alias') for f in ('u8', 'hits')]


@pytest.mark.parametrize('case,fmt', ORACLE_CASES)
def test_episode_end_against_the_oracle(case, fmt):
    """Before every step the GPU state and ep_len go to the oracle, which steps without truncation; the GPU steps with
    auto-reset and max_episode_steps T.  done == terminated | (ep_len + 1 >= T), truncated only where the env did not
    terminate, final_obs == the oracle's observation on every done row (byte for byte against a twin stepped without
    auto-reset: narrow rows too), every other row keeps its sentinel.  Half of the envs the oracle sees terminate are put
    one step before the limit, so terminating on the limit's step is covered: it must report terminated."""
    compiled, n, cfg_id = _oracle_inputs(case)
    T = 4
    h = _handle(compiled, n, cfg_id, seed=17, fmt=fmt)
    twin = _handle(compiled, n, cfg_id, seed=17, fmt=fmt, episode_end=False)     # the same step without auto-reset
    h.reset()
    ob = OracleBatch(compiled, n, cfg_id=cfg_id)
    assert ob.inv_stride == h.inv_stride
    n_act = _n_act(compiled, n, cfg_id)
    rng = np.random.RandomState(23)
    both = n_trunc = n_term = 0
    for t in range(10):
        m, p, v = h.export_state()
        ob.map[:] = m.reshape(n, -1).cpu().numpy()
        ob.pose[:] = p.cpu().numpy()
        ob.inv[:] = v.cpu().numpy()
        twin.load_state(m, p, v)
        a = (rng.randint(0, 1 << 30, size=n) % n_act).astype(np.int32)
        o_obs, _, o_done, _, _ = ob.step(a, n_threads=8)
        term = o_done.astype(bool)
        late = np.nonzero(term)[0][::2]
        if late.size:
            h.ep_len[torch.from_numpy(late).cuda()] = T - 1
        ep_len = h.ep_len.cpu().numpy()
        _fill(h)
        a_dev = torch.from_numpy(a).cuda()
        obs, rew, done, cost, res = h.step(a_dev, auto_reset=True, max_episode_steps=T)
        want_rows = twin.step(a_dev)[0].cpu().numpy()
        expect_trunc = ep_len + 1 >= T
        where = "%s %s step %d" % (case, fmt, t)
        done = done.cpu().numpy().astype(bool)
        trunc = h.truncated.cpu().numpy()
        assert set(np.unique(trunc)) <= {0, 1}, where
        assert np.array_equal(done, term | expect_trunc), where
        assert np.array_equal(trunc.astype(bool), expect_trunc & ~term), where
        fo = h.final_obs.cpu().numpy()
        assert np.array_equal(fo[done], want_rows[done]), where
        assert (fo[~done].view(np.uint8) == SENTINEL).all(), where
        if fmt == 'i32':
            assert np.array_equal(fo[done][:, :ob.obs_dim], o_obs[done]), where
        else:
            assert np.array_equal(obs_to_vector(fo[done], compiled, fmt), o_obs[done]), where
        both += int((term & expect_trunc).sum())
        n_trunc += int(trunc.sum())
        n_term += int(term.sum())
    assert n_trunc > 0 and int(h.stats()[5].item()) > 0
    if case == 'firewall':
        assert n_term > 0 and both > 0, (n_term, both)


def _profiled_step(h, a, tmp_path):
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        h.step(a)
        torch.cuda.synchronize()
    trace = str(tmp_path / 'step.json')
    prof.export_chrome_trace(trace)
    with open(trace) as f:
        events = json.load(f)['traceEvents']
    steps = [(e['name'], e['args']['block'][0]) for e in events if e.get('cat') == 'kernel' and 'step1' in e['name']]
    assert len(steps) == 1, steps
    return steps[0]


def _same_state(a, b):
    for name in ('map', 'pose', 'inventory', 'episode', 'ep_len', 'error_flags'):
        assert torch.equal(getattr(a, name), getattr(b, name)), name


@pytest.mark.parametrize('case', sorted(ROUTES))
def test_buffers_change_no_other_output(case, tmp_path):
    """A handle without the buffers and a twin with them, same seed and actions, auto-reset and truncation on: every
    existing output and the whole state stay byte-identical; with the buffers set, the step still runs the kernel shape
    the routing table lists."""
    compiled, n, cfg_id = _inputs(case)
    off = _handle(compiled, n, cfg_id, seed=29, episode_end=False)
    on = _handle(compiled, n, cfg_id, seed=29)
    for h in (off, on):
        h.reset()
    n_act = _n_act(compiled, n, cfg_id)
    rng = np.random.RandomState(3)
    n_trunc = 0
    for t in range(20):
        a = torch.from_numpy((rng.randint(0, 1 << 30, size=n) % n_act).astype(np.int32)).cuda()
        for x, y in zip(off.step(a, auto_reset=True, max_episode_steps=3), on.step(a, auto_reset=True, max_episode_steps=3)):
            assert torch.equal(x, y), "step %d" % t
        _same_state(off, on)
        n_trunc += int(on.truncated.sum().item())
    assert n_trunc > 0
    name, threads = _profiled_step(on, torch.zeros(n, dtype=torch.int32, device='cuda'), tmp_path)
    kernel, want_threads = ROUTES[case]
    assert kernel + '(' in name and threads == want_threads, (name, threads)


@pytest.mark.parametrize('case', ['C2', 'ms40', 'C3-waves-two'])
def test_overlapped_steps_with_episode_end_buffers(case):
    """test_overlapped_steps_with_queued_resets_in_a_graph with the buffers set on every handle: 11 of 12 captured
    launches still overlap and every output, truncated and final_obs included, equals one-at-a-time stepping.  When handle
    B's actions alias handle A's truncated or final_obs buffer, B's launch does not overlap A's."""
    H = 2 if case.endswith('-two') else 3
    if case.startswith('C2'):
        cc, n = _compiled(C2_DESC), 32 * 90 + 5
    elif case.startswith('C3'):
        cc, n = _compiled(golden_util.get('bow_C3_axe_medium_fence_hard')['meta']), 32 * 148 * 28 + 17
    else:
        cc, n = _compiled(golden_util.get(C5)['meta']), 32 * 20 + 3
    rng = np.random.RandomState(12)
    hs = [_handle([cc], n, seed=70 + k) for k in range(H)]
    ref = [_handle([cc], n, seed=70 + k) for k in range(H)]
    for x in hs + ref:
        x.reset()
    torch.cuda.synchronize()
    acts = [torch.from_numpy(rng.randint(0, cc.c.n_actions, size=n).astype(np.int32)).cuda() for _ in range(12)]
    stream = torch.cuda.Stream()
    graph = torch.cuda.CUDAGraph()
    keep = []
    c0 = sum(x.concurrent_launch_count() for x in hs)
    with torch.cuda.stream(stream):
        with torch.cuda.graph(graph, stream=stream):
            for t in range(12):
                keep.append(hs[t % H].step(acts[t], auto_reset=True, max_episode_steps=3))
    assert sum(x.concurrent_launch_count() for x in hs) - c0 == 11
    for rep in range(3):
        graph.replay()
        torch.cuda.synchronize()
        for t in range(12):
            want = ref[t % H].step(acts[t], auto_reset=True, max_episode_steps=3)
            torch.cuda.synchronize()
            if t >= 12 - H:
                for x, y in zip(keep[t], want):
                    assert torch.equal(x, y), "replay %d launch %d" % (rep, t)
        for a, b in zip(hs, ref):
            _same_state(a, b)
            assert torch.equal(a.truncated, b.truncated) and torch.equal(a.final_obs, b.final_obs), "replay %d" % rep
    assert int(hs[0].episode.min().item()) >= 4 and sum(int(x.truncated.sum().item()) for x in hs) > 0

    A, B = hs[0], hs[1]
    alias = torch.zeros(n, dtype=torch.int32, device='cuda')      # int32 [n] whose first n bytes are A's truncated flags
    capi.check(A.lib, A.lib.ngw_set_episode_end_buffers(A._h, C.c_void_p(alias.data_ptr()),
                                                        C.c_void_p(A.final_obs.data_ptr())))
    for b_actions, should_overlap in ((acts[1], True), (alias, False), (A.final_obs.view(-1)[:n], False)):
        c0 = A.concurrent_launch_count() + B.concurrent_launch_count()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.stream(stream):
            with torch.cuda.graph(g, stream=stream):
                A.step(acts[0], auto_reset=True, max_episode_steps=3)
                B.step(b_actions, auto_reset=True, max_episode_steps=3)
        got = A.concurrent_launch_count() + B.concurrent_launch_count() - c0
        assert got == (1 if should_overlap else 0), (should_overlap, got)
    A.enable_episode_end()


def test_host_paths_and_step_group_write_the_same_buffers():
    """ngw_step_host and _begin/_end write the same truncated flags and final_obs rows as the device path; a StepGroup
    writes each handle's own buffers."""
    cc = _compiled(C2_DESC)
    n = 32 * 50 + 7
    hd, hh, hb = [_handle([cc], n, seed=5) for _ in range(3)]
    for h in (hd, hh, hb):
        h.reset()
    rng = np.random.RandomState(4)
    n_trunc = 0
    for t in range(8):
        a = rng.randint(0, cc.c.n_actions, size=n).astype(np.int32)
        dev = [x.cpu().numpy() for x in hd.step(torch.from_numpy(a).cuda(), auto_reset=True, max_episode_steps=3)]
        host = hh.step_host(a, auto_reset=True, max_episode_steps=3)
        hb.step_host_begin(a, auto_reset=True, max_episode_steps=3)
        begin_end = hb.step_host_end()
        for got in (host, begin_end):
            for x, y in zip(got, dev):
                assert np.array_equal(x, y), "step %d" % t
        for h in (hh, hb):
            assert torch.equal(h.truncated, hd.truncated) and torch.equal(h.final_obs, hd.final_obs), "step %d" % t
        n_trunc += int(hd.truncated.sum().item())
    assert n_trunc > 0

    hs = [_handle([cc], n, seed=60 + k) for k in range(3)]
    ref = [_handle([cc], n, seed=60 + k) for k in range(3)]
    for x in hs + ref:
        x.reset()
    group = StepGroup(hs)
    for t in range(6):
        acts = [torch.from_numpy(rng.randint(0, cc.c.n_actions, size=n).astype(np.int32)).cuda() for _ in range(3)]
        group.step(acts, auto_reset=True, max_episode_steps=3)
        for k in range(3):
            ref[k].step(acts[k], auto_reset=True, max_episode_steps=3)
        torch.cuda.synchronize()
        for a, b in zip(hs, ref):
            assert torch.equal(a.truncated, b.truncated) and torch.equal(a.final_obs, b.final_obs), "group step %d" % t
            _same_state(a, b)


def test_other_calls_leave_the_buffers_alone_and_edge_cases():
    """ngw_rollout (given and device-random actions), the closed-loop rollout, ngw_observe and ngw_reset never write the
    buffers; a misaligned final_obs is refused; invalid-action lanes write truncated 0; without auto-reset an env past the
    limit reports done and truncated on every step; a batch without LidarInFront gets truncated flags only."""
    cc = _compiled(C2_DESC)
    n = 32 * 40 + 9
    h = _handle([cc], n, seed=8)
    h.reset()
    _fill(h)
    acts = torch.from_numpy(np.random.RandomState(1).randint(0, cc.c.n_actions, size=(7, n)).astype(np.int32)).cuda()
    h.rollout(7, actions=acts, auto_reset=True, max_episode_steps=3)
    h.rollout(7, policy_seed=3, auto_reset=True, max_episode_steps=3)
    w = torch.ones((h.obs_dim, 4), dtype=torch.int32, device='cuda')
    h.rollout(7, policy=(w, torch.zeros(4, dtype=torch.int32, device='cuda')), auto_reset=True, max_episode_steps=3)
    h.observe()
    h.reset()
    torch.cuda.synchronize()
    assert int(h.episode.min().item()) >= 3                           # the rollouts did reset envs
    assert (h.truncated.cpu().numpy() == SENTINEL).all() and (h.final_obs.view(torch.uint8).cpu().numpy() == SENTINEL).all()

    with pytest.raises(RuntimeError, match='aligned'):
        capi.check(h.lib, h.lib.ngw_set_episode_end_buffers(h._h, None, C.c_void_p(h.final_obs.data_ptr() + 4)))

    # invalid-action lanes at the limit: done 0, truncated 0; the others are truncated unless they terminated
    h.ep_len.fill_(5)
    a = torch.randint(0, cc.c.n_actions, (n,), dtype=torch.int32, device='cuda')
    bad = torch.arange(n, device='cuda') % 3 == 0
    a[bad] = -1
    _, _, done, _, _ = h.step(a, auto_reset=False, max_episode_steps=4)
    trunc = h.truncated.bool()
    assert not trunc[bad].any() and not done[bad].bool().any()
    assert torch.equal(trunc[~bad], done[~bad].bool())                # (C2 random actions do not terminate in one step)
    assert bool(trunc[~bad].all())
    h.error_flags.zero_()
    for _ in range(2):                                                # no auto-reset: past the limit, every step again
        _, _, done, _, _ = h.step(torch.zeros(n, dtype=torch.int32, device='cuda'), max_episode_steps=4)
        assert bool(done.bool().all()) and torch.equal(h.truncated.bool(), done.bool())
    h.enable_episode_end(False)
    assert h.truncated is None and h.final_obs is None
    h.step(torch.zeros(n, dtype=torch.int32, device='cuda'), auto_reset=True, max_episode_steps=4)

    nolidar = _compiled({'env': scenarios.POGO, 'map_size': 10, 'chain': [['limit', scenarios.C2_SET]]})
    hd = _handle([nolidar], 300, seed=2)
    assert hd.obs_dim == 0
    hd.reset(want_obs=False)
    for t in range(4):
        _, _, done, _, _ = hd.step(torch.zeros(300, dtype=torch.int32, device='cuda'), auto_reset=True, max_episode_steps=2)
        assert torch.equal(hd.truncated.bool(), done.bool()) and bool(done.bool().all()) == (t % 2 == 1)


def test_gym_api_episode_end_info():
    """make(..., num_envs=n, auto_reset=True, max_episode_steps=T, episode_end_info=True): info['TimeLimit.truncated']
    and info['terminal_observation'] are the handle's buffers on the device path and the host path; at the first limit
    the terminal observations equal what an env without auto-reset returns.  Without the keyword neither key exists."""
    import gym_novel_gridworlds_b200 as gym
    n, T = 1000, 5

    def env_of(**kw):
        env = gym.make('NovelGridworld-Pogostick-v1', num_envs=n, device='cuda:0', seed=6, **kw)
        env = gym.LimitActions(env, set(scenarios.C2_SET))
        return gym.LidarInFront(env, num_beams=8)

    e = env_of(auto_reset=True, max_episode_steps=T, episode_end_info=True)
    plain = env_of(max_episode_steps=T)
    for x in (e, plain):
        x.reset()
    h = e.unwrapped._runtime.handle
    rng = np.random.RandomState(3)
    for t in range(12):
        a = rng.randint(0, len(scenarios.C2_SET), size=n).astype(np.int32)
        if t % 2 == 0:                                                # device path
            obs, rew, done, info = e.step(torch.from_numpy(a).cuda())
            trunc, term_obs = info['TimeLimit.truncated'], info['terminal_observation']
            assert trunc.dtype == torch.bool and torch.equal(trunc, h.truncated.bool())
            assert torch.equal(term_obs, h.final_obs[:, :h.obs_dim])
            trunc, term_obs, done = trunc.cpu().numpy(), term_obs.cpu().numpy(), done.cpu().numpy()
        else:                                                         # host path: fetched on access
            obs, rew, done, info = e.step(a)
            trunc, term_obs = info['TimeLimit.truncated'], info['terminal_observation']
            assert trunc.dtype == np.bool_ and np.array_equal(trunc, h.truncated.cpu().numpy().astype(bool))
            assert np.array_equal(term_obs, h.final_obs[:, :h.obs_dim].cpu().numpy())
        assert 'TimeLimit.truncated' in info and info.get('terminal_observation') is not None
        assert not (trunc & ~done).any()
        if t < T:
            p_obs, _, p_done, _ = plain.step(torch.from_numpy(a).cuda())
            if t == T - 1:                                            # every env ends its first episode here
                assert done.all() and np.array_equal(term_obs, p_obs.cpu().numpy())
                assert trunc.sum() > 0
    _, _, _, info = plain.step(torch.zeros(n, dtype=torch.int32, device='cuda'))
    assert 'TimeLimit.truncated' not in info.keys() and 'terminal_observation' not in info
    with pytest.raises(KeyError):
        info['TimeLimit.truncated']
    assert info.get('terminal_observation') is None
