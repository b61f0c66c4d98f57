"""NGW_OBS_HITS observation rows on the GPU (run on the B200 box: pytest -m gpu): byte for byte against the C oracle's
vector through the format's encoder, and against an int32 twin handle on every kernel shape and every entry point that
writes observation rows."""
import json

import numpy as np
import pytest
import torch

import golden_util
import scenarios
from gym_novel_gridworlds_b200.runtime import BatchHandle, StepGroup, obs_to_vector
from oracle.oracle_lib import OracleBatch
from test_gpu_kernel_routing import ROUTES, _inputs
from test_gpu_parity import C2_DESC, _compiled, tile_group_inputs
from test_obs_hits_format import encode_hits

pytestmark = pytest.mark.gpu

C4_CHAINS = [dict(C2_DESC, chain=[['limit', scenarios.C2_SET + ex], ['lidar', 8], nov]) for ex, nov in (
    (['Chop'], ['novelty', 'addchop', 'hard', '', '']), (['Jump'], ['novelty', 'addjump', 'hard', '', '']),
    ([], ['novelty', 'additem', 'medium', 'spring', '']), ([], ['novelty', 'remapaction', 'hard', '', '']))]
BOW16 = {'env': scenarios.BOW, 'map_size': 12, 'chain': [['lidar', 16]]}


def _expected_rows(h, vec, cfg_id=None):
    """The oracle's vectors -> the hits rows the handle must write (padding included)."""
    rows = np.zeros((vec.shape[0], h.obs_row_bytes), np.uint8)
    ids = np.zeros(vec.shape[0], np.int64) if cfg_id is None else np.asarray(cfg_id, np.int64)
    for k, cc in enumerate(h.compiled):
        sel = ids == k
        if sel.any():
            rows[sel] = encode_hits(vec[sel, :cc.obs_dim], cc.c, h.obs_row_bytes)
    return rows


def _np(x):
    return x.cpu().numpy() if hasattr(x, 'cpu') else np.asarray(x)


def _handles(compiled, n, cfg_id=None, seed=0):
    ids = None if cfg_id is None else np.asarray(cfg_id).astype(np.int32)
    return (BatchHandle(compiled, n, seed=seed, cfg_id=ids, obs_format='hits'),
            BatchHandle(compiled, n, seed=seed, cfg_id=ids))


def _same_state(a, b):
    for name in ('map', 'pose', 'inventory', 'episode', 'ep_len', 'error_flags'):
        assert torch.equal(getattr(a, name), getattr(b, name)), name


def _same_outputs(hits_out, i32_out, h):
    assert torch.equal(h.obs_vector(hits_out[0]), i32_out[0][:, :h.obs_dim])
    for x, y in zip(hits_out[1:], i32_out[1:]):
        assert torch.equal(x, y)


@pytest.mark.parametrize('case', ['C2', 'C4', 'C5', 'Bow16'])
def test_hits_rows_equal_the_oracle(case):
    """Device path and host-buffer path, a new step every time; C4 mixes four configs (env i -> config i mod 4,
    partial last tile), C5 is map 40 (also with auto-reset and truncation, against an int32 twin), Bow16 takes the
    generic LUT walk."""
    cfg_id = None
    if case == 'C2':
        compiled, n, steps = [_compiled(C2_DESC)], 3000 + 11, 24
    elif case == 'C4':
        compiled, n, steps = [_compiled(d) for d in C4_CHAINS], 2048 + 9, 24
        cfg_id = (np.arange(n) % 4).astype(np.uint8)
    elif case == 'C5':
        compiled, n, steps = [_compiled(golden_util.get('pogo_ms40_additem_hard')['meta'])], 200, 24
    else:
        compiled, n, steps = [_compiled(BOW16)], 500, 24
    ob = OracleBatch(compiled, n, cfg_id=cfg_id)
    ob.reset_legacy(909)
    ids = None if cfg_id is None else cfg_id.astype(np.int32)
    hd, hh = [BatchHandle(compiled, n, cfg_id=ids, obs_format='hits') for _ in range(2)]   # device path, host path
    for h in (hd, hh):
        h.load_state(ob.map, ob.pose, ob.inv)
    assert hd.obs.dtype == torch.uint8 and hd.obs.shape == (n, hd.obs_row_bytes)
    want_bytes = max(((2 * cc.c.n_beams + 3) & ~3) + 4 * cc.c.n_inv_obs for cc in compiled)
    assert hd.obs_row_bytes == want_bytes
    assert np.array_equal(_np(hd.observe()), _expected_rows(hd, ob.observe(), cfg_id))
    n_act = np.array([cc.c.n_actions for cc in compiled])[ob.cfg_id.astype(np.int64)]
    rng = np.random.RandomState(5)
    for t in range(steps):
        a = (rng.randint(0, 1 << 30, size=n) % n_act).astype(np.int32)
        o_obs, o_rew, o_done, o_cost, o_res = ob.step(a, n_threads=8)
        want = _expected_rows(hd, o_obs, cfg_id)
        for path, (obs, rew, done, cost, res) in (('device', hd.step(torch.from_numpy(a).cuda())), ('host', hh.step_host(a))):
            where = "%s step %d" % (path, t)
            assert np.array_equal(_np(obs), want), where
            assert np.array_equal(_np(rew), o_rew) and np.array_equal(_np(done), o_done), where
            assert np.array_equal(_np(res), o_res), where
            np.testing.assert_allclose(_np(cost), o_cost, rtol=1e-6, err_msg=where)
    assert np.array_equal(hd.map.cpu().numpy().reshape(n, -1), ob.map) and np.array_equal(hh.inventory.cpu().numpy(), ob.inv)
    if case == 'C5':                                                  # queued auto-reset rows, truncation
        hi = BatchHandle(compiled, n)
        hi.load_state(*hd.export_state())
        hi.episode.copy_(hd.episode)
        for t in range(6):
            a = torch.zeros(n, dtype=torch.int32, device='cuda')
            got = hd.step(a, auto_reset=True, max_episode_steps=3)
            ref = hi.step(a, auto_reset=True, max_episode_steps=3)
            _same_outputs(got, ref, hd)
        assert (hd.episode.cpu().numpy() == 2).all()
        _same_state(hd, hi)


def _hits_inputs(case):
    """ROUTES inputs; where hits rows (smaller than int32 rows) let the launcher pack more tiles per CTA, a larger batch
    that reaches the listed shape again."""
    if case == 'G2-waves':
        compiled, _, cfg_id = tile_group_inputs(case)
        return compiled, 32 * 4500 + 5, cfg_id
    return _inputs(case)


def _step_kernel_of(h, a, tmp_path):
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


@pytest.mark.parametrize('case', sorted(ROUTES))
def test_every_kernel_shape_writes_hits_rows(case, tmp_path):
    """A hits handle and an int32 handle from the same seed through the same actions with auto-reset: decoded rows,
    every other output and the state arrays identical; one hits step is recorded to show which shape ran."""
    compiled, n, cfg_id = _hits_inputs(case)
    hh, hi = _handles(compiled, n, cfg_id, seed=31)
    for h in (hh, hi):
        h.reset()
    assert torch.equal(hh.obs_vector(), hi.obs[:, :hh.obs_dim])
    n_act = np.array([cc.c.n_actions for cc in compiled])[(np.zeros(n, np.int64) if cfg_id is None else cfg_id.astype(np.int64))]
    rng = np.random.RandomState(8)
    for t in range(6):
        a = torch.from_numpy((rng.randint(0, 1 << 30, size=n) % n_act).astype(np.int32)).cuda()
        _same_outputs(hh.step(a, auto_reset=True, max_episode_steps=3), hi.step(a, auto_reset=True, max_episode_steps=3), hh)
    _same_state(hh, hi)
    assert int(hh.stats()[5].item()) > 0                              # auto-resets happened (NGW_STAT_RESETS)
    name, threads = _step_kernel_of(hh, torch.zeros(n, dtype=torch.int32, device='cuda'), tmp_path)
    kernel, want_threads = ROUTES[case]
    assert kernel + '(' in name and threads == want_threads, (name, threads)


@pytest.mark.parametrize('case', ['C2', 'C4', 'Bow16', 'ms40'])
def test_other_entry_points_write_hits_rows(case):
    """ngw_reset observations (masked and full), ngw_observe, ngw_rollout's final observation with given and
    device-random actions (lane-pair rollout2_kernel for C2 / C4, rollout_kernel for Bow16 / ms40), ngw_step_host and
    _begin/_end: each against an int32 twin.  ngw_rollout_policy refuses hits rows."""
    cfg_id = None
    if case == 'C2':
        compiled, n = [_compiled(C2_DESC)], 32 * 50 + 7
    elif case == 'C4':
        compiled, n = [_compiled(d) for d in C4_CHAINS], 32 * 40 + 9
        cfg_id = (np.arange(n) % 4).astype(np.uint8)
    elif case == 'Bow16':
        compiled, n = [_compiled(BOW16)], 300
    else:
        compiled, n = [_compiled(golden_util.get('pogo_ms40_additem_hard')['meta'])], 32 * 4 + 3
    hh, hi = _handles(compiled, n, cfg_id, seed=44)
    assert torch.equal(hh.obs_vector(hh.reset()), hi.reset()[:, :hh.obs_dim])
    _same_state(hh, hi)
    mask = torch.from_numpy((np.arange(n) % 3 == 0).astype(np.uint8)).cuda()
    assert torch.equal(hh.obs_vector(hh.reset(mask)), hi.reset(mask)[:, :hh.obs_dim])
    assert torch.equal(hh.obs_vector(hh.observe()), hi.observe()[:, :hh.obs_dim])
    n_act = np.array([cc.c.n_actions for cc in compiled])[(np.zeros(n, np.int64) if cfg_id is None else cfg_id.astype(np.int64))]
    rng = np.random.RandomState(2)
    acts = torch.from_numpy((rng.randint(0, 1 << 30, size=(7, n)) % n_act).astype(np.int32)).cuda()
    for kw in ({'actions': acts}, {'policy_seed': 77}):
        got = hh.rollout(7, auto_reset=True, max_episode_steps=4, record_actions=True, **kw)
        ref = hi.rollout(7, auto_reset=True, max_episode_steps=4, record_actions=True, **kw)
        _same_outputs(got, ref, hh)
        _same_state(hh, hi)
    for t in range(3):
        a = (rng.randint(0, 1 << 30, size=n) % n_act).astype(np.int32)
        got = hh.step_host(a, auto_reset=True, max_episode_steps=2)
        ref = hi.step_host(a, auto_reset=True, max_episode_steps=2)
        assert np.array_equal(hh.obs_vector(got[0]), ref[0][:, :hh.obs_dim]), "step_host %d" % t
        for x, y in zip(got[1:], ref[1:]):
            assert np.array_equal(x, y)
        hh.step_host_begin(a)
        hi.step_host_begin(a)
        got, ref = hh.step_host_end(), hi.step_host_end()
        assert np.array_equal(hh.obs_vector(got[0]), ref[0][:, :hh.obs_dim]), "step_host_begin/end %d" % t
        for x, y in zip(got[1:], ref[1:]):
            assert np.array_equal(x, y)
    _same_state(hh, hi)
    w = torch.zeros((hh.obs_dim, 4), dtype=torch.int32, device='cuda')
    b = torch.zeros(4, dtype=torch.int32, device='cuda')
    with pytest.raises(RuntimeError, match='NGW_OBS_I32'):
        hh.rollout(2, policy=(w, b))


def test_captured_and_grouped_hits_handles_overlap():
    """Three rotating hits handles in one CUDA graph and in a StepGroup: launches overlap and the results equal
    stepping each handle one launch at a time."""
    cc, n, H = _compiled(C2_DESC), 32 * 90 + 5, 3
    hs = [BatchHandle([cc], n, seed=70 + k, obs_format='hits') for k in range(H)]
    ref = [BatchHandle([cc], n, seed=70 + k, obs_format='hits') for k in range(H)]
    for x in hs + ref:
        x.reset()
    torch.cuda.synchronize()
    rng = np.random.RandomState(13)
    acts = [torch.from_numpy(rng.randint(0, cc.c.n_actions, size=n).astype(np.int32)).cuda() for _ in range(12)]
    stream = torch.cuda.Stream()
    graph = torch.cuda.CUDAGraph()
    keep = []
    c0 = sum(x.concurrent_launch_count() for x in hs)
    with torch.cuda.stream(stream):
        with torch.cuda.graph(graph, stream=stream):
            for t in range(12):
                keep.append(hs[t % H].step(acts[t], auto_reset=True, max_episode_steps=3))
    assert sum(x.concurrent_launch_count() for x in hs) - c0 > 0
    for rep in range(2):
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
    group = StepGroup(hs)
    c0 = sum(x.concurrent_launch_count() for x in hs)
    for t in range(4):
        a3 = [acts[(t + k) % 12] for k in range(H)]
        outs = group.step(a3, auto_reset=True, max_episode_steps=3)
        torch.cuda.synchronize()
        for k in range(H):
            want = ref[k].step(a3[k], auto_reset=True, max_episode_steps=3)
            for x, y in zip(outs[k], want):
                assert torch.equal(x, y), "group step %d handle %d" % (t, k)
    assert sum(x.concurrent_launch_count() for x in hs) - c0 > 0
    for a, b in zip(hs, ref):
        _same_state(a, b)


def test_make_with_hits_rows():
    """make(..., num_envs=n, obs_format='hits') wrapped in LidarInFront: reset / step return hits rows whose decoded
    form equals what an int32 env returns."""
    import gym_novel_gridworlds_b200 as gym

    def env_of(fmt):
        env = gym.make('NovelGridworld-Pogostick-v1', num_envs=1000, device='cuda:0', seed=6, obs_format=fmt,
                       auto_reset=True, max_episode_steps=5)
        env = gym.LimitActions(env, set(scenarios.C2_SET))
        return gym.LidarInFront(env, num_beams=8)

    eh, ei = env_of('hits'), env_of('i32')
    oh, oi = eh.reset(), ei.reset()
    h = eh.unwrapped._runtime.handle
    assert oh.dtype == torch.uint8 and oh.shape == (1000, h.obs_row_bytes) and h.obs_row_bytes == 44
    assert torch.equal(obs_to_vector(oh, h.compiled, 'hits'), oi)
    rng = np.random.RandomState(3)
    for t in range(8):
        a = torch.from_numpy(rng.randint(0, len(scenarios.C2_SET), size=1000).astype(np.int32)).cuda()
        (oh, rh, dh, ih), (oi, ri, di, ii) = eh.step(a), ei.step(a)
        assert torch.equal(h.obs_vector(oh), oi), "step %d" % t
        assert torch.equal(rh, ri) and torch.equal(dh, di) and torch.equal(ih['result'], ii['result'])
        ah = rng.randint(0, len(scenarios.C2_SET), size=1000).astype(np.int32)
        (oh, rh, dh, _), (oi, ri, di, _) = eh.step(ah), ei.step(ah)     # host-buffer path
        assert np.array_equal(h.obs_vector(oh), oi), "host step %d" % t
        assert np.array_equal(rh, ri) and np.array_equal(dh, di)
