"""GPU parity (run on the B200 box: pytest -m gpu).  Everything goes through the C-ABI (libngw_b200.so):
   1. every golden trace of the unmodified reference, replayed on the GPU, compared at every step;
   2. >= 10^6 env-steps against the C oracle from reference-exact (legacy-stream) reset states;
   3. layout / API edge cases: partial tiles, host-buffer path, invalid actions, N == 1;
   4. every kernel shape the launch code selects from the input (test_gpu_kernel_routing.py proves the routes)."""
import os

import numpy as np
import pytest
import torch

import golden_util
import scenarios
from gym_novel_gridworlds_b200.compiler import compile_chain
from gym_novel_gridworlds_b200.runtime import BatchHandle, MixedBatch
from oracle.oracle_lib import OracleBatch

pytestmark = pytest.mark.gpu
NAMES = golden_util.names()


def _compiled(desc):
    return compile_chain(scenarios.build_chain(scenarios.b200_namespace(), desc))


@pytest.mark.parametrize('name', NAMES)
def test_gpu_replays_reference_golden_trace(name):
    g = golden_util.get(name)
    cc = _compiled(g['meta'])
    E, T = g['actions'].shape
    n_items = g['init_inv'].shape[1]
    h = BatchHandle([cc], E, seed=1)
    h.load_state(g['init_map'], g['init_pose'], g['init_inv'])
    h.enable_messages()
    from gym_novel_gridworlds_b200.runtime import decode_message
    kind = g['meta']['reset_kind']
    has_obs = g['obs'].shape[2] > 0 and kind != 'agent_map'
    amap = torch.empty((E, 11, 11), dtype=torch.int8, device='cuda')
    for t in range(T):
        obs, reward, done, cost, result = h.step(torch.from_numpy(g['actions'][:, t].copy()).cuda())
        if kind == 'agent_map':
            from gym_novel_gridworlds_b200 import capi
            import ctypes as C
            capi.check(h.lib, h.lib.ngw_agent_map(h._h, C.c_void_p(amap.data_ptr()), 5, h._stream()))
            assert np.array_equal(amap.cpu().numpy().reshape(E, -1), g['obs'][:, t]), "%s step %d" % (name, t)
        where = "%s step %d" % (name, t)
        assert np.array_equal(reward.cpu().numpy(), g['reward'][:, t].astype(np.float32)), where
        assert np.array_equal(done.cpu().numpy(), g['done'][:, t]), where
        assert np.array_equal(result.cpu().numpy(), g['result'][:, t]), where
        np.testing.assert_allclose(cost.cpu().numpy(), g['cost'][:, t], rtol=1e-6, err_msg=where)
        assert [decode_message(c, cc) for c in h.msg.cpu().numpy()] == list(g['message'][:, t]), where   # info['message']
        assert np.array_equal(h.map.cpu().numpy().reshape(E, -1), g['map'][:, t]), where
        assert np.array_equal(h.pose.cpu().numpy(), g['pose'][:, t]), where
        assert np.array_equal(h.inventory.cpu().numpy()[:, :n_items], g['inv'][:, t]), where
        if has_obs:
            assert np.array_equal(obs.cpu().numpy()[:, :cc.obs_dim], g['obs'][:, t].astype(np.int32)), where
    assert int(h.error_flags.abs().sum().item()) == 0
    h.close()


def _parity_vs_oracle(compiled, n, steps, seed0, cfg_id=None, rng_seed=0):
    ob = OracleBatch(compiled, n, cfg_id=cfg_id)
    err = ob.reset_legacy(seed0)
    assert not err.any()
    h = BatchHandle(compiled, n, seed=3, cfg_id=None if cfg_id is None else cfg_id.astype(np.int32))
    h.load_state(ob.map, ob.pose, ob.inv)
    n_act = np.array([cc.c.n_actions for cc in compiled])[ob.cfg_id.astype(np.int64)]
    rng = np.random.RandomState(rng_seed)
    obs0 = h.observe().cpu().numpy()
    assert np.array_equal(obs0[:, :ob.obs_dim], ob.observe())
    for t in range(steps):
        actions = (rng.randint(0, 1 << 30, size=n) % n_act).astype(np.int32)
        o_obs, o_rew, o_done, o_cost, o_res = ob.step(actions, n_threads=8)
        obs, rew, done, cost, res = h.step(torch.from_numpy(actions).cuda())
        where = "step %d" % t
        assert np.array_equal(rew.cpu().numpy(), o_rew), where
        assert np.array_equal(done.cpu().numpy(), o_done), where
        assert np.array_equal(res.cpu().numpy(), o_res), where
        np.testing.assert_allclose(cost.cpu().numpy(), o_cost, rtol=1e-6, err_msg=where)
        if ob.obs_dim:
            assert np.array_equal(obs.cpu().numpy()[:, :ob.obs_dim], o_obs), where
        if t % 16 == 15 or t == steps - 1:
            assert np.array_equal(h.map.cpu().numpy().reshape(n, -1), ob.map), where
            assert np.array_equal(h.pose.cpu().numpy(), ob.pose), where
            assert np.array_equal(h.inventory.cpu().numpy(), ob.inv), where
    h.close()
    return n * steps


def test_million_steps_c2_vs_oracle():
    """BASELINE config C2 (Pogostick-v1 + LimitActions + LidarInFront): 4096 reference-exact resets x 256 steps."""
    cc = _compiled({'env': scenarios.POGO, 'map_size': 10, 'chain': [['limit', scenarios.C2_SET], ['lidar', 8]]})
    assert _parity_vs_oracle([cc], 4096, 256, seed0=1000) >= 10 ** 6


def test_c3_bow_axe_fence_vs_oracle():
    cc = _compiled(golden_util.get('bow_C3_axe_medium_fence_hard')['meta'])
    _parity_vs_oracle([cc], 2048, 128, seed0=5000)


def test_c4_mixed_novelties_one_launch_vs_oracle():
    """addchop / addjump / additem(medium) / remapaction(hard), env i -> config i mod 4, one launch per step."""
    base = [['limit', scenarios.C2_SET + ['Chop', 'Jump']], ['lidar', 8]]
    descs = [{'env': scenarios.POGO, 'map_size': 10, 'chain': base + [extra]} for extra in (
        ['novelty', 'addchop', 'hard', '', ''], ['novelty', 'addjump', 'hard', '', ''],
        ['novelty', 'additem', 'medium', 'spring', ''], ['novelty', 'remapaction', 'hard', '', ''])]
    # Chop/Jump are only valid where the novelty exists: use per-config limited sets
    descs[0]['chain'][0] = ['limit', scenarios.C2_SET + ['Chop']]
    descs[1]['chain'][0] = ['limit', scenarios.C2_SET + ['Jump']]
    descs[2]['chain'][0] = ['limit', scenarios.C2_SET]
    descs[3]['chain'][0] = ['limit', scenarios.C2_SET]
    compiled = [_compiled(d) for d in descs]
    n = 4096 + 7                                  # exercises the partial last tile and heterogeneous warps
    cfg_id = (np.arange(n) % 4).astype(np.uint8)
    _parity_vs_oracle(compiled, n, 96, seed0=9000, cfg_id=cfg_id)


def test_c5_map40_additem_hard_vs_oracle():
    cc = _compiled(golden_util.get('pogo_ms40_additem_hard')['meta'])
    _parity_vs_oracle([cc], 256, 64, seed0=100)


def test_host_buffer_path_matches_device_path():
    cc = _compiled({'env': scenarios.POGO, 'map_size': 10, 'chain': [['limit', scenarios.C2_SET], ['lidar', 8]]})
    n = 40000 + 13
    ob = OracleBatch([cc], n)
    ob.reset_legacy(42)
    h1, h2 = BatchHandle([cc], n), BatchHandle([cc], n)
    for h in (h1, h2):
        h.load_state(ob.map, ob.pose, ob.inv)
    rng = np.random.RandomState(1)
    for t in range(12):
        a = rng.randint(0, cc.c.n_actions, size=n).astype(np.int32)
        d = [x.cpu().numpy() for x in h1.step(torch.from_numpy(a).cuda())]
        if t % 2:
            hb = h2.step_host(a)
        else:
            h2.step_host_begin(a)
            hb = h2.step_host_end()
        for x, y in zip(d, hb):
            assert np.array_equal(x, y)
    assert np.array_equal(h1.map.cpu().numpy(), h2.map.cpu().numpy())
    assert np.array_equal(h1.inventory.cpu().numpy(), h2.inventory.cpu().numpy())


def test_invalid_action_sets_flag_and_leaves_state():
    cc = _compiled({'env': scenarios.POGO, 'map_size': 10, 'chain': [['limit', scenarios.C2_SET], ['lidar', 8]]})
    h = BatchHandle([cc], 64)
    h.reset()
    before = [x.clone() for x in (h.map, h.pose, h.inventory)]
    a = torch.full((64,), 10, dtype=torch.int32, device='cuda')      # limited ids are 0..9 (wrappers.py:76)
    a[::2] = -3
    h.step(a)
    assert (h.error_flags.cpu().numpy() & 1).all()
    for x, y in zip(before, (h.map, h.pose, h.inventory)):
        assert torch.equal(x, y)
    assert h.stats().cpu().numpy()[6] == 64


def test_single_env_api_reproduces_survey_kat():
    """SURVEY §8c seed-0 known-answer test through the drop-in gym API with num_envs == 1."""
    import gym_novel_gridworlds_b200 as gym
    env = gym.make('NovelGridworld-Pogostick-v1')
    env = gym.LimitActions(env, set(scenarios.C2_SET))
    env = gym.LidarInFront(env, num_beams=8)
    env.reset()
    rt = env.unwrapped._runtime
    ob = OracleBatch([rt.compiled], 1)
    ob.reset_one(0, 0)                       # np.random.seed(0) reset of the reference
    rt.handle.load_state(ob.map, ob.pose, ob.inv)
    obs = env.observation()
    nz = np.nonzero(obs)[0]
    assert list(nz) == [6, 13, 18, 25, 28, 41, 48, 55] and list(obs[nz]) == [2, 3, 4, 4, 3, 3, 2, 3]
    rewards, costs, results = [], [], []
    for a in [6, 6, 9, 6, 0, 7, 6, 0, 1, 1, 3, 8, 5]:
        obs, r, d, info = env.step(a)
        rewards.append(r); costs.append(info['step_cost']); results.append(info['result'])
    assert rewards == [-1, -1, -1, -1, -1, -1, -1, 10, 10, -1, 10, -1, -1]
    np.testing.assert_allclose(costs, [27.906975, 27.906975, 24, 27.906975, 3600, 24, 27.906975, 3600, 1200, 0, 2400,
                                       300, 120], rtol=1e-6)
    assert results == [True, True, True, True, False, True, True, True, True, False, True, False, False]
    assert env.agent_location == (3, 5) and env.agent_facing_str == 'EAST'
    assert [env.inventory_items_quantity[k] for k in sorted(env.inventory_items_quantity)] == [0, 0, 2, 0, 0, 4, 0, 0, 0]
    nz = np.nonzero(obs)[0]
    assert list(nz) == [6, 11, 18, 27, 34, 41, 42, 55, 57, 60] and list(obs[nz]) == [5, 4, 2, 5, 4, 4, 1, 4, 2, 4]
    with pytest.raises(AssertionError):
        env.step(10)


def test_rollout_kernel_equals_repeated_steps():
    """SURVEY §8f N1: T steps in one launch == T launches (same states, observation, sums), given and random policy."""
    cc = _compiled({'env': scenarios.POGO, 'map_size': 10, 'chain': [['limit', scenarios.C2_SET], ['lidar', 8]]})
    n, T = 3000 + 9, 40
    ob = OracleBatch([cc], n)
    ob.reset_legacy(31337)
    h1, h2, h3 = BatchHandle([cc], n), BatchHandle([cc], n), BatchHandle([cc], n)
    for h in (h1, h2, h3):
        h.load_state(ob.map, ob.pose, ob.inv)
    rng = np.random.RandomState(5)
    acts = rng.randint(0, cc.c.n_actions, size=(T, n)).astype(np.int32)
    rew = np.zeros(n); cost = np.zeros(n); dones = np.zeros(n, int)
    for t in range(T):
        o, r, d, c, res = h1.step(torch.from_numpy(acts[t]).cuda())
        rew += r.cpu().numpy(); cost += c.cpu().numpy().astype(np.float64); dones += d.cpu().numpy()
    obs2, r2, c2, dc2, d2, res2 = h2.rollout(T, torch.from_numpy(acts).cuda())
    assert torch.equal(h1.map, h2.map) and torch.equal(h1.pose, h2.pose) and torch.equal(h1.inventory, h2.inventory)
    assert torch.equal(obs2, o) and torch.equal(d2, d) and torch.equal(res2, res)
    assert np.array_equal(r2.cpu().numpy(), rew) and np.array_equal(dc2.cpu().numpy(), dones)
    np.testing.assert_allclose(c2.cpu().numpy(), cost, rtol=1e-5)
    # on-device random policy: replay the recorded actions through the oracle
    out = h3.rollout(T, None, policy_seed=99, record_actions=True)
    taken = out[-1].cpu().numpy()
    assert taken.min() >= 0 and taken.max() < cc.c.n_actions
    counts = np.bincount(taken.ravel(), minlength=cc.c.n_actions) / taken.size
    assert np.abs(counts - 1.0 / cc.c.n_actions).max() < 0.01         # uniform policy
    for t in range(T):
        o_obs, o_rew, o_done, o_cost, o_res = ob.step(taken[t])
    assert np.array_equal(h3.map.cpu().numpy().reshape(n, -1), ob.map)
    assert np.array_equal(h3.inventory.cpu().numpy(), ob.inv) and np.array_equal(h3.pose.cpu().numpy(), ob.pose)
    assert np.array_equal(out[0].cpu().numpy()[:, :cc.obs_dim], o_obs)


def test_env_restore_chaining_and_save_trajectories(tmp_path):
    """SURVEY §8f N3: the `env=` restore branch of reset (pogostick_v1_env.py:89-109) and the SaveTrajectories schema."""
    import pickle
    import gym_novel_gridworlds_b200 as gym
    for n in (1, 300):
        first = gym.LidarInFront(gym.make('NovelGridworld-Pogostick-v1', num_envs=n, seed=3))
        first.reset()
        a = 3 if n == 1 else torch.full((n,), 3, dtype=torch.int32, device='cuda')
        first.step(a)
        second = gym.LidarInFront(gym.make('NovelGridworld-Pogostick-v1', num_envs=n, env=first))
        obs = second.reset()
        h1, h2 = first.unwrapped._runtime.handle, second.unwrapped._runtime.handle
        assert torch.equal(h1.map, h2.map) and torch.equal(h1.inventory, h2.inventory)
        assert torch.equal(h1.pose[:, :3], h2.pose[:, :3])
        o1 = first.observation()
        assert np.array_equal(np.asarray(obs if n == 1 else obs.cpu().numpy()), np.asarray(o1 if n == 1 else o1.cpu().numpy()))
    env = gym.SaveTrajectories(gym.make('NovelGridworld-Bow-v1'), str(tmp_path))
    env.reset()
    for a in (0, 1, 3):
        env.step(a)
    path = env.save()
    with open(path, 'rb') as f:
        traj = pickle.load(f)
    assert len(traj) == 3
    assert set(traj[0]) == {"map_size", "map", "agent_location", "agent_facing_str", "block_in_front_id", "items_id",
                            "items_quantity", "inventory_items_quantity", "action_str", "last_action", "last_done"}


def test_batched_gym_api_auto_reset_messages_and_mixed_batch():
    import gym_novel_gridworlds_b200 as gym
    n = 2000
    env = gym.make('NovelGridworld-Pogostick-v1', num_envs=n, seed=7, auto_reset=True, max_episode_steps=8, messages=True)
    env = gym.LidarInFront(gym.LimitActions(env, set(scenarios.C2_SET)))
    obs = env.reset()
    assert obs.shape == (n, 63) and obs.dtype == torch.int32
    dones = 0
    for t in range(16):
        a = torch.randint(0, 10, (n,), device='cuda', dtype=torch.int32)
        obs, reward, done, info = env.step(a)
        dones += int(done.sum().item())
        assert len(info['message']) == n and info['step_cost'].shape == (n,) and info['result'].dtype == torch.bool
    assert dones == 2 * n                                         # truncated (and regenerated) at steps 8 and 16
    assert env.seed(11) == [11]
    # host-buffer path through the same API: numpy in, numpy out
    obs = env.reset()
    o, r, d, info = env.step(np.zeros(n, np.int32))
    assert isinstance(o, np.ndarray) and o.shape == (n, 63) and isinstance(r, np.ndarray)
    # several chains in one batch
    chains = [gym.LidarInFront(gym.LimitActions(gym.make('NovelGridworld-Pogostick-v1'), set(scenarios.C2_SET))),
              gym.inject_novelty(gym.LidarInFront(gym.LimitActions(gym.make('NovelGridworld-Pogostick-v1'),
                                                                   set(scenarios.C2_SET + ['Chop']))), 'addchop')]
    mb = MixedBatch(chains, 1000, assignment='blocked')
    assert (mb.cfg_id_host[:500] == 0).all() and (mb.cfg_id_host[500:] == 1).all()
    obs = mb.reset()
    out = mb.step(torch.full((1000,), 10, dtype=torch.int32, device='cuda'))      # id 10 = Right (cfg 1) / invalid (cfg 0)
    flags = mb.handle.error_flags.cpu().numpy()
    assert (flags[:500] & 1).all() and not (flags[500:] & 1).any()
    st = mb.handle.stats().cpu().numpy()
    assert st[0] == 500 and st[6] == 500


def many_config_inputs(n_cfg):
    """(compiled configs, batch size, cfg_id) of a batch of n_cfg novelty variants of C2, env i -> config 7 i mod n_cfg."""
    variants = [('addchop', 'hard', '', '', ['Chop']), ('addjump', 'hard', '', '', ['Jump']),
                ('additem', 'easy', 'spring', '', []), ('breakincrease', 'hard', '', '', []),
                ('axe', 'easy', 'wooden', 'true', ['Select_wooden_axe']), ('fence', 'medium', 'oak', '', [])]
    compiled = []
    for i in range(n_cfg):
        name, diff, a1, a2, extra = variants[i % len(variants)]
        desc = {'env': scenarios.POGO, 'map_size': 10, 'build_seed': 100 + i,
                'chain': [['limit', scenarios.C2_SET + extra], ['lidar', 8], ['novelty', name, diff, a1, a2]]}
        compiled.append(_compiled(desc))
    n = 64 * n_cfg + 5
    return compiled, n, (np.arange(n) * 7 % n_cfg).astype(np.uint8)


@pytest.mark.parametrize('n_cfg', [6, 20])
def test_many_configs_in_one_batch_inline_and_global_tables(n_cfg):
    """NC = 16 inline-config kernel (6 configs) and the global-memory fallback (20 configs > 16)."""
    compiled, n, cfg_id = many_config_inputs(n_cfg)
    _parity_vs_oracle(compiled, n, 40, seed0=777, cfg_id=cfg_id)


@pytest.mark.parametrize('ms,beams,n', [(64, 8, 70), (12, 16, 600), (9, 5, 600), (11, 8, 333), (23, 1, 200), (40, 5, 70)])
def test_map_sizes_and_beam_counts_vs_oracle(ms, beams, n):
    """Largest grid (one tile per SM, 8 warps per tile), generic lidar LUT path (beam counts != 8, also on a grid above
    32x32), tiny grids."""
    cc = _compiled({'env': scenarios.BOW, 'map_size': ms, 'chain': [['lidar', beams]]})
    _parity_vs_oracle([cc], n, 48, seed0=4242)


def test_no_lidar_dict_observation_batch_with_auto_reset():
    cc = _compiled({'env': scenarios.POGO, 'map_size': 10, 'chain': []})
    assert cc.obs_dim == 0
    n = 1500
    ob = OracleBatch([cc], n)
    ob.reset_legacy(1)
    h = BatchHandle([cc], n)
    h.load_state(ob.map, ob.pose, ob.inv)
    rng = np.random.RandomState(0)
    for t in range(24):
        a = rng.randint(0, cc.c.n_actions, size=n).astype(np.int32)
        o_obs, o_rew, o_done, o_cost, o_res = ob.step(a)
        obs, rew, done, cost, res = h.step(torch.from_numpy(a).cuda())
        assert np.array_equal(rew.cpu().numpy(), o_rew) and np.array_equal(res.cpu().numpy(), o_res)
    assert np.array_equal(h.map.cpu().numpy().reshape(n, -1), ob.map) and np.array_equal(h.inventory.cpu().numpy(), ob.inv)
    for t in range(6):
        h.step(torch.zeros(n, dtype=torch.int32, device='cuda'), auto_reset=True, max_episode_steps=3)
    assert (h.episode.cpu().numpy() == 2).all() and int(h.error_flags.abs().sum().item()) == 0


def test_placement_failure_rate_matches_reference_on_a_crowded_grid():
    """AxeHard(iron) puts 11 items into the 6x6 interior: the reference sometimes asserts 'Cannot place items'
    (pogostick_v1_env.py:167); the GPU generator must fail at the same rate and flag it."""
    cc = _compiled(golden_util.get('pogo_A_axe_hard_iron_inc')['meta'])
    n = 20000
    h = BatchHandle([cc], n, seed=12)
    h.reset()
    gpu_fail = ((h.error_flags.cpu().numpy() & 2) != 0).mean()
    ref = OracleBatch([cc], n)
    ref_fail = (ref.reset_legacy(31) != 0).mean()
    assert abs(gpu_fail - ref_fail) < 4 * np.sqrt(max(ref_fail, 1e-4) / n) + 2e-4, (gpu_fail, ref_fail)


def test_closed_loop_policy_rollout_matches_host_replay():
    """N1 policy hook: observations consumed and actions produced on the device (integer linear policy, greedy)."""
    cc = _compiled({'env': scenarios.POGO, 'map_size': 10, 'chain': [['limit', scenarios.C2_SET], ['lidar', 8]]})
    n, T, A = 1500 + 3, 48, cc.c.n_actions
    ob = OracleBatch([cc], n)
    ob.reset_legacy(2718)
    h = BatchHandle([cc], n)
    h.load_state(ob.map, ob.pose, ob.inv)
    rng = np.random.RandomState(3)
    W = rng.randint(-9, 10, size=(cc.obs_dim, A)).astype(np.int32)
    b = rng.randint(-30, 31, size=A).astype(np.int32)
    out = h.rollout(T, policy=(W, b), record_actions=True)
    taken = out[-1].cpu().numpy()
    rew = np.zeros(n)
    for t in range(T):
        obs = ob.observe().astype(np.int64)
        a = np.argmax(obs @ W.astype(np.int64) + b, axis=1).astype(np.int32)       # first maximum, like the kernel
        assert np.array_equal(a, taken[t]), "step %d" % t
        o_obs, o_rew, o_done, o_cost, o_res = ob.step(a)
        rew += o_rew
    assert len(np.unique(taken)) >= 4                                             # the policy is not degenerate
    assert np.array_equal(h.map.cpu().numpy().reshape(n, -1), ob.map) and np.array_equal(h.pose.cpu().numpy(), ob.pose)
    assert np.array_equal(h.inventory.cpu().numpy(), ob.inv)
    assert np.array_equal(out[0].cpu().numpy()[:, :cc.obs_dim], o_obs) and np.array_equal(out[1].cpu().numpy(), rew)


# ---------------------------------------------------------------------------------------------- round 2 additions
C2_DESC = {'env': scenarios.POGO, 'map_size': 10, 'chain': [['limit', scenarios.C2_SET], ['lidar', 8]]}


def _u8_rows_to_vector(h, rows, cfg_ids=None):
    """NGW_OBS_U8 rows -> the reference's int32 vector (lidar ranges then inventory tail), per env."""
    rows = rows.cpu().numpy() if hasattr(rows, 'cpu') else rows
    out = np.zeros((rows.shape[0], h.obs_dim), np.int32)
    ids = np.zeros(rows.shape[0], np.int64) if cfg_ids is None else np.asarray(cfg_ids, np.int64)
    for k, cc in enumerate(h.compiled):
        sel = ids == k
        if not sel.any():
            continue
        lidar, tail = h.split_obs(rows, cfg=k)
        nl, ni = lidar.shape[1], tail.shape[1]
        out[sel, :nl] = lidar[sel]
        out[sel, nl:nl + ni] = np.ascontiguousarray(tail)[sel]
    return out


@pytest.mark.parametrize('case', ['C2', 'C4', 'C5', 'generic16'])
def test_compact_u8_observation_rows_equal_the_int32_vector(case):
    """NGW_OBS_U8 (uint8 lidar ranges + int32 inventory tail) carries exactly the reference's vector: every step
    compared with the oracle, device path and host-buffer path, single and mixed configs, map 40 with auto-reset."""
    cfg_id = None
    if case == 'C2':
        compiled, n, steps = [_compiled(C2_DESC)], 3000 + 11, 48
    elif case == 'C4':
        descs = [dict(C2_DESC, chain=[['limit', scenarios.C2_SET + ex], ['lidar', 8], nov]) for ex, nov in (
            (['Chop'], ['novelty', 'addchop', 'hard', '', '']), (['Jump'], ['novelty', 'addjump', 'hard', '', '']),
            ([], ['novelty', 'additem', 'medium', 'spring', '']), ([], ['novelty', 'remapaction', 'hard', '', '']))]
        compiled, n, steps = [_compiled(d) for d in descs], 2048 + 9, 40
        cfg_id = (np.arange(n) % 4).astype(np.uint8)
    elif case == 'C5':
        compiled, n, steps = [_compiled(golden_util.get('pogo_ms40_additem_hard')['meta'])], 200, 40
    else:
        compiled, n, steps = [_compiled({'env': scenarios.BOW, 'map_size': 12, 'chain': [['lidar', 16]]})], 500, 32
    ob = OracleBatch(compiled, n, cfg_id=cfg_id)
    ob.reset_legacy(808)
    hd = BatchHandle(compiled, n, cfg_id=None if cfg_id is None else cfg_id.astype(np.int32), obs_format='u8')
    hh = BatchHandle(compiled, n, cfg_id=None if cfg_id is None else cfg_id.astype(np.int32), obs_format='u8')
    for h in (hd, hh):
        h.load_state(ob.map, ob.pose, ob.inv)
    assert hd.obs.dtype == torch.uint8 and hd.obs_row_bytes < 4 * hd.obs_dim
    assert np.array_equal(_u8_rows_to_vector(hd, hd.observe(), cfg_id), ob.observe())
    n_act = np.array([cc.c.n_actions for cc in compiled])[ob.cfg_id.astype(np.int64)]
    rng = np.random.RandomState(4)
    for t in range(steps):
        a = (rng.randint(0, 1 << 30, size=n) % n_act).astype(np.int32)
        o_obs, o_rew, o_done, o_cost, o_res = ob.step(a, n_threads=8)
        obs, rew, done, cost, res = hd.step(torch.from_numpy(a).cuda())
        assert np.array_equal(_u8_rows_to_vector(hd, obs, cfg_id), o_obs), "device step %d" % t
        assert np.array_equal(rew.cpu().numpy(), o_rew) and np.array_equal(done.cpu().numpy(), o_done)
        hobs, hrew, hdone, hcost, hres = hh.step_host(a)
        assert np.array_equal(_u8_rows_to_vector(hh, hobs, cfg_id), o_obs), "host step %d" % t
        assert np.array_equal(hrew, o_rew) and np.array_equal(hres, o_res)
    assert np.array_equal(hd.map.cpu().numpy().reshape(n, -1), ob.map) and np.array_equal(hh.inventory.cpu().numpy(), ob.inv)
    if case == 'C5':                                                  # the queued auto-reset writes u8 rows too
        hi = BatchHandle(compiled, n)                                 # int32 twin: same seed, same state, same steps
        hi.load_state(*hd.export_state())
        hi.episode.copy_(hd.episode)
        for t in range(6):
            a = torch.zeros(n, dtype=torch.int32, device='cuda')
            obs = hd.step(a, auto_reset=True, max_episode_steps=3)[0]
            ref = hi.step(a, auto_reset=True, max_episode_steps=3)[0]
            assert np.array_equal(_u8_rows_to_vector(hd, obs), ref.cpu().numpy()[:, :hd.obs_dim]), "auto-reset step %d" % t
        assert (hd.episode.cpu().numpy() == 2).all() and torch.equal(hd.map, hi.map)


TILE_GROUP_CHAINS = [C2_DESC, 'bow_C3_axe_medium_fence_hard', 'pogo_crate_over_fr_hard', 'pogo_ms40_additem_hard']
SINGLE = [[0], [1], [2], [3]]
# Inputs that send a one-step launch to each shape of the tile-group kernel (step1_kernel<NC, kOne, kAlias>): map size,
# beam count, batch size, and the batches to run — lists of TILE_GROUP_CHAINS indices, interleaved env by env when a
# batch has several configs.  G = warps per tile.
TILE_GROUP_SHAPES = {
    'G4-alias': (40, 8, 32 * 9 + 3, SINGLE),                # > 32x32: pointer-walking lidar, one tile per CTA, alias plan
    'G4-multi': (33, 8, 32 * 300 + 5, SINGLE),              # one wave of 2-tile CTAs (named barriers)
    'G2-multi': (12, 16, 32 * 300 + 5, SINGLE),             # generic lidar LUT: one wave of 2-tile CTAs
    'G2-waves': (12, 16, 32 * 1500 + 5, SINGLE),            # several waves: one tile per CTA
    'G1-mixed': (12, 16, 32 * 37 + 5, [[0, 2], [3, 2]]),    # two configs per batch: one warp per tile
}


def tile_group_inputs(case, batch=0):
    """(compiled configs, batch size, cfg_id or None) of batch `batch` of a TILE_GROUP_SHAPES case."""
    ms, beams, n, batches = TILE_GROUP_SHAPES[case]
    compiled = []
    for k in batches[batch]:
        d = TILE_GROUP_CHAINS[k]
        d = d if isinstance(d, dict) else golden_util.get(d)['meta']
        chain = [['lidar', beams] if step[0] == 'lidar' else step for step in d['chain']]
        compiled.append(_compiled(dict(d, map_size=ms, chain=chain)))
    cfg_id = (np.arange(n) % len(compiled)).astype(np.uint8) if len(compiled) > 1 else None
    return compiled, n, cfg_id


@pytest.mark.parametrize('case', sorted(TILE_GROUP_SHAPES))
def test_tile_group_kernel_shapes(case):
    """Every shape of the tile-group kernel that an input selects: with >= 2 warps per tile the step is split by action
    class (warp 0: turns / crafts / selects, warp 1: moves and block-in-front actions) and the lidar is shared out over
    the warps; a CTA runs several tile groups side by side (named barriers).  Same results as the oracle for single and
    mixed configs, layered novelties, partial last tile / partial last CTA, auto-reset queueing from both stepping warps,
    CTA-level statistics."""
    for batch in range(len(TILE_GROUP_SHAPES[case][3])):
        compiled, n, cfg_id = tile_group_inputs(case, batch)
        _parity_vs_oracle(compiled, n, 12 if n > 20000 else 24, seed0=100 * batch + 1, cfg_id=cfg_id)
    compiled, n, cfg_id = tile_group_inputs(case)
    h = BatchHandle(compiled, n, seed=2, cfg_id=None if cfg_id is None else cfg_id.astype(np.int32))
    h.reset()
    n_act = np.array([cc.c.n_actions for cc in compiled])[np.zeros(n, np.int64) if cfg_id is None else cfg_id]
    rng = np.random.RandomState(1)
    dones = 0
    for t in range(12):
        a = torch.from_numpy((rng.randint(0, 1 << 30, size=n) % n_act).astype(np.int32)).cuda()
        dones += int(h.step(a, auto_reset=True, max_episode_steps=4)[2].sum().item())
    st = h.stats().cpu().numpy()
    assert dones == 3 * n and (h.episode.cpu().numpy() == 4).all() and st[0] == 12 * n and st[5] == 3 * n
    assert st[1] == dones


# one tile per CTA / several tiles per CTA in a one-wave launch that waits for its predecessor / several waves
WARP_PER_TILE_BATCHES = [32 * 37 + 5, 32 * 400 + 5, 32 * 148 * 15 + 5]


@pytest.mark.parametrize('n0', WARP_PER_TILE_BATCHES)
def test_warp_per_tile_shape(n0):
    """step1w_kernel: one warp per tile, the observation tile aliases the grid / inventory rows in shared memory (hits and
    inventory tail wait in registers), two consecutive launches share an SM.  Same results as the oracle for single and
    mixed configs, layered novelties, partial last tile / partial last CTA, u8 rows, observe-only launches, auto-reset
    queueing and CTA-level statistics; back-to-back launches of rotating handles (early state loads under PDL)."""
    _parity_vs_oracle([_compiled(C2_DESC)], n0, 40, seed0=n0 % 1000)
    _parity_vs_oracle([_compiled(golden_util.get('bow_C3_axe_medium_fence_hard')['meta'])], n0 - 4, 24, seed0=n0 % 7)
    _parity_vs_oracle([_compiled(golden_util.get('pogo_crate_over_fr_hard')['meta'])], n0 + 11, 24, seed0=3)
    _parity_vs_oracle([_compiled({'env': scenarios.POGO, 'map_size': 23, 'chain': [['lidar', 8]]})], n0 - 32, 24, seed0=11)
    cc = _compiled(C2_DESC)
    n = n0
    h = BatchHandle([cc], n, seed=2)
    h.reset()
    rng = np.random.RandomState(1)
    dones = 0
    for t in range(12):
        a = torch.from_numpy(rng.randint(0, cc.c.n_actions, size=n).astype(np.int32)).cuda()
        dones += int(h.step(a, auto_reset=True, max_episode_steps=4)[2].sum().item())
    st = h.stats().cpu().numpy()
    assert dones == 3 * n and (h.episode.cpu().numpy() == 4).all() and st[0] == 12 * n and st[5] == 3 * n
    assert st[1] == dones
    # rotating handles back to back on one stream, no host synchronisation in between (early state loads, co-resident
    # launches), u8 and i32 rows, against handles stepped one at a time with a synchronise after every launch
    n = 32 * 150 + 7
    rng = np.random.RandomState(5)
    for fmt in ('i32', 'u8'):
        hs = [BatchHandle([cc], n, seed=40 + k, obs_format=fmt) for k in range(3)]
        ref = [BatchHandle([cc], n, seed=40 + k, obs_format=fmt) for k in range(3)]
        for x in hs + ref:
            x.reset()
        torch.cuda.synchronize()
        acts = [torch.from_numpy(rng.randint(0, cc.c.n_actions, size=n).astype(np.int32)).cuda() for _ in range(30)]
        outs = []
        for t in range(30):
            outs.append([x.clone() for x in hs[t % 3].step(acts[t])])
        torch.cuda.synchronize()
        for t in range(30):
            want = ref[t % 3].step(acts[t])
            torch.cuda.synchronize()
            for x, y in zip(outs[t], want):
                assert torch.equal(x, y), "launch %d (%s)" % (t, fmt)
        for a, b in zip(hs, ref):
            assert torch.equal(a.map, b.map) and torch.equal(a.inventory, b.inventory) and torch.equal(a.pose, b.pose)
        # the same rotation as ONE captured graph: launches 2.. are proven independent of their predecessor and overlap
        # it (gate warp); replayed three times against the one-at-a-time handles
        stream = torch.cuda.Stream()
        graph = torch.cuda.CUDAGraph()
        keep = []
        c0 = sum(x.concurrent_launch_count() for x in hs)
        with torch.cuda.stream(stream):
            with torch.cuda.graph(graph, stream=stream):
                for t in range(12):
                    keep.append(hs[t % 3].step(acts[t]))
        n_conc = sum(x.concurrent_launch_count() for x in hs) - c0
        assert n_conc == 11, n_conc
        for rep in range(3):
            graph.replay()
            torch.cuda.synchronize()
            for t in range(12):
                want = ref[t % 3].step(acts[t])
                torch.cuda.synchronize()
                if t >= 9:                                        # each handle's buffers hold its latest step
                    for x, y in zip(keep[t], want):
                        assert torch.equal(x, y), "graph replay %d launch %d (%s)" % (rep, t, fmt)
            for a, b in zip(hs, ref):
                assert torch.equal(a.map, b.map) and torch.equal(a.inventory, b.inventory) and torch.equal(a.pose, b.pose)
                np.testing.assert_allclose(a.stats(reset=False).cpu().numpy(), b.stats(reset=False).cpu().numpy(), rtol=1e-6)   # cost sums: float partials per CTA, the CTA shape depends on the launch mode
        # a handle stepped twice in a row, or buffers shared between neighbours, are never overlapped
        c0 = hs[0].concurrent_launch_count() + hs[1].concurrent_launch_count()
        g2 = torch.cuda.CUDAGraph()
        with torch.cuda.stream(stream):
            with torch.cuda.graph(g2, stream=stream):
                hs[0].step(acts[0]); hs[0].step(acts[1])
                hs[1].step(hs[0].reward.view(torch.int32))        # actions alias the predecessor's output
        assert hs[0].concurrent_launch_count() + hs[1].concurrent_launch_count() == c0


@pytest.mark.parametrize('case', ['C2', 'ms40', 'bow12_16beams', 'C2-two', 'ms40-two', 'C3-waves-two'])
def test_overlapped_steps_with_queued_resets_in_a_graph(case):
    """Inside one captured graph, handle B's step is independent of handle A's step AND of A's queued-reset kernel behind
    it: the library proves adjacency and overlaps them (gate warp / gate CTA keep stream order).  Rotating handles with
    auto-reset and truncation, replayed several times, against handles stepped one launch at a time."""
    H = 2 if case.endswith('-two') else 3      # two handles: launch N + 2 steps the handle of launch N again
    if case.startswith('C2'):
        cc, n = _compiled(C2_DESC), 32 * 90 + 5                        # warp-per-tile kernel, one wave
    elif case.startswith('C3'):
        cc, n = _compiled(golden_util.get('bow_C3_axe_medium_fence_hard')['meta']), 32 * 148 * 28 + 17   # several waves
    elif case.startswith('ms40'):
        cc, n = _compiled(golden_util.get('pogo_ms40_additem_hard')['meta']), 32 * 20 + 3   # tile-group kernel, alias plan
    else:
        cc, n = _compiled({'env': scenarios.BOW, 'map_size': 12, 'chain': [['lidar', 16]]}), 500   # generic lidar, no alias
    rng = np.random.RandomState(12)
    hs = [BatchHandle([cc], n, seed=70 + k) for k in range(H)]
    ref = [BatchHandle([cc], n, seed=70 + k) for k in range(H)]
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
    n_conc = sum(x.concurrent_launch_count() for x in hs) - c0
    assert n_conc == 11, n_conc
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
            assert torch.equal(a.map, b.map) and torch.equal(a.inventory, b.inventory) and torch.equal(a.pose, b.pose)
            assert torch.equal(a.episode, b.episode) and torch.equal(a.ep_len, b.ep_len)
            np.testing.assert_allclose(a.stats(reset=False).cpu().numpy(), b.stats(reset=False).cpu().numpy(), rtol=1e-6)   # cost sums: float partials per CTA, the CTA shape depends on the launch mode
    assert int(hs[0].episode.min().item()) >= 4


def test_reset_then_host_step_is_ordered_after_the_reset():
    """ADVICE r1 (high): env.reset(); env.step(numpy_actions) — the host-buffer step runs on the handle's own stream and
    must see the reset that was enqueued on the caller's stream.  Large batch, many rounds, compared with a handle
    driven through the device path with explicit synchronisation."""
    cc = _compiled(golden_util.get('pogo_ms40_additem_hard')['meta'])     # 1600-cell grids: a slow reset
    n = 20000
    a_host = np.random.RandomState(0).randint(0, cc.c.n_actions, size=n).astype(np.int32)
    h1, h2 = BatchHandle([cc], n, seed=5), BatchHandle([cc], n, seed=5)
    for rnd in range(4):
        h1.reset()                                                    # no synchronize: step_host must order itself
        got = [np.array(x) for x in h1.step_host(a_host)]
        h2.reset()
        torch.cuda.synchronize()
        ref = [x.cpu().numpy() for x in h2.step(torch.from_numpy(a_host).cuda())]
        torch.cuda.synchronize()
        for x, y in zip(got, ref):
            assert np.array_equal(x, y), "round %d" % rnd
        assert torch.equal(h1.map, h2.map) and torch.equal(h1.inventory, h2.inventory) and torch.equal(h1.pose, h2.pose)
        # and the other direction: a device-path call right after an unfinished host-path call
        h1.step_host_begin(a_host)
        d1 = [x.clone() for x in h1.step(torch.from_numpy(a_host).cuda())]
        h1.step_host_end()
        h2.step(torch.from_numpy(a_host).cuda())
        d2 = h2.step(torch.from_numpy(a_host).cuda())
        for x, y in zip(d1, d2):
            assert torch.equal(x, y)


def test_export_state_device_and_host_subrange():
    cc = _compiled(C2_DESC)
    n = 700
    h = BatchHandle([cc], n, seed=9)
    h.reset()
    m, p, v = h.export_state()
    assert torch.equal(m, h.map) and torch.equal(p, h.pose) and torch.equal(v, h.inventory)
    m2, p2, v2 = h.export_state(first=100, count=333, host=True)
    assert not m2.is_cuda and np.array_equal(m2.numpy(), h.map[100:433].cpu().numpy())
    assert np.array_equal(p2.numpy(), h.pose[100:433].cpu().numpy()) and np.array_equal(v2.numpy(), h.inventory[100:433].cpu().numpy())
    h2 = BatchHandle([cc], 333)
    h2.load_state(m2, p2, v2)                                         # export -> load round trip
    assert torch.equal(h2.map, h.map[100:433]) and torch.equal(h2.pose, h.pose[100:433])
    with pytest.raises(RuntimeError):
        h.export_state(first=600, count=200)


def test_auto_reset_observation_is_the_reference_reset_observation():
    """Quirk Q3 under auto-reset: AxeEasy wrapped outside LidarInFront patches the inventory AFTER the reset observation
    was computed (novelty_wrappers.py:29-35), so the observation row of a regenerated env shows axe count 0 while the
    state has 1 — the queued auto-reset must return what ngw_reset (and the reference's reset()) returns."""
    cc = _compiled(golden_util.get('pogo_A_axe_easy_wooden')['meta'])
    assert cc.c.reset_obs_after_ops < cc.c.n_reset_ops
    n = 600
    h = BatchHandle([cc], n, seed=21)
    h.reset()
    axe = [i for i, nm in enumerate(cc.item_names) if nm == 'wooden_axe'][0]
    tail_pos = cc.c.n_lidar_items * cc.c.n_beams + [cc.c.inv_obs_item[i] for i in range(cc.c.n_inv_obs)].index(axe)
    for t in range(4):
        obs = h.step(torch.full((n,), 1, dtype=torch.int32, device='cuda'), auto_reset=True, max_episode_steps=2)[0]
    o = obs.cpu().numpy()
    assert (h.episode.cpu().numpy() == 3).all()
    assert (h.inventory.cpu().numpy()[:, axe] == 1).all() and (o[:, tail_pos] == 0).all()
    # the same rows from ngw_reset on a twin handle whose Philox counters are at the same episode
    twin = BatchHandle([cc], n, seed=21)
    for _ in range(3):
        robs = twin.reset()
    assert torch.equal(twin.map, h.map) and torch.equal(twin.pose, h.pose)
    assert np.array_equal(robs.cpu().numpy(), o)


def test_closed_loop_rollout_final_observation_is_clean():
    """ADVICE r1 (medium): the observation returned by ngw_rollout_policy must not keep lidar slots of the previous
    step's policy observation.  T is short so that most envs still move on the last step."""
    cc = _compiled(C2_DESC)
    n, A = 2000, cc.c.n_actions
    rng = np.random.RandomState(8)
    W = rng.randint(-9, 10, size=(cc.obs_dim, A)).astype(np.int32)
    b = rng.randint(-30, 31, size=A).astype(np.int32)
    for T in (1, 2, 3, 5):
        ob = OracleBatch([cc], n)
        ob.reset_legacy(4000 + T)
        h = BatchHandle([cc], n)
        h.load_state(ob.map, ob.pose, ob.inv)
        out = h.rollout(T, policy=(W, b), record_actions=True)
        changed = 0
        for t in range(T):
            before = ob.observe().astype(np.int64)
            a = np.argmax(before @ W.astype(np.int64) + b, axis=1).astype(np.int32)
            after = ob.step(a)[0]
            changed = int((after != before).any(axis=1).sum())
        if T == 1:
            assert changed > n // 20, "the last step must still change observations for this test to bite"
        assert np.array_equal(out[0].cpu().numpy()[:, :cc.obs_dim], after), "T=%d" % T


def test_step_many_overlaps_handles_in_eager_mode():
    """ngw_step_many: one call steps several handles back to back, so the library knows the launches are adjacent and
    overlaps them without a stream capture; same results as one ngw_step per handle with a synchronise in between.  The
    same handle twice in one call, or a shared output buffer, are never overlapped."""
    from gym_novel_gridworlds_b200.runtime import step_many
    for desc, n in ((C2_DESC, 32 * 120 + 9), (golden_util.get('pogo_ms40_additem_hard')['meta'], 32 * 12 + 1)):
        cc = _compiled(desc)
        hs = [BatchHandle([cc], n, seed=90 + k) for k in range(4)]
        ref = [BatchHandle([cc], n, seed=90 + k) for k in range(4)]
        for x in hs + ref:
            x.reset()
        torch.cuda.synchronize()
        rng = np.random.RandomState(2)
        c0 = sum(x.concurrent_launch_count() for x in hs)
        for rnd in range(8):
            acts = [torch.from_numpy(rng.randint(0, cc.c.n_actions, size=n).astype(np.int32)).cuda() for _ in range(4)]
            outs = step_many(hs, acts, auto_reset=True, max_episode_steps=5)
            torch.cuda.synchronize()
            for k in range(4):
                want = ref[k].step(acts[k], auto_reset=True, max_episode_steps=5)
                torch.cuda.synchronize()
                for x, y in zip(outs[k], want):
                    assert torch.equal(x, y), "round %d handle %d" % (rnd, k)
        assert sum(x.concurrent_launch_count() for x in hs) - c0 == 8 * 3          # items 2..4 of every call
        for a, b in zip(hs, ref):
            assert torch.equal(a.map, b.map) and torch.equal(a.inventory, b.inventory) and torch.equal(a.pose, b.pose)
            assert torch.equal(a.episode, b.episode)
        c0 = sum(x.concurrent_launch_count() for x in hs)
        a0 = torch.zeros(n, dtype=torch.int32, device='cuda')
        step_many([hs[0], hs[0], hs[1]], [a0, a0, a0])                                # same handle twice: item 2 waits
        assert sum(x.concurrent_launch_count() for x in hs) - c0 == 1


def test_step_many_mixes_kernel_shapes():
    """One ngw_step_many call over handles that take DIFFERENT kernels (warp-per-tile, tile groups with the alias plan,
    tile groups with the generic lidar, mixed configs): launches of neighbouring items overlap across kernel shapes (gate
    warp next to gate CTA); same results as stepping every handle alone."""
    from gym_novel_gridworlds_b200.runtime import StepGroup
    specs = [([_compiled(C2_DESC)], 32 * 70 + 3, None),
             ([_compiled(golden_util.get('pogo_ms40_additem_hard')['meta'])], 32 * 6 + 1, None),
             ([_compiled({'env': scenarios.BOW, 'map_size': 12, 'chain': [['lidar', 16]]})], 300, None),
             ([_compiled(d) for d in _c4_descs()], 32 * 40 + 5, 4),
             ([_compiled(golden_util.get('bow_C3_axe_medium_fence_hard')['meta'])], 32 * 148 * 14 + 9, None)]
    hs, ref = [], []
    for k, (compiled, n, ncfg) in enumerate(specs):
        cfg_id = None if ncfg is None else (np.arange(n) % ncfg).astype(np.int32)
        for group in (hs, ref):
            h = BatchHandle(compiled, n, seed=300 + k, cfg_id=cfg_id)
            h.reset()
            group.append(h)
    torch.cuda.synchronize()
    group = StepGroup(hs)
    rng = np.random.RandomState(9)
    c0 = sum(x.concurrent_launch_count() for x in hs)
    for rnd in range(10):
        acts = []
        for h in hs:
            n_act = torch.tensor([cc.c.n_actions for cc in h.compiled], device='cuda')[h.cfg_id.long()]
            acts.append((torch.from_numpy(rng.randint(0, 1 << 30, size=h.n)).cuda() % n_act).to(torch.int32))
        outs = group.step(acts, auto_reset=True, max_episode_steps=4)
        torch.cuda.synchronize()
        for k, h in enumerate(ref):
            want = h.step(acts[k], auto_reset=True, max_episode_steps=4)
            torch.cuda.synchronize()
            for x, y in zip(outs[k], want):
                assert torch.equal(x, y), "round %d handle %d" % (rnd, k)
    assert sum(x.concurrent_launch_count() for x in hs) - c0 == 10 * (len(hs) - 1)
    for a, b in zip(hs, ref):
        assert torch.equal(a.map, b.map) and torch.equal(a.inventory, b.inventory) and torch.equal(a.pose, b.pose)
        assert torch.equal(a.episode, b.episode) and torch.equal(a.ep_len, b.ep_len)


def _c4_descs():
    return [dict(C2_DESC, chain=[['limit', scenarios.C2_SET + ex], ['lidar', 8], nov]) for ex, nov in (
        (['Chop'], ['novelty', 'addchop', 'hard', '', '']), (['Jump'], ['novelty', 'addjump', 'hard', '', '']),
        ([], ['novelty', 'additem', 'medium', 'spring', '']), ([], ['novelty', 'remapaction', 'hard', '', '']))]


def rollout_case_inputs(case):
    """(compiled configs, batch size, cfg_id or None) of a case of test_rollout_kernels_equal_repeated_steps_on_other_shapes:
    grids up to 32x32 take the lane-pair rollout kernel (rollout2_kernel), 40x40 grids and 16 beams the one-warp-per-tile
    kernel (rollout_kernel)."""
    cfg_id = None
    if case == 'c2_u8':
        compiled, n = [_compiled(C2_DESC)], 32 * 20 + 11
    elif case == 'pogo_ms40_u8':
        compiled, n = [_compiled(golden_util.get('pogo_ms40_additem_hard')['meta'])], 32 * 2 + 9
    elif case == 'pogo_ms23':
        compiled, n = [_compiled({'env': scenarios.POGO, 'map_size': 23, 'chain': [['limit', scenarios.C2_SET], ['lidar', 8]]})], 32 * 9 + 7
    elif case == 'bow_ms13':
        compiled, n = [_compiled(golden_util.get('bow_ms13_lidar')['meta'])], 32 * 11 + 1
    elif case == 'c4_mixed':
        compiled, n = [_compiled(d) for d in _c4_descs()], 32 * 14 + 19
        cfg_id = (np.arange(n) % 4).astype(np.int32)
    elif case == 'c3_layers':
        compiled, n = [_compiled(golden_util.get('bow_C3_axe_medium_fence_hard')['meta'])], 32 * 8 + 3
    elif case == 'pogo_ms40':
        compiled, n = [_compiled(golden_util.get('pogo_ms40_additem_hard')['meta'])], 32 * 3 + 5
    else:
        compiled, n = [_compiled({'env': scenarios.BOW, 'map_size': 12, 'chain': [['lidar', 16]]})], 200
    return compiled, n, cfg_id


@pytest.mark.parametrize('case', ['pogo_ms23', 'bow_ms13', 'c4_mixed', 'c3_layers', 'pogo_ms40', 'bow12_16beams', 'c2_u8', 'pogo_ms40_u8'])
@pytest.mark.parametrize('mode', ['given', 'given+autoreset', 'policy', 'random'])
def test_rollout_kernels_equal_repeated_steps_on_other_shapes(case, mode):
    """The K-step rollout kernels (lane-pair kernel on grids up to 32x32 incl. its generic-size lidar, mixed configs through
    the global config table, layered novelties; the one-warp-per-tile kernel on 40x40 grids and 16 beams) against the same
    steps issued one launch at a time: states, sums, final observation, episode counters; closed loop: every action is the
    argmax of the integer policy on the twin's observation; auto-reset with truncation regenerates the same episodes."""
    fmt = 'u8' if case.endswith('_u8') else 'i32'
    if fmt == 'u8' and mode == 'policy':
        pytest.skip("the device policy reads int32 observation rows")
    compiled, n, cfg_id = rollout_case_inputs(case)
    T = 24
    kw = dict(auto_reset=True, max_episode_steps=7) if mode == 'given+autoreset' else {}
    h1 = BatchHandle(compiled, n, seed=21, cfg_id=cfg_id, obs_format=fmt)   # one launch per step
    h2 = BatchHandle(compiled, n, seed=21, cfg_id=cfg_id, obs_format=fmt)   # one launch for all T steps
    h1.reset(); h2.reset()
    n_act = torch.tensor([cc.c.n_actions for cc in compiled], device='cuda')[h1.cfg_id.long()]
    A = int(n_act.max().item())
    rng = np.random.RandomState(17)
    if mode == 'policy':
        if A > 16:
            pytest.skip("the device policy scores at most 16 actions")
        W = torch.from_numpy(rng.randint(-9, 10, size=(h1.obs_dim, A)).astype(np.int32)).cuda()
        b = torch.from_numpy(rng.randint(-30, 31, size=A).astype(np.int32)).cuda()
        out = h2.rollout(T, policy=(W, b), record_actions=True, **kw)
        acts = out[-1]
    elif mode == 'random':
        out = h2.rollout(T, None, policy_seed=5, record_actions=True, **kw)
        acts = out[-1]
        assert int(acts.min().item()) >= 0 and bool((acts < n_act[None, :]).all().item())
    else:
        acts = torch.from_numpy((rng.randint(0, 1 << 30, size=(T, n)) % n_act.cpu().numpy()[None, :]).astype(np.int32)).cuda()
        out = h2.rollout(T, acts, **kw)
    rew = torch.zeros(n, device='cuda'); cost = torch.zeros(n, dtype=torch.float64, device='cuda')
    dones = torch.zeros(n, dtype=torch.int64, device='cuda')
    obs = h1.observe().clone()
    for t in range(T):
        if mode == 'policy':                                          # the action the device must have taken: first maximum
            score = obs[:, :h1.obs_dim].double() @ W.double() + b.double()[None, :]      # exact: small integers
            score = torch.where(torch.arange(A, device='cuda')[None, :] < n_act[:, None], score, torch.full_like(score, -1e18))
            assert torch.equal(torch.argmax(score, dim=1).to(torch.int32), acts[t]), "step %d" % t
        o, r, d, c, res = h1.step(acts[t].contiguous(), **kw)
        obs = o.clone()
        rew += r; cost += c.double(); dones += d.long()
    assert torch.equal(h1.map, h2.map) and torch.equal(h1.pose, h2.pose) and torch.equal(h1.inventory, h2.inventory)
    assert torch.equal(h1.episode, h2.episode) and torch.equal(h1.ep_len, h2.ep_len)
    assert torch.equal(out[0], o) and torch.equal(out[4], d) and torch.equal(out[5], res)
    assert torch.equal(out[1], rew) and torch.equal(out[3].long(), dones)
    np.testing.assert_allclose(out[2].cpu().numpy(), cost.cpu().numpy(), rtol=1e-5)
    s1, s2 = h1.stats().cpu().numpy(), h2.stats().cpu().numpy()
    assert np.array_equal(s1[[0, 1, 2, 3, 5, 6]], s2[[0, 1, 2, 3, 5, 6]])
    np.testing.assert_allclose(s1[4], s2[4], rtol=1e-6)


def _long_case(names):
    """(compiled configs, cfg ids, per-env trace rows) for one or several long-trace configs run as ONE batch; several
    configs are interleaved env i -> config i mod len(names), like BASELINE config C4."""
    gs = [golden_util.long_get(nm) for nm in names]
    compiled = [_compiled(g['meta']) for g in gs]
    E, T = gs[0]['actions'].shape
    assert all(g['actions'].shape == (E, T) for g in gs)
    k = len(names)
    n = E * k
    cfg = (np.arange(n) % k).astype(np.uint8)
    ms2 = gs[0]['init_map'].shape[1]
    width = max(cc.n_items for cc in compiled)
    init_map = np.zeros((n, ms2), np.int8); init_pose = np.zeros((n, 4), np.uint8); init_inv = np.zeros((n, width), np.int32)
    actions = np.zeros((n, T), np.int32); hashes = np.zeros((n, T), np.uint64)
    for j, g in enumerate(gs):
        init_map[j::k] = g['init_map']; init_pose[j::k] = g['init_pose']
        init_inv[j::k, :g['init_inv'].shape[1]] = g['init_inv']
        actions[j::k] = g['actions']; hashes[j::k] = g['hash']
    return gs, compiled, cfg, init_map, init_pose, init_inv, actions, hashes


@pytest.mark.skipif(not golden_util.long_names(), reason="tests/golden/long_traces.npz is missing")
@pytest.mark.parametrize('case', ['C2', 'C3', 'C4', 'C5'])
def test_gpu_replays_hashed_long_reference_traces(case):
    """DIRECT GPU-vs-reference parity at volume: 983,040 steps of the unmodified reference (C2 524k, C3 131k, C4 262k in
    ONE mixed batch with env i -> novelty i mod 4, C5 65k on 40x40 grids), every step's observation / reward / done /
    result / step_cost / inventory / pose / map compared through the 64-bit hash recorded on the reference side."""
    names = ['C4_0', 'C4_1', 'C4_2', 'C4_3'] if case == 'C4' else [case]
    gs, compiled, cfg, init_map, init_pose, init_inv, actions, hashes = _long_case(names)
    n, T = actions.shape
    h = BatchHandle(compiled, n, cfg_id=cfg.astype(np.int32) if len(compiled) > 1 else None)
    h.load_state(init_map, init_pose, init_inv)
    groups = [(np.nonzero(cfg == j)[0], cc, g['init_inv'].shape[1]) for j, (cc, g) in enumerate(zip(compiled, gs))]
    acts = torch.from_numpy(actions.T.copy()).cuda()
    for t in range(T):
        obs, rew, done, cost, res = h.step(acts[t])
        o, r, d, c, s = (x.cpu().numpy() for x in (obs, rew, done, cost, res))
        m, p, v = h.map.cpu().numpy().reshape(n, -1), h.pose.cpu().numpy(), h.inventory.cpu().numpy()
        for idx, cc, n_items in groups:
            got = golden_util.trace_hash(o[idx, :cc.obs_dim], r[idx], d[idx], s[idx], c[idx], v[idx, :n_items], p[idx], m[idx])
            bad = got != hashes[idx, t]
            assert not bad.any(), "%s step %d: %d envs differ from the reference" % (case, t, int(bad.sum()))
    assert int((h.error_flags != 0).sum().item()) == 0
    h.close()


def test_c5_map40_volume_vs_oracle():
    """VERDICT r1 weak #2: C5 (40x40 grids, lidar range 53) at volume: 2,048 envs x 256 steps against the oracle, every
    step; random policies wander far on the large grid, so long beams are sampled."""
    cc = _compiled(golden_util.get('pogo_ms40_additem_hard')['meta'])
    assert _parity_vs_oracle([cc], 2048, 256, seed0=31000) == 2048 * 256


# ---------------------------------------------------------------------------------------------- N3 / N4 against the reference
def _aux_golden():
    import json
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'aux.json')) as f:
        return json.load(f)


def _load_single(env, state):
    """put a recorded reference state into a num_envs == 1 env (after its own reset) and refresh the attribute mirrors"""
    rt = env.unwrapped._runtime
    h = rt.handle
    inv = np.zeros((1, h.inv_stride), np.int32)
    inv[0, :len(state['inv'])] = state['inv']
    h.load_state(np.asarray(state['map'], np.int8).reshape(1, -1), np.asarray([state['pose']], np.uint8), inv)
    rt._sync_single()


def _spec_equal(got, want, info_panel=True):
    assert got['title'] == want['title'] and got['grid'] == want['grid'] and got['vmax'] == want['vmax']
    assert [float(x) for x in got['arrow']] == want['arrow'] and list(got['axis']) == want['axis']
    g = [[float(x), float(y), s] for x, y, s in got['texts']]
    w = [list(t) for t in want['texts']]
    if not info_panel:          # quirk Q12: under a step-intercepting novelty the reference's own step_count / last_* drift
        g, w = g[:1] + g[2:], w[:1] + w[2:]
        assert got['texts'][1][2].split('\n')[2] == want['texts'][1][2].split('\n')[2]        # "Agent Facing: ..."
    assert g == w
    assert [[a, b] for a, b in got['legend']] == want['legend']


def test_render_through_the_env_matches_the_reference():
    """SURVEY §8f N4 end to end: the same states and actions as the reference run through the GPU env; render(mode='spec')
    must list exactly what the reference's render() drew at the same points (info panel with steps / last action /
    reward / step cost / done, banner, legend)."""
    for case in _aux_golden()['render']:
        env = scenarios.build_chain(scenarios.b200_namespace(), case['desc'])
        env.reset()
        _load_single(env, case['reset_state'])
        shots = iter(case['shots'])
        exact = case['tag'] == 'pogo'       # bow_axe: AxeEasy intercepts Break, the reference's bookkeeping drifts (Q12)
        _spec_equal(env.render(mode='spec'), next(shots)['spec'], exact)
        for i, a in enumerate(case['actions']):
            env.step(a)
            if i % 4 == 3:
                shot = next(shots)
                _spec_equal(env.render(mode='spec', title=shot['title_arg']), shot['spec'], exact)
        base = env.unwrapped
        st = dict(next(shots)['state'])                      # the reference put the goal item into the inventory, then stepped
        h = base._runtime.handle
        inv = h.inventory.clone()
        inv[0, base.items_id[case['goal']]] = 1
        h.load_state(h.map.clone(), h.pose.clone(), inv)
        obs, r, d, info = env.step(case['actions'][0])
        assert d and r == 50
        spec = env.render(mode='spec')
        assert spec['texts'][-1][2].startswith('YOU WIN') and 'Done: True' in spec['texts'][1][2]
        if exact:
            assert 'Steps: %d' % st['step_count'] in spec['texts'][1][2]
        assert isinstance(env.render(mode='ansi'), str)
        env.close()


def test_save_trajectories_pickle_matches_the_reference(tmp_path):
    """SURVEY §8f N3: the list SaveTrajectories pickles (wrappers.py:29-54) — keys, per-step values, the aliased live map —
    equals what the unmodified reference wrote for the same episode."""
    import pickle
    import gym_novel_gridworlds_b200 as gym
    g = _aux_golden()['trajectories']
    env = gym.SaveTrajectories(gym.make(g['env']), str(tmp_path))
    env.reset()
    _load_single(env, g['reset_state'])
    for a in g['actions']:
        env.step(a)
    path = env.save()
    assert os.path.basename(path)[19:] == g['file_suffix']
    with open(path, 'rb') as f:
        traj = pickle.load(f)
    assert len(traj) == len(g['trajectory'])
    assert all(t['map'] is traj[0]['map'] for t in traj) == g['map_aliased']
    for got, want in zip(traj, g['trajectory']):
        assert sorted(got) == sorted(want)
        for k, v in want.items():
            x = got[k]
            x = np.asarray(x, int).tolist() if k == 'map' else (list(x) if k == 'agent_location' else x)
            assert x == v, k


def test_env_restore_chain_matches_the_reference():
    """SURVEY §8f N3: gym.make(id, env=previous).reset() (pogostick_v1_env.py:89-109, tests/test_multi_agent.py:55-57): the
    restored state, the bookkeeping copied with it, the observation returned and the following steps equal the
    reference's."""
    import gym_novel_gridworlds_b200 as gym
    g = _aux_golden()['restore']
    first = gym.LidarInFront(gym.make(g['env']), num_beams=8)
    first.reset()
    _load_single(first, g['reset_state'])
    for a in g['actions']:
        first.step(a)
    second = gym.LidarInFront(gym.make(g['env'], env=first), num_beams=8)
    obs = second.reset()
    assert np.asarray(obs).tolist() == g['restored_obs']
    b2, want = second.unwrapped, g['restored_state']
    assert np.asarray(b2.map).tolist() == want['map'] and list(b2.agent_location) == want['pose'][:2]
    assert b2.agent_facing_id == want['pose'][2] and b2.selected_item == want['selected_item']
    assert (b2.last_action, b2.step_count, b2.last_reward, b2.last_done) == (want['last_action'], want['step_count'],
                                                                                  want['last_reward'], want['last_done'])
    inv = [b2.inventory_items_quantity[n] for n in sorted(b2.items_id, key=b2.items_id.get)]
    assert inv == want['inv']
    for a, o in zip(g['more_actions'], g['more_outputs']):
        obs, r, d, info = second.step(a)
        assert np.asarray(obs).tolist() == o['obs'] and r == o['reward'] and d == o['done']
        assert info['result'] == o['result'] and info['step_cost'] == o['step_cost'] and info['message'] == o['message']
    assert np.asarray(b2.map).tolist() == g['final_state']['map'] and b2.step_count == g['final_state']['step_count']
    assert b2.block_in_front_id == g['block_in_front_id']
    assert np.asarray(first.unwrapped.map).tolist() == g['first_state']['map']        # the source env is untouched


def test_batched_invalid_actions_surface():
    """ADVICE r1 (low): a batched step must not swallow rejected action ids.  info['invalid'] marks the envs;
    strict_actions=True raises what the reference raises (wrappers.py:76) and names the first offender; the u8 observation
    format is reachable through gym.make."""
    import gym_novel_gridworlds_b200 as gym
    n = 500
    env = gym.LidarInFront(gym.LimitActions(gym.make('NovelGridworld-Pogostick-v1', num_envs=n, obs_format='u8'),
                                            set(scenarios.C2_SET)))
    obs = env.reset()
    assert obs.dtype == torch.uint8 and obs.shape == (n, 84)
    a = torch.zeros(n, dtype=torch.int32, device='cuda')
    a[17] = 10
    a[400] = -1
    obs, r, d, info = env.step(a)
    bad = info['invalid'].cpu().numpy()
    assert bad.sum() == 2 and bad[17] and bad[400] and obs.shape == (n, 84)
    strict = gym.LidarInFront(gym.LimitActions(gym.make('NovelGridworld-Pogostick-v1', num_envs=n, strict_actions=True),
                                               set(scenarios.C2_SET)))
    strict.reset()
    strict.step(torch.zeros(n, dtype=torch.int32, device='cuda'))
    with pytest.raises(AssertionError, match="env 17 of 2"):
        strict.step(a)
    strict.step(torch.zeros(n, dtype=torch.int32, device='cuda'))       # the flags were cleared by the raise
    with pytest.raises(AssertionError, match="env 400 of 1"):
        strict.step(np.where(np.arange(n) == 400, 11, 0).astype(np.int32))      # host-buffer path too


def test_torch_policy_rollout_graph_matches_host_replay():
    """N1 with a general policy: a CUDA graph of K x [torch policy on the device observation -> ngw_step]; replayed twice;
    the recorded actions are replayed through the oracle and every output must agree."""
    cc = _compiled(C2_DESC)
    n, K, A = 3000 + 17, 12, cc.c.n_actions
    ob = OracleBatch([cc], n)
    ob.reset_legacy(606)
    h = BatchHandle([cc], n)
    h.load_state(ob.map, ob.pose, ob.inv)
    h.observe()
    gen = torch.Generator(device='cuda').manual_seed(0)
    W = torch.randn((cc.obs_dim, A), generator=gen, device='cuda')
    policy = lambda obs: torch.argmax(obs[:, :cc.obs_dim].float() @ W, dim=1).to(torch.int32)     # noqa: E731
    graph, rec = h.capture_policy_rollout(policy, K)
    h.load_state(ob.map, ob.pose, ob.inv)                      # the capture's warm-up did not step, but be explicit
    h.observe()
    for rep in range(2):
        graph.replay()
        torch.cuda.synchronize()
        acts = rec['actions'].cpu().numpy()
        rew = np.zeros(n)
        for t in range(K):
            obs_before = ob.observe()
            want = torch.argmax(torch.from_numpy(obs_before).cuda().float() @ W, dim=1).cpu().numpy()
            assert np.array_equal(acts[t], want), "replay %d step %d" % (rep, t)
            o_obs, o_rew, o_done, o_cost, o_res = ob.step(acts[t])
            rew += o_rew
        assert np.array_equal(rec['obs'].cpu().numpy()[:, :cc.obs_dim], o_obs)
        assert np.array_equal(rec['reward_sum'].cpu().numpy(), rew)
        assert np.array_equal(h.map.cpu().numpy().reshape(n, -1), ob.map) and np.array_equal(h.inventory.cpu().numpy(), ob.inv)
    assert len(np.unique(acts)) >= 3
