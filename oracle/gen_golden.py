#!/usr/bin/env python
"""Golden-trace generator: runs the UNMODIFIED reference (via oracle/gymstub) and
records reset states, actions and every step's outputs into tests/golden/traces.npz.

Run where the reference is installed under baseline/_ref (see __graft_entry__.install_reference):

    python oracle/gen_golden.py            # ~1-2 min, rewrites tests/golden/traces.npz

The output is reproducible byte for byte: every iteration over a hash-ordered container is sorted, PYTHONHASHSEED is
pinned to 0 (the script re-executes itself if needed), and tests/test_oracle_golden.py regenerates a few scenarios and
compares them with the committed file.

For each scenario of tests/scenarios.py and each episode:
  * np.random.seed(ep_seed); obs0 = env.reset()          -> reset observation + reset state (pins the
    oracle's legacy-stream reset and the reset-observation quirks Q1/Q3)
  * most episodes then perturb the state directly on the reference object (random inventory, a selected
    item, a few extra blocks) so that rare branches (crafting, tree taps, rubber, sticky done) are reached
    by a random policy; the perturbed state is stored as `init_*`
  * T uniformly random valid actions; obs / reward / done / info and the full state after every step.
"""
import json
import os
import sys

if __name__ == '__main__' and os.environ.get('PYTHONHASHSEED') != '0':
    os.environ['PYTHONHASHSEED'] = '0'
    os.execv(sys.executable, [sys.executable] + sys.argv)

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, '..', 'tests'))
sys.path.insert(0, os.path.join(HERE, '..'))
import scenarios  # noqa: E402

EPISODES = 3
STEPS = 120


def snapshot(base):
    ids = base.items_id
    n = max(ids.values()) + 1
    inv = np.zeros(n, np.int32)
    for name, q in base.inventory_items_quantity.items():
        inv[ids[name]] = q
    sel = ids.get(base.selected_item, 0) if base.selected_item else 0
    r, c = base.agent_location
    pose = np.array([r, c, base.agent_facing_id, sel], np.uint8)
    return np.asarray(base.map, np.int8).reshape(-1).copy(), pose, inv


def perturb(base, rng):
    ids = base.items_id
    # sorted: inventory_items_quantity is built from a set (pogostick_v1_env.py:119-120), its order follows the string hash
    names = sorted(n for n in base.inventory_items_quantity if n not in ('air', 'wall'))
    for name in names:
        if rng.rand() < 0.6:
            hi = 2 if name == base.goal_item_to_craft else 9
            base.inventory_items_quantity[name] = int(rng.randint(0, hi))
    if rng.rand() < 0.25:
        base.inventory_items_quantity[base.goal_item_to_craft] = 0
    held = [n for n in names if base.inventory_items_quantity[n] >= 1]
    if held and rng.rand() < 0.6:
        axes = [n for n in held if n.endswith('_axe')]
        base.selected_item = axes[0] if (axes and rng.rand() < 0.7) else held[rng.randint(len(held))]
    ms = base.map_size
    placeable = sorted(i for n, i in ids.items() if n not in ('air', 'wall'))
    for _ in range(rng.randint(0, 5)):
        r, c = rng.randint(1, ms - 1), rng.randint(1, ms - 1)
        if (r, c) != tuple(base.agent_location) and base.map[r][c] == 0:
            base.map[r][c] = placeable[rng.randint(len(placeable))]
    base.update_block_in_front()           # keep the cached front block consistent, as every step does


def run_scenario(ns, desc, out):
    env = scenarios.build_chain(ns, desc)
    base = env.unwrapped
    key = desc['name']
    ext = (sorted(set(env.limited_actions_id.values())) if hasattr(env, 'limited_actions_id')
           else sorted(set(env.actions_id.values())))
    meta = dict(desc)
    rec = {k: [] for k in ('reset_map', 'reset_pose', 'reset_inv', 'reset_obs', 'init_map', 'init_pose', 'init_inv',
                           'actions', 'obs', 'reward', 'done', 'cost', 'result', 'map', 'pose', 'inv', 'message')}
    seeds = []
    reset_kind = None
    for ep in range(EPISODES):
        ep_seed = (abs(hash(key)) % 100000) * 10 + ep if False else (sum(map(ord, key)) * 31 + ep * 7919) % (2 ** 31)
        seeds.append(ep_seed)
        np.random.seed(ep_seed)
        obs0 = env.reset()
        m, p, v = snapshot(base)
        rec['reset_map'].append(m); rec['reset_pose'].append(p); rec['reset_inv'].append(v)
        if isinstance(obs0, dict) and 'agent_map' in obs0:
            reset_kind = 'agent_map'
            rec['reset_obs'].append(np.asarray(obs0['agent_map'], np.int64).ravel())
        elif isinstance(obs0, dict):
            reset_kind = 'dict'
            assert obs0['map'] is base.map and obs0['inventory_items_quantity'] is base.inventory_items_quantity
            rec['reset_obs'].append(np.zeros(0, np.int64))
        else:
            reset_kind = 'lidar'
            rec['reset_obs'].append(np.asarray(obs0, np.int64))
        rng = np.random.RandomState(ep_seed ^ 0x5bd1e995)
        if ep > 0:
            perturb(base, rng)
        m, p, v = snapshot(base)
        rec['init_map'].append(m); rec['init_pose'].append(p); rec['init_inv'].append(v)
        A, O, R, D, Cst, Res, M, P, V, Msg = [], [], [], [], [], [], [], [], [], []
        for t in range(STEPS):
            a = int(ext[rng.randint(len(ext))])
            obs, reward, done, info = env.step(a)
            A.append(a); R.append(reward); D.append(bool(done)); Cst.append(float(info['step_cost']))
            Res.append(bool(info['result'])); Msg.append(str(info['message']))
            if isinstance(obs, dict) and 'agent_map' in obs:
                assert obs['agent_facing_id'] == base.agent_facing_id
                O.append(np.asarray(obs['agent_map'], np.int64).ravel())
            else:
                O.append(np.zeros(0, np.int64) if isinstance(obs, dict) else np.asarray(obs, np.int64))
            m, p, v = snapshot(base)
            M.append(m); P.append(p); V.append(v)
        rec['actions'].append(np.array(A, np.int32)); rec['obs'].append(np.stack(O))
        rec['reward'].append(np.array(R, np.int32)); rec['done'].append(np.array(D, np.uint8))
        rec['cost'].append(np.array(Cst, np.float64)); rec['result'].append(np.array(Res, np.uint8))
        rec['map'].append(np.stack(M)); rec['pose'].append(np.stack(P)); rec['inv'].append(np.stack(V))
        rec['message'].append(np.array(Msg, dtype='U96'))
    # tables the host layer must reproduce
    meta.update({
        'seeds': seeds, 'reset_kind': reset_kind, 'external_ids': ext,
        'items_id': dict(base.items_id), 'base_actions_id': dict(base.actions_id),
        'top_actions_id': dict(env.actions_id),
        'limited_actions_id': dict(env.limited_actions_id) if hasattr(env, 'limited_actions_id') else None,
        'unbreakable': sorted(base.unbreakable_items), 'entities': sorted(base.entities),
        'items_quantity': dict(base.items_quantity),
        'lidar_items_id': dict(env.lidar_items_id) if hasattr(env, 'lidar_items_id') else None,
        'crate_ingredients': [str(x) for x in env.crate_ingredients] if hasattr(env, 'crate_ingredients') else None,
    })
    out[key + '/meta'] = np.frombuffer(json.dumps(meta).encode(), np.uint8)
    for k, v in rec.items():
        arr = np.stack(v)
        if k in ('obs', 'reset_obs'):
            assert arr.size == 0 or (arr.min() >= 0 and arr.max() < 32767)
            arr = arr.astype(np.int16)
        out[key + '/' + k] = arr


def generate(names=None, verbose=False):
    """{npz key: array} for the named scenarios (all when None), straight from the unmodified reference."""
    ns = scenarios.reference_namespace()
    import io
    import contextlib
    out = {}
    S = [d for d in scenarios.all_scenarios() if names is None or d['name'] in names]
    for i, desc in enumerate(S):
        with contextlib.redirect_stdout(io.StringIO()):       # the reference prints remapped action tables
            run_scenario(ns, desc, out)
        if verbose and i % 25 == 0:
            print('%d/%d %s' % (i, len(S), desc['name']), flush=True)
    return out, S


def main():
    out, S = generate(verbose=True)
    path = os.path.join(HERE, '..', 'tests', 'golden', 'traces.npz')
    np.savez_compressed(path, **out)
    print('wrote', path, os.path.getsize(path) // 1024, 'KiB,', len(S), 'scenarios,',
          len(S) * EPISODES * STEPS, 'reference steps')


if __name__ == '__main__':
    main()
