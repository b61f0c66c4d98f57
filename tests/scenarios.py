"""Wrapper-chain descriptors shared by the golden generator (run against the reference) and the tests
(run against this package).  A descriptor is plain JSON so it travels inside the .npz fixtures:

    {"name": ..., "env": gym id, "map_size": int, "chain": [step, ...]}
    step = ["limit", [action names]] | ["lidar", num_beams] | ["novelty", name, difficulty, arg1, arg2]

`build_chain(ns, desc)` builds it inside a namespace that offers make / LimitActions / LidarInFront /
inject_novelty — the reference's modules or gym_novel_gridworlds_b200's.  The global legacy np.random
stream is re-seeded before every chain step so construction-time draws (Crate, remapaction) coincide
even though the reference also burns draws in constructor-time resets."""
import numpy as np

POGO = 'NovelGridworld-Pogostick-v1'
BOW = 'NovelGridworld-Bow-v1'
POGO0 = 'NovelGridworld-Pogostick-v0'
BOW0 = 'NovelGridworld-Bow-v0'

C2_SET = ['Forward', 'Left', 'Right', 'Break', 'Place_tree_tap', 'Extract_rubber',
          'Craft_plank', 'Craft_stick', 'Craft_tree_tap', 'Craft_pogo_stick']
BOW_SET = ['Forward', 'Left', 'Right', 'Break', 'Extract_string', 'Craft_plank', 'Craft_stick', 'Craft_bow']


def build_chain(ns, desc, **make_kwargs):
    env = ns['make'](desc['env'], **make_kwargs)
    if desc.get('map_size', 10) != 10:
        env.map_size = desc['map_size']            # plain attribute on the base env (SURVEY §5 config row)
    for i, step in enumerate(desc['chain']):
        np.random.seed(desc.get('build_seed', 7) * 1000 + i)
        kind = step[0]
        if kind == 'limit':
            env = ns['LimitActions'](env, set(step[1]))
        elif kind == 'lidar':
            env = ns['LidarInFront'](env, num_beams=step[1])
        elif kind == 'agentmap':
            env = ns['AgentMap'](env)
        elif kind == 'novelty':
            env = ns['inject_novelty'](env, step[1], step[2], step[3], step[4])
        else:
            raise ValueError(kind)
    return env


def reference_root():
    """Where the unmodified reference package lives: the copy that __graft_entry__.build() installs under git-ignored
    baseline/_ref when the upstream sources are at hand; None when it is not installed."""
    import os
    root = os.path.join(os.path.dirname(os.path.abspath(__file__)), '..', 'baseline', '_ref')
    return os.path.abspath(root) if os.path.isdir(os.path.join(root, 'gym_novel_gridworlds')) else None


def reference_namespace(ref_root=None):
    """The unmodified reference through oracle/gymstub (a ~150-line gym-0.18 / matplotlib stand-in)."""
    import os
    import sys
    here = os.path.dirname(os.path.abspath(__file__))
    stub = os.path.abspath(os.path.join(here, '..', 'oracle', 'gymstub'))
    root = ref_root or reference_root()
    if root is None:
        raise RuntimeError("the reference package is not installed under baseline/_ref")
    for p in (stub, root):
        if p not in sys.path:
            sys.path.insert(0, p)
    import gym
    import gym_novel_gridworlds  # noqa: F401  (registers the ids)
    from gym_novel_gridworlds.wrappers import LimitActions
    from gym_novel_gridworlds.observation_wrappers import LidarInFront, AgentMap
    from gym_novel_gridworlds.novelty_wrappers import inject_novelty
    return {'make': gym.make, 'LimitActions': LimitActions, 'LidarInFront': LidarInFront, 'AgentMap': AgentMap,
            'inject_novelty': inject_novelty}


def b200_namespace():
    import gym_novel_gridworlds_b200 as g
    return {'make': g.make, 'LimitActions': g.LimitActions, 'LidarInFront': g.LidarInFront, 'AgentMap': g.AgentMap,
            'inject_novelty': g.inject_novelty}


def _nov(name, difficulty='hard', a1='', a2=''):
    return ['novelty', name, difficulty, a1, a2]


def _novelty_variants(env_id):
    """(tag, novelty step, extra limited action names) for every novelty the env accepts."""
    out = []
    for d in ('easy', 'medium', 'hard'):
        extra = ['Select_wooden_axe'] + (['Craft_wooden_axe'] if d == 'hard' else [])
        out.append(('axe_%s_wooden' % d, _nov('axe', d, 'wooden', ''), extra))
        out.append(('axetobreak_%s_wooden' % d, _nov('axetobreak', d, 'wooden'), extra))
        out.append(('fence_%s' % d, _nov('fence', d, 'oak'), []))
        out.append(('fencerestriction_%s' % d, _nov('fencerestriction', d, 'oak'), ['Select_oak_fence']))
        out.append(('additem_%s' % d, _nov('additem', d, 'spring'), []))
        out.append(('crate_%s' % d, _nov('crate', d), []))
        out.append(('firewall_%s' % d, _nov('firewall', d), []))
        out.append(('remapaction_%s' % d, _nov('remapaction', d), []))
        out.append(('replaceitem_%s_wall' % d, _nov('replaceitem', d, 'wall', 'brick'), []))
        out.append(('replaceitem_%s_log' % d, _nov('replaceitem', d, 'tree_log', 'birch_log'), []))
    out.append(('axe_hard_iron_inc', _nov('axe', 'hard', 'iron', 'true'), ['Select_iron_axe', 'Craft_iron_axe']))
    out.append(('axe_easy_iron_inc', _nov('axe', 'easy', 'iron', 'true'), ['Select_iron_axe']))
    out.append(('axe_medium_wooden_inc', _nov('axe', 'medium', 'wooden', 'true'), ['Select_wooden_axe']))
    out.append(('axetobreak_hard_iron', _nov('axetobreak', 'hard', 'iron'), ['Select_iron_axe', 'Craft_iron_axe']))
    out.append(('addchop', _nov('addchop'), ['Chop']))
    out.append(('addjump', _nov('addjump'), ['Jump']))
    out.append(('breakincrease_all', _nov('breakincrease'), []))
    out.append(('breakincrease_log', _nov('breakincrease', 'hard', 'tree_log'), []))
    if env_id == BOW:
        out.append(('extractincdec_dec', _nov('extractincdec', 'hard', 'decrease'), []))
    return out


def all_scenarios():
    S = []

    def add(name, env, chain, map_size=10):
        S.append({'name': name, 'env': env, 'map_size': map_size, 'chain': chain})

    for env_id, tag, base_set in ((POGO, 'pogo', C2_SET), (BOW, 'bow', BOW_SET)):
        add(tag + '_bare', env_id, [])
        add(tag + '_lidar', env_id, [['lidar', 8]])
        add(tag + '_limit_lidar', env_id, [['limit', base_set], ['lidar', 8]])
        for vt, nov, extra in _novelty_variants(env_id):
            # A: canonical order of every reference script: make -> LimitActions -> LidarInFront -> novelty
            add('%s_A_%s' % (tag, vt), env_id, [['limit', base_set + extra], ['lidar', 8], nov])
            # B: novelty under the lidar (lidar sees the new items), no LimitActions
            add('%s_B_%s' % (tag, vt), env_id, [nov, ['lidar', 8]])
            # C: lidar first, novelty outermost, no LimitActions
            add('%s_C_%s' % (tag, vt), env_id, [['lidar', 8], nov])
    # other beam counts and map sizes
    add('pogo_lidar_b5', POGO, [['limit', C2_SET], ['lidar', 5]])
    add('pogo_lidar_b16', POGO, [['limit', C2_SET], ['lidar', 16]])
    add('pogo_ms20_c2', POGO, [['limit', C2_SET], ['lidar', 8]], map_size=20)
    add('pogo_ms40_additem_hard', POGO, [['limit', C2_SET], ['lidar', 8], _nov('additem', 'hard', 'spring')], map_size=40)
    add('bow_ms13_lidar', BOW, [['lidar', 8]], map_size=13)
    # stacked novelties (BASELINE config C3 first)
    add('bow_C3_axe_medium_fence_hard', BOW, [['lidar', 8], _nov('axe', 'medium', 'wooden', ''), _nov('fence', 'hard', 'oak')])
    add('pogo_crate_over_axe', POGO, [['lidar', 8], _nov('axe', 'easy', 'wooden', ''), _nov('crate', 'easy')])
    add('pogo_axe_over_crate', POGO, [['lidar', 8], _nov('crate', 'easy'), _nov('axe', 'easy', 'wooden', '')])
    add('pogo_firewall_over_addchop', POGO, [['lidar', 8], _nov('addchop'), _nov('firewall', 'hard')])
    add('pogo_addchop_over_firewall', POGO, [['lidar', 8], _nov('firewall', 'hard'), _nov('addchop')])
    # (fence/fencerestriction OUTSIDE a wall-replacing novelty is not a scenario: the reference's Fence.reset then
    #  fences around border cells and dies with IndexError in add_fence_around, pogostick_v1_env.py:533)
    add('pogo_firewall_over_fr_medium', POGO, [['lidar', 8], _nov('fencerestriction', 'medium', 'oak'), _nov('firewall', 'medium')])
    add('pogo_fr_hard_over_axetobreak', POGO, [['lidar', 8], _nov('axetobreak', 'easy', 'wooden'), _nov('fencerestriction', 'hard', 'oak')])
    add('pogo_fr_medium_over_crate', POGO, [['lidar', 8], _nov('crate', 'medium'), _nov('fencerestriction', 'medium', 'jungle')])
    add('pogo_crate_over_fr_hard', POGO, [['lidar', 8], _nov('fencerestriction', 'hard', 'jungle'), _nov('crate', 'hard')])
    add('pogo_fence_over_additem', POGO, [['limit', C2_SET], ['lidar', 8], _nov('additem', 'medium', 'spring'), _nov('fence', 'medium', 'oak')])
    add('pogo_breakinc_over_axe', POGO, [['lidar', 8], _nov('axe', 'easy', 'iron', ''), _nov('breakincrease')])
    add('pogo_remap_over_addjump_limit', POGO, [['limit', C2_SET + ['Jump']], ['lidar', 8], _nov('addjump'), _nov('remapaction', 'hard')])
    add('pogo_addchop_addjump', POGO, [['limit', C2_SET + ['Chop', 'Jump']], ['lidar', 8], _nov('addchop'), _nov('addjump')])
    add('bow_axehard_wooden_limit', BOW, [['limit', BOW_SET + ['Craft_wooden_axe', 'Select_wooden_axe']], ['lidar', 8], _nov('axe', 'hard', 'wooden', 'true')])
    add('bow_extractdec_over_firewall', BOW, [['lidar', 8], _nov('firewall', 'easy'), _nov('extractincdec', 'hard', 'decrease')])
    # SURVEY §8f N2: the v0 envs (ingredients pre-placed, tree_tap placed at reset, other reward items) and AgentMap
    add('pogo0_bare', POGO0, [])
    add('pogo0_lidar', POGO0, [['lidar', 8]])
    add('pogo0_limit_lidar', POGO0, [['limit', C2_SET], ['lidar', 8]])
    add('pogo0_A_axe_easy', POGO0, [['limit', C2_SET + ['Select_wooden_axe']], ['lidar', 8], _nov('axe', 'easy', 'wooden', '')])
    add('pogo0_C_fence_hard', POGO0, [['lidar', 8], _nov('fence', 'hard', 'oak')])
    add('pogo0_ms16_lidar', POGO0, [['lidar', 8]], map_size=16)
    add('bow0_bare', BOW0, [])
    add('bow0_limit_lidar', BOW0, [['limit', BOW_SET], ['lidar', 8]])
    add('bow0_C_firewall_hard', BOW0, [['lidar', 8], _nov('firewall', 'hard')])
    add('bow0_B_additem_medium', BOW0, [_nov('additem', 'medium', 'spring'), ['lidar', 8]])
    add('pogo_agentmap', POGO, [['limit', C2_SET], ['agentmap']])
    add('bow_agentmap', BOW, [['agentmap']])
    add('pogo0_agentmap_additem', POGO0, [_nov('additem', 'hard', 'spring'), ['agentmap']])
    add('pogo_ms20_agentmap', POGO, [['agentmap']], map_size=20)
    return S
