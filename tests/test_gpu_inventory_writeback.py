"""step1w_kernel stores back only the 32-byte sectors of a tile's inventory rows that hold a row the step changed (run on
the B200 box: pytest -m gpu).  Every case is compared with the oracle through the C-ABI, on batches that end in a partial
tile: one changed row per tile at every lane position, through every inventory change a step can make, at inventory
strides 9, 10 and 11 (rows of 36, 40 and 44 bytes: some rows straddle a sector, some start on one); a captured rotation of
handles whose launches overlap; inventory edits on clean rows between steps."""
import numpy as np
import pytest
import torch

import scenarios
from gym_novel_gridworlds_b200 import opcodes as oc
from gym_novel_gridworlds_b200.compiler import compile_chain
from gym_novel_gridworlds_b200.runtime import BatchHandle
from oracle.oracle_lib import OracleBatch
from test_gpu_graph_branches import World, _assert_same, _capture
from test_gpu_kernel_routing import _step_kernel

pytestmark = pytest.mark.gpu

N = 32 * 10 + 5                                   # ten full tiles and a partial one, one wave
AR, AC = 4, 4                                     # the agent, facing north: front (3, 4), two ahead (2, 4)
NORTH = 0

CHAINS = {                                        # name -> (env, chain); inventory stride in the comment
    'c2': (scenarios.POGO, [['limit', scenarios.C2_SET], ['lidar', 8]]),                                   # 9
    'breakincrease': (scenarios.POGO, [['lidar', 8], ['novelty', 'breakincrease', 'hard', '', '']]),       # 9
    'addchop': (scenarios.POGO, [['limit', scenarios.C2_SET + ['Chop']], ['lidar', 8], ['novelty', 'addchop', 'hard', '', '']]),   # 9
    'additem': (scenarios.POGO, [['limit', scenarios.C2_SET], ['lidar', 8], ['novelty', 'additem', 'medium', 'spring', '']]),      # 10
    'crate': (scenarios.POGO, [['lidar', 8], ['novelty', 'crate', 'easy', '', '']]),                       # 10
    'axe_iron_inc': (scenarios.POGO, [['lidar', 8], ['novelty', 'axe', 'easy', 'iron', 'true']]),          # 10
    'bow_axe_fence': (scenarios.BOW, [['lidar', 8], ['novelty', 'axe', 'medium', 'wooden', ''],
                                      ['novelty', 'fence', 'hard', 'oak', '']]),                           # 11
}


def _compiled(name):
    env, chain = CHAINS[name]
    return compile_chain(scenarios.build_chain(scenarios.b200_namespace(), {'env': env, 'map_size': 10, 'chain': chain}))


def _id(cc, name):
    return cc.item_names.index(name)


def _action(cc, op):
    return next(a for a in range(cc.c.n_actions) if cc.c.actions[a].op == op)


def mutations(cc):
    """(action, front item, selected item, extra cells) of every way a step of this config changes the inventory: each
    opcode that writes it, each break variant, the crate layer and grabbing an entity."""
    c = cc.c
    axe = c.id_wooden_axe if c.id_wooden_axe != oc.NONE else c.id_iron_axe
    out = []
    for a in range(c.n_actions):
        e = c.actions[a]
        if e.op == oc.OP_BREAK:
            if oc.LAYER_CRATE in list(e.layers):
                out.append((a, c.id_crate, 0, {}))
            if e.variant in (oc.BRK_AXE, oc.BRK_AXE_INC, oc.BRK_AXETOBREAK):
                out.append((a, c.id_tree_log, axe, {}))                  # with the axe selected
            if e.variant != oc.BRK_AXETOBREAK:
                out.append((a, c.id_tree_log, 0, {}))                    # base / increase / axe variant without the axe
        elif e.op == oc.OP_PLACE_TREE_TAP:
            out.append((a, 0, 0, {}))
        elif e.op == oc.OP_EXTRACT_RUBBER:
            out.append((a, c.id_tree_tap, 0, {(AR - 2, AC): c.id_tree_log}))
        elif e.op == oc.OP_EXTRACT_STRING:
            out.append((a, c.id_wool, 0, {}))
        elif e.op in (oc.OP_CRAFT, oc.OP_CHOP):
            out.append((a, c.id_crafting_table if e.op == oc.OP_CRAFT else c.id_tree_log, 0, {}))
    if c.entity_mask:
        ent = next(i for i in range(cc.n_items) if (c.entity_mask >> i) & 1)
        out.append((_action(cc, oc.OP_LEFT), 0, 0, {(AR + 1, AC + 1): ent}))
    return out


def base_state(cc, seed, inv=8):
    """Reset maps with the agent at (AR, AC) facing north and air around it; `inv` of every item but the goal."""
    ob = OracleBatch([cc], N)
    ob.reset_legacy(seed)
    ms = cc.map_size
    m = ob.map.reshape(N, ms, ms)
    m[:, AR - 2:AR + 2, AC - 1:AC + 2] = 0
    ob.pose[:] = (AR, AC, NORTH, 0)
    ob.inv[:, 1:] = inv
    ob.inv[:, cc.c.id_goal] = 0
    return ob


def apply(ob, cc, lanes_to_mut):
    """Actions of the batch: env e takes mutation lanes_to_mut[e] (its front cell, selection and extra cells set up in the
    oracle's state), or turns left when that is None."""
    ms = cc.map_size
    m = ob.map.reshape(N, ms, ms)
    acts = np.full(N, _action(cc, oc.OP_LEFT), np.int32)
    for e, mut in enumerate(lanes_to_mut):
        if mut is None:
            continue
        a, front, sel, extra = mut
        acts[e] = a
        m[e, AR - 1, AC] = front
        ob.pose[e, 3] = sel
        for (r, c), v in extra.items():
            m[e, r, c] = v
    return acts


def _compare_outputs(got, want, what):
    obs, rew, done, cost, res = [x.cpu().numpy() for x in got]
    o_obs, o_rew, o_done, o_cost, o_res = want
    assert np.array_equal(obs, o_obs), what + ": obs"
    assert np.array_equal(rew, o_rew) and np.array_equal(done, o_done) and np.array_equal(res, o_res), what
    np.testing.assert_allclose(cost, o_cost, rtol=1e-6, err_msg=what)


def _compare_state(h, ob, what):
    m, p, v = h.export_state()
    assert np.array_equal(v.cpu().numpy(), ob.inv), what + ": inventory"
    assert np.array_equal(m.cpu().numpy().reshape(N, -1), ob.map), what + ": map"
    assert np.array_equal(p.cpu().numpy(), ob.pose), what + ": pose"


@pytest.mark.parametrize('name', sorted(CHAINS))
def test_one_changed_row_per_tile_at_every_lane(name, tmp_path):
    cc = _compiled(name)
    assert 'step1w_kernel<' in _step_kernel([cc], N, None, tmp_path)[0]
    muts = mutations(cc)
    assert len(muts) >= 3
    h = BatchHandle([cc], N, device='cuda:0')
    for lane in range(32):
        # tile k's lane `lane` takes mutation (lane + k) mod len(muts): each lane position meets every mutation
        ob = base_state(cc, 100 + lane)
        plan = [muts[(lane + e // 32) % len(muts)] if e % 32 == lane else None for e in range(N)]
        acts = apply(ob, cc, plan)
        h.load_state(ob.map, ob.pose, ob.inv)
        inv0 = ob.inv.copy()
        want = ob.step(acts)
        changed = (ob.inv != inv0).any(1)
        assert np.array_equal(changed, np.array([p is not None for p in plan])), "every planned row changes, no other"
        got = h.step(torch.from_numpy(acts).cuda())
        _compare_outputs(got, want, "%s lane %d" % (name, lane))
        _compare_state(h, ob, "%s lane %d" % (name, lane))


def test_edits_of_clean_rows_persist():
    cc = _compiled('c2')
    left = _action(cc, oc.OP_LEFT)
    craft = next(a for a in range(cc.c.n_actions)
                 if cc.c.actions[a].op == oc.OP_CRAFT and not cc.c.recipes[cc.c.actions[a].arg].needs_table)
    brk = next(m for m in mutations(cc) if m[0] == _action(cc, oc.OP_BREAK))
    ob = base_state(cc, 7)
    lane3 = np.arange(N) % 32 == 3
    acts0 = apply(ob, cc, [brk if x else None for x in lane3])
    h = BatchHandle([cc], N, device='cuda:0')
    h.load_state(ob.map, ob.pose, ob.inv)
    rng = np.random.RandomState(5)
    # lane 3 of every tile breaks, crafts, does nothing, crafts; the other lanes turn
    for t, acts in enumerate([acts0, np.where(lane3, craft, left), np.full(N, left), np.where(lane3, craft, left)]):
        acts = acts.astype(np.int32)
        inv0 = ob.inv.copy()
        want = ob.step(acts)
        assert np.array_equal((ob.inv != inv0).any(1), lane3 & (t != 2))
        got = h.step(torch.from_numpy(acts).cuda())
        _compare_outputs(got, want, "step %d" % t)
        _compare_state(h, ob, "step %d" % t)
        # rows 2 and 4 share sectors with the changed row 3 (rows of 36 bytes); tile 10 is the partial one
        for e in (2, 4, 32 + 2, 32 * 10 + 1):
            item = rng.randint(1, cc.n_items)
            h.inventory[e, item] += 5                                 # zero-copy state view
            ob.inv[e, item] += 5
        e = 32 * 5 + 4                                                # ngw_load_state of one env
        ob.inv[e] = rng.randint(0, 50, size=ob.inv.shape[1])
        h.load_state(ob.map[e:e + 1], ob.pose[e:e + 1], ob.inv[e:e + 1], first=e)
    _compare_state(h, ob, "after the last edits")


@pytest.mark.parametrize('name', ['c2', 'bow_axe_fence'])
def test_captured_rotation(name):
    """4 handles rotated inside one capture (their launches overlap on the graph's branches): replays against eager twins,
    and both against the oracle."""
    cc = _compiled(name)
    R, L = 4, 12
    crafts = [a for a in range(cc.c.n_actions) if cc.c.actions[a].op == oc.OP_CRAFT]
    left = _action(cc, oc.OP_LEFT)
    states = []
    for k in range(R):
        ob = base_state(cc, 30 + k, inv=1000)
        m = ob.map.reshape(N, cc.map_size, cc.map_size)
        for r, c in ((AR - 1, AC), (AR + 1, AC), (AR, AC - 1), (AR, AC + 1)):   # a table in front, whichever way it faces
            m[:, r, c] = cc.c.id_crafting_table
        states.append(ob)
    acts = []
    for s in range(8):                                                 # set s: lane 7 s mod 32 of each tile crafts
        a = np.full(N, left, np.int32)
        for e in range(N):
            if e % 32 == (7 * s) % 32:
                a[e] = crafts[(e // 32 + s) % len(crafts)]
        acts.append(a)

    def setup(w):
        for h, ob in zip(w.hs, states):
            h.load_state(ob.map, ob.pose, ob.inv)
        w.acts = [torch.from_numpy(a).cuda() for a in acts]

    ops = [('step', t % R, t % 8, 'o%d' % t, False) for t in range(L)]
    got, want = World(cc, N, R, setup=setup), World(cc, N, R, setup=setup)
    want.prepare(ops)
    c0 = sum(h.concurrent_launch_count() for h in got.hs)
    g = _capture(got, ops)
    assert sum(h.concurrent_launch_count() for h in got.hs) - c0 == L - 1
    for rep in range(2):
        g.replay()
        torch.cuda.synchronize()
        want.run(ops, eager=True)
        _assert_same(got, want, "replay %d" % rep)
        for t, (_, k, s, nm, _) in enumerate(ops):
            inv0 = states[k].inv.copy()
            o = states[k].step(acts[s])
            assert np.array_equal((states[k].inv != inv0).any(1), acts[s] != left)
            _compare_outputs(want.outs(nm), o, "replay %d step %d" % (rep, t))
        for k in range(R):
            _compare_state(want.hs[k], states[k], "replay %d handle %d" % (rep, k))
