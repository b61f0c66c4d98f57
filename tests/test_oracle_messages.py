"""CPU suite: the C oracle's info['message'] codes against the strings of the unmodified reference in every golden trace.
The GPU tests compare the kernels' codes with the oracle's, so the oracle itself is pinned here first."""
import numpy as np

import golden_util
import scenarios
from gym_novel_gridworlds_b200 import opcodes as oc
from gym_novel_gridworlds_b200.compiler import compile_chain
from gym_novel_gridworlds_b200.runtime import decode_message
from oracle.oracle_lib import OracleBatch


def _replay(name):
    """Yields (step, oracle codes, reference strings) for every step of a golden trace."""
    g = golden_util.get(name)
    cc = compile_chain(scenarios.build_chain(scenarios.b200_namespace(), g['meta']))
    E, T = g['actions'].shape
    n_items = g['init_inv'].shape[1]
    ob = OracleBatch([cc], E)
    ob.map[:] = g['init_map']
    ob.pose[:] = g['init_pose']
    ob.inv[:, :n_items] = g['init_inv']
    for t in range(T):
        ob.step(g['actions'][:, t], want_obs=False)
        assert not ob.err.any(), "%s step %d" % (name, t)
        yield t, cc, ob.msg.copy(), g['message'][:, t]


def test_oracle_messages_equal_the_reference_strings():
    """Every step of every golden trace (271 traces, 97,560 env-steps): the decoded code is the reference's string, and
    every message kind of enum ngw_msg occurs."""
    kinds = set()
    steps = 0
    for name in golden_util.names():
        for t, cc, codes, want in _replay(name):
            got = [decode_message(c, cc) for c in codes]
            assert got == list(want), "%s step %d: %s vs %s" % (name, t, got, list(want))
            kinds.update(int(k) for k in codes & 31)
            steps += len(codes)
    assert steps == 97560
    assert kinds == set(range(16)), sorted(set(range(16)) - kinds)


def test_invalid_action_id_gives_message_code_zero():
    """A rejected id (negative, >= n_actions) writes code 0 over the previous step's code and leaves the state alone."""
    g = golden_util.get('pogo_lidar')
    cc = compile_chain(scenarios.build_chain(scenarios.b200_namespace(), g['meta']))
    n = 4
    ob = OracleBatch([cc], n)
    ob.map[:] = g['init_map'][0]
    ob.pose[:] = g['init_pose'][0]
    ob.inv[:, :g['init_inv'].shape[1]] = g['init_inv'][0]
    forward = [a for a in range(cc.c.n_actions) if cc.c.actions[a].op == oc.OP_FORWARD][0]
    for _ in range(cc.map_size):                       # walk into the wall: "Block in path" on every env
        ob.step(np.full(n, forward, np.int32), want_obs=False)
    assert (ob.msg == 1).all() and not ob.err.any()
    state = (ob.map.copy(), ob.pose.copy(), ob.inv.copy())
    _, reward, done, cost, result = ob.step(np.array([-1, cc.c.n_actions, 1 << 20, -(1 << 20)], np.int32))
    assert (ob.msg == 0).all() and (ob.err == 1).all()
    assert not reward.any() and not done.any() and not cost.any() and not result.any()
    for a, b in zip(state, (ob.map, ob.pose, ob.inv)):
        assert np.array_equal(a, b)
