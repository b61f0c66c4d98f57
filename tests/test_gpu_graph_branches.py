"""One-step launches captured on ONE stream are spread over parallel branches of the graph (ngw_capi.cu, claim_stream):
every program below is captured and replayed, and compared bit for bit with identical twins driven eagerly, one call at a
time with a synchronise after each.  The graph's topology is read back through the driver."""
import ctypes as C
import os
import threading

import numpy as np
import pytest
import torch

import golden_util
import scenarios
from gym_novel_gridworlds_b200 import capi
from gym_novel_gridworlds_b200.compiler import compile_chain
from gym_novel_gridworlds_b200.runtime import BatchHandle

pytestmark = pytest.mark.gpu

C2_DESC = {'env': scenarios.POGO, 'map_size': 10,
           'chain': [['limit', ['Forward', 'Left', 'Right', 'Break', 'Place_tree_tap', 'Extract_rubber', 'Craft_plank',
                                'Craft_stick', 'Craft_tree_tap', 'Craft_pogo_stick']], ['lidar', 8]]}
W = 3                     # branches of a capture chain (kBranches in ngw_capi.cu)
N = 32 * 90 + 5           # one wave, warp-per-tile kernel


def _compiled(desc):
    return compile_chain(scenarios.build_chain(scenarios.b200_namespace(), desc))


class World(object):
    """R handles, their action sets and named output buffers; programs refer to buffers by name."""

    def __init__(self, cc, n, R, fmt='i32', episode_end=False, setup=None):
        self.cc, self.n = cc, n
        self.hs = [BatchHandle([cc], n, seed=50 + k, obs_format=fmt) for k in range(R)]
        for h in self.hs:
            h.reset()
            h.enable_messages()
            if episode_end:
                h.enable_episode_end()
            h._done_count = torch.zeros(n, dtype=torch.int32, device='cuda')
        rng = np.random.RandomState(3)
        self.acts = [torch.from_numpy(rng.randint(0, cc.c.n_actions, size=n).astype(np.int32)).cuda() for _ in range(8)]
        self.sets, self.extra = {}, {}
        if setup is not None:
            setup(self)
        self.side = torch.cuda.Stream()
        torch.cuda.synchronize()

    def outs(self, name):
        if name not in self.sets:
            h = self.hs[0]
            self.sets[name] = (torch.zeros_like(h.obs), torch.zeros_like(h.reward), torch.zeros_like(h.done),
                               torch.zeros_like(h.step_cost), torch.zeros_like(h.result))
        return self.sets[name]

    def prepare(self, ops):
        for op in ops:
            if op[0] == 'step':
                self.outs(op[3])
            elif op[0] in ('mix', 'event', 'fork'):
                self.extra.setdefault(op[0], torch.zeros(self.n, dtype=torch.float32, device='cuda'))

    def run(self, ops, eager):
        stream = torch.cuda.current_stream()
        for op in ops:
            kind = op[0]
            if kind == 'step':
                _, k, a, name, auto = op
                h, (obs, rew, done, cost, res) = self.hs[k], self.outs(name)
                capi.check(h.lib, h.lib.ngw_step(h._h, self.acts[a].data_ptr(), obs.data_ptr(), rew.data_ptr(),
                                                 done.data_ptr(), cost.data_ptr(), res.data_ptr(), int(auto), 3 if auto else 0,
                                                 h._stream()))
            elif kind == 'mix':                       # a torch op that reads the outputs of earlier launches
                o = [self.outs(nm) for nm in op[1]]
                self.extra['mix'].copy_(o[0][1] + 2 * o[1][1] + o[2][0].view(torch.uint8).float().sum(1) + o[2][4].float())
            elif kind == 'event':                     # an event record on the capturing stream, read on a second stream
                ev = torch.cuda.Event()
                ev.record(stream)
                self.side.wait_event(ev)
                with torch.cuda.stream(self.side):
                    o = [self.outs(nm) for nm in op[1]]
                    self.extra['event'].copy_(o[0][1] - o[1][3] + o[0][2].float())
            elif kind == 'fork':                      # a second stream starts from here, with work of its own
                self.side.wait_stream(stream)
                with torch.cuda.stream(self.side):
                    self.extra['fork'].copy_(self.acts[0].float() * 2)
            elif kind == 'join':                      # ... and the capturing stream waits for it
                stream.wait_stream(self.side)
            elif kind == 'reset':
                self.hs[op[1]].reset()
            elif kind == 'observe':
                self.hs[op[1]].observe()
            elif kind == 'rollout':
                self.hs[op[1]].rollout(4, None, policy_seed=7)
            if eager:
                torch.cuda.synchronize()
        if any(op[0] == 'event' for op in ops):
            stream.wait_stream(self.side)


def _assert_same(got, want, what):
    for name in want.sets:
        for x, y in zip(got.sets[name], want.sets[name]):
            assert torch.equal(x, y), "%s: buffers %s" % (what, name)
    for name in want.extra:
        assert torch.equal(got.extra[name], want.extra[name]), "%s: %s" % (what, name)
    for a, b in zip(got.hs, want.hs):
        for f in ('map', 'pose', 'inventory', 'error_flags', 'episode', 'ep_len', 'obs', 'msg'):
            assert torch.equal(getattr(a, f), getattr(b, f)), "%s: %s" % (what, f)
        if getattr(b, 'truncated', None) is not None:
            assert torch.equal(a.truncated, b.truncated) and torch.equal(a.final_obs, b.final_obs), what
        # cost sums: float partials per CTA, the CTA shape depends on the launch mode
        np.testing.assert_allclose(a.stats().cpu().numpy(), b.stats().cpu().numpy(), rtol=1e-6)


def _capture(world, ops):
    """ops captured on one stream (keep_graph: the topology can be read back)."""
    world.prepare(ops)
    stream = torch.cuda.Stream()
    g = torch.cuda.CUDAGraph(keep_graph=True)
    with torch.cuda.stream(stream):
        with torch.cuda.graph(g, stream=stream):
            world.run(ops, eager=False)
    return g


def _check(ops, R, fmt='i32', episode_end=False, setup=None, cc=None, n=N, replays=2):
    cc = cc or _compiled(C2_DESC)
    got = World(cc, n, R, fmt, episode_end, setup)
    want = World(cc, n, R, fmt, episode_end, setup)
    want.prepare(ops)
    c0 = sum(h.concurrent_launch_count() for h in got.hs)
    g = _capture(got, ops)
    n_conc = sum(h.concurrent_launch_count() for h in got.hs) - c0
    for rep in range(replays):
        g.replay()
        torch.cuda.synchronize()
        want.run(ops, eager=True)
        _assert_same(got, want, "replay %d" % rep)
    return g, n_conc


# ---------------------------------------------------------------------------------------------- graph topology
def _driver():
    cu = C.CDLL('libcuda.so.1')
    cu.cuGraphGetNodes.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(C.c_size_t)]
    cu.cuGraphGetEdges_v2.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_size_t)]
    cu.cuGraphNodeGetType.argtypes = [C.c_void_p, C.POINTER(C.c_int)]
    return cu


def topology(g):
    """(node -> driver node type, list of (from, to) edges) of a captured graph."""
    cu, raw = _driver(), C.c_void_p(g.raw_cuda_graph())
    n = C.c_size_t(0)
    assert cu.cuGraphGetNodes(raw, None, C.byref(n)) == 0
    nodes = (C.c_void_p * n.value)()
    assert cu.cuGraphGetNodes(raw, nodes, C.byref(n)) == 0
    types = {}
    for x in nodes:
        t = C.c_int(0)
        assert cu.cuGraphNodeGetType(C.c_void_p(x), C.byref(t)) == 0
        types[x] = t.value
    m = C.c_size_t(0)
    assert cu.cuGraphGetEdges_v2(raw, None, None, None, C.byref(m)) == 0
    src, dst, data = (C.c_void_p * m.value)(), (C.c_void_p * m.value)(), (C.c_uint64 * m.value)()
    assert cu.cuGraphGetEdges_v2(raw, src, dst, data, C.byref(m)) == 0
    return types, list(zip(src, dst))


def chains(types, edges):
    """Number of parallel chains of a graph in which every node has at most one predecessor and one successor."""
    ins = {x: 0 for x in types}
    outs = dict(ins)
    for a, b in edges:
        outs[a] += 1
        ins[b] += 1
    assert max(ins.values()) <= 1 and max(outs.values()) <= 1, "not a set of chains"
    return sum(1 for x in types if ins[x] == 0)


def _rotation(R, L, auto=False):
    return [('step', t % R, t % 8, 'o%d' % t, auto) for t in range(L)]


# ---------------------------------------------------------------------------------------------- cases
@pytest.mark.parametrize('R', [1, 2, 3, 4, 7, 18])
def test_rotation_of_handles(R):
    L = max(12, 2 * R + 3)
    g, n_conc = _check(_rotation(R, L), R)
    assert n_conc == (0 if R == 1 else L - 1), n_conc
    types, edges = topology(g)
    assert len(types) == L and chains(types, edges) == min(R, W)


def test_u8_rows_and_irregular_order():
    order = [0, 1, 0, 2, 1, 0, 2, 2, 1, 0, 3, 0, 1]                 # a handle again at distance 1, 2 and 3
    ops = [('step', k, t % 8, 'o%d' % t, False) for t, k in enumerate(order)]
    g, _ = _check(ops, 4, fmt='u8')
    types, edges = topology(g)
    assert len(types) == len(order) and chains(types, edges) == W


def test_auto_reset_steps_stay_on_their_branch():
    g, n_conc = _check(_rotation(5, 15, auto=True), 5, episode_end=True, replays=3)
    assert n_conc == 14
    types, edges = topology(g)
    assert len(types) == 30 and chains(types, edges) == W           # each step followed by its queued-reset kernel


def _alias_outputs(w):
    """o1 writes the reward tensor of o0; the obs rows of o2 overlap those of o1 by half."""
    o0, o1, o2 = w.outs('o0'), w.outs('o1'), w.outs('o2')
    half = w.n // 2 & ~3                                             # (rows stay 16-byte aligned)
    big = torch.zeros((w.n + half,) + tuple(o0[0].shape[1:]), dtype=o0[0].dtype, device='cuda')
    w.sets['o1'] = (big[:w.n], o0[1]) + o1[2:]
    w.sets['o2'] = (big[half:half + w.n],) + o2[1:]
    w.extra['big'] = big


def test_aliased_outputs_keep_stream_order():
    # o1 and o2 conflict with the branch of their predecessor: each starts a new chain behind it, the last writer wins
    ops = [('step', 0, 0, 'o0', False), ('step', 1, 1, 'o1', False), ('step', 2, 2, 'o2', False),
           ('step', 3, 3, 'o3', False), ('step', 1, 4, 'o4', False)]
    g, _ = _check(ops, 4, setup=_alias_outputs)
    types, edges = topology(g)
    assert len(types) == 5 and len({b for a, b in edges}) == 4       # every launch after the first waits for something


def test_actions_written_by_another_branch_are_ordered():
    # launch 2 reads as actions the observation rows launch 1 wrote on another branch: it joins both branches and does
    # not count as overlapped
    def setup(w):
        w.acts[5] = w.outs('o1')[0].view(-1)[:w.n]
    ops = [('step', 0, 0, 'o0', False), ('step', 1, 1, 'o1', False), ('step', 2, 5, 'o2', False)]
    g, n_conc = _check(ops, 3, setup=setup)
    assert n_conc == 1
    types, edges = topology(g)
    assert len(types) == 3 and len(edges) == 2 and len({b for a, b in edges}) == 1     # launch 2 joins 0 and 1


def test_torch_op_and_event_join_every_branch():
    ops = _rotation(4, 6) + [('mix', ['o3', 'o4', 'o5'])] + [('step', (t + 6) % 4, t % 8, 'p%d' % t, False) for t in range(5)]
    ops += [('event', ['p3', 'p4'])] + [('step', (t + 1) % 4, t % 8, 'q%d' % t, False) for t in range(4)]
    g, _ = _check(ops, 4)
    types, edges = topology(g)
    n_preds = {}
    for a, b in edges:
        n_preds[b] = n_preds.get(b, 0) + 1
    # exactly two nodes wait for the tip of every branch: the torch op's first kernel and the second stream's op.  (Had
    # the event record ended the chain, the launch after it would be a third.)
    assert sorted(n_preds.values()).count(W) == 2, sorted(n_preds.values())
    assert max(n_preds.values()) == W


def test_launches_after_a_join_from_another_stream():
    # the join adds the second stream's node to the chain's tips: every handle of the chain may still be a direct
    # predecessor, so a step, an observe and a rollout of a handle whose launch is a tip other than the last wait for it
    ops = [('fork',)] + _rotation(4, 7) + [('join',), ('step', 0, 1, 'a', False), ('step', 1, 2, 'b', False)]
    ops += [('fork',)] + _rotation(4, 6) + [('join',), ('observe', 3), ('step', 2, 3, 'c', False)]
    ops += [('fork',)] + _rotation(4, 5) + [('join',), ('rollout', 2), ('step', 3, 4, 'd', False)]
    _, n_conc = _check(ops, 4, replays=3)
    # overlapped: the first rotation but its first launch; 'b' and the second rotation, which continue the chain 'a'
    # started (a fork records an event, no node); the third rotation.  'a', 'c' and 'd' start chains behind a join.
    assert n_conc == 6 + 1 + 6 + 5, n_conc


def test_reset_observe_and_rollout_in_a_chain():
    ops = _rotation(4, 5) + [('reset', 1), ('step', 2, 1, 'a', False), ('observe', 3), ('step', 0, 2, 'b', False),
                             ('step', 1, 3, 'c', False), ('rollout', 2), ('step', 3, 4, 'd', False),
                             ('step', 2, 5, 'e', False)]
    _check(ops, 4)


def test_no_concurrent_is_one_chain():
    os.environ['NGW_NO_CONCURRENT'] = '1'
    try:
        g, n_conc = _check(_rotation(7, 14), 7)
    finally:
        del os.environ['NGW_NO_CONCURRENT']
    assert n_conc == 0
    types, edges = topology(g)
    assert chains(types, edges) == 1


def test_multi_wave_launches():
    # launches of several waves keep the two-deep chain on one stream; the results are the same
    cc = _compiled(golden_util.get('bow_C3_axe_medium_fence_hard')['meta'])
    _check(_rotation(4, 9), 4, cc=cc, n=32 * 148 * 20 + 17)


def test_two_threads_capture_at_once():
    cc = _compiled(C2_DESC)
    ops = _rotation(5, 12)
    pairs = [(World(cc, N, 5), World(cc, N, 5)) for _ in range(2)]
    for got, want in pairs:
        got.prepare(ops)
        want.prepare(ops)
    graphs, errors = [None, None], []
    barrier = threading.Barrier(2)

    def capture(i):
        try:
            got = pairs[i][0]
            stream = torch.cuda.Stream()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.stream(stream):
                g.capture_begin(capture_error_mode='thread_local')
                try:
                    barrier.wait()
                    for op in ops:                    # both captures advance op by op, interleaved
                        got.run([op], eager=False)
                        barrier.wait()
                finally:
                    g.capture_end()
            graphs[i] = g
        except Exception as e:                        # re-raised in the main thread
            errors.append(e)
            barrier.abort()

    threads = [threading.Thread(target=capture, args=(i,)) for i in range(2)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert not errors, errors
    for rep in range(2):
        for g, (got, want) in zip(graphs, pairs):
            g.replay()
            torch.cuda.synchronize()
            want.run(ops, eager=True)
            _assert_same(got, want, "replay %d" % rep)
