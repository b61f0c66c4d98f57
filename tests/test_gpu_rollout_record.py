"""Per-step record of the K-step rollouts (ngw_set_rollout_record, BatchHandle.rollout(..., record=)), run on the B200
box with pytest -m gpu.  Every recorded field is compared exactly against a twin handle that takes the same steps one
ngw_step at a time with its episode-end buffers on and an observe() after every step; a third handle runs the same rollout
without a record, and everything a rollout returned before the record existed must be identical to the recording one's."""
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from gym_novel_gridworlds_b200 import capi
from gym_novel_gridworlds_b200.runtime import BatchHandle, obs_to_vector
from test_gpu_parity import C2_DESC, _compiled, rollout_case_inputs

pytestmark = pytest.mark.gpu

LANE_PAIR = ['c2', 'pogo_ms23', 'bow_ms13', 'c4_mixed', 'c3_layers']     # rollout2_kernel
ONE_WARP = ['pogo_ms40', 'bow12_16beams']                                 # rollout_kernel
SENTINEL = 0xA5
T = 24


def _inputs(case):
    return rollout_case_inputs('c2_u8' if case == 'c2' else case)


def _fill(rec, byte=SENTINEL):
    for t in rec.padded.values():
        if t is not None:
            t.view(torch.uint8).fill_(byte)


def _handles(compiled, n, cfg_id, fmt, k=3, seed=21):
    hs = [BatchHandle(compiled, n, seed=seed, cfg_id=cfg_id, obs_format=fmt) for _ in range(k)]
    for h in hs:
        h.reset()
    return hs


def _policy(h, compiled, rng):
    n_act = torch.tensor([cc.c.n_actions for cc in compiled], device='cuda')[h.cfg_id.long()]
    A = int(n_act.max().item())
    W = torch.from_numpy(rng.randint(-9, 10, size=(h.obs_dim, A)).astype(np.int32)).cuda()
    b = torch.from_numpy(rng.randint(-30, 31, size=A).astype(np.int32)).cuda()
    return n_act, W, b


def _argmax(obs, W, b, n_act):
    score = obs.double() @ W.double() + b.double()[None, :]                      # exact: small integers
    A = W.shape[1]
    score = torch.where(torch.arange(A, device='cuda')[None, :] < n_act[:, None], score, torch.full_like(score, -1e18))
    return torch.argmax(score, dim=1).to(torch.int32)


def _check_against_twin(tw, rec, acts, K, kw, first_obs=None, policy=None):
    """Step the twin K times with `acts` and compare every recorded field at every step.  policy=(W, b, n_act): the
    recorded actions must be the argmax of the policy on the previous recorded observation."""
    auto = kw.get('auto_reset', False)
    for t in range(K):
        if policy is not None:
            prev = first_obs if t == 0 else rec.obs[t - 1]
            assert torch.equal(_argmax(prev, *policy), acts[t]), "action, step %d" % t
        o, r, d, c, res = tw.step(acts[t].contiguous(), **kw)
        assert torch.equal(rec.reward[t], r), "reward, step %d" % t
        assert torch.equal(rec.step_cost[t], c), "step_cost, step %d" % t
        assert torch.equal(rec.done[t], d), "done, step %d" % t
        assert torch.equal(rec.result[t], res), "result, step %d" % t
        assert torch.equal(rec.truncated[t], tw.truncated), "truncated, step %d" % t
        if tw.obs_dim:
            regen = d.bool() if auto else torch.zeros_like(d, dtype=torch.bool)
            if rec.final_obs is not None:
                assert torch.equal(rec.final_obs[t][regen], tw.final_obs[regen]), "final_obs, step %d" % t
                assert bool((rec.final_obs[t][~regen].view(torch.uint8) == SENTINEL).all().item()), "final_obs touched, step %d" % t
            assert torch.equal(rec.obs[t], tw.observe()), "obs, step %d" % t


def _same_outputs(h1, out1, h2, out2):
    for a, b in zip(out1, out2):
        assert torch.equal(a, b)
    for name in ('map', 'pose', 'inventory', 'episode', 'ep_len', 'error_flags'):
        assert torch.equal(getattr(h1, name), getattr(h2, name)), name
    s1, s2 = h1.stats().cpu().numpy(), h2.stats().cpu().numpy()
    assert np.array_equal(s1[[0, 1, 2, 3, 5, 6]], s2[[0, 1, 2, 3, 5, 6]])
    np.testing.assert_allclose(s1[4], s2[4], rtol=1e-6)


def _record_vs_twin(case, fmt, mode, invalid=False):
    compiled, n, cfg_id = _inputs(case)
    h, tw, plain = _handles(compiled, n, cfg_id, fmt)
    tw.enable_episode_end()
    kw = {} if mode == 'given' else dict(auto_reset=True, max_episode_steps=7)
    rng = np.random.RandomState(17)
    n_act, W, b = _policy(h, compiled, rng)
    if mode == 'policy' and int(n_act.max().item()) > 16:
        pytest.skip("the device policy scores at most 16 actions")
    rec = h.rollout_record(T, final_obs=True)
    _fill(rec)
    first_obs = h.observe().clone() if mode == 'policy' else None
    if mode == 'policy':
        call = dict(policy=(W, b))
    elif mode == 'random':
        call = dict(actions=None, policy_seed=5)
    else:
        acts = (rng.randint(0, 1 << 30, size=(T, n)) % n_act.cpu().numpy()[None, :]).astype(np.int32)
        if invalid:
            bad = rng.rand(T, n) < 0.02
            acts[bad] = (n_act.cpu().numpy()[None, :] + 3).repeat(T, 0)[bad]
        call = dict(actions=torch.from_numpy(acts).cuda())
    out = h.rollout(T, record_actions=True, record=rec, **call, **kw)
    ref = plain.rollout(T, record_actions=True, **call, **kw)
    assert out[-1] is rec and len(out) == len(ref) + 1
    _same_outputs(h, out[:-1], plain, ref)
    acts = out[6]
    _check_against_twin(tw, rec, acts, T, kw, first_obs, (W, b, n_act) if mode == 'policy' else None)
    for name in ('map', 'pose', 'inventory', 'episode', 'ep_len'):
        assert torch.equal(getattr(h, name), getattr(tw, name)), name
    # consistency inside the launch
    assert torch.equal(rec.reward.sum(0), out[1])
    assert torch.equal(rec.done.long().sum(0), out[3].long())
    assert torch.equal(rec.done[T - 1], out[4]) and torch.equal(rec.result[T - 1], out[5])
    if h.obs_dim:
        assert torch.equal(rec.obs[T - 1], out[0])
    return acts, n_act, rec


@pytest.mark.parametrize('case', LANE_PAIR + ONE_WARP)
@pytest.mark.parametrize('fmt', ['i32', 'u8', 'hits'])
@pytest.mark.parametrize('mode', ['given', 'given+autoreset', 'random', 'policy'])
def test_record_equals_the_one_step_twin(case, fmt, mode):
    """Every recorded field at every step equals the twin's, both rollout kernels, every observation format; final_obs
    only where the auto-reset regenerated an env; the rollout's own outputs, state and statistics do not change."""
    if mode == 'policy' and fmt != 'i32':
        pytest.skip("the device policy reads int32 observation rows")
    _record_vs_twin(case, fmt, mode)


@pytest.mark.parametrize('case', ['c2', 'pogo_ms40'])
def test_invalid_actions_record_zeros_and_no_truncation(case):
    acts, n_act, rec = _record_vs_twin(case, 'hits', 'given+autoreset', invalid=True)
    bad = acts >= n_act[None, :]
    assert bool(bad.any().item()) and not bool(rec.truncated[bad].any().item())
    assert not bool(rec.reward[bad].any().item()) and not bool(rec.done[bad].any().item())


def test_hits_record_decodes_to_the_i32_record():
    compiled, n, cfg_id = _inputs('c4_mixed')
    hh = BatchHandle(compiled, n, seed=3, cfg_id=cfg_id, obs_format='hits')
    hi = BatchHandle(compiled, n, seed=3, cfg_id=cfg_id, obs_format='i32')
    rh, ri = hh.rollout_record(T), hi.rollout_record(T)
    for h, r in ((hh, rh), (hi, ri)):
        h.reset()
        h.rollout(T, None, policy_seed=9, auto_reset=True, max_episode_steps=5, record=r)
    cfg = hh.cfg_id.long().repeat(T)
    vec = obs_to_vector(rh.obs.reshape(T * n, -1), hh.compiled, 'hits', cfg)
    assert torch.equal(vec, ri.obs.reshape(T * n, -1))


ROUTES = {'c2': 'rollout2_kernel<1, 0, true>', 'c4_mixed': 'rollout2_kernel<0, 0, true>',
          'pogo_ms40': 'rollout_kernel<1, true>', 'bow12_16beams': 'rollout_kernel<1, true>'}

# one recorded rollout under torch.profiler, in a process of its own (kernel activity records of a fresh profiler session
# do not depend on what earlier tests of this process did); prints the names of the rollout kernels it ran
_PROFILE_CHILD = """
import json, sys, torch
from gym_novel_gridworlds_b200.runtime import BatchHandle
from test_gpu_rollout_record import _inputs
compiled, n, cfg_id = _inputs(sys.argv[1])
h = BatchHandle(compiled, n, seed=1, cfg_id=cfg_id)
h.reset()
rec = h.rollout_record(4)
torch.cuda.synchronize()
with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
    h.rollout(4, None, policy_seed=1, record=rec)
    torch.cuda.synchronize()
prof.export_chrome_trace(sys.argv[2])
with open(sys.argv[2]) as f:
    print(json.dumps([e['name'] for e in json.load(f)['traceEvents'] if e.get('cat') == 'kernel' and 'rollout' in e['name']]))
"""


@pytest.mark.parametrize('case', sorted(ROUTES))
def test_recording_kernel_routing(case, tmp_path):
    """The recording instance of the lane-pair kernel runs for C2 / C4 shapes, of the one-warp kernel for 40x40 and 16 beams."""
    here = os.path.dirname(os.path.abspath(__file__))
    env = dict(os.environ, PYTHONPATH=os.pathsep.join([os.path.dirname(here), here]))
    cmd = [sys.executable] + (['-s'] if sys.flags.no_user_site else []) + ['-c', _PROFILE_CHILD, case, str(tmp_path / 'r.json')]
    out = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    names = json.loads(out.stdout.strip().splitlines()[-1])
    assert len(names) == 1 and ROUTES[case] + '(' in names[0], names


def test_record_in_a_cuda_graph_and_switched_off():
    compiled, n, _ = _inputs('c2')
    h, tw = _handles(compiled, n, None, 'u8', k=2)
    kw = dict(auto_reset=True, max_episode_steps=7)
    n_a = compiled[0].c.n_actions
    acts = torch.from_numpy(np.random.RandomState(4).randint(0, n_a, size=(T, n)).astype(np.int32)).cuda()
    rec, rec_tw = h.rollout_record(T, final_obs=True), tw.rollout_record(T, final_obs=True)
    for hh, r in ((h, rec), (tw, rec_tw)):                            # eager warm-up (allocates the rollout's outputs)
        hh.rollout(T, acts, record=r, **kw)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    g = torch.cuda.CUDAGraph()
    with torch.cuda.stream(s):
        with torch.cuda.graph(g, stream=s):
            h.rollout(T, acts, record=rec, **kw)
    torch.cuda.current_stream().wait_stream(s)
    for _ in range(2):
        _fill(rec); _fill(rec_tw)
        g.replay()
        out_tw = tw.rollout(T, acts, record=rec_tw, **kw)
        torch.cuda.synchronize()
        for k, t in rec.padded.items():
            if t is not None:
                assert torch.equal(getattr(rec, k), getattr(rec_tw, k)), k
        assert torch.equal(h.obs, out_tw[0]) and torch.equal(h.map, tw.map) and torch.equal(h.ep_len, tw.ep_len)
    _fill(rec)
    h.rollout(T, acts, **kw)                                          # the record is off again after a recorded call
    capi.check(h.lib, h.lib.ngw_set_rollout_record(h._h, None))
    h.rollout(T, None, policy_seed=2, **kw)
    torch.cuda.synchronize()
    for t in rec.padded.values():
        if t is not None:
            assert bool((t.view(torch.uint8) == SENTINEL).all().item())


def test_record_errors_enqueue_nothing():
    compiled, n, _ = _inputs('c2')
    h = BatchHandle(compiled, n, seed=1)
    hu = BatchHandle(compiled, n, seed=1, obs_format='u8')
    h.reset()
    acts = torch.zeros((5, n), dtype=torch.int32, device='cuda')
    rec = h.rollout_record(4, final_obs=True)
    before = h.launch_count()
    with pytest.raises(RuntimeError, match='max_steps'):
        h.rollout(5, acts, record=rec)
    with pytest.raises(ValueError, match='format'):
        h.rollout(4, acts[:4], record=hu.rollout_record(4))
    for field in ('obs', 'final_obs'):
        c = capi.RolloutRecordC.from_buffer_copy(rec._c)
        setattr(c, field, getattr(c, field) + 4)
        assert h.lib.ngw_set_rollout_record(h._h, C.byref(c)) != 0
        assert b'aligned' in h.lib.ngw_last_error()
    c = capi.RolloutRecordC.from_buffer_copy(rec._c)
    c.max_steps = 0
    assert h.lib.ngw_set_rollout_record(h._h, C.byref(c)) != 0
    assert h.launch_count() == before


def test_record_at_launch_size():
    """C2 at 65,536 envs, K = 64, hits rows, random policy with auto-reset at 32 steps: full tiles, whole-tile stores."""
    n, K = 65536, 64
    compiled = [_compiled(C2_DESC)]
    h, tw = _handles(compiled, n, None, 'hits', k=2, seed=8)
    tw.enable_episode_end()
    kw = dict(auto_reset=True, max_episode_steps=32)
    rec = h.rollout_record(K, final_obs=True)
    _fill(rec)
    out = h.rollout(K, None, policy_seed=77, record_actions=True, record=rec, **kw)
    _check_against_twin(tw, rec, out[6], K, kw)
    assert torch.equal(h.map, tw.map) and torch.equal(rec.obs[K - 1], out[0])


@pytest.mark.parametrize('case', ['c2', 'pogo_ms40'])
@pytest.mark.parametrize('fields', ['final_obs_only_rows', 'scalars_only'])
def test_partial_records_through_the_c_abi(case, fields):
    """A C-ABI record may leave any field NULL: without obs (final_obs alone, or no rows at all) the other fields are
    still the twin's, and the buffers of the NULL fields are never written."""
    compiled, n, cfg_id = _inputs(case)
    h, tw = _handles(compiled, n, cfg_id, 'hits', k=2)
    tw.enable_episode_end()
    kw = dict(auto_reset=True, max_episode_steps=7)
    rec = h.rollout_record(T, final_obs=True)
    _fill(rec)
    c = capi.RolloutRecordC.from_buffer_copy(rec._c)
    c.obs = None
    if fields == 'scalars_only':
        c.final_obs = None
    capi.check(h.lib, h.lib.ngw_set_rollout_record(h._h, C.byref(c)))
    out = h.rollout(T, None, policy_seed=3, record_actions=True, **kw)
    capi.check(h.lib, h.lib.ngw_set_rollout_record(h._h, None))
    acts = out[6]
    for t in range(T):
        o, r, d, cost, res = tw.step(acts[t].contiguous(), **kw)
        assert torch.equal(rec.reward[t], r) and torch.equal(rec.step_cost[t], cost) and torch.equal(rec.done[t], d)
        assert torch.equal(rec.result[t], res) and torch.equal(rec.truncated[t], tw.truncated), "step %d" % t
        regen = d.bool()
        if fields == 'final_obs_only_rows':
            assert torch.equal(rec.final_obs[t][regen], tw.final_obs[regen]), "final_obs, step %d" % t
            assert bool((rec.final_obs[t][~regen] == SENTINEL).all().item())
    assert bool((rec.padded['obs'] == SENTINEL).all().item())
    if fields == 'scalars_only':
        assert bool((rec.padded['final_obs'] == SENTINEL).all().item())
    assert bool(rec.done.any().item())
