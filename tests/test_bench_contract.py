"""bench.py without a GPU: the algorithmic-bytes formula reproduces SURVEY §8d, the workloads compile, and the
`--impl reference` arm prints the contract's JSON line.  With one: `--dump-outputs` writes the last timed step."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import bench

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_algorithmic_bytes_match_survey_8d():
    got = {}
    for w in ('C2', 'C3', 'C4', 'C5'):
        desc, compiled, envs, rule, kw = bench.build_workload(w)
        got[w] = ([bench.algorithmic_bytes_per_env_step(cc) for cc in compiled], envs)
    assert got['C2'] == ([446], 65536)                       # 144 read + 302 written
    assert got['C3'] == ([470], 262144)                      # I = 11, I_obs = 9
    assert got['C4'] == ([446, 446, 458, 446], 1048576)      # + 1 byte config id per env in bench.py (uint8, not int32)
    assert got['C5'] == ([1958], 524288)                     # map 40, I = 10


def test_reference_arm_prints_the_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--steps', '4',
                          '--warmup', '1'], capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 0, out.stderr
    line = json.loads(out.stdout.strip().splitlines()[-1])
    for key in ('impl', 'metric', 'value', 'unit', 'n_gpus', 'steps', 'warmup', 'ms_per_step', 'higher_is_better',
                'scaling', 'vs_baseline', 'dtype', 'data', 'config', 'cpu_baseline', 'e2e'):
        assert key in line, key
    assert line['impl'] == 'reference' and line['vs_baseline'] is None and line['value'] > 0
    assert line['cpu_baseline']['kind'] == 'port' and line['cpu_baseline']['cores'] >= 1
    assert line['e2e']['h2d_bytes_per_step'] == 0 and line['e2e']['d2h_bytes_per_step'] == 0
    assert line['metric'] == json.load(open(os.path.join(ROOT, 'BASELINE.json')))['metric']


@pytest.mark.gpu
def test_dump_outputs_hold_the_last_of_exactly_k_timed_steps(tmp_path):
    """`--steps K --warmup W --dump-outputs DIR`: the headline batches take W eager steps, lead_in_regions(K) untimed and
    one timed replay of the K-step graph, and DIR holds what the last of those steps returned — the same arrays an
    in-process replay of that step sequence produces."""
    import torch
    K, W = 5, 3
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--steps', str(K), '--warmup', str(W),
                          '--no-workloads', '--no-cpu-baseline', '--dump-outputs', str(tmp_path)],
                         capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line['steps'] == K and line['timing']['regions'] == 1
    got = {name: np.load(str(tmp_path / (name + '.npy'))) for name in ('obs', 'reward', 'done', 'step_cost', 'result')}
    assert sorted(os.listdir(str(tmp_path))) == sorted(name + '.npy' for name in got)
    assert got['obs'].shape == (bench.ENVS_PER_BATCH, 63)
    assert all(a.dtype == np.float32 for a in got.values()) and sum(a.nbytes for a in got.values()) <= bench.DUMP_LIMIT_BYTES

    wl = bench.Workload('C2', 0, 1, torch.device('cuda', 0))
    for i in range(W):
        wl.step(i)
    for _ in range(bench.lead_in_regions(K) + 1):
        for i in range(K):
            wl.step(i)
    h = wl.batches[(K - 1) % wl.n_batches]
    want = {'obs': h.obs[:, :h.obs_dim], 'reward': h.reward, 'done': h.done, 'step_cost': h.step_cost,
            'result': h.result}
    for name, t in want.items():
        assert np.array_equal(got[name], t.cpu().numpy().astype(np.float32)), name
    wl.close()
