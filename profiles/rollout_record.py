"""Cost of the per-step rollout record (ngw_set_rollout_record) on the C2 K-step rollouts.
    python profiles/rollout_record.py [--out profiles/rollout_record.jsonl] [--rounds R] [--window-ms W]
Workload: C2 (bench.py), 4 batches of 65,536 envs, K = 64 steps per launch, auto-reset; the device random policy
(ngw_rollout) and the closed loop (ngw_rollout_policy, int32 rows only: the device policy reads them), as
profiles/rollout_probe.py runs them.  Arms: no record, then records of every field but final_obs in hits, u8 and i32
rows; and, for each row format, the same transitions from the one-step route: one CUDA graph of K ngw_step launches per
batch (the 4 batches interleaved, uniform random actions drawn beforehand, auto-reset, episode-end buffers on), replayed.
That route leaves every step's outputs in the handle's buffers; copying them out per step is not included.  The arms alternate in one process for --rounds rounds, each timed with CUDA events over enough launches (cycling
through the batches) to fill --window-ms; the record holds the median env-steps/s of each arm, every round's figure, the
record's bytes per env-step (computed from its shapes) and the write bandwidth that implies, next to the 6552 GB/s
device-to-device copy peak DESIGN.md §7 uses.  One JSON line is printed and appended to --out, with the card's name and
power limit (a read-only nvidia-smi query in the same run)."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), '..')
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from gym_novel_gridworlds_b200.runtime import BatchHandle  # noqa: E402

K, N_BATCHES = 64, 4
COPY_PEAK_GBS = 6552.0


def gpu_info():
    out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'], capture_output=True,
                         text=True, check=True).stdout.strip().splitlines()[0]
    name, power = [x.strip() for x in out.split(',')]
    return {"name": name, "power_limit": power}


def record_bytes(h):
    """Bytes the record writes per env-step: observation row + reward + step_cost + done + result + truncated."""
    return h.obs_row_bytes + 4 + 4 + 1 + 1 + 1


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'rollout_record.jsonl'))
    ap.add_argument('--rounds', type=int, default=3)
    ap.add_argument('--window-ms', type=float, default=500.0)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("rollout_record.py measures on a CUDA device; none is present")
    t_start = time.time()
    desc, compiled, envs, rule, kw = bench.build_workload('C2')
    handles = {fmt: [BatchHandle(compiled, envs, seed=0, first_env_gid=b * envs, obs_format=fmt) for b in range(N_BATCHES)]
               for fmt in ('i32', 'u8', 'hits')}
    for hs in handles.values():
        for h in hs:
            h.reset()
    records = {fmt: [h.rollout_record(K) for h in hs] for fmt, hs in handles.items()}
    cc = compiled[0]
    rng = np.random.RandomState(0)
    W = torch.from_numpy(rng.randint(-9, 10, size=(cc.obs_dim, cc.c.n_actions)).astype(np.int32)).cuda()
    b = torch.from_numpy(rng.randint(-30, 31, size=cc.c.n_actions).astype(np.int32)).cuda()

    def random_arm(fmt, rec):
        hs, rs = handles[fmt], records[fmt]
        return lambda i: hs[i % N_BATCHES].rollout(K, None, policy_seed=i, auto_reset=True,
                                                     record=rs[i % N_BATCHES] if rec else None)

    def policy_arm(rec):
        hs, rs = handles['i32'], records['i32']
        return lambda i: hs[i % N_BATCHES].rollout(K, policy=(W, b), auto_reset=True,
                                                     record=rs[i % N_BATCHES] if rec else None)

    gen = torch.Generator(device='cuda')
    gen.manual_seed(5)
    acts = torch.randint(0, cc.c.n_actions, (K, envs), generator=gen, device='cuda', dtype=torch.int32)
    stream = torch.cuda.Stream()
    stream.wait_stream(torch.cuda.current_stream())

    def onestep_arm(fmt):
        hs = handles[fmt]
        with torch.cuda.stream(stream):
            for h in hs:
                h.enable_episode_end()
                h.step(acts[0], auto_reset=True)                      # warm-up outside the capture
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=stream):
                for t in range(K):
                    for h in hs:
                        h.step(acts[t], auto_reset=True)
        torch.cuda.current_stream().wait_stream(stream)

        def run(i):
            if i % N_BATCHES == 0:                                    # one replay steps all N_BATCHES batches K times
                g.replay()
        return run

    arms = {'random/off': random_arm('i32', False), 'random/hits': random_arm('hits', True),
            'random/u8': random_arm('u8', True), 'random/i32': random_arm('i32', True),
            'policy/off': policy_arm(False), 'policy/i32': policy_arm(True),
            'onestep/hits': onestep_arm('hits'), 'onestep/u8': onestep_arm('u8'), 'onestep/i32': onestep_arm('i32')}
    reps = {}
    for name, fn in arms.items():                                     # warm-up, then launches per window
        for i in range(N_BATCHES):
            fn(i)
        torch.cuda.synchronize()
        t0 = time.time()
        for i in range(N_BATCHES):
            fn(i)
        torch.cuda.synchronize()
        per = (time.time() - t0) * 1e3 / N_BATCHES
        reps[name] = max(N_BATCHES, int(np.ceil(args.window_ms / per / N_BATCHES)) * N_BATCHES)
    runs = {name: [] for name in arms}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for r in range(args.rounds):
        order = list(arms) if r % 2 == 0 else list(reversed(list(arms)))
        for name in order:
            fn = arms[name]
            e0.record()
            for i in range(reps[name]):
                fn(100 + i)
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1)
            runs[name].append(envs * K * reps[name] / (ms * 1e-3))
    res = {}
    for name, v in runs.items():
        rate = float(np.median(v))
        fmt = name.split('/')[1]
        row = {"env_steps_per_s": rate, "runs": v, "launches_per_window": reps[name]}
        if fmt != 'off' and not name.startswith('onestep'):
            nb = record_bytes(handles[fmt][0])
            row.update(record_bytes_per_env_step=nb, write_GBps=rate * nb / 1e9,
                       write_share_of_copy_peak=rate * nb / 1e9 / COPY_PEAK_GBS, obs_row_bytes=handles[fmt][0].obs_row_bytes)
        res[name] = row
    line = {"script": "profiles/rollout_record.py", "gpu": gpu_info(), "torch": torch.__version__,
            "cuda": torch.version.cuda, "date": time.strftime('%Y-%m-%d'),
            "desc": desc + "; %d envs/batch x %d batches, K = %d steps per launch, auto-reset" % (envs, N_BATCHES, K),
            "rounds": args.rounds, "arms": res, "copy_peak_GBps": COPY_PEAK_GBS,
            "timing": "CUDA events around each arm's launches, arms alternated, median over rounds",
            "seconds": time.time() - t_start}
    print(json.dumps(line), flush=True)
    with open(args.out, 'a') as f:
        f.write(json.dumps(line) + '\n')


if __name__ == '__main__':
    main()
