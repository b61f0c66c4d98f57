"""Cost of the numpy reset stream (ngw_set_reset_rng(NGW_RNG_NUMPY)) against the default Philox generator.
    python profiles/numpy_reset.py [--out profiles/numpy_reset.jsonl] [--rounds R]
Arms, each on a Philox handle and on a numpy-stream handle of the same workload (bench.py's configs), alternated in one
process for --rounds rounds:
  reset/C2, reset/C5   one ngw_reset of every env (C2: 65,536 envs on 10x10, C5: 524,288 envs on 40x40), CUDA events
                       around enough resets to fill --window-ms;
  step/C2, step/C5     graph replay of G ngw_step launches with auto-reset and uniform random actions, in microseconds per
                       step; the numpy stream pays in the queued-reset kernel, as often as episodes end.
The numpy stream draws the reference's sequential MT19937 stream (candidate-list pops, Fisher-Yates shuffles) where the
Philox generator samples without lists, so it is expected to be slower; the record holds what was measured.  One JSON
line is printed and appended to --out, with the card's name and power limit (a read-only nvidia-smi query in the same
run)."""
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

RESET_ENVS = {'C2': 65536, 'C5': 524288}
STEPS_PER_GRAPH = 32


def gpu_info():
    out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'], capture_output=True,
                         text=True, check=True).stdout.strip().splitlines()[0]
    name, power = [x.strip() for x in out.split(',')]
    return {"name": name, "power_limit": power}


def timed(fn, window_ms):
    """ms per call of fn over enough calls to fill window_ms (after one warm-up call)."""
    fn()
    torch.cuda.synchronize()
    t0 = time.time()
    fn()
    torch.cuda.synchronize()
    reps = max(1, int(np.ceil(window_ms / max((time.time() - t0) * 1e3, 1e-3))))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'numpy_reset.jsonl'))
    ap.add_argument('--rounds', type=int, default=3)
    ap.add_argument('--window-ms', type=float, default=400.0)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("numpy_reset.py measures on a CUDA device; none is present")
    arms, keep = {}, []
    for cfg in ('C2', 'C5'):
        _, compiled, envs, _, _ = bench.build_workload(cfg)
        for rng_kind in ('philox', 'numpy'):
            h = BatchHandle(compiled, RESET_ENVS[cfg], seed=1, reset_rng=rng_kind)
            arms['reset/%s/%s' % (cfg, rng_kind)] = (lambda h=h: h.reset(want_obs=True), 1)
            s = BatchHandle(compiled, envs, seed=2, reset_rng=rng_kind)
            s.reset()
            gen = torch.Generator(device='cuda')
            gen.manual_seed(3)
            acts = torch.randint(0, compiled[0].c.n_actions, (STEPS_PER_GRAPH, envs), generator=gen, device='cuda',
                                 dtype=torch.int32)
            stream = torch.cuda.Stream()
            stream.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(stream):
                s.step(acts[0], auto_reset=True)
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g, stream=stream):
                    for t in range(STEPS_PER_GRAPH):
                        s.step(acts[t], auto_reset=True)
            torch.cuda.current_stream().wait_stream(stream)
            arms['step/%s/%s' % (cfg, rng_kind)] = (g.replay, STEPS_PER_GRAPH)
            keep.append((s, acts, g))                                      # the graph replays these buffers
    runs = {k: [] for k in arms}
    for r in range(args.rounds):
        order = sorted(runs) if r % 2 == 0 else sorted(runs, reverse=True)
        for name in order:
            fn, per = arms[name]
            runs[name].append(timed(fn, args.window_ms) * 1e3 / per)      # microseconds per reset call / per step
    med = {k: float(np.median(v)) for k, v in runs.items()}
    rec = {"what": "numpy reset stream vs Philox", "gpu": gpu_info(), "date": time.strftime('%Y-%m-%d'),
           "reset_envs": RESET_ENVS, "steps_per_graph": STEPS_PER_GRAPH, "rounds": args.rounds,
           "us_median": med, "us_runs": runs,
           "numpy_over_philox": {k.replace('/philox', ''): med[k.replace('/philox', '/numpy')] / med[k]
                                 for k in med if k.endswith('/philox')}}
    line = json.dumps(rec)
    print(line)
    with open(args.out, 'a') as f:
        f.write(line + '\n')


if __name__ == '__main__':
    main()
