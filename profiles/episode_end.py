"""Cost of the episode-end outputs (ngw_set_episode_end_buffers: truncated flags + the last observation of every
auto-reset env) on the batched auto-reset step, in CUDA-graph replay.
    python profiles/episode_end.py [--out profiles/episode_end.jsonl] [--rounds R] [--graph-steps K]
Per workload, the same rotating batches (bench.Workload, as bench.py builds them) are captured twice: one graph of K
steps with the buffers off, then one with them on.  The two graphs are replayed alternately in one process (the order
flips every round), each timed with CUDA events over enough replays to fill --window-ms; the record holds the median us
per step of each arm, every round's figure, and the auto-resets per step the library counted (NGW_STAT_RESETS).
Workloads:
  - C2: 65,536 envs per batch, auto-reset with max_episode_steps 256, episode ages staggered as bench.py does for C5;
  - C5: bench.py's C5 (map 40 + additem(hard), 524,288 envs, auto-reset, max_episode_steps 256).
One JSON line per workload is printed and appended to --out, with the card's name and power limit (a read-only
nvidia-smi query in the same run)."""
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

T_MAX = 256


def gpu_info():
    out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'], capture_output=True,
                         text=True, check=True).stdout.strip().splitlines()[0]
    name, power = [x.strip() for x in out.split(',')]
    return {"name": name, "power_limit": power}


def workload(name, dev):
    wl = bench.Workload(name, 0, 1, dev)
    if name == 'C2':                                   # bench.py's C2 steps without auto-reset: add it, ages staggered
        wl.kw = {'auto_reset': True, 'max_episode_steps': T_MAX}
        gen = torch.Generator(device=dev)
        gen.manual_seed(99)
        for h in wl.batches:
            h.ep_len.copy_(torch.randint(0, T_MAX, (wl.envs,), generator=gen, device=dev, dtype=torch.int32))
    assert wl.kw == {'auto_reset': True, 'max_episode_steps': T_MAX}
    return wl


def capture(wl, K, stream):
    g = torch.cuda.CUDAGraph()
    with torch.cuda.stream(stream):
        with torch.cuda.graph(g, stream=stream):
            for i in range(K):
                wl.step(i)
    return g


def time_replays(g, reps, stream):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.cuda.stream(stream):
        e0.record(stream)
        for _ in range(reps):
            g.replay()
        e1.record(stream)
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def measure(name, K, rounds, window_ms, dev):
    wl = workload(name, dev)
    K = max(K - K % wl.n_batches, wl.n_batches)        # whole rotations: every batch steps equally often
    stream = torch.cuda.Stream(dev)
    stream.wait_stream(torch.cuda.current_stream(dev))
    graphs = {'off': capture(wl, K, stream)}
    for h in wl.batches:                               # the off graph keeps null pointers; the buffers outlive both graphs
        h.enable_episode_end()
    graphs['on'] = capture(wl, K, stream)
    for g in graphs.values():                          # upload + warm-up
        for _ in range(2):
            time_replays(g, 1, stream)
    reps = max(1, int(np.ceil(window_ms / max(time_replays(graphs['off'], 1, stream), 1e-3))))
    for h in wl.batches:
        h.stats(reset=True)
    runs = {'off': [], 'on': []}
    for r in range(rounds):
        for arm in (('off', 'on') if r % 2 == 0 else ('on', 'off')):
            runs[arm].append(time_replays(graphs[arm], reps, stream) / (reps * K) * 1e3)
    steps = 2 * rounds * reps * K
    resets = sum(float(h.stats()[5].item()) for h in wl.batches)
    off, on = float(np.median(runs['off'])), float(np.median(runs['on']))
    rec = {"workload": name, "desc": wl.desc + ("; here with auto-reset, max_episode_steps 256, staggered episode ages"
                                                if name == 'C2' else ""),
           "envs_per_batch": wl.envs, "batches_rotated": wl.n_batches, "steps_per_graph": K, "replays_per_window": reps,
           "rounds": rounds, "us_per_step_off": off, "us_per_step_on": on, "delta_us": on - off,
           "delta_pct": 100.0 * (on - off) / off, "runs_off": runs['off'], "runs_on": runs['on'],
           "auto_resets_per_step": resets / steps,
           "obs_row_bytes": wl.batches[0].obs_row_bytes,
           "timing": "CUDA-graph replay on one stream, CUDA events around each arm's replays, median over rounds"}
    wl.close()
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=os.path.join(os.path.dirname(os.path.abspath(__file__)), 'episode_end.jsonl'))
    ap.add_argument('--workloads', default='C2,C5')
    ap.add_argument('--graph-steps', type=int, default=256)
    ap.add_argument('--rounds', type=int, default=7)
    ap.add_argument('--window-ms', type=float, default=100.0)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("episode_end.py measures on a CUDA device; none is visible")
    dev = torch.device('cuda', 0)
    torch.cuda.set_device(dev)
    gpu = gpu_info()
    for name in args.workloads.split(','):
        t0 = time.time()
        rec = measure(name, args.graph_steps if name != 'C5' else min(args.graph_steps, 64), args.rounds,
                      args.window_ms, dev)
        line = {"script": "profiles/episode_end.py", "gpu": gpu, "torch": torch.__version__, "cuda": torch.version.cuda,
                "date": time.strftime('%Y-%m-%d', time.gmtime())}
        line.update(rec)
        line["seconds"] = time.time() - t0
        s = json.dumps(line)
        print(s, flush=True)
        with open(args.out, 'a') as f:
            f.write(s + '\n')


if __name__ == '__main__':
    main()
