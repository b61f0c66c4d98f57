"""A/B sweep of environment settings read by ngw_create on the BASELINE workloads.
    python profiles/sweep.py C2 "" "NGW_NO_CONCURRENT=1" ...     -> one JSON line per variant
Timing = bench.py's: rotating batches (> L2), CUDA-graph replay on one stream, CUDA events, >= 40 ms per measurement."""
import json
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), '..'))
import bench  # noqa: E402
from gym_novel_gridworlds_b200.runtime import BatchHandle  # noqa: E402


def measure(workload, knobs, obs_format='i32'):
    saved = {}
    for kv in knobs.split():
        k, v = kv.split('=')
        saved[k] = os.environ.get(k)
        os.environ[k] = v
    try:
        size = None
        if '@' in workload:                          # "C4@131072": the workload at another batch size (per-GPU share of a strong-scaled job)
            workload, size = workload.split('@')[0], int(workload.split('@')[1])
        desc, compiled, envs, rule, kw = bench.build_workload(workload.replace('-noreset', ''))
        if size:
            envs = size
        if workload.endswith('-noreset'):
            kw = {}
        bytes_step = float(np.mean([bench.algorithmic_bytes_per_env_step(cc, obs_format) for cc in compiled])) + (1 if len(compiled) > 1 else 0)
        n_b = max(2, int(np.ceil(1.6 * 126e6 / (envs * bytes_step))))
        batches = []
        for b in range(n_b):
            cfg_id = None
            if len(compiled) > 1:
                idx = np.arange(envs)
                cfg_id = (idx % len(compiled)) if rule == 'interleaved' else np.minimum(idx * len(compiled) // envs, len(compiled) - 1)
            h = BatchHandle(compiled, envs, seed=0, first_env_gid=b * envs, cfg_id=cfg_id, obs_format=obs_format)
            h.reset()
            if kw.get('max_episode_steps', 0):
                h.ep_len.copy_(torch.randint(0, kw['max_episode_steps'], (envs,), device='cuda', dtype=torch.int32))
            batches.append(h)
    finally:
        for k, v in saved.items():
            if v is None:
                del os.environ[k]
            else:
                os.environ[k] = v
    g = torch.Generator(device='cuda')
    g.manual_seed(1234)
    n_act = torch.tensor([cc.c.n_actions for cc in compiled], device='cuda')[batches[0].cfg_id.long()]
    acts = [(torch.randint(0, 1 << 30, (envs,), generator=g, device='cuda') % n_act).to(torch.int32) for _ in range(4)]
    for i in range(2 * n_b):
        batches[i % n_b].step(acts[i % 4], **kw)
    torch.cuda.synchronize()
    stream = torch.cuda.Stream()
    n_graph = n_b * max(1, 56 // n_b)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.stream(stream):
        with torch.cuda.graph(graph, stream=stream):
            for i in range(n_graph):
                batches[i % n_b].step(acts[i % 4], **kw)
        graph.replay()
    torch.cuda.synchronize()
    best = []
    for rep in range(3):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        replays = 1
        while True:
            with torch.cuda.stream(stream):
                e0.record(stream)
                for _ in range(replays):
                    graph.replay()
                e1.record(stream)
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1)
            if ms >= 40.0 or replays >= 4096:
                break
            replays *= 2
        best.append(ms / (replays * n_graph) * 1e3)
    us = float(np.median(best))
    peak, _ = bench.measured_hbm_peak()
    out = {"workload": workload, "knobs": knobs, "obs_format": obs_format, "us_per_step": round(us, 3),
           "env_steps_per_s": envs / (us * 1e-6), "frac_of_hbm_peak": round(envs * bytes_step / (us * 1e-6) / 1e9 / peak, 4),
           "bytes_per_env_step": bytes_step, "batches": n_b, "us_all": [round(x, 3) for x in best]}
    for h in batches:
        h.close()
    return out


if __name__ == '__main__':
    workload = sys.argv[1]
    fmt = 'i32'
    variants = sys.argv[2:] or ['']
    if variants and variants[0] in ('i32', 'u8'):
        fmt, variants = variants[0], variants[1:] or ['']
    for knobs in variants:
        try:
            print(json.dumps(measure(workload, knobs, fmt)), flush=True)
        except Exception as e:                      # a knob combination the library refuses must not end the sweep
            print(json.dumps({"workload": workload, "knobs": knobs, "obs_format": fmt, "error": str(e)[:200]}), flush=True)
