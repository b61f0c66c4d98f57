"""C2 (and C5) with the three observation row layouts of include/ngw.h: int32 vector, NGW_OBS_U8, NGW_OBS_HITS.
    python profiles/obs_formats.py [--out profiles/obs_formats.jsonl] [--batches N] [--e2e-steps S] [--rounds R]
prints one JSON line and appends it to --out.  Uses bench.py's own machinery (imported as profiles/sweep.py does):
  - graph: launch-to-launch us per step in CUDA-graph replay (bench.time_regions) for each layout, the same number of
    rotating batches for all three (default: what bench.py rotates for int32 rows);
  - e2e: bench.e2e_run (ngw_step_host_begin/_end pipelined over the batches, then the blocking ngw_step_host) for u8 vs
    hits rows, alternated in the same process for --rounds rounds, each beside bench.pcie_probe with that layout's D2H
    bytes per step (a plain cudaMemcpyAsync of the same bytes: the link's ceiling for it);
  - the same e2e comparison on C5 (map 40, auto-reset rows).
The card's name and power limit are read with a read-only nvidia-smi query in the same run."""
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

FORMATS = ('i32', 'u8', 'hits')


def gpu_info():
    out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'], capture_output=True,
                         text=True, check=True).stdout.strip().splitlines()[0]
    name, power = [x.strip() for x in out.split(',')]
    return {"name": name, "power_limit": power}


def row_bytes(cc, fmt):
    """observation row bytes of one env of this config (include/ngw.h)"""
    c = cc.c
    if c.n_beams <= 0:
        return 0
    L, B, ni = c.n_lidar_items, c.n_beams, c.n_inv_obs
    if fmt == 'i32':
        return 4 * (L * B + ni)
    return ((L * B if fmt == 'u8' else 2 * B) + 3) // 4 * 4 + 4 * ni


def algorithmic_bytes(compiled, fmt):
    """bench.algorithmic_bytes_per_env_step with the row of `fmt` (bench counts every non-int32 layout as u8 rows)"""
    per = [bench.algorithmic_bytes_per_env_step(cc, 'i32') - row_bytes(cc, 'i32') + row_bytes(cc, fmt) for cc in compiled]
    return float(np.mean(per)) + (1 if len(compiled) > 1 else 0)


def graph_us_per_step(name, fmt, n_batches, K, dev):
    wl = bench.Workload(name, 0, 1, dev, obs_format=fmt, n_batches=n_batches)
    for i in range(max(3, wl.n_batches)):
        wl.step(i)
    torch.cuda.synchronize(dev)
    reg = bench.time_regions(wl, K, dev, 1)[0]
    us = float(np.median(reg)) / K * 1e3
    rec = {"us_per_step": us, "regions": len(reg), "obs_row_bytes": wl.batches[0].obs_row_bytes,
           "algorithmic_bytes_per_env_step": algorithmic_bytes(wl.compiled, fmt),
           "achieved_gbs": wl.envs * algorithmic_bytes(wl.compiled, fmt) / (us * 1e-6) / 1e9}
    wl.close()
    return rec


def e2e_compare(name, n_batches, n_steps, rounds, dev):
    """u8 vs hits through the host-buffer path, alternated; median over the rounds of each figure"""
    if not n_batches:                                     # as bench.py rotates this workload with int32 rows, for both
        _, compiled, envs, _, _ = bench.build_workload(name)
        n_batches = bench.batches_to_exceed_l2(envs, bench.workload_bytes_per_env_step(compiled, 'i32'))
    wls = {f: bench.Workload(name, 0, 1, dev, obs_format=f, n_batches=n_batches) for f in ('u8', 'hits')}
    host_acts = [a.cpu().numpy() for a in wls['u8'].act_sets]
    envs = wls['u8'].envs
    runs = {f: {"pipelined": [], "blocking": [], "pcie_ms": []} for f in wls}
    for _ in range(rounds):
        for f, wl in wls.items():
            t_pipe, t_block, _ = bench.e2e_run(wl, n_steps, dev, 1, host_acts)
            runs[f]["pipelined"].append(envs * n_steps / t_pipe)
            runs[f]["blocking"].append(envs * n_steps / t_block)
            d2h = (wl.batches[0].obs_row_bytes + 10) * envs
            runs[f]["pcie_ms"].append(bench.pcie_probe(dev, d2h, 4 * envs, 1)["ms_per_step_bytes"])
    out = {}
    for f, wl in wls.items():
        d2h = (wl.batches[0].obs_row_bytes + 10) * envs
        pcie_ms = float(np.median(runs[f]["pcie_ms"]))
        pipe, block = float(np.median(runs[f]["pipelined"])), float(np.median(runs[f]["blocking"]))
        limit = envs / (pcie_ms * 1e-3)
        out[f] = {"obs_row_bytes": wl.batches[0].obs_row_bytes, "d2h_bytes_per_env_step": d2h / envs,
                  "h2d_bytes_per_env_step": 4, "pipelined_env_steps_per_s": pipe, "blocking_env_steps_per_s": block,
                  "pipelined_runs": runs[f]["pipelined"], "blocking_runs": runs[f]["blocking"],
                  "pcie_probe": {"ms_per_step_bytes": pcie_ms, "d2h_gbs": d2h / (pcie_ms * 1e-3) / 1e9,
                                 "limit_env_steps_per_s": limit},
                  "frac_of_pcie_limit": max(pipe, block) / limit}
    out["hits_over_u8"] = {"pipelined": out['hits']["pipelined_env_steps_per_s"] / out['u8']["pipelined_env_steps_per_s"],
                           "blocking": out['hits']["blocking_env_steps_per_s"] / out['u8']["blocking_env_steps_per_s"],
                           "pcie_limit": out['hits']["pcie_probe"]["limit_env_steps_per_s"]
                           / out['u8']["pcie_probe"]["limit_env_steps_per_s"]}
    out.update(envs=envs, batches_rotated=n_batches, steps=n_steps, rounds=rounds, workload=wls['u8'].desc)
    for wl in wls.values():
        wl.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=os.path.join(os.path.dirname(os.path.abspath(__file__)), 'obs_formats.jsonl'))
    ap.add_argument('--batches', type=int, default=0, help='rotating C2 batches for every layout (0: as bench.py, int32)')
    ap.add_argument('--graph-steps', type=int, default=256)
    ap.add_argument('--e2e-steps', type=int, default=400)
    ap.add_argument('--c5-e2e-steps', type=int, default=40)
    ap.add_argument('--rounds', type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("obs_formats.py measures on a CUDA device; none is visible")
    dev = torch.device('cuda', 0)
    torch.cuda.set_device(dev)
    t0 = time.time()
    gpu = gpu_info()
    desc, compiled, envs, _, _ = bench.build_workload('C2')
    n_b = args.batches or bench.batches_to_exceed_l2(envs, bench.workload_bytes_per_env_step(compiled, 'i32'))
    graph = {f: graph_us_per_step('C2', f, n_b, args.graph_steps, dev) for f in FORMATS}
    graph.update(envs=envs, batches_rotated=n_b, steps_per_region=args.graph_steps,
                 timing="bench.time_regions: CUDA-graph replay on one stream, CUDA events, median region")
    line = {"script": "profiles/obs_formats.py", "gpu": gpu, "torch": torch.__version__, "cuda": torch.version.cuda,
            "date": time.strftime('%Y-%m-%d', time.gmtime()),
            "C2_graph": graph,
            "C2_e2e": e2e_compare('C2', n_b, args.e2e_steps, args.rounds, dev),
            "C5_e2e": e2e_compare('C5', 0, args.c5_e2e_steps, args.rounds, dev)}
    line["seconds"] = time.time() - t0
    s = json.dumps(line)
    print(s)
    with open(args.out, 'a') as f:
        f.write(s + '\n')


if __name__ == '__main__':
    main()
