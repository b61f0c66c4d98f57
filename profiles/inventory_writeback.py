"""CPU model of step1w_kernel's inventory write-back (store 1): how many envs, tiles and 32-byte inventory sectors a step
changes, at the episode ages bench.py times, with uniform random actions, on the oracle (no GPU, no timing).

    python profiles/inventory_writeback.py [C2 C3 C4] [--envs 8192] [--from 230] [--to 460]

A step stores back only the sectors of a tile's inventory span that hold a changed row; sector s of a tile with rows of
R = 4 inv_stride bytes holds rows 32 s / R .. (32 s + 31) / R.  Prints one table row per workload: changed envs, tiles
with any change, sectors stored, and the bytes saved per env-step against bench.py's algorithmic bytes (which count the
whole inventory write), for sector stores and for skipping unchanged tiles only."""
import argparse
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402
from oracle.oracle_lib import OracleBatch  # noqa: E402


def model(name, n, t_lo, t_hi):
    desc, compiled, _, _, _ = bench.build_workload(name)
    cfg_id = None if len(compiled) == 1 else (np.arange(n) % len(compiled)).astype(np.uint8)   # C4: env i -> i mod 4
    ob = OracleBatch(compiled, n, cfg_id=cfg_id)
    ob.reset_legacy(1)
    n_actions = np.array([cc.c.n_actions for cc in compiled])[ob.cfg_id]
    rng = np.random.RandomState(0)
    row = 4 * ob.inv_stride
    first = 32 * np.arange(row)                                     # a tile's span is 32 rows = `row` sectors
    lo, hi = first // row, (first + 31) // row
    acc = []
    for t in range(t_hi):
        inv0 = ob.inv.copy()
        ob.step((rng.randint(0, 1 << 30, size=n) % n_actions).astype(np.int32), want_obs=False)
        if t < t_lo:
            continue
        dirty = (ob.inv != inv0).any(1).reshape(-1, 32)
        acc.append((dirty.mean(), dirty.any(1).mean(), (dirty[:, lo] | dirty[:, hi]).mean()))
    env_f, tile_f, sec_f = np.mean(acc, 0)
    total = bench.workload_bytes_per_env_step(compiled)
    saved, saved_tiles = row * (1 - sec_f), row * (1 - tile_f)
    return ob.inv_stride, env_f, tile_f, sec_f, saved, total, saved_tiles


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('workloads', nargs='*', default=['C2', 'C3', 'C4'])
    ap.add_argument('--envs', type=int, default=8192)
    ap.add_argument('--from', dest='t_lo', type=int, default=230)
    ap.add_argument('--to', dest='t_hi', type=int, default=460)
    args = ap.parse_args()
    print("| workload | inv_stride | envs whose inventory changes | tiles with any change | 32-B inventory sectors "
          "that must be stored | bytes saved / algorithmic bytes | tile skip only |")
    print("|---|---|---|---|---|---|---|")
    for name in args.workloads:
        stride, env_f, tile_f, sec_f, saved, total, saved_tiles = model(name, args.envs, args.t_lo, args.t_hi)
        print("| %s | %d | %.2f %% | %.1f %% | %.1f %% | %.1f / %.0f B = %.1f %% | %.1f %% |" % (
            name, stride, 100 * env_f, 100 * tile_f, 100 * sec_f, saved, total, 100 * saved / total,
            100 * saved_tiles / total))


if __name__ == '__main__':
    main()
