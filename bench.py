#!/usr/bin/env python
"""bench.py — env-steps/sec of the fused step + LidarInFront hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
    torchrun --nproc-per-node N bench.py --gpus N ...          (one rank per GPU)

A "step" is ONE pass of the hot path over ONE batch of 65,536 envs of BASELINE config C2
(NovelGridworld-Pogostick-v1 + LimitActions(10 actions) + LidarInFront(8 beams)), random actions.
To keep L2 cold between timed iterations the run rotates over several independent batches whose combined
working set (state + outputs) exceeds the 126 MB L2 ("inputs larger than L2").

Prints ONE JSON line (rank 0):
  value       device-timed throughput, inputs resident in HBM: CUDA-graph replay of exactly K launches on one stream,
              CUDA events on that stream around those K steps (after W eager warm-up steps and untimed replays of the
              graph right ahead of them, lead_in_regions(K)), MAX over ranks.
  e2e         the same metric through the host-buffer C-ABI call (ngw_step_host_begin/_end): pinned H2D of the actions,
              one launch, D2H of obs/reward/done/step_cost/result every step, >= 200 steps; observation rows in the
              compact NGW_OBS_U8 layout (uint8 lidar ranges + int32 inventory tail; `int32_rows` = the default layout);
              `pcie` = a plain cudaMemcpyAsync probe of the same bytes on every rank at the same time.
  roofline    algorithmic bytes per launch / average launch duration vs the measured HBM copy peak.
  workloads   BASELINE configs C3, C4 (1,048,576 envs sharded over the ranks, env i -> novelty i mod 4) and C5
              (524,288 envs per GPU, fused auto-reset), same timing method, per-GPU roofline fraction.
  cpu_baseline  the C port of the reference path (oracle/ngw_oracle.c) on all host threads, and — when the unmodified
              Python reference is installed under baseline/_ref — its single-process and process-pool throughput.
`--impl reference` times the C port alone (rank 0 only), same config keys.
`--dump-outputs DIR` writes what the last timed step of `value` returned (rank 0) as DIR/<name>.npy, see dump_outputs().
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
if os.environ.get('NCCL_DEBUG', 'VERSION').upper() == 'VERSION':
    os.environ['NCCL_DEBUG'] = 'WARN'                  # keep NCCL's version banner off stdout: ONE JSON line only

ENVS_PER_BATCH = 65536
C2_SET = ['Forward', 'Left', 'Right', 'Break', 'Place_tree_tap', 'Extract_rubber',
          'Craft_plank', 'Craft_stick', 'Craft_tree_tap', 'Craft_pogo_stick']
METRIC = "env-steps/sec, Pogostick-v1+LidarInFront, 1/2/4/8 B200 vs host-CPU reference"
N_ACTION_SETS = 16
GRAPH_STEPS = 1024
L2_BYTES = 126e6
VALUE_FLOOR_MS = 50.0            # the K-step region is repeated until this much was timed
E2E_MIN_STEPS = 400
E2E_CHUNK = 50                # e2e loops are timed in chunks of this many steps, median chunk reported
REFERENCE_FLOOR_S = 2.0
C4_TOTAL_ENVS = 1048576
DUMP_LIMIT_BYTES = 64 << 20       # --dump-outputs: above this a fixed, seeded sample of env rows is written
QUEUE_SLEEP_CYCLES = 4000000      # ~2 ms of device spin ahead of a timed region, see time_regions
LEAD_IN_STEPS = 2048              # untimed steps replayed right ahead of the exactly-K-step `value` region


def lead_in_regions(K):
    """Untimed replays of the K-step region ahead of the timed one (a function of K alone, so that the batches always
    advance by the same number of steps): the timed steps run in the steady state that the 2nd .. nth region of a
    longer run sees (on a B200 at its 1000 W limit, 1965 MHz, a 20-step C2 region measured 1-3 % slower right behind a
    single untimed replay than in a long back-to-back run)."""
    return max(1, -(-LEAD_IN_STEPS // K))


def build_c2_chain(num_envs=1, device=None):
    import gym_novel_gridworlds_b200 as gym
    env = gym.make('NovelGridworld-Pogostick-v1', num_envs=num_envs, device=device)
    env = gym.LimitActions(env, set(C2_SET))
    return gym.LidarInFront(env, num_beams=8)


def build_workload(name):
    """BASELINE.json configs -> (description, [compiled configs], envs per batch per GPU, cfg-id rule, step kwargs).
    C2 is the headline; C3-C5 are measured into `workloads` (or alone with `--workload`)."""
    import gym_novel_gridworlds_b200 as gym
    from gym_novel_gridworlds_b200.compiler import compile_chain

    def pogo(extra_actions=(), map_size=10):
        env = gym.make('NovelGridworld-Pogostick-v1')
        env.map_size = map_size
        env = gym.LimitActions(env, set(C2_SET) | set(extra_actions))
        return gym.LidarInFront(env, num_beams=8)

    if name == 'C2':
        return ("C2: NovelGridworld-Pogostick-v1 + LimitActions(10) + LidarInFront(8), 65536 envs/batch, "
                "uniform random actions", [compile_chain(pogo())], 65536, None, {})
    if name == 'C3':
        env = gym.make('NovelGridworld-Bow-v1')
        env = gym.LidarInFront(env, num_beams=8)
        env = gym.inject_novelty(env, 'axe', 'medium', 'wooden', '')
        env = gym.inject_novelty(env, 'fence', 'hard', 'oak', '')
        return ("C3: NovelGridworld-Bow-v1 + LidarInFront(8) + axe(medium, wooden) + fence(hard, oak), 262144 envs/batch",
                [compile_chain(env)], 262144, None, {})
    if name in ('C4', 'C4-blocked'):
        np.random.seed(4)
        chains = [gym.inject_novelty(pogo(['Chop']), 'addchop'), gym.inject_novelty(pogo(['Jump']), 'addjump'),
                  gym.inject_novelty(pogo(), 'additem', 'medium', 'spring'),
                  gym.inject_novelty(pogo(), 'remapaction', 'hard')]
        rule = 'interleaved' if name == 'C4' else 'blocked'
        return ("C4: Pogostick-v1 + LimitActions + LidarInFront(8), per-env novelty addchop / addjump / additem(medium) / "
                "remapaction(hard), config ids %s, 1048576 envs/batch, one launch per step" % rule,
                [compile_chain(c) for c in chains], C4_TOTAL_ENVS, rule, {})
    if name == 'C5':
        env = gym.inject_novelty(pogo(map_size=40), 'additem', 'hard', 'spring')
        return ("C5: Pogostick-v1 map_size 40 + additem(hard) + LidarInFront(8), 524288 envs/batch per GPU, fused "
                "auto-reset, max_episode_steps 256 (harness truncation knob)",
                [compile_chain(env)], 524288, None, {'auto_reset': True, 'max_episode_steps': 256})
    raise ValueError(name)


def algorithmic_bytes_per_env_step(cc, obs_format='i32'):
    """SURVEY §8d with the dtypes actually written: read ms^2 + 4 (pose) + 4 I (inventory) + 4 (action); write 4 (pose)
    + 4 I + observation row + 4 (reward) + 4 (step_cost) + 1 (done) + 1 (result); grid write-back counted as 0.
    Observation row: int32 [L B + I_obs], or (NGW_OBS_U8) uint8 [L B] padded to 4 + int32 [I_obs]."""
    ms, n_items, d = cc.map_size, cc.n_items, cc.obs_dim
    n_lidar = cc.c.n_lidar_items * cc.c.n_beams
    row = 4 * d if obs_format == 'i32' else ((n_lidar + 3) // 4 * 4 + 4 * cc.c.n_inv_obs if d else 0)
    return (ms * ms + 4 + 4 * n_items + 4) + (4 + 4 * n_items + row + 4 + 4 + 1 + 1)


def workload_bytes_per_env_step(compiled, obs_format='i32'):
    """mean over the configs of a batch (+1 byte config id per env when the batch is mixed)"""
    return float(np.mean([algorithmic_bytes_per_env_step(cc, obs_format) for cc in compiled])) + (1 if len(compiled) > 1 else 0)


L2_FACTOR = 4.0                  # rotating working set >= 4 x L2: with 1.6 x (7 C2 batches) ncu still shows 28 % of the
                                 # algorithmic bytes served by L2 (profiles/step_kernel_traffic.json), with 4 x about 10 %


def batches_to_exceed_l2(envs, bytes_step, factor=L2_FACTOR):
    return max(2, int(np.ceil(factor * L2_BYTES / (envs * bytes_step))))


def c2_config(n_gpus):
    """The `config` object of the JSON line — static, so that both arms (--impl ours / reference) print the same one."""
    n_b = batches_to_exceed_l2(ENVS_PER_BATCH, 446.0)
    return {"workload": "C2: NovelGridworld-Pogostick-v1 + LimitActions(10) + LidarInFront(8), 65536 envs/batch, "
                        "uniform random actions",
            "envs_per_batch": ENVS_PER_BATCH, "batches_rotated": n_b,
            "l2": "inputs larger than L2: %d rotating batches, %.0f MB combined working set = %.1f x the 126 MB L2"
                  % (n_b, n_b * ENVS_PER_BATCH * 446.0 / 1e6, n_b * ENVS_PER_BATCH * 446.0 / L2_BYTES),
            "obs_dtype": "int32 rows for value/roofline (446 B/env-step); e2e moves NGW_OBS_U8 rows",
            "parallelism": "independent shards, one process per GPU x%d, no collective on the step path" % n_gpus}


def measured_hbm_peak():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    try:
        with open(path) as f:
            return float(json.load(f)['hbm_gbs']), 'measured (MEASURED_PEAKS.json hbm_gbs)'
    except Exception:
        return 6650.0, 'fallback (B200_PROFILING.md 6.65 TB/s)'


def measured_traffic(workload):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed multi-launch ncu capture."""
    try:
        with open(os.path.join(ROOT, 'profiles', 'step_kernel_traffic.json')) as f:
            rec = json.load(f).get(workload)
        return (rec or {}).get('dram_bytes_per_launch'), (rec or {}).get('source')
    except Exception:
        return None, None


class ClockSampler(threading.Thread):
    """Samples SM clock + throttle reasons with NVML while the timed regions run."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag, self.max_mhz, self.ok = index, [], False, None, False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.ok = False

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        while not self.stop_flag:
            try:
                mhz = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                try:
                    reasons = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    reasons = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                util = nv.nvmlDeviceGetUtilizationRates(self.h).gpu
                self.samples.append((time.perf_counter(), mhz, reasons, util))
            except Exception:
                pass
            time.sleep(0.02)

    def summary(self, t0, t1):
        names = {0x2: 'applications_clocks_setting', 0x4: 'sw_power_cap', 0x8: 'hw_slowdown', 0x10: 'sync_boost',
                 0x20: 'sw_thermal_slowdown', 0x40: 'hw_thermal_slowdown', 0x80: 'hw_power_brake_slowdown',
                 0x100: 'display_clock_setting'}
        if not self.samples:                            # NVML unavailable: one nvidia-smi reading as a last resort
            try:
                import subprocess
                q = subprocess.run(['nvidia-smi', '-i', str(self.index), '--query-gpu=clocks.sm,clocks.max.sm,'
                                    'clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
                                    'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap',
                                    '--format=csv,noheader,nounits'], capture_output=True, text=True, timeout=20)
                f = [x.strip() for x in q.stdout.strip().split(',')]
                labels = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
                return {"sm_mhz": float(f[0]), "sm_max_mhz": float(f[1]),
                        "reasons": [n for n, v in zip(labels, f[2:]) if v.lower().startswith('active')],
                        "samples": 1, "source": "nvidia-smi after the timed region"}
            except Exception:
                return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "samples": 0}
        inside = [s for s in self.samples if t0 <= s[0] <= t1] or [s for s in self.samples if s[3] > 0] or self.samples
        busy = [s for s in inside if s[3] > 0] or inside
        reasons = 0
        for s in inside:
            reasons |= s[2]
        return {"sm_mhz": float(np.median([s[1] for s in busy])), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(n for b, n in names.items() if reasons & b), "samples": len(inside)}


# ---------------------------------------------------------------------------------------------- host-side helpers
def pin_to_gpu_numa(local_rank):
    """One process per GPU: run this rank's host threads — and therefore first-touch its pinned buffers — on the CPUs
    NVML reports as local to the GPU (its NUMA node), when the container's cpuset allows any of them."""
    info = {"applied": False}
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(local_rank)
        allowed = os.sched_getaffinity(0)
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (max(allowed | {os.cpu_count() or 1}) // 64) + 1)
        ideal = {64 * i + b for i, w in enumerate(words) for b in range(64) if (int(w) >> b) & 1}
        pci = pynvml.nvmlDeviceGetPciInfo(h).busId
        pci = pci.decode() if isinstance(pci, bytes) else pci
        node = None
        try:
            with open('/sys/bus/pci/devices/%s/numa_node' % pci.lower()[-12:]) as f:
                node = int(f.read().strip())
        except Exception:
            pass
        info.update({"gpu_numa_node": node, "gpu_local_cpus": len(ideal), "allowed_cpus": len(allowed)})
        both = ideal & allowed
        if both and both != allowed:
            os.sched_setaffinity(0, both)
            info["applied"] = True
        info["cpus_used"] = len(os.sched_getaffinity(0))
    except Exception as e:                                    # no NVML / no permission: stay where the launcher put us
        info["error"] = str(e)[:80]
    return info


def cpu_port_regions(cc, envs, K, warmup, threads, floor_s, max_regions=400):
    """Times the C oracle port (oracle/ngw_oracle.c): a region = K steps over `envs` environments with all host threads
    (threads own contiguous env slices, no per-step barrier — the fastest honest CPU arrangement of the reference
    algorithm; every step still writes obs/reward/done/step_cost/result).  Regions repeat until floor_s seconds were
    timed; returns the list of region durations."""
    from oracle.oracle_lib import OracleBatch
    ob = OracleBatch([cc], envs)
    ob.reset_legacy(1)
    rng = np.random.RandomState(1234)
    acts = np.stack([rng.randint(0, cc.c.n_actions, size=envs).astype(np.int32) for _ in range(N_ACTION_SETS)])
    if warmup:
        ob.rollout(acts, warmup, n_threads=threads)
    regions, total = [], 0.0
    while (total < floor_s or len(regions) < 3) and len(regions) < max_regions:
        t0 = time.perf_counter()
        ob.rollout(acts, K, n_threads=threads)
        dt = time.perf_counter() - t0
        regions.append(dt)
        total += dt
    return regions


def _python_reference_worker(args):
    seconds, seed, ref_root, repo_root = args
    import contextlib
    import io
    for p in (os.path.join(repo_root, 'tests'), repo_root):
        if p not in sys.path:
            sys.path.insert(0, p)
    import scenarios
    desc = {'env': scenarios.POGO, 'map_size': 10, 'chain': [['limit', scenarios.C2_SET], ['lidar', 8]]}
    with contextlib.redirect_stdout(io.StringIO()):
        env = scenarios.build_chain(scenarios.reference_namespace(ref_root), desc)
        n_act = len(env.limited_actions_id)
        np.random.seed(seed)
        env.reset()
        rng = np.random.RandomState(seed)
        steps, t0 = 0, time.perf_counter()
        while time.perf_counter() - t0 < seconds:
            for _ in range(100):                                  # tests/random_action.py:51-55 without render/prints
                obs, r, done, info = env.step(int(rng.randint(n_act)))
                if done:
                    env.reset()
            steps += 100
        return steps / (time.perf_counter() - t0)


def python_reference_baseline(seconds=4.0):
    """The UNMODIFIED Python reference (installed under git-ignored baseline/_ref by __graft_entry__.build(), imported
    through oracle/gymstub) on C2: one process, and a pool of os.cpu_count() worker processes with one env each
    (SubprocVecEnv style: stable-baselines is not installed)."""
    ref_root = os.path.join(ROOT, 'baseline', '_ref')
    if not os.path.isdir(os.path.join(ref_root, 'gym_novel_gridworlds')):
        return {"unavailable": "baseline/_ref/gym_novel_gridworlds is not installed (run __graft_entry__.build() where "
                               "/root/reference exists)"}
    import multiprocessing as mp
    try:
        ctx = mp.get_context('spawn')                             # never fork a process that holds a CUDA context
        workers = os.cpu_count() or 1
        with ctx.Pool(1) as pool:
            single = pool.map(_python_reference_worker, [(seconds, 0, ref_root, ROOT)])[0]
        with ctx.Pool(workers) as pool:
            pooled = sum(pool.map(_python_reference_worker, [(seconds, i, ref_root, ROOT) for i in range(workers)]))
        model = ''
        try:
            with open('/proc/cpuinfo') as f:
                model = [ln.split(':', 1)[1].strip() for ln in f if ln.startswith('model name')][0]
        except Exception:
            pass
        return {"single_process": single, "pool": pooled, "pool_workers": workers, "unit": "env-steps/s",
                "seconds_each": seconds, "cpu": model, "python": sys.version.split()[0], "numpy": np.__version__,
                "what": "gtatiya/gym-novel-gridworlds, unmodified, C2 chain, random actions, reset on done"}
    except Exception as e:
        return {"unavailable": "python reference failed: %s" % str(e)[:120]}


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU implementation of the path = its C port (the oracle) with every host
    thread; the unmodified Python reference is reported beside it by the main arm (cpu_baseline.python_reference).
    A step is one pass over S envs of the same C2 workload, S bounded so that K steps end within a few minutes; the
    K-step region is repeated for >= 2 s and the median region is reported."""
    if rank != 0:
        return
    from gym_novel_gridworlds_b200.compiler import compile_chain
    cc = compile_chain(build_c2_chain())
    threads = os.cpu_count() or 1
    K = max(args.steps, 1)
    envs = ENVS_PER_BATCH
    while envs > 1024 and envs * K > 4e8:
        envs //= 2
    regions = cpu_port_regions(cc, envs, K, args.warmup, threads, REFERENCE_FLOOR_S)
    dt = float(np.median(regions))
    value = K * envs / dt
    sample = ("%d regions of %d steps x %d envs of C2 (%.1f s timed, median region), C port of the reference path "
              "(oracle/ngw_oracle.c), %d threads, no per-step barrier" % (len(regions), K, envs, sum(regions), threads))
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "env-steps/s", "n_gpus": args.gpus,
        "steps": K, "warmup": args.warmup, "ms_per_step": dt / K * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "int32", "data": "synthetic",
        "config": c2_config(args.gpus),
        "cpu_baseline": {"value": value, "unit": "env-steps/s", "cores": threads, "kind": "port", "sample": sample,
                         "envs_per_step": envs},
        "e2e": {"value": value, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------- GPU side
class Workload(object):
    """Rotating batches of one BASELINE workload on this rank, sharded by global env id."""

    def __init__(self, name, rank, world, dev, obs_format='i32', n_batches=None):
        import torch
        from gym_novel_gridworlds_b200.runtime import BatchHandle
        from gym_novel_gridworlds_b200.sharding import shard_range
        self.name = name
        self.desc, self.compiled, total, self.rule, self.kw = build_workload(name)
        n_cfg = len(self.compiled)
        self.bytes_step = workload_bytes_per_env_step(self.compiled, obs_format)
        if name.startswith('C4'):                      # strong scaling: the 1M-env job is cut into contiguous id ranges
            lo, hi = shard_range(total, rank, world)
            self.scaling, self.total_envs = 'strong', total
        else:                                          # weak scaling: every GPU runs the configured batch
            lo, hi = rank * total, (rank + 1) * total
            self.scaling, self.total_envs = 'weak', total * world
        self.envs = hi - lo
        self.n_batches = n_batches or batches_to_exceed_l2(self.envs, self.bytes_step)
        gen = torch.Generator(device=dev)
        gen.manual_seed(1234 + rank)
        self.batches = []
        for b in range(self.n_batches):
            gid0 = b * self.total_envs + lo            # global env id of this shard's first env in rotation slot b
            cfg_id = None
            if n_cfg > 1:
                gid = lo + np.arange(self.envs, dtype=np.int64)
                cfg_id = (gid % n_cfg) if self.rule == 'interleaved' else np.minimum(gid * n_cfg // total, n_cfg - 1)
            h = BatchHandle(self.compiled, self.envs, device=dev, seed=0, first_env_gid=gid0, cfg_id=cfg_id,
                            obs_format=obs_format)
            h.reset()
            if self.kw.get('max_episode_steps', 0) > 0:        # stagger episode ages so truncation-resets spread evenly
                h.ep_len.copy_(torch.randint(0, self.kw['max_episode_steps'], (self.envs,), generator=gen, device=dev,
                                             dtype=torch.int32))
            self.batches.append(h)
        n_act = torch.tensor([cc.c.n_actions for cc in self.compiled], device=dev, dtype=torch.int64)
        self.max_actions = int(n_act.max().item())
        per_env_n = n_act[self.batches[0].cfg_id.long()]
        self.n_sets = N_ACTION_SETS if self.envs <= 262144 else 4
        self.act_sets = []
        for _ in range(self.n_sets):
            r = torch.randint(0, 1 << 30, (self.envs,), generator=gen, device=dev, dtype=torch.int64)
            self.act_sets.append((r % per_env_n).to(torch.int32))
        self.reset_error_flags = sum(int((h.error_flags != 0).sum().item()) for h in self.batches)
        self.last = None                                # batch of the latest step() call (in a capture: the last replayed)

    def step(self, i):
        self.last = i % self.n_batches
        self.batches[self.last].step(self.act_sets[i % self.n_sets], **self.kw)

    def launches(self):
        return sum(h.launch_count() for h in self.batches)

    def concurrent_launches(self):
        return sum(h.concurrent_launch_count() for h in self.batches)

    def close(self):
        for h in self.batches:
            h.close()
        self.batches = []


def time_regions(wl, K, dev, world, floor_ms=VALUE_FLOOR_MS, n_streams=1, max_regions=4000, n_regions=None):
    """Exactly K steps per region as CUDA-graph replays on one launching stream, CUDA events on that stream around every
    region; barrier + synchronize on both sides of the whole measurement.  The region is repeated until floor_ms were
    timed, or exactly n_regions times when that is given (then the batches advance by a number of steps that does not
    depend on the speed of the build).  Returns (region durations in ms, wall bracket, launches per step, steps per
    graph)."""
    import torch
    import torch.distributed as dist
    n_b = wl.n_batches
    if K <= GRAPH_STEPS:
        g_steps = K                                                     # the whole region is ONE graph of exactly K launches
    else:
        g_steps = GRAPH_STEPS - GRAPH_STEPS % n_b                       # whole rotations per replay
    g_steps = max(g_steps, 1)
    stream = torch.cuda.Stream(dev)

    def capture(n, first=0):
        g = torch.cuda.CUDAGraph()
        side = [torch.cuda.Stream(dev) for _ in range(n_streams)] if n_streams > 1 else []
        with torch.cuda.stream(stream):
            with torch.cuda.graph(g, stream=stream):
                if not side:
                    for i in range(n):
                        wl.step(first + i)
                else:                                   # independent batches on parallel branches of the graph
                    for s_ in side:
                        s_.wait_stream(stream)
                    for i in range(n):
                        with torch.cuda.stream(side[((first + i) % n_b) % n_streams]):
                            wl.step(first + i)
                    for s_ in side:
                        stream.wait_stream(s_)
        return g

    before, before_c = wl.launches(), wl.concurrent_launches()
    graph = capture(g_steps)
    launches_per_step = (wl.launches() - before) / g_steps
    wl.overlapped_launches_per_graph = wl.concurrent_launches() - before_c     # launches proven independent of their predecessor
    replays, rem = K // g_steps, K % g_steps
    graph_rem = capture(rem, replays * g_steps) if rem else None

    def region():
        for _ in range(replays):
            graph.replay()
        if graph_rem:
            graph_rem.replay()

    fixed = n_regions is not None
    if not fixed:
        with torch.cuda.stream(stream):
            region()                                                     # graph warm-up (uploads the exec graphs)
        torch.cuda.synchronize(dev)
        # how many regions make the floor: probe one
        p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(stream):
            p0.record(stream)
            region()
            p1.record(stream)
        torch.cuda.synchronize(dev)
        n_regions = int(min(max_regions, max(3, np.ceil(floor_ms / max(p0.elapsed_time(p1), 1e-3)))))
        if world > 1:
            t = torch.tensor([n_regions], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            n_regions = int(t.item())
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize(dev)
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(n_regions + 1)]
    t0 = time.perf_counter()
    with torch.cuda.stream(stream):
        if fixed:
            # the graph warm-up (uploads the exec graphs; lead_in_regions(K) replays) runs right ahead of the timed
            # regions, and both wait behind a device spin while the host enqueues them: the first event does not time
            # the host's graph launch
            torch.cuda._sleep(QUEUE_SLEEP_CYCLES)
            for _ in range(lead_in_regions(K)):
                region()
        evs[0].record(stream)
        for r in range(n_regions):
            region()
            evs[r + 1].record(stream)
    torch.cuda.synchronize(dev)
    if world > 1:
        dist.barrier()
    t1 = time.perf_counter()
    return [evs[r].elapsed_time(evs[r + 1]) for r in range(n_regions)], (t0, t1), launches_per_step, g_steps


def dump_outputs(wl, out_dir):
    """What the last timed step returned to its caller, for comparing two builds output by output: the observation rows,
    reward, done, step_cost and result of the batch that step advanced, as float32 DIR/<name>.npy.  When they would
    exceed DUMP_LIMIT_BYTES, the same fixed, seeded sample of env rows is kept of each (its indices: env_index.npy)."""
    import torch
    h = wl.batches[wl.last]
    torch.cuda.synchronize(h.device)
    outs = {'obs': h.obs[:, :h.obs_dim], 'reward': h.reward, 'done': h.done, 'step_cost': h.step_cost,
            'result': h.result}
    if not h.obs_dim:
        del outs['obs']
    row_bytes = 4 * sum(t[0].numel() for t in outs.values())
    index = None
    if h.n * row_bytes > DUMP_LIMIT_BYTES:
        index = np.sort(np.random.RandomState(0).choice(h.n, DUMP_LIMIT_BYTES // row_bytes, replace=False))
        rows = torch.from_numpy(index).to(h.device)
        outs = {name: t[rows] for name, t in outs.items()}
    os.makedirs(out_dir, exist_ok=True)
    for name, t in outs.items():
        np.save(os.path.join(out_dir, name + '.npy'), t.cpu().numpy().astype(np.float32))
    if index is not None:
        np.save(os.path.join(out_dir, 'env_index.npy'), index.astype(np.float64))


def pcie_probe(dev, d2h_bytes, h2d_bytes, world, reps=60):
    """Plain cudaMemcpyAsync of one step's worth of bytes between pinned host memory and HBM, both directions at once
    (two streams), on every rank at the same time: the PCIe roofline of the host-buffer path at this N."""
    import torch
    import torch.distributed as dist
    dsrc = torch.empty(d2h_bytes, dtype=torch.uint8, device=dev)
    hdst = torch.empty(d2h_bytes, dtype=torch.uint8).pin_memory()
    hsrc = torch.empty(max(h2d_bytes, 1), dtype=torch.uint8).pin_memory()
    ddst = torch.empty(max(h2d_bytes, 1), dtype=torch.uint8, device=dev)
    s_out, s_in = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
    for _ in range(3):
        with torch.cuda.stream(s_out):
            hdst.copy_(dsrc, non_blocking=True)
    torch.cuda.synchronize(dev)
    if world > 1:
        dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.cuda.stream(s_out):
        e0.record(s_out)
    for _ in range(reps):
        with torch.cuda.stream(s_in):
            ddst.copy_(hsrc, non_blocking=True)
        with torch.cuda.stream(s_out):
            hdst.copy_(dsrc, non_blocking=True)
    with torch.cuda.stream(s_out):
        e1.record(s_out)
    torch.cuda.synchronize(dev)
    if world > 1:
        dist.barrier()
    ms = e0.elapsed_time(e1) / reps
    return {"d2h_gbs": d2h_bytes / (ms * 1e-3) / 1e9, "ms_per_step_bytes": ms}


E2E_PIPELINE_DEPTH = int(os.environ.get('NGW_E2E_DEPTH', '3'))   # measured 1 / 2 / 3 / 4 ahead: 5.31 / 5.72 / 5.69 / 5.72 x 10^8


def e2e_run(wl, n_steps, dev, world, host_acts):
    """ngw_step_host_begin/_end over the rotating batches as a software pipeline: batches i+1 .. i+depth are enqueued (H2D,
    launch, D2H, each on its handle's own stream) before the host waits for batch i, so the PCIe link never idles — with
    only one batch ahead the link waits for the host to wake up after every copy (0.92 of a plain copy instead of 0.99);
    every step copies its inputs in and its complete results out, and the results are read on the host."""
    import torch
    import torch.distributed as dist
    n_b, n_sets, kw = wl.n_batches, wl.n_sets, wl.kw
    for i in range(max(3, n_b)):                                        # every handle allocates its pinned buffers here
        wl.batches[i % n_b].step_host(host_acts[i % n_sets], **kw)
    torch.cuda.synchronize(dev)
    if world > 1:
        dist.barrier()
    checksum = 0.0

    def robust_total(stamps):
        # the loop is timed in chunks of E2E_CHUNK steps and reported as (median chunk) x (number of chunks), like `value`
        # (median region): a host hiccup in one chunk of a 25-50 ms measurement does not decide the figure
        chunks = np.diff(np.asarray(stamps))
        return float(np.median(chunks)) * len(chunks) * (n_steps / (len(chunks) * E2E_CHUNK)) if len(chunks) >= 3 \
            else float(stamps[-1] - stamps[0])

    depth = max(1, min(E2E_PIPELINE_DEPTH, n_b - 1))                    # batches enqueued ahead of the one being waited for
    stamps = [time.perf_counter()]
    for j in range(min(depth, n_steps)):
        wl.batches[j % n_b].step_host_begin(host_acts[j % n_sets], **kw)
    for i in range(n_steps):
        if i + depth < n_steps:
            wl.batches[(i + depth) % n_b].step_host_begin(host_acts[(i + depth) % n_sets], **kw)
        obs, rew, dn, cost, res = wl.batches[i % n_b].step_host_end()
        checksum += float(rew[0]) + float(obs[0, 0])                    # touch the results on the host
        if (i + 1) % E2E_CHUNK == 0:
            stamps.append(time.perf_counter())
    t_pipe = robust_total(stamps) if n_steps % E2E_CHUNK == 0 else time.perf_counter() - stamps[0]
    torch.cuda.synchronize(dev)
    if world > 1:
        dist.barrier()
    stamps = [time.perf_counter()]                                      # the plain blocking call, one batch at a time
    for i in range(n_steps):
        obs, rew, dn, cost, res = wl.batches[i % n_b].step_host(host_acts[i % n_sets], **kw)
        checksum += float(rew[0]) + float(obs[0, 0])
        if (i + 1) % E2E_CHUNK == 0:
            stamps.append(time.perf_counter())
    t_block = robust_total(stamps) if n_steps % E2E_CHUNK == 0 else time.perf_counter() - stamps[0]
    return t_pipe, t_block, checksum


def run_ours(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist

    numa = pin_to_gpu_numa(local_rank)                                  # before any pinned allocation
    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    if world > 1:
        # NCCL prints its version banner to stdout when the communicator is created (NCCL_DEBUG=VERSION is set in this
        # image); stdout must carry ONE JSON line, so fd 1 points at stderr while the communicator comes up
        sys.stdout.flush()
        saved_fd = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group('nccl', device_id=dev)
            warm = torch.zeros(1, device=dev)
            dist.all_reduce(warm)
            torch.cuda.synchronize(dev)
        finally:
            sys.stdout.flush()
            os.dup2(saved_fd, 1)
            os.close(saved_fd)

    def reduce_max(values):
        t = torch.tensor([float(v) for v in values], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)                     # device-timed durations: max over ranks
        return [float(x) for x in t.cpu().numpy()]

    W, K = max(args.warmup, 3), max(args.steps, 1)
    peak, peak_src = measured_hbm_peak()
    sampler = ClockSampler(local_rank)
    sampler.start()

    # ================= headline workload (C2 unless --workload says otherwise), int32 observation rows
    wl = Workload(args.workload, rank, world, dev)
    envs, n_batches, bytes_step = wl.envs, wl.n_batches, wl.bytes_step
    for i in range(W):                                                  # warm-up: eager launches
        wl.step(i)
    torch.cuda.synchronize(dev)
    regions, (t_wall0, t_wall1), launches_per_step, g_steps = time_regions(wl, K, dev, world, n_regions=1)
    if args.dump_outputs and rank == 0:
        dump_outputs(wl, args.dump_outputs)                             # before anything else steps these batches
    ms_region = float(np.median(regions))
    overlapped_per_graph = wl.overlapped_launches_per_graph
    ov_regions = time_regions(wl, K, dev, world, n_streams=min(3, n_batches))[0]
    ms_overlap = float(np.median(ov_regions))

    # ---- how much the rotation size matters (L2 keeps part of a small rotation): the same measurement with 7 and 32 batches
    l2_sens = {}
    if args.workload == 'C2' and not args.no_workloads:
        for nb in (7, 32):
            w2 = Workload('C2', rank, world, dev, n_batches=nb)
            for i in range(nb):
                w2.step(i)
            torch.cuda.synchronize(dev)
            reg2 = time_regions(w2, K, dev, world, floor_ms=20.0)[0]
            l2_sens[nb] = float(np.median(reg2)) / K
            w2.close()

    # ---- the same K-step graph with every launch waiting for its predecessor (NGW_NO_CONCURRENT): what the overlap buys
    ms_serial = 0.0
    if args.workload == 'C2' and not args.no_workloads:
        os.environ['NGW_NO_CONCURRENT'] = '1'
        try:
            w3 = Workload('C2', rank, world, dev, n_batches=n_batches)
        finally:
            del os.environ['NGW_NO_CONCURRENT']
        for i in range(n_batches):
            w3.step(i)
        torch.cuda.synchronize(dev)
        ms_serial = float(np.median(time_regions(w3, K, dev, world, floor_ms=20.0)[0]))
        w3.close()

    # ---- K-step rollout kernel (SURVEY §8f N1): 64 steps per launch, uniform random policy drawn on the device
    roll_T = 64
    for h in wl.batches:
        h.rollout(roll_T, None, policy_seed=1, **wl.kw)
    torch.cuda.synchronize(dev)
    r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n_roll = max(2 * n_batches, 8)
    r0.record()
    for i in range(n_roll):
        wl.batches[i % n_batches].rollout(roll_T, None, policy_seed=2 + i, **wl.kw)
    r1.record()
    torch.cuda.synchronize(dev)
    roll_ms = r0.elapsed_time(r1)
    # ---- closed-loop rollout: integer linear policy evaluated on the device from each step's observation
    roll_policy_ms = 0.0
    if wl.batches[0].obs_dim > 0 and wl.max_actions <= 16:
        gw = torch.Generator(device=dev)
        gw.manual_seed(7)
        w_pol = torch.randint(-9, 10, (wl.batches[0].obs_dim, wl.max_actions), generator=gw, device=dev, dtype=torch.int32)
        b_pol = torch.randint(-30, 31, (wl.max_actions,), generator=gw, device=dev, dtype=torch.int32)
        for h in wl.batches:
            h.rollout(roll_T, policy=(w_pol, b_pol), **wl.kw)
        torch.cuda.synchronize(dev)
        q0, q1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        q0.record()
        for i in range(n_roll):
            wl.batches[i % n_batches].rollout(roll_T, policy=(w_pol, b_pol), **wl.kw)
        q1.record()
        torch.cuda.synchronize(dev)
        roll_policy_ms = q0.elapsed_time(q1)
    # ---- general policy hook: one CUDA graph of 32 x [torch policy on the device observation -> ngw_step], one batch
    torch_policy_ms, tp_T = 0.0, 32
    if wl.batches[0].obs_dim > 0:
        gw = torch.Generator(device=dev)
        gw.manual_seed(11)
        w_f = torch.randn((wl.batches[0].obs_dim, wl.max_actions), generator=gw, device=dev)
        n_valid = torch.tensor([cc.c.n_actions for cc in wl.compiled], device=dev)[wl.batches[0].cfg_id.long()]
        d0 = wl.batches[0].obs_dim

        def torch_policy(obs):
            return torch.remainder(torch.argmax(obs[:, :d0].float() @ w_f, dim=1), n_valid).to(torch.int32)

        tp_graph, _ = wl.batches[0].capture_policy_rollout(torch_policy, tp_T, **wl.kw)
        tp_graph.replay()
        torch.cuda.synchronize(dev)
        t0_, t1_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0_.record()
        for _ in range(8):
            tp_graph.replay()
        t1_.record()
        torch.cuda.synchronize(dev)
        torch_policy_ms = t0_.elapsed_time(t1_) / 8
        del tp_graph
    # ---- eager (one python call per launch) figure, for the launch-bound picture
    n_eager = min(max(K, 200), 2000)
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(n_eager):
        wl.step(i)
    e1.record()
    torch.cuda.synchronize(dev)
    eager_ms = e0.elapsed_time(e1) / n_eager
    # ---- the same eager stepping through ngw_step_many: one library call per rotation of the batches (launches overlap)
    from gym_novel_gridworlds_b200.runtime import StepGroup
    group = StepGroup(wl.batches)
    rotation = [[wl.act_sets[(c * n_batches + i) % wl.n_sets] for i in range(n_batches)] for c in range(wl.n_sets)]
    for c in range(2):
        group.step(rotation[c % wl.n_sets], **wl.kw)
    n_calls = max(8, n_eager // n_batches)
    torch.cuda.synchronize(dev)
    m0, m1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    m0.record()
    for c in range(n_calls):
        group.step(rotation[c % wl.n_sets], **wl.kw)
    m1.record()
    torch.cuda.synchronize(dev)
    eager_many_ms = m0.elapsed_time(m1) / (n_calls * n_batches)
    stats = torch.zeros(8, dtype=torch.float64, device=dev)
    for h in wl.batches:
        stats += h.stats()
    host_acts = [a.cpu().numpy() for a in wl.act_sets]
    d_obs = wl.batches[0].obs_dim
    headline_flags = wl.reset_error_flags
    headline_compiled = wl.compiled

    # ================= end to end through the host-buffer C-ABI call, compact rows (and the int32 rows for comparison)
    n_e2e = max(K, E2E_MIN_STEPS) if envs <= 65536 else max(min(K, 40), 20)
    if n_e2e >= 3 * E2E_CHUNK:
        n_e2e -= n_e2e % E2E_CHUNK                                      # whole chunks
    n_e2e_i32 = max(n_e2e // 2, 20)
    t_e2e_i32, t_block_i32, _ = e2e_run(wl, n_e2e_i32, dev, world, host_acts)
    wl.close()
    wl8 = Workload(args.workload, rank, world, dev, obs_format='u8', n_batches=n_batches)
    row8 = wl8.batches[0].obs_row_bytes if d_obs else 0
    t_e2e, t_block, _ = e2e_run(wl8, n_e2e, dev, world, host_acts)
    d2h_u8, d2h_i32, h2d = (row8 + 10) * envs, (4 * d_obs + 10) * envs, 4 * envs
    probe = pcie_probe(dev, d2h_u8, h2d, world)
    wl8.close()

    # ================= the other BASELINE workloads at this N (skipped when a single workload was asked for)
    extra, extra_times = {}, []
    names = [] if (args.workload != 'C2' or args.no_workloads) else ['C3', 'C4', 'C5']
    K_x = min(K, 256)
    for name in names:
        w = Workload(name, rank, world, dev)
        for i in range(max(3, w.n_batches)):
            w.step(i)
        torch.cuda.synchronize(dev)
        reg, _, lps, _ = time_regions(w, K_x, dev, world)
        extra[name] = {"workload": w.desc, "scaling": w.scaling, "envs_per_gpu": w.envs, "total_envs": w.total_envs,
                       "batches_rotated": w.n_batches, "steps": K_x, "regions": len(reg),
                       "launches_per_step": lps, "algorithmic_bytes_per_env_step": w.bytes_step,
                       "overlapped_launches_per_graph": w.overlapped_launches_per_graph,
                       "reset_error_flags": w.reset_error_flags}
        extra_times.append(float(np.median(reg)))
        st = torch.zeros(8, dtype=torch.float64, device=dev)
        for h in w.batches:
            st += h.stats()
        if world > 1:
            dist.all_reduce(st, op=dist.ReduceOp.SUM)
        extra[name]["episode_stats"] = {"steps": float(st[0].item()), "episodes": float(st[1].item()),
                                        "resets": float(st[5].item())}
        w.close()
    t_timed_end = time.perf_counter()

    sampler.stop_flag = True
    sampler.join(timeout=1.0)
    clocks = sampler.summary(t_wall0, t_timed_end)

    if world > 1:
        dist.all_reduce(stats, op=dist.ReduceOp.SUM)                     # episode statistics over NCCL
    red = reduce_max([ms_region, ms_overlap, t_e2e, t_block, t_e2e_i32, t_block_i32, roll_ms, roll_policy_ms, eager_ms,
                      probe["ms_per_step_bytes"], torch_policy_ms, ms_serial, eager_many_ms] + extra_times)
    (ms_region, ms_overlap, t_e2e, t_block, t_e2e_i32, t_block_i32, roll_ms, roll_policy_ms, eager_ms, probe_ms,
     torch_policy_ms, ms_serial, eager_many_ms) = red[:13]
    extra_times = red[13:]

    if rank == 0:
        ms_per_step = ms_region / K
        total_envs = wl.total_envs if wl.scaling == 'strong' else world * envs
        value = total_envs * K / (ms_region * 1e-3)
        achieved = envs * bytes_step / (ms_per_step * 1e-3) / 1e9
        ov_achieved = envs * bytes_step / (ms_overlap / K * 1e-3) / 1e9
        traffic, traffic_src = measured_traffic(args.workload)
        # two ways to call the host-buffer API: pipelined over the batches (_begin/_end) or one blocking call per step.
        # On one GPU the pipeline wins (the link never idles); with 8 ranks sharing the host's PCIe / memory system the
        # blocking call does (fewer copies in flight).  A caller picks the faster one; both are in the line.
        e2e_pipe, e2e_block = total_envs * n_e2e / t_e2e, total_envs * n_e2e / t_block
        e2e_value = max(e2e_pipe, e2e_block)
        pcie_gbs = d2h_u8 / (probe_ms * 1e-3) / 1e9
        pcie_limit = world * envs / (probe_ms * 1e-3)
        for name, ms in zip(names, extra_times):
            x = extra[name]
            x["us_per_step"] = ms / K_x * 1e3
            x["value"] = x["total_envs"] * K_x / (ms * 1e-3)
            x["unit"] = "env-steps/s"
            x["achieved_gbs_per_gpu"] = x["envs_per_gpu"] * x["algorithmic_bytes_per_env_step"] / (ms / K_x * 1e-3) / 1e9
            x["frac_of_hbm_peak"] = x["achieved_gbs_per_gpu"] / peak
        cfg = c2_config(world) if args.workload == 'C2' else {"workload": wl.desc, "envs_per_batch": envs,
                                                                "batches_rotated": n_batches}
        line = {
            "metric": METRIC, "value": value, "unit": "env-steps/s", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": wl.scaling, "vs_baseline": None,
            "dtype": "int32", "data": "synthetic", "config": cfg,
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": "env-steps/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h_u8,
                    "steps": n_e2e, "timing": "wall clock over the whole loop in chunks of %d steps, median chunk x chunks" % E2E_CHUNK, "obs_format": "NGW_OBS_U8 (uint8 lidar ranges + int32 inventory tail, %d B/env)" % row8,
                    "api": "ngw_step_host (blocking) / ngw_step_host_begin+_end (batches i+1..i+%d enqueued before waiting for "
                           "batch i), pinned host buffers: H2D actions, one launch, one D2H of obs|reward|step_cost|done|result "
                           "per step" % E2E_PIPELINE_DEPTH,
                    "mode": "pipelined" if e2e_pipe >= e2e_block else "blocking",
                    "pipelined_value": e2e_pipe, "blocking_value": e2e_block,
                    "achieved_d2h_gbs_total": e2e_value * (row8 + 10) / 1e9,
                    "pcie": {"d2h_gbs_per_gpu": pcie_gbs, "d2h_gbs_total": pcie_gbs * world,
                             "limit_env_steps_per_s": pcie_limit, "frac": e2e_value / pcie_limit,
                             "note": "probe = plain cudaMemcpyAsync of one step's bytes, both directions at once, on every "
                                     "rank at the same time; the host side of this box delivers that much in aggregate"},
                    "int32_rows": {"value": total_envs * n_e2e_i32 / t_e2e_i32, "d2h_bytes_per_step": d2h_i32,
                                   "blocking_value": total_envs * n_e2e_i32 / t_block_i32, "steps": n_e2e_i32},
                    "numa": numa},
            "gpu_launches": int(round(launches_per_step * K)),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "traffic_source": traffic_src, "kernel": "ngw::step1w_kernel",
                         "launch_overlap": {
                             "overlapped_launches_per_graph": overlapped_per_graph, "launches_per_graph": g_steps,
                             "note": "consecutive launches of the K-step graph step DIFFERENT batches (rotation) and share no "
                                     "buffer; inside a stream capture the library proves they are adjacent and lets the "
                                     "second start while the first computes (one gate warp per CTA keeps stream order); "
                                     "avg_launch_us = region / K, i.e. the launch-to-launch interval",
                             "serialized": None if not ms_serial else {
                                 "note": "same graph with NGW_NO_CONCURRENT=1 (every launch waits for its predecessor)",
                                 "us_per_step": ms_serial / K * 1e3,
                                 "frac": envs * bytes_step / (ms_serial / K * 1e-3) / 1e9 / peak}},
                         "peak_source": peak_src, "algorithmic_bytes_per_env_step": bytes_step,
                         "algorithmic_bytes_per_launch": envs * bytes_step, "avg_launch_us": ms_per_step * 1e3,
                         "l2_sensitivity": {"%d_batches_%.0f_MB" % (nb, nb * envs * bytes_step / 1e6):
                                            {"us_per_step": ms * 1e3, "frac": envs * bytes_step / (ms * 1e-3) / 1e9 / peak}
                                            for nb, ms in sorted(l2_sens.items())}},
            "timing": {"regions": len(regions),
                       "region_ms_min_med_max": [min(regions), float(np.median(regions)), max(regions)],
                       "timed_ms_total": float(sum(regions)), "graph_steps": g_steps,
                       "launch": "one stream, CUDA-graph replay (one kernel launch per step; launches of different batches overlap)",
                       "reset_error_flags": headline_flags, "per_gpu_envs_resident": n_batches * envs},
            "overlapped": {"note": "same K steps, independent batches on %d parallel graph branches (launches overlap)"
                                   % min(3, n_batches), "value": total_envs * K / (ms_overlap * 1e-3), "unit": "env-steps/s",
                           "us_per_step": ms_overlap / K * 1e3, "achieved_gbs": ov_achieved,
                           "frac_of_hbm_peak": ov_achieved / peak},
            "rollout": {"note": "ngw_rollout: %d steps per launch, on-device uniform random policy, tile resident in "
                                "shared memory; outputs are per-env sums + final observation" % roll_T,
                        "value": total_envs * roll_T * n_roll / (roll_ms * 1e-3), "unit": "env-steps/s"},
            "rollout_policy": None if not roll_policy_ms else {
                "note": "ngw_rollout_policy: %d steps per launch, action = argmax(b + obs @ W) on the device from each "
                        "step's lidar observation" % roll_T,
                "value": total_envs * roll_T * n_roll / (roll_policy_ms * 1e-3), "unit": "env-steps/s"},
            "torch_policy_graph": None if not torch_policy_ms else {
                "note": "BatchHandle.capture_policy_rollout: ONE CUDA graph of %d x [torch policy (float matmul + argmax on the "
                        "device observation) -> ngw_step] on one batch: the closed loop with a general policy, host out of "
                        "the loop" % tp_T,
                "value": total_envs * tp_T / (torch_policy_ms * 1e-3), "unit": "env-steps/s",
                "us_per_step": torch_policy_ms / tp_T * 1e3},
            "eager": {"value": total_envs / (eager_ms * 1e-3), "unit": "env-steps/s", "us_per_step": eager_ms * 1e3,
                      "note": "no CUDA graph: one python -> ctypes -> ngw_step call per launch (bound by the host)"},
            "eager_many": {"value": total_envs / (eager_many_ms * 1e-3), "unit": "env-steps/s",
                           "us_per_step": eager_many_ms * 1e3,
                           "note": "no CUDA graph: one ngw_step_many call per rotation of the %d batches; the library issues "
                                   "the launches back to back and overlaps them" % n_batches},
            "workloads": extra,
            "episode_stats": dict(zip(('steps', 'episodes', 'successes', 'reward_sum', 'cost_sum', 'resets',
                                       'invalid'), [float(x) for x in stats.cpu().numpy()[:7]])),
            "wall_ms_timed_region": (t_wall1 - t_wall0) * 1e3,
        }
        if world == 1 and not args.no_cpu_baseline and args.workload == 'C2':
            threads = os.cpu_count() or 1
            reg = cpu_port_regions(headline_compiled[0], ENVS_PER_BATCH, 64, 16, threads, 3.0)
            dt = float(np.median(reg))
            line["cpu_baseline"] = {
                "value": 64 * ENVS_PER_BATCH / dt, "unit": "env-steps/s", "cores": threads, "kind": "port",
                "sample": "%d regions of 64 steps x %d envs (%.1f s wall, ~%.0f s of CPU work, median region), C port of "
                          "the reference path (oracle/ngw_oracle.c), %d threads, no per-step barrier"
                          % (len(reg), ENVS_PER_BATCH, sum(reg), sum(reg) * threads, threads),
                "python_reference": python_reference_baseline()}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=4096)
    ap.add_argument('--warmup', type=int, default=64)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-workloads', action='store_true', help='skip the C3/C4/C5 measurements of the default line')
    ap.add_argument('--workload', default='C2', choices=['C2', 'C3', 'C4', 'C4-blocked', 'C5'])
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='write the outputs of the last timed step as DIR/<name>.npy (float32, at most 64 MB)')
    args = ap.parse_args()
    if args.dump_outputs and args.impl == 'reference':
        ap.error('--dump-outputs writes the outputs of the GPU path (--impl ours)')
    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    if args.impl == 'reference':
        run_reference(args, rank, world)
        return
    run_ours(args, rank, world, local_rank)


if __name__ == '__main__':
    main()
