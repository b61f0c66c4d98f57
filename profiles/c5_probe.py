import os, sys, time
import numpy as np, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench
from gym_novel_gridworlds_b200.runtime import BatchHandle
desc, compiled, envs, rule, kw = bench.build_workload('C5')
hs = []
for b in range(2):
    h = BatchHandle(compiled, envs, seed=0, first_env_gid=b*envs); h.reset(); hs.append(h)
acts = [torch.randint(0, 10, (envs,), device='cuda', dtype=torch.int32) for _ in range(4)]
def run(kw, n=60):
    for i in range(6): hs[i%2].step(acts[i%4], **kw)
    torch.cuda.synchronize(); e0=torch.cuda.Event(enable_timing=True); e1=torch.cuda.Event(enable_timing=True); e0.record()
    for i in range(n): hs[i%2].step(acts[i%4], **kw)
    e1.record(); torch.cuda.synchronize(); return e0.elapsed_time(e1)/n*1e3
print('no reset us/step', run({}), ' with staggered reset', end=' ')
for h in hs: h.ep_len.copy_(torch.randint(0,256,(envs,),device='cuda',dtype=torch.int32))
print(run(dict(auto_reset=True, max_episode_steps=256)))
# time of a full reset of the batch
torch.cuda.synchronize(); t0=time.perf_counter(); hs[0].reset(want_obs=False); torch.cuda.synchronize(); print('full reset of %d envs: %.2f ms' % (envs, (time.perf_counter()-t0)*1e3))
