import os, time, cProfile, pstats, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from examples.random_action import build
env = build(65536); env.reset()
a = torch.zeros(65536, dtype=torch.int32, device='cuda')
for _ in range(50): env.step(a)
torch.cuda.synchronize()
t0 = time.perf_counter()
for _ in range(2000): env.step(a)
torch.cuda.synchronize(); dt = time.perf_counter() - t0
print('env.step: %.1f us/step' % (dt / 2000 * 1e6))
h = env.unwrapped._runtime.handle
t0 = time.perf_counter()
for _ in range(2000): h.step(a)
torch.cuda.synchronize(); dt = time.perf_counter() - t0
print('handle.step: %.1f us/step' % (dt / 2000 * 1e6))
pr = cProfile.Profile(); pr.enable()
for _ in range(2000): env.step(a)
pr.disable(); torch.cuda.synchronize()
pstats.Stats(pr).sort_stats('cumulative').print_stats(12)
