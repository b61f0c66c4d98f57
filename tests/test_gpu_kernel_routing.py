"""Which one-step kernel the library launches for a given input (run on the B200 box: pytest -m gpu).  The launch code
picks the kernel and its CTA shape from the map size, the lidar geometry, the configs of the batch and the batch size
alone; each case records one step with torch.profiler and checks the kernel's template name and block size, so that
the parity tests of every shape (test_gpu_parity.py) are known to run the shape they are meant for."""
import json

import numpy as np
import pytest
import torch

import scenarios
from gym_novel_gridworlds_b200.runtime import BatchHandle
from test_gpu_parity import C2_DESC, TILE_GROUP_SHAPES, WARP_PER_TILE_BATCHES, _compiled, tile_group_inputs

pytestmark = pytest.mark.gpu


def _step_kernel(compiled, n, cfg_id, tmp_path):
    """(demangled name, threads per block) of the step kernel that one ngw_step launch of this batch runs."""
    h = BatchHandle(compiled, n, seed=1, cfg_id=None if cfg_id is None else cfg_id.astype(np.int32))
    h.reset()
    a = torch.zeros(n, dtype=torch.int32, device='cuda')
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        h.step(a)
        torch.cuda.synchronize()
    trace = str(tmp_path / 'step.json')
    prof.export_chrome_trace(trace)
    with open(trace) as f:
        events = json.load(f)['traceEvents']
    steps = [(e['name'], e['args']['block'][0]) for e in events if e.get('cat') == 'kernel' and 'step1' in e['name']]
    h.close()
    assert len(steps) == 1, steps
    return steps[0]


# case -> (kernel, threads per block = 32 x warps per tile x tiles per CTA, + 1 gate warp for step1w_kernel)
ROUTES = {
    'G4-alias': ('step1_kernel<1, true, true>', 32 * 4),
    'G4-multi': ('step1_kernel<1, false, false>', 32 * 4 * 2),
    'G2-multi': ('step1_kernel<1, false, false>', 32 * 2 * 2),
    'G2-waves': ('step1_kernel<1, true, false>', 32 * 2),
    'G1-mixed': ('step1_kernel<4, true, false>', 32),
    'generic-40': ('step1_kernel<1, true, false>', 32 * 4),
    'warp-1': ('step1w_kernel<1, 8>', 32 * (1 + 1)),
    'warp-3': ('step1w_kernel<1, 8>', 32 * (3 + 1)),
    'warp-waves': ('step1w_kernel<1, 8>', 32 * (8 + 1)),
}


def _inputs(case):
    if case in TILE_GROUP_SHAPES:
        return tile_group_inputs(case)
    if case == 'generic-40':                         # test_map_sizes_and_beam_counts_vs_oracle(40, 5, 70)
        return [_compiled({'env': scenarios.BOW, 'map_size': 40, 'chain': [['lidar', 5]]})], 70, None
    n = WARP_PER_TILE_BATCHES[['warp-1', 'warp-3', 'warp-waves'].index(case)]
    return [_compiled(C2_DESC)], n, None


@pytest.mark.parametrize('case', sorted(ROUTES))
def test_input_selects_the_kernel_shape(case, tmp_path):
    name, threads = _step_kernel(*_inputs(case), tmp_path)
    kernel, want_threads = ROUTES[case]
    assert kernel + '(' in name and threads == want_threads, (name, threads)
