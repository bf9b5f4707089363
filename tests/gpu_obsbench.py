"""Times k_obs2 alone (observe_only) and the step kernel alone for the 2v2 workload."""
import torch
import parity
from parity import make_config
from masurvival import _lib
rec = make_config('2v2', auto_reset=True)
N = 16384
h = _lib.Handle(rec, N, 0, 1, 0); h.reset()
torch.manual_seed(1234)
acts = torch.randint(0, 2, (8, N, 4, 6), dtype=torch.uint8, device='cuda')
acts[..., 0:3] = torch.randint(0, 3, (8, N, 4, 3), dtype=torch.uint8, device='cuda')
for t in range(200): h.step(acts[t % 8].data_ptr())
torch.cuda.synchronize()
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record()
for t in range(200): h.observe_only()
e1.record(); torch.cuda.synchronize()
print('k_obs2 %.1f us' % (e0.elapsed_time(e1) / 200 * 1e3))
e0.record()
for t in range(200): h.step_kernel_only(acts[t % 8].data_ptr())
e1.record(); torch.cuda.synchronize()
print('k_step %.1f us' % (e0.elapsed_time(e1) / 200 * 1e3))
