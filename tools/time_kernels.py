"""Per-step device times of step_kernel and ff_kernel over one lock-step SwingRacket episode (events inside the library).
usage: time_kernels.py precision n_envs"""
import sys
import os
import torch
RING = int(os.environ.get("TB_RING", 32))  # pre-drawn action batches the steps cycle through (>= 26: i.i.d. within an episode)
sys.path.insert(0, ".")
from tennisbot_rl_b200.batch import TennisBatch
prec = sys.argv[1]; n = int(sys.argv[2])
torch.manual_seed(0)  # the same action ring in every process: variants are compared on identical work
b = TennisBatch("SwingRacket-v0", n, precision=prec, seed=0)
b.reset()
acts = [torch.empty((n, b.act_dim), device="cuda").uniform_(-1, 1) for _ in range(RING)]
for t in range(26): b.step(acts[t % RING])
torch.cuda.synchronize()
b.set_kernel_timing(True)
rows = []
for t in range(26):
    b.step(acts[t % RING])
    rows.append(b.kernel_timing())
for t, r in enumerate(rows):
    if t % 26 >= 23 or t % 26 in (0, 12): print(t, "step_kernel %.4f ms ff_kernel %.4f ms" % (r[0], r[1]))
d = b.ff_diagnostics()
print("ff diagnostics: ran %d, visits to the server path %d, flights over after %d ns, fault %d" % (d[0], d[1], d[2], d[15]))
