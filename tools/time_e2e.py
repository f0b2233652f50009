"""End-to-end step time through tb_step_host (pinned host buffers in and out) for the two transports.
usage: time_e2e.py [n_envs] [env] [mode,mode,...]"""
import os, sys, time
import numpy as np
import torch
sys.path.insert(0, ".")
from tennisbot_rl_b200.batch import TennisBatch
n = int(sys.argv[1]) if len(sys.argv) > 1 else 1 << 20
env = sys.argv[2] if len(sys.argv) > 2 else "SwingRacket-v0"
modes = sys.argv[3].split(",") if len(sys.argv) > 3 else ("zero_copy", "staging")
for mode in modes:
    os.environ["TB_HOST_MODE"] = mode
    b = TennisBatch(env, n, seed=0)
    b.reset_host()
    hb = b.host_buffers()
    np.copyto(hb["actions"], np.random.default_rng(0).uniform(-1, 1, hb["actions"].shape).astype(np.float32))
    for _ in range(26): b.step_host(want_terminal=False, want_events=False)
    torch.cuda.synchronize(); t0 = time.perf_counter()
    for _ in range(52): b.step_host(want_terminal=False, want_events=False)
    dt = (time.perf_counter() - t0) / 52
    t1 = time.perf_counter()
    for _ in range(26): b.step_host(want_terminal=True, want_events=True)
    dt2 = (time.perf_counter() - t1) / 26
    print("%-10s %s n=%d: %.3f ms/step -> %.3e env-steps/s (with terminal obs + events: %.3f ms)" % (mode, env, n, dt * 1e3, n / dt, dt2 * 1e3), flush=True)
    b.close()
