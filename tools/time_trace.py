"""Kernel time of tb_trace_step (trace_kernel) on SwingRacket-v0's 26th env step, the one that fast-forwards the ball's
flight, from CUDA events over repeated launches after a warm-up.

  python tools/time_trace.py [--reps 20] [--precision f64]

For M = 16, 1 024 and 16 384 envs, the records before the 26th step come from an episode of the saved PPO policy
(tests/golden/ppo_swing_policy.npz, deterministic) and of uniform random actions.  Printed per case: ms per launch, traced
substeps per second (the sum of `substeps` over the envs, divided by the time) and the largest `substeps`.  Every launch
writes the full [776, M, 32] float64 block (0.2 MB per env), padding included."""
import argparse
import subprocess
import sys
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
from tennisbot_rl_b200 import _lib  # noqa: E402
from tennisbot_rl_b200.batch import TennisBatch  # noqa: E402
from tennisbot_rl_b200.ppo import load_sb3_policy_npz  # noqa: E402

GOLDEN = Path(__file__).resolve().parent.parent / "tests" / "golden" / "ppo_swing_policy.npz"
SIZES = (16, 1024, 16384)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[torch.cuda.current_device()] if q else torch.cuda.get_device_name()


def before_the_flight(m, source, precision):
    """(batch, records before the 26th step, the actions that step takes)."""
    b = TennisBatch("SwingRacket-v0", m, seed=1, precision=precision, auto_reset=False)
    obs = torch.zeros((1, m, 6), device=b.device)
    obs[0].copy_(b.reset())
    g = torch.Generator(b.device).manual_seed(1)
    if source == "policy":
        b.set_policy(load_sb3_policy_npz(GOLDEN).to(b.device))
        rew, done = torch.zeros((1, m), device=b.device), torch.zeros((1, m), dtype=torch.uint8, device=b.device)
        last, act = torch.zeros((m, 6), device=b.device), torch.zeros((1, m, 6), device=b.device)
    for _ in range(26):
        states = b.get_state()
        if source == "policy":
            b.policy_rollout(obs, rew, done, last, actions=act, deterministic=True)
            obs[0].copy_(last)
            taken = act[0].clamp(-1, 1).contiguous()
        else:
            taken = torch.empty((m, 6), device=b.device).uniform_(-1, 1, generator=g)
            b.step(taken)
    return b, states, taken


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--precision", default="f64")
    a = ap.parse_args()
    print("card (name, power limit, max SM clock):", card(), flush=True)
    S = _lib.TRACE_MAX_SUBSTEPS
    for m in SIZES:
        for source in ("policy", "random"):
            b, states, taken = before_the_flight(m, source, a.precision)
            trace = torch.empty((S, m, _lib.STATE_WORDS), dtype=torch.float64, device=b.device)
            bits = torch.empty((S, m), dtype=torch.uint8, device=b.device)
            sub = torch.empty(m, dtype=torch.int32, device=b.device)
            stream = b._stream()

            def call():
                _lib.check(b.lib.tb_trace_step(b.h, states.data_ptr(), taken.data_ptr(), m, S, trace.data_ptr(), bits.data_ptr(),
                                               sub.data_ptr(), None, None, None, stream))

            for _ in range(3):
                call()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            for _ in range(a.reps):
                call()
            e1.record()
            torch.cuda.synchronize()
            s = e0.elapsed_time(e1) / a.reps * 1e-3
            total, longest = int(sub.sum()), int(sub.max())
            print(f"SwingRacket-v0 {a.precision} M={m:6d} {source:>6s}: {s * 1e3:8.3f} ms per launch, {total / s:.3e} substeps/s, "
                  f"{total / m:.1f} substeps per env on average, largest {longest}; "
                  f"{trace.numel() * 8 / 1e9:.2f} GB written per launch", flush=True)
            b.close()
            del trace, bits, sub, states, taken
            torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
