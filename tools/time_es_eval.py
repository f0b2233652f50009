"""Time of one ES generation through EsEvaluator (in-kernel rollout) and through batched_fitness_static (the torch adapter) on
the same population, over a sweep of population sizes with 10 repeats, and where the evaluator's device time goes.

For each size: the wall time of one generation (host clock around calls that end in a device synchronise, median of `reps`
after one warm-up generation), its env-steps/s (envs x env steps run), and, from a separate torch.profiler run of one
evaluator generation, the device time of es_kernel, of the env step (step_kernel + ff_kernel) and of the rest (the weight
transpose, reset and begin kernels).  The card's name and power limit are read in the same run.
SwingRacket-v0 runs the saved ES policy with antithetic perturbations; Tennisbot-v0 random weights (scale 0.3).
usage: time_es_eval.py ENV [individuals ...]      (default individuals: 1639 6554 26215, i.e. up to 262 150 envs)"""
import json
import statistics
import subprocess
import sys
import time
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
from tennisbot_rl_b200 import es_eval  # noqa: E402
from tennisbot_rl_b200.batch import TennisBatch  # noqa: E402

REPEATS = 10


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[torch.cuda.current_device()] if q else torch.cuda.get_device_name()


def population(env_id, individuals):
    rng = np.random.default_rng(0)
    if env_id == "SwingRacket-v0":
        saved = np.load(ROOT / "tests" / "golden" / "es_swing_weights.npz")["weights"].astype(np.float32)
        eps = rng.standard_normal(((individuals + 1) // 2, saved.size)).astype(np.float32)
        return np.concatenate([saved + 0.05 * eps, saved - 0.05 * eps])[:individuals]
    return (0.3 * rng.standard_normal((individuals, 858))).astype(np.float32)


def timed(fn, reps):
    out = []
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        out.append(time.perf_counter() - t0)
    return statistics.median(out)


class StepCounter:
    """Counts TennisBatch.step calls: the env steps batched_fitness_static runs before its envs are all done."""

    def __enter__(self):
        self.calls, self._orig = 0, TennisBatch.step

        def step(b, *a, **k):
            self.calls += 1
            return self._orig(b, *a, **k)

        TennisBatch.step = step
        return self

    def __exit__(self, *exc):
        TennisBatch.step = self._orig


def split(ev, w, state):
    """(es_kernel ms, env-step ms, other ms) of one generation, from torch.profiler's kernel records."""
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        ev.evaluate(w, state)
        torch.cuda.synchronize()
    es = env = other = 0.0
    for e in prof.key_averages():
        us = getattr(e, "device_time_total", None)
        us = e.cuda_time_total if us is None else us
        if us <= 0:
            continue
        if "es_kernel" in e.key:
            es += us
        elif "step_kernel" in e.key or "ff_kernel" in e.key:
            env += us
        else:
            other += us
    return es / 1e3, env / 1e3, other / 1e3


def main():
    env_id = sys.argv[1] if len(sys.argv) > 1 else "SwingRacket-v0"
    sizes = [int(x) for x in sys.argv[2:]] or [1639, 6554, 26215]
    print("card (name, power limit, max SM clock):", card(), flush=True)
    od = TennisBatch(env_id, 1).obs_dim
    m = np.random.default_rng(1)
    state = (np.full(od, 50.0), m.normal(0, 0.5, od), np.full(od, 50.0), np.ones(od))
    rows = []
    for individuals in sizes:
        n = individuals * REPEATS
        w = torch.from_numpy(population(env_id, individuals)).cuda()
        ev = es_eval.EsEvaluator(env_id, individuals, REPEATS, seed=0)
        ev.evaluate(w, state)  # warm-up
        t_ev = timed(lambda: ev.evaluate(w, state), 5)
        steps_ev = ev.steps_run
        es_ms, env_ms, other_ms = split(ev, w, state)
        reps_t = 3 if env_id == "SwingRacket-v0" else 1
        es_eval.batched_fitness_static(w, env_id, repeats=REPEATS, normalizer_state=state, seed=0)  # warm-up
        with StepCounter() as sc:
            t_t = timed(lambda: es_eval.batched_fitness_static(w, env_id, repeats=REPEATS, normalizer_state=state, seed=0), reps_t)
        steps_t = sc.calls // reps_t
        row = dict(env=env_id, envs=n, individuals=individuals, repeats=REPEATS,
                   evaluator=dict(ms=round(t_ev * 1e3, 3), steps=steps_ev, env_steps_per_s=n * steps_ev / t_ev,
                                  es_kernel_ms=round(es_ms, 3), env_step_ms=round(env_ms, 3), other_ms=round(other_ms, 3)),
                   torch_adapter=dict(ms=round(t_t * 1e3, 3), steps=steps_t, env_steps_per_s=n * steps_t / t_t),
                   speedup=round(t_t / t_ev, 2))
        rows.append(row)
        print(json.dumps(row), flush=True)
        ev.close()
        del w
        torch.cuda.empty_cache()
    return rows


if __name__ == "__main__":
    main()
