#!/usr/bin/env python3
"""bench.py - env-steps/s of the SwingRacket-v0 step path on B200 (BASELINE.json metric), one JSON line.

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...   # CPU arm (restated oracle; PyBullet is not in the image)
    torchrun --nproc-per-node N bench.py --gpus N ...         # one rank per GPU, weak scaling
    python bench.py ... --dump-outputs DIR                    # also write the last timed step's outputs (two builds compare)

A "step" is one pass of the hot path over the batch: one agent-visible env step for every env of the batch
(SwingRacket's 26th step, which fast-forwards up to 776 physics substeps, counts once).  Workload = config 5's
per-GPU slice: 1 048 576 SwingRacket-v0 envs per GPU, uniform random actions, initial states from the env's own
reset ranges.  Every SwingRacket episode is exactly 26 agent steps (25 one-substep control steps + the fast-forward
step), so the timed region must cover whole episodes to weight the two kinds of step correctly:
Episodes run in lock step (all envs reset together, as a VecEnv starts).  With --steps a multiple of 26 (default
1040 = 40 episodes, ~0.4 s) the timed region spans K/26 whole episodes.  For any other K the region is placed so
that it ENDS right after a fast-forward step and therefore contains ceil(K/26) of them: the expensive step is then
weighted at least as heavily as in whole episodes and the number can only come out pessimistic.  The NCCL all-reduce
of the episode statistics follows every fast-forward step of the timed region, so any K contains ceil(K/26) reductions.
`--stagger on` instead offsets the episode phases per 128-env group (g mod 26) so that every launch carries the same
25:1 mix (slower: each launch then waits for its own 800-substep time-out flights).

Actions: a ring of 32 pre-drawn U(-1,1) batches in HBM, i.e. i.i.d. within every 26-step episode (SURVEY 8(d)).
`extras` (N = 1 only): the other BASELINE.json configs measured in the same process - Tennisbot-v0 at 65 536 envs with a
scripted ball-tracking policy (config 3 with racket-ball contact), the TennisVecEnv host loop at 16 384 envs (config 4's
env side), the fused tb_rollout at K = 26 and the policy rollout the PPO trainer uses.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

METRIC = "env-steps/sec SwingRacket-v0"
UNIT = "env-steps/s"
ALGO_BYTES = {  # SURVEY.md 8(d): action + obs + reward + done + state read + state written, per env step
    ("SwingRacket-v0", "f32"): 24 + 24 + 4 + 1 + 128 + 128,
    ("SwingRacket-v0", "f64"): 24 + 24 + 4 + 1 + 256 + 256,
    ("Tennisbot-v0", "f32"): 8 + 48 + 4 + 1 + 128 + 128,
    ("Tennisbot-v0", "f64"): 8 + 48 + 4 + 1 + 256 + 256,
}
MOVED_BYTES = {  # what a control step actually moves per env (profiles/r2_traffic.json): packs 0-3 + 7 each way, I/O
    ("SwingRacket-v0", "f64"): 160 + 160 + 53, ("SwingRacket-v0", "f32"): 80 + 80 + 53,
    ("Tennisbot-v0", "f64"): 224 + 224 + 61, ("Tennisbot-v0", "f32"): 112 + 112 + 61,
}
ALGO_BYTES_F32_STATE = {"SwingRacket-v0": 24 + 24 + 4 + 1 + 128 + 128, "Tennisbot-v0": 8 + 48 + 4 + 1 + 128 + 128}  # BASELINE.md's yardstick
EPISODE_STEPS = 26
GROUP = 128
RING = 32  # pre-drawn action batches: >= 26, so the actions of an episode are i.i.d. (a ring of 4 repeats every 4 steps and
           # drives the racket in one direction: many more racket-ball contacts than action_space.sample() gives)
DUMP_LIMIT = 64 * 10**6  # bytes of all files --dump-outputs writes; beyond it a seeded sample of envs is written


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=1040)
    ap.add_argument("--warmup", type=int, default=26)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--env", default="SwingRacket-v0", choices=["SwingRacket-v0", "Tennisbot-v0"])
    ap.add_argument("--envs-per-gpu", type=int, default=1 << 20)
    ap.add_argument("--precision", default="f64", choices=["f32", "f64"])
    ap.add_argument("--e2e-steps", type=int, default=26)
    ap.add_argument("--cpu-sample-envs", type=int, default=65536)
    ap.add_argument("--stagger", default="off", choices=["on", "off"],
                    help="episode phases: off = lock-step (all envs reset together), on = staggered per 128-env group")
    ap.add_argument("--skip-cpu-baseline", action="store_true")
    ap.add_argument("--extras", default="auto", choices=["auto", "on", "off"],
                    help="measure the other BASELINE configs too (auto: at N = 1)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last of them returned (rank 0's envs) as DIR/<name>.npy, "
                         "at most 64 MB: obs, reward, done, terminal_obs, events, one row per env")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    return args


# ---------------------------------------------------------------------------------------------- helpers
class ClockSampler:
    """SM clock, throttle reasons and power while the timed region runs (B200_PROFILING.md's clocks line).  NVML from a
    polling thread (a row per millisecond: the driver's 20-step window lasts under 4 ms) plus one row taken by the launching
    thread itself once the whole window is queued and the device is still working through it (sample_now), so that a window of
    any length holds a sample; without the NVML
    bindings, one long-running `nvidia-smi -lms 50` whose rows between start() and stop() are kept."""

    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap,power.draw")
    REASONS = (("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20), ("sw_power_cap", 0x4))

    def __init__(self, index, uuid=None):
        self.rows, self.proc, self.thread, self.nvml, self.handle = [], None, None, None, None
        self.keep, self.quit, self.source = False, False, None
        try:
            import pynvml

            pynvml.nvmlInit()
            try:
                self.handle = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + str(uuid)) if uuid and not str(uuid).startswith("GPU-") else str(uuid))
            except Exception:
                self.handle = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.nvml = pynvml
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM)
            self._nvml_row()  # (fails here, not in the timed region, if a query is unsupported)
            self.rows.clear()
            self.source = "nvml"
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            return
        self.source = "nvidia-smi"
        self.thread = threading.Thread(target=self._pump, daemon=True)
        self.thread.start()

    def _nvml_row(self):
        n, h = self.nvml, self.handle
        sm = n.nvmlDeviceGetClockInfo(h, n.NVML_CLOCK_SM)
        try:
            bits = n.nvmlDeviceGetCurrentClocksEventReasons(h)
        except Exception:
            bits = n.nvmlDeviceGetCurrentClocksThrottleReasons(h)
        try:
            watts = n.nvmlDeviceGetPowerUsage(h) / 1000.0
        except Exception:
            watts = None
        self.rows.append((sm, self.max_mhz, bits, watts))

    def _poll(self):
        while not self.quit:
            if self.keep:
                try:
                    self._nvml_row()
                except Exception:
                    pass
            time.sleep(0.001)

    def _pump(self):
        for line in self.proc.stdout:
            if self.keep:
                parts = [p.strip() for p in line.strip().split(",")]
                if len(parts) >= 7:
                    bits = sum(bit for (_, bit), v in zip(self.REASONS, parts[2:6]) if v.lower().startswith("active"))
                    if parts[0].isdigit():
                        self.rows.append((int(parts[0]), int(parts[1]) if parts[1].isdigit() else None, bits,
                                          float(parts[6]) if parts[6].replace(".", "", 1).isdigit() else None))

    def start(self):
        if self.source == "nvidia-smi":
            time.sleep(0.15)  # let nvidia-smi reach its sampling loop
        self.keep = True

    def sample_now(self):
        """one row from the calling thread"""
        if self.nvml is not None and self.keep:
            try:
                self._nvml_row()
            except Exception:
                pass

    def stop(self):
        self.keep = False
        self.quit = True
        if self.proc is not None:
            self.proc.terminate()
        rows = list(self.rows)
        sm = sorted(r[0] for r in rows)
        bits = 0
        for r in rows:
            bits |= r[2]
        watts = [r[3] for r in rows if r[3] is not None]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": rows[0][1] if rows else None,
                "reasons": sorted(name for name, bit in self.REASONS if bits & bit), "samples": len(rows),
                "power_w_max": max(watts) if watts else None, "source": self.source}


def measured_traffic(env, precision, n):
    """DRAM bytes of one env step of the whole batch (dram__bytes_read.sum + dram__bytes_write.sum of a step_kernel launch
    + 1/26 of a fast-forward ff_kernel launch) from the committed ncu captures of the same workload, else None."""
    p = ROOT / "profiles" / "r2_traffic.json"
    key = {"SwingRacket-v0": "dram_bytes_per_env_step_launch_pair", "Tennisbot-v0": "hit_step_kernel_dram_bytes_per_launch"}[env]
    if precision == "f64" and n == 1 << 20 and p.exists():
        try:
            return float(json.loads(p.read_text())[key])
        except Exception:
            pass
    return None


def measured_peak():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "measured"
        except Exception:
            pass
    return 6650.0, "fallback"


def dump_outputs(out_dir, arrays):
    """Write {name: array with one row per env} as out_dir/<name>.npy in float32 (float64 arrays stay float64), so that
    two builds can be compared output for output.  When the files would exceed DUMP_LIMIT, the same seeded sample of envs
    is taken from every array and the sampled env indices go to env_index.npy."""
    import numpy as np

    arrays = {k: (v if v.dtype in (np.float32, np.float64) else v.astype(np.float32)) for k, v in arrays.items()}
    n = len(next(iter(arrays.values())))
    row_bytes = sum(v.nbytes for v in arrays.values()) // n
    budget = DUMP_LIMIT - 4096  # room for the .npy headers
    if n * row_bytes > budget:
        idx = np.sort(np.random.default_rng(0).choice(n, budget // (row_bytes + 8), replace=False))
        arrays = {k: v[idx] for k, v in arrays.items()}
        arrays["env_index"] = idx.astype(np.float64)
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    for k, v in arrays.items():
        np.save(out / f"{k}.npy", v)


class CpuOracleRun:
    """The restated CPU oracle (PyBullet is not installable here) on `threads` host threads: one env batch, one
    pre-drawn action tape; step() timings exclude construction and action generation."""

    def __init__(self, env, n_envs, threads):
        import numpy as np

        from oracle import binding as ob

        ob.build()
        self.n = n_envs
        self.o = ob.OracleEnv(env, n_envs, seed=0, threads=threads)
        self.o.reset()
        rng = np.random.default_rng(0)
        self.acts = rng.uniform(-1, 1, (EPISODE_STEPS, n_envs, self.o.act_dim)).astype(np.float32)
        self.t = 0
        self.last = None

    def run(self, steps):
        """`steps` env steps for every env of the sample; returns (seconds, env steps done).  self.last: the last step's outputs."""
        t0 = time.perf_counter()
        for _ in range(steps):
            self.last = self.o.step(self.acts[self.t % EPISODE_STEPS])
            self.t += 1
        return time.perf_counter() - t0, self.n * steps


# ---------------------------------------------------------------------------------------------- reference arm
def real_reference():
    """(path, None) when the unmodified reference can run here - pybullet, gym and stable-baselines3 importable and the
    reference installed under baseline/_ref - else (None, why).  Never true in this image (SURVEY 8(c)): kept so that the
    arm switches to the real thing, kind = "reference", wherever those packages exist."""
    ref = ROOT / "baseline" / "_ref"
    if not (ref / "tennisbot").exists():
        return None, "baseline/_ref absent (the reference needs the pybullet wheel, which cannot be installed offline)"
    try:
        import gym  # noqa: F401
        import pybullet  # noqa: F401
        import stable_baselines3  # noqa: F401
    except Exception as e:  # pragma: no cover - not reachable in this image
        return None, f"{type(e).__name__}: {e}"
    return ref, None


def _ref_env_factory(ref_path, env_id):  # pragma: no cover - needs pybullet
    def make():
        import sys as _sys
        _sys.path.insert(0, str(ref_path))
        import gym
        import tennisbot  # noqa: F401  (the reference's own package: registers the ids)
        return gym.make(env_id, use_gui=False)
    return make


def run_real_reference(args, ref_path):  # pragma: no cover - needs pybullet
    """SURVEY 8(d): the reference env (GUI off) under SB3 SubprocVecEnv with one worker per host core, random actions."""
    import numpy as np
    from stable_baselines3.common.vec_env import SubprocVecEnv

    cores = os.cpu_count() or 1
    venv = SubprocVecEnv([_ref_env_factory(ref_path, args.env) for _ in range(cores)])
    venv.reset()
    rng = np.random.default_rng(0)
    ad = venv.action_space.shape[0]
    last = {}
    def episode():
        t0 = time.perf_counter()
        for _ in range(EPISODE_STEPS):
            obs, reward, done, _ = venv.step(rng.uniform(-1, 1, (cores, ad)).astype(np.float32))
        last.update(obs=obs, reward=reward, done=done)
        return time.perf_counter() - t0
    for _ in range(max(args.warmup, 0)):
        episode()
    wall = sum(episode() for _ in range(args.steps))
    venv.close()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, last)
    return cores * EPISODE_STEPS * args.steps / wall, wall, cores


def run_reference(args, rank):
    """CPU arm: the oracle port on all host cores, same workload (random actions, auto-reset), each bench step =
    one whole 26-step episode of a bounded sample so the fast-forward step is weighted as in the GPU arm."""
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    ref_path, why = real_reference()
    if ref_path is not None:  # pragma: no cover - needs pybullet
        value, wall, cores = run_real_reference(args, ref_path)
        emit({"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
              "warmup": args.warmup, "ms_per_step": 1e3 * wall / args.steps, "higher_is_better": True, "scaling": "weak",
              "vs_baseline": None, "dtype": "f64", "data": "synthetic",
              "config": {"workload": f"{args.env} random actions, unmodified reference under SB3 SubprocVecEnv, {cores} workers x "
                                     f"{EPISODE_STEPS} env steps per bench step"},
              "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "reference",
                               "sample": f"{cores} envs x {EPISODE_STEPS} env steps x {args.steps} repeats (PyBullet DIRECT)"},
              "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}})
        return
    n = args.cpu_sample_envs
    run = CpuOracleRun(args.env, n, cores)
    for _ in range(max(args.warmup, 0)):
        run.run(EPISODE_STEPS)
    wall, total = 0.0, 0
    for _ in range(args.steps):
        dt, k = run.run(EPISODE_STEPS)
        wall += dt
        total += k
    value = total / wall
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, run.last)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * wall / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"{args.env} random actions, CPU sample of {n} envs x {EPISODE_STEPS} env steps per bench step",
                   "note": "restated double-precision CPU oracle (oracle/tb_oracle.c) - NOT PyBullet: " + why},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": f"{n} envs x {EPISODE_STEPS} env steps x {args.steps} repeats, "
                                   f"{run.o.physics_steps()} physics substeps incl. warm-up"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    emit(line)


# ---------------------------------------------------------------------------------------------- extras (N = 1)
def _timed(torch, fn, reps):
    """CUDA-event time of `reps` calls of fn() on the current stream, in seconds."""
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e-3


def run_extras(args, torch, np):
    """The other BASELINE.json configs, each a few hundred milliseconds: numbers the driver can see next to the headline."""
    from tennisbot_rl_b200 import _lib
    from tennisbot_rl_b200.batch import TennisBatch
    from tennisbot_rl_b200.vec_env import TennisVecEnv

    out = {}
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", 0)))
    # ---- config 3: Tennisbot-v0, 65 536 envs, WITH racket-ball contact: scripted tracker (a1 follows the ball's y)
    try:
        n = 65536
        b = TennisBatch("Tennisbot-v0", n, device=dev.index, seed=0, precision=args.precision)
        obs = b.reset()
        act = torch.zeros((n, 2), device=dev)

        def tracked_step():  # the action law of TB_ACT_TRACK, formed by torch from the observation (API mode: tb_step per step)
            act[:, 0].uniform_(-0.2, 0.2)
            torch.clamp(4.0 * (obs[:, 7] - obs[:, 1]) - 1.5 * obs[:, 4], -1, 1, out=act[:, 1])
            b.step(act)

        for _ in range(700):  # desynchronise: episodes last 380 .. 1001 steps
            tracked_step()
        b.read_stats(clear=True)
        k = 300
        sec = _timed(torch, tracked_step, k)
        st = b.read_stats(clear=True)
        api = {"env_steps_per_s": n * k / sec, "ms_per_step": 1e3 * sec / k, "racket_hit_steps": int(st[2]), "episodes": int(st[0])}
        sec = _timed(torch, lambda: b.rollout(100, action_mode=_lib.ACT_TRACK, want_outputs=False), 3)
        st = b.read_stats(clear=True)
        out["tennisbot_v0_65536_tracking"] = {
            "workload": "Tennisbot-v0, 65 536 envs, desynchronised episodes, scripted ball tracker (BASELINE config 3 with contact)",
            "api_mode": api,
            "fused_rollout_k100": {"env_steps_per_s": n * 300 / sec, "racket_hit_steps": int(st[2]), "episodes": int(st[0])}}
        b.close()
    except Exception as e:  # an extra must never cost the headline line
        out["tennisbot_v0_65536_tracking"] = {"error": f"{type(e).__name__}: {e}"}
    # ---- config 4, env side: the VecEnv host loop SB3 drives (numpy in / out, terminal observations and infos on)
    try:
        n = 16384
        env = TennisVecEnv("SwingRacket-v0", n, device=dev.index, seed=0, precision=args.precision)
        env.reset()
        rng = np.random.default_rng(0)
        acts = rng.uniform(-1, 1, (8, n, 6)).astype(np.float32)
        for t in range(EPISODE_STEPS):
            env.step(acts[t % 8])
        t0 = time.perf_counter()
        k = 4 * EPISODE_STEPS
        for t in range(k):
            env.step(acts[t % 8])
        sec = time.perf_counter() - t0
        out["swingracket_v0_16384_vecenv"] = {
            "workload": "TennisVecEnv.step (SB3 VecEnv contract: numpy actions in, obs / rewards / dones / infos with terminal_observation "
                        "and episode records out), 16 384 envs, 4 episodes, wall clock",
            "env_steps_per_s": n * k / sec, "ms_per_step": 1e3 * sec / k}
        env.close()
    except Exception as e:
        out["swingracket_v0_16384_vecenv"] = {"error": f"{type(e).__name__}: {e}"}
    # ---- fused K = 26 rollout with in-kernel random actions (state in registers across the episode), 1 Mi envs
    try:
        n = args.envs_per_gpu
        b = TennisBatch("SwingRacket-v0", n, device=dev.index, seed=0, precision=args.precision)
        b.reset()
        b.rollout(EPISODE_STEPS, want_outputs=False)
        sec = _timed(torch, lambda: b.rollout(EPISODE_STEPS, want_outputs=False), 3)
        out["swingracket_v0_tb_rollout_k26"] = {"workload": f"tb_rollout(TB_ACT_RANDOM, 26), {n} envs, one launch per episode",
                                                "env_steps_per_s": n * EPISODE_STEPS * 3 / sec, "ms_per_episode": 1e3 * sec / 3}
        b.close()
    except Exception as e:
        out["swingracket_v0_tb_rollout_k26"] = {"error": f"{type(e).__name__}: {e}"}
    # ---- config 4, rollout side: the policy evaluated in-kernel (tb_policy_rollout), 16 384 envs, CUDA graph
    try:
        from tennisbot_rl_b200.ppo import SwingPPO

        ppo = SwingPPO(num_envs=16384, seed=0, use_graph=True, fused_policy=True, device=dev.index)
        for _ in range(3):
            ppo.rollout()
        ppo.rollout_s = 0.0
        reps = 20
        for _ in range(reps):
            ppo.rollout()
        out["swingracket_v0_16384_policy_rollout"] = {
            "workload": "26-step rollouts of the (untrained) MlpPolicy through tb_policy_rollout, 16 384 envs, replayed CUDA graph; "
                        "tests/test_ppo_gpu.py trains it to the reference return",
            "env_steps_per_s": 16384 * EPISODE_STEPS * reps / ppo.rollout_s, "ms_per_rollout": 1e3 * ppo.rollout_s / reps}
        ppo.env.close()
    except Exception as e:
        out["swingracket_v0_16384_policy_rollout"] = {"error": f"{type(e).__name__}: {e}"}
    return out


# ---------------------------------------------------------------------------------------------- B200 arm
def stagger_phases(batch, torch, gen):
    """Group g (128 envs) starts g mod 26 steps late: step everyone, then restart the groups whose turn it is."""
    n = batch.num_envs
    group = torch.arange(n, device=batch.device) // GROUP % EPISODE_STEPS
    act = torch.zeros((n, batch.act_dim), dtype=torch.float32, device=batch.device)
    batch.reset()
    for p in range(1, EPISODE_STEPS):
        act.uniform_(-1, 1, generator=gen)
        batch.step(act)
        batch.reset(mask=(group == p))
    return EPISODE_STEPS - 1


def run_b200(args, rank, world):
    import numpy as np
    import torch

    from tennisbot_rl_b200.batch import TennisBatch

    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    n = args.envs_per_gpu
    batch = TennisBatch(args.env, n, device=local, seed=0, precision=args.precision, env_id_offset=rank * n)
    dev = batch.device
    stats = batch.stats_tensor()

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    # action buffers: a ring of pre-drawn U(-1,1) batches resident in HBM (synthetic actions = action_space.sample())
    gen = torch.Generator(device=dev).manual_seed(0)  # same actions in every run, so that --dump-outputs can be compared
    ring = [torch.empty((n, batch.act_dim), dtype=torch.float32, device=dev).uniform_(-1, 1, generator=gen) for _ in range(RING)]
    pre_launch = 0
    stagger = args.stagger == "on" and args.env == "SwingRacket-v0"
    if not stagger:
        batch.reset()
    else:
        pre_launch = stagger_phases(batch, torch, gen)
    # lock-step: start the timed region at episode phase (-K mod 26) so that it ends right after a fast-forward step
    swing_lockstep = args.env == "SwingRacket-v0" and not stagger
    align = (-args.steps - args.warmup) % EPISODE_STEPS if swing_lockstep else 0
    for w in range(args.warmup + align):  # `align` extra untimed steps put the timed region on an episode boundary
        batch.step(ring[w % len(ring)])
    reduced = stats.clone()  # the all-reduce works on a snapshot: the live vector keeps accumulating in the kernels
    if dist is not None:
        dist.all_reduce(reduced)  # warm the NCCL communicator
    batch.read_stats(clear=True)
    l0 = batch.launch_count()

    sampler = ClockSampler(local, getattr(torch.cuda.get_device_properties(local), "uuid", None)) if rank == 0 else None
    if sampler:
        sampler.start()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    n_reductions = 0
    for k in range(args.steps):
        out = batch.step(ring[k % len(ring)])
        # the per-iteration reduction of the episode statistics (10 x int64, NCCL) follows every step that ends an episode:
        # in lock step those are the fast-forward steps, and the region ends on one
        if dist is not None and ((args.steps - 1 - k) % EPISODE_STEPS == 0 if swing_lockstep else (k + 1) % EPISODE_STEPS == 0):
            reduced.copy_(stats)
            dist.all_reduce(reduced)
            n_reductions += 1
    e1.record()
    if sampler:
        sampler.sample_now()  # everything is queued and the device is still working through it (the window ends on a fast-forward step)
    barrier()
    ms = e0.elapsed_time(e1)
    clocks = sampler.stop() if sampler else None
    launches = batch.launch_count() - l0
    st = batch.read_stats() if dist is None else None
    if dist is not None:
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
        reduced.copy_(stats)
        dist.all_reduce(reduced)
        st = reduced.cpu().numpy()
    if args.dump_outputs and rank == 0:  # before the steps below overwrite the batch's output buffers
        dump_outputs(args.dump_outputs, dict(zip(("obs", "reward", "done", "terminal_obs", "events"), (t.cpu().numpy() for t in out))))

    # ---- per-kernel device times over one more episode (events inside the library, stream synchronised per step:
    #      outside the timed region by construction)
    batch.set_kernel_timing(True)
    for k in range(EPISODE_STEPS if args.env == "SwingRacket-v0" else 8):
        batch.step(ring[k % len(ring)])
    ms_a, ms_b, nk = batch.kernel_timing()
    batch.set_kernel_timing(False)

    # ---- end to end through the host-buffer entry point (pinned numpy in, pinned numpy out)
    hb = batch.host_buffers()
    rng = np.random.default_rng(rank)
    host_actions = rng.uniform(-1, 1, (n, batch.act_dim)).astype(np.float32)
    np.copyto(hb["actions"], host_actions)
    for _ in range(3 if stagger or args.env != "SwingRacket-v0" else EPISODE_STEPS):  # warm-up, whole episode in lock-step
        batch.step_host(want_terminal=False, want_events=False)
    barrier()
    t0 = time.perf_counter()
    ret_sum = 0.0
    for _ in range(args.e2e_steps):
        out = batch.step_host(want_terminal=False, want_events=False)
        ret_sum += float(out["reward"][0])  # the result is consumed on the host
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    if dist is not None:
        t = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t.item())
    h2d = n * batch.act_dim * 4
    d2h = n * (batch.obs_dim * 4 + 4 + 1)

    if rank == 0:
        total_envs = n * world
        value = total_envs * args.steps / (ms * 1e-3)
        peak, peak_src = measured_peak()
        algo = ALGO_BYTES[(args.env, args.precision)]
        achieved = n * algo / (ms * 1e-3 / args.steps) / 1e9
        ms_step = ms_a / max(nk, 1)
        step_gbs = n * algo / (ms_step * 1e-3) / 1e9
        line = {
            "metric": METRIC if args.env == "SwingRacket-v0" else "env-steps/sec Tennisbot-v0",
            "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": args.precision, "data": "synthetic",
            "config": {"workload": f"{args.env} batched {n} envs per GPU (config 5 slice), uniform random actions, "
                                   f"reset ranges of the env, auto-reset",
                       "envs_per_gpu": n, "total_envs": total_envs,
                       "phase_stagger": f"per {GROUP}-env group, g mod {EPISODE_STEPS}" if stagger else
                       f"none: lock-step episodes, timed region holds {-(-args.steps // EPISODE_STEPS)} fast-forward steps in {args.steps} steps",
                       "alignment_steps": align,
                       "l2_policy": "working set per launch %.0f MB > 126 MB L2 (inputs larger than L2)" % (n * algo / 1e6),
                       "actions": f"ring of {RING} pre-drawn U(-1,1) batches in HBM: i.i.d. within every 26-step episode",
                       "parallelism": f"env-sharded x{world}, no data-path collective; int64[10] stats all-reduce (NCCL) after every "
                                      f"episode-ending step: {n_reductions} inside the timed region"},
            # One env step is a pair of launches whose shares shift with the precision and the step of the episode, so the
            # headline roofline figure is the whole step: algorithmic bytes of an env step (SURVEY 8(d): action + obs +
            # reward + done + state read + state written) over the mean step time of the timed region.  Per kernel:
            # step_kernel is HBM-bound (its own algorithmic fraction and the DRAM bytes ncu saw per launch are given);
            # ff_kernel is bound by the FP64 pipe / latency, not by memory (profiles/).
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         # the same step time on BASELINE.md's float32-state yardstick (309 B per SwingRacket env step): the
                         # 60 % target of the north star is quoted on that one and is out of reach for an f64 state (26 x the
                         # state traffic alone exceeds the time it allows) - see DESIGN.md section 4
                         "frac_fp32_bytes": n * ALGO_BYTES_F32_STATE[args.env] / (ms * 1e-3 / args.steps) / 1e9 / peak,
                         "traffic": measured_traffic(args.env, args.precision, n), "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": n * algo, "algorithmic_bytes_per_env_step": algo,
                         "scope": "whole env step = step_kernel + ff_kernel: algorithmic bytes of the step / mean step time",
                         "kernels": {
                             "step_kernel": {"ms_per_launch": ms_step, "achieved_gbs": step_gbs, "frac": step_gbs / peak, "bound": "hbm",
                                             "share_of_step_time": ms_a / max(ms_a + ms_b, 1e-9),
                                             "moved_bytes_per_env_step": MOVED_BYTES.get((args.env, args.precision)),
                                             "wire_gbs": n * MOVED_BYTES.get((args.env, args.precision), algo) / (ms_step * 1e-3) / 1e9,
                                             "wire_frac": n * MOVED_BYTES.get((args.env, args.precision), algo) / (ms_step * 1e-3) / 1e9 / peak,
                                             "note": "achieved_gbs / frac: ALGORITHMIC bytes (SURVEY 8(d)) of all envs over this kernel's mean launch "
                                                     "time - above the peak because the kernel moves fewer: it re-derives the episode constants "
                                                     "from the RNG counters and tabulates the free-falling ball's velocity instead of loading them; "
                                                     "wire_*: the bytes a control step actually moves (profiles/r2_traffic.json)"},
                             "ff_kernel": {"ms_per_launch": ms_b / max(nk, 1), "share_of_step_time": ms_b / max(ms_a + ms_b, 1e-9),
                                           "ms_per_episode": ms_b / max(nk, 1) * (EPISODE_STEPS if args.env == "SwingRacket-v0" else 1),
                                           "bound": "instruction issue / fp64 pipe: ~335 instructions (160 FP64) per physics substep, ~106 substeps per env "
                                                    "on its 26th step; not memory-bound (profiles/r2_ff_kernel_f64_ncu.txt, DESIGN.md 4.2)"}}},
            "e2e": {"value": total_envs * args.e2e_steps / e2e_s, "unit": UNIT, "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h, "steps": args.e2e_steps, "api": "TennisBatch.step_host -> tb_step_host: pinned host buffers in and out; the kernels read the actions from and write obs/reward/done to host memory over PCIe themselves (both directions concurrent with the compute)"},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "episode_stats": {"episodes": int(st[0]), "mean_length": float(st[1]) / max(int(st[0]), 1),
                              "mean_return": float(st[6]) / 1048576.0 / max(int(st[0]), 1),
                              "physics_substeps": int(st[8]), "env_steps": int(st[9]),
                              "physics_substeps_per_s": float(st[8]) / (ms * 1e-3)},
        }
        if args.extras == "on" or (args.extras == "auto" and world == 1 and args.env == "SwingRacket-v0"):
            batch.close()
            line["extras"] = run_extras(args, torch, np)
        if not args.skip_cpu_baseline and world == 1:  # (rank 0 at N = 1 only: the other ranks of a multi-GPU run would wait)
            cores = os.cpu_count() or 1
            cpu_n = args.cpu_sample_envs
            run = CpuOracleRun(args.env, cpu_n, cores)
            run.run(EPISODE_STEPS)
            reps, total, t_cpu = 0, 0, 0.0
            while t_cpu < 12.0 and reps < 200:
                dt, k = run.run(EPISODE_STEPS)
                t_cpu += dt
                total += k
                reps += 1
            line["cpu_baseline"] = {"value": total / t_cpu, "unit": UNIT, "cores": cores, "kind": "port",
                                    "sample": f"{cpu_n} envs x {EPISODE_STEPS} env steps x {reps} episodes on {cores} threads "
                                              f"({t_cpu:.1f} s); restated CPU oracle, not PyBullet (absent from the image)"}
        emit(line)
    batch.close()
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


_REAL_STDOUT = None


def emit(line):
    """The ONE JSON line of the contract, on the process's original stdout."""
    out = _REAL_STDOUT if _REAL_STDOUT is not None else sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def main():
    global _REAL_STDOUT
    sys.dont_write_bytecode = True  # the tree may be read-only: bench.py writes nothing there
    args = parse()
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    # libraries write to fd 1 behind Python's back (NCCL prints its version banner there when NCCL_DEBUG is set on the
    # box): keep the original stdout for the JSON line and send everything else to stderr
    sys.stdout.flush()
    _REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    if args.impl == "reference":
        run_reference(args, rank)
        return
    if world == 1 and args.gpus > 1:
        # launched without torchrun: re-exec under torch.distributed.run
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", os.environ.get("MASTER_PORT", "29517"), __file__] + sys.argv[1:]
        sys.exit(subprocess.call(cmd, stdout=_REAL_STDOUT))
    run_b200(args, rank, world)


if __name__ == "__main__":
    main()
