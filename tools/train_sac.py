"""Train with GpuSAC and time the in-kernel SAC actor.

usage: train_sac.py ENV [--envs N] [--steps K] [--batch B] [--gradient-steps G] [--slots S] [--iters I] [--eval-every E]
                        [--seed N] [--normalize] [--save FILE.npz] [--sweep] [--throughput] [--sizes N ...] [--no-train]
                        [--out FILE.json]

Prints the card's name and power limit, then:
  - training (unless --no-train): the curve (collection returns and deterministic evaluations) and the per-phase split of an
    iteration (collect / update wall seconds, torch.cuda.synchronize at every boundary);
  - --sweep: the same for each batch geometry of SWEEP (same iterations budget in gradient steps), one JSON line each;
  - --throughput: at each size, collection env-steps/s of tb_sac_rollout (in-kernel actor) against SacActor in torch float32 with
    TennisBatch.step in one CUDA graph (K steps per graph), the actor kernel's own time from torch.profiler (sac_kernel launches
    that evaluate the network) and its achieved TFLOP/s on the tensor cores (2 x N x 256 x 256 per step) against the BF16
    data-sheet rate of one B200 (2250 dense TFLOP/s at 1000 W);
  - --throughput --normalize: instead, at each size, collection env-steps/s of tb_sac_rollout with and without TB_SAC_VECNORM
    (a training normaliser: the statistics pass after every step), alternating the two graphs, and once the GpuSAC update
    graph's time per gradient step with and without tb_vecnorm_apply on the sampled batch.
--normalize trains with GpuSAC(normalize=True); --save writes GpuSAC.save's npz (actor, and the record with --normalize).
"""
import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
from tennisbot_rl_b200 import _lib  # noqa: E402
from tennisbot_rl_b200.batch import TennisBatch  # noqa: E402
from tennisbot_rl_b200.sac import GpuSAC, SacActor, pack_sac_actor  # noqa: E402

BF16_DENSE_TFLOPS = 2250.0
# (envs, steps per collection, batch, gradient steps per collection, slots)
SWEEP = [(256, 1, 256, 8, 4096), (256, 1, 1024, 8, 4096), (1024, 1, 1024, 8, 1024), (64, 1, 256, 4, 16384)]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[torch.cuda.current_device()] if q else torch.cuda.get_device_name()


def train(args, envs, steps, batch, grad, slots, iters, eval_every):
    s = GpuSAC(args.env, num_envs=envs, steps=steps, batch_size=batch, gradient_steps=grad, slots=slots, seed=args.seed,
               normalize=args.normalize)
    out = s.train(iters, log=lambda m: print(m, flush=True), eval_every=eval_every)
    if args.save:
        s.save(args.save)
    s.env.close()
    out.pop("history")
    per_it = iters or 1
    out["collect_ms_per_iter"] = round(out["collect_s"] / per_it * 1e3, 3)
    out["update_ms_per_iter"] = round(out["update_s"] / per_it * 1e3, 3)
    return out


def throughput(env_id, n, K=26, reps=5):
    """(in-kernel env-steps/s, torch-actor env-steps/s, sac_kernel ms per env step)."""
    b = TennisBatch(env_id, n, seed=1)
    od, ad = b.obs_dim, b.act_dim
    torch.manual_seed(0)
    actor = SacActor(od, ad).cuda()
    b.set_sac_actor(pack_sac_actor(actor).cuda())
    b.sac_begin()
    b.sac_rollout(K, "sample", None)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        b.sac_rollout(K, "sample", None)
    g.replay()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(reps):
        g.replay()
    torch.cuda.synchronize()
    fused = reps * K * n / (time.perf_counter() - t0)
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        g.replay()
        torch.cuda.synchronize()
    us = sum(e.device_time_total for e in prof.key_averages() if "sac_kernel" in e.key)
    kernel_ms = us / 1e3 / K  # (includes the fold-only launch ending the call: one per K steps)
    # the same actor in torch float32, TennisBatch.step in the same graph
    obs = b.reset().clone()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())

    def body():
        with torch.no_grad():
            for _ in range(K):
                a = actor(obs)
                o, _, _, _, _ = b.step(a)
                obs.copy_(o)
    with torch.cuda.stream(s):
        body()
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    g2 = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g2):
        body()
    g2.replay()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(reps):
        g2.replay()
    torch.cuda.synchronize()
    eager = reps * K * n / (time.perf_counter() - t0)
    b.close()
    return fused, eager, kernel_ms


def _graph_rate(b, K, reps, normalize):
    """Captures K steps of tb_sac_rollout (sample, no ring) and returns a function timing `reps` replays: env-steps/s."""
    b.sac_rollout(K, "sample", None, normalize=normalize)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        b.sac_rollout(K, "sample", None, normalize=normalize)
    g.replay()
    torch.cuda.synchronize()

    def rate():
        t0 = time.perf_counter()
        for _ in range(reps):
            g.replay()
        torch.cuda.synchronize()
        return reps * K * b.num_envs / (time.perf_counter() - t0)
    return rate


def throughput_normalize(env_id, n, K=26, reps=5, rounds=5):
    """(env-steps/s without, with the normaliser): two contexts, the same actor, best of `rounds` alternating timings."""
    torch.manual_seed(0)
    rates = []
    for normalize in (False, True):
        b = TennisBatch(env_id, n, seed=1)
        actor = SacActor(b.obs_dim, b.act_dim).cuda()
        b.set_sac_actor(pack_sac_actor(actor).cuda())
        if normalize:
            b.set_vecnorm()
        b.sac_begin()
        rates.append((b, _graph_rate(b, K, reps, normalize)))
    best = [0.0, 0.0]
    for _ in range(rounds):
        for j, (_, rate) in enumerate(rates):
            best[j] = max(best[j], rate())
    for b, _ in rates:
        b.close()
    return best


def update_ms(env_id, rounds=5, reps=50):
    """GpuSAC's update graph (the defaults: batch 1024), ms per gradient step without and with tb_vecnorm_apply, best of
    `rounds` alternating timings of `reps` gradient steps."""
    runs = []
    for normalize in (False, True):
        s = GpuSAC(env_id, seed=0, normalize=normalize)
        s.update()  # captures the graph
        torch.cuda.synchronize()
        runs.append(s)
    best = [float("inf")] * 2
    for _ in range(rounds):
        for j, s in enumerate(runs):
            t0 = time.perf_counter()
            for _ in range(reps):
                s.update_graph.replay()
            torch.cuda.synchronize()
            best[j] = min(best[j], (time.perf_counter() - t0) / reps * 1e3)
    for s in runs:
        s.env.close()
    return best


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("env", nargs="?", default="SwingRacket-v0")
    ap.add_argument("--envs", type=int, default=1024)
    ap.add_argument("--steps", type=int, default=1)
    ap.add_argument("--batch", type=int, default=1024)
    ap.add_argument("--gradient-steps", type=int, default=8)
    ap.add_argument("--slots", type=int, default=1024)
    ap.add_argument("--iters", type=int, default=5000)
    ap.add_argument("--eval-every", type=int, default=1000)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--normalize", action="store_true")
    ap.add_argument("--save", default=None)
    ap.add_argument("--sweep", action="store_true")
    ap.add_argument("--throughput", action="store_true")
    ap.add_argument("--no-train", action="store_true")
    ap.add_argument("--sizes", type=int, nargs="*", default=[4096, 16384, 65536, 1 << 20])
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    print("card:", card(), flush=True)
    results = {"card": card(), "env": args.env}
    if not args.no_train:
        r = train(args, args.envs, args.steps, args.batch, args.gradient_steps, args.slots, args.iters, args.eval_every)
        print(json.dumps(r), flush=True)
        results["train"] = r
    if args.sweep:
        budget = args.iters * args.gradient_steps  # gradient steps per configuration (the sweep in DESIGN: 10 000 x 4)
        results["sweep"] = []
        for envs, steps, batch, grad, slots in SWEEP:
            iters = max(1, budget // grad)
            r = train(args, envs, steps, batch, grad, slots, iters, max(1, iters // 6))
            row = {k: r[k] for k in ("envs", "steps", "batch_size", "gradient_steps", "slots", "iters", "eval_mean_return",
                                     "evaluations", "wall_s", "collect_s", "update_s")}
            print(json.dumps(row), flush=True)
            results["sweep"].append(row)
    if args.throughput and args.normalize:
        results["throughput_normalize"] = []
        for n in args.sizes:
            plain, norm = throughput_normalize(args.env, n)
            row = {"envs": n, "env_steps_per_s": plain, "env_steps_per_s_normalize": norm,
                   "us_per_step": 1e6 * n / plain, "us_per_step_normalize": 1e6 * n / norm}
            print(json.dumps(row), flush=True)
            results["throughput_normalize"].append(row)
        plain, norm = update_ms(args.env)
        row = {"update_ms_per_gradient_step": plain, "update_ms_per_gradient_step_normalize": norm}
        print(json.dumps(row), flush=True)
        results["update_normalize"] = row
    elif args.throughput:
        results["throughput"] = []
        for n in args.sizes:
            fused, eager, kms = throughput(args.env, n)
            tflops = 2.0 * n * _lib.SAC_HIDDEN * _lib.SAC_HIDDEN / (kms * 1e-3) / 1e12
            row = {"envs": n, "in_kernel_env_steps_per_s": fused, "torch_actor_env_steps_per_s": eager,
                   "sac_kernel_ms_per_step": kms, "layer2_tflops": tflops, "share_of_bf16_datasheet": tflops / BF16_DENSE_TFLOPS}
            print(json.dumps(row), flush=True)
            results["throughput"].append(row)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(json.dumps(results, indent=1))


if __name__ == "__main__":
    main()
