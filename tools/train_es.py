"""Train with the device-resident ES trainer (es_train.EsTrainer, ARS V2-t) and time where a generation goes.

usage: train_es.py ENV [--directions D] [--generations G] [--repeats R] [--top-k K] [--sigma S] [--lr A] [--seed N]
                       [--noise-seed N] [--theta FILE.npz] [--save FILE.pt] [--print-step P] [--split-directions D ...]

Prints the card's name and power limit, then one JSON line per generation (mean and max fitness, sigma_R, the master
normaliser's count, env steps, wall ms).  With --save, the trainer's state (theta, master normaliser, generation, seeds) and
the last generation's fitness are written every --print-step generations and at the end.  Then, in a separate run per
--split-directions value, the wall-time split of a generation (median of 5 after 2 warm-up generations, torch.cuda.synchronize
at every boundary): drawing the population (tb_es_begin_noise: perturbation, reset, normaliser seeding), the rollout, the
update (ARS selection and tb_es_noise_combine) and the master-normaliser merge (tb_es_normalizer_stats).  Default split sizes:
819 and 13 107 directions, i.e. 16 380 and 262 140 envs at 10 repeats (the nearest even populations to 16 390 and 262 150)."""
import argparse
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
from tennisbot_rl_b200.es_train import EsTrainer  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[torch.cuda.current_device()] if q else torch.cuda.get_device_name()


def make(args, directions):
    theta = None if args.theta is None else np.load(args.theta)["weights"]
    return EsTrainer(args.env, directions, repeats=args.repeats, top_k=args.top_k, sigma=args.sigma, lr=args.lr, seed=args.seed,
                     noise_seed=args.noise_seed, theta=theta)


def train(args):
    tr = make(args, args.directions)
    for g in range(args.generations):
        t0 = time.perf_counter()
        row = tr.step()
        row["ms"] = round((time.perf_counter() - t0) * 1e3, 3)
        print(json.dumps(dict(env=args.env, directions=args.directions, repeats=args.repeats, **row)), flush=True)
        if args.save and ((g + 1) % args.print_step == 0 or g + 1 == args.generations):
            torch.save(dict(tr.state_dict(), fitness=tr.fitness.cpu()), args.save)
    tr.close()


def split(args, directions):
    tr = make(args, directions)
    for _ in range(2):
        tr.step()
    runs = []
    for _ in range(5):
        t = {}
        tr.step(timings=t)
        runs.append(t)
    row = dict(env=args.env, directions=directions, envs=2 * directions * args.repeats, steps=tr.ev.steps_run,
               **{k: round(statistics.median(r[k] for r in runs) * 1e3, 3) for k in runs[0]})
    row["total_ms"] = round(sum(row[k] for k in runs[0]), 3)
    print(json.dumps(dict(split_ms=row)), flush=True)
    tr.close()
    torch.cuda.empty_cache()


def main():
    p = argparse.ArgumentParser()
    p.add_argument("env", nargs="?", default="SwingRacket-v0")
    p.add_argument("--directions", type=int, default=256)
    p.add_argument("--generations", type=int, default=30)
    p.add_argument("--repeats", type=int, default=10)
    p.add_argument("--top-k", type=int, default=66)
    p.add_argument("--sigma", type=float, default=0.05)
    p.add_argument("--lr", type=float, default=0.1)
    p.add_argument("--seed", type=int, default=0)
    p.add_argument("--noise-seed", type=int, default=0)
    p.add_argument("--theta", default=None, help="npz with a 'weights' vector to start from (default zeros)")
    p.add_argument("--save", default=None)
    p.add_argument("--print-step", type=int, default=10)
    p.add_argument("--split-directions", type=int, nargs="*", default=[819, 13107])
    args = p.parse_args()
    print("card (name, power limit, max SM clock):", card(), flush=True)
    if args.generations > 0:
        train(args)
    for d in args.split_directions:
        split(args, d)


if __name__ == "__main__":
    main()
