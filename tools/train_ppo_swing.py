#!/usr/bin/env python3
"""CLI of tennisbot_rl_b200.ppo: GPU-resident PPO on SwingRacket-v0 (BASELINE config 4) or Tennisbot-v0 (train.py, with
its racket-scale curriculum over --curriculum TOTAL env steps).

    python tools/train_ppo_swing.py --iters 150 --out gpurun_out/ppo_swing_b200.json
    python tools/train_ppo_swing.py --env Tennisbot-v0 --rollout-len 128 --curriculum 200000000 --iters 100
    python tools/train_ppo_swing.py --env Tennisbot-v0 --iters 60 --normalize --save hit_norm.npz
"""
import argparse
import json
import sys
from pathlib import Path

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
from tennisbot_rl_b200.ppo import HitPPO, SwingPPO  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--env", default="SwingRacket-v0", choices=("SwingRacket-v0", "Tennisbot-v0"))
    ap.add_argument("--envs", type=int, default=16384)
    ap.add_argument("--iters", type=int, default=150)
    ap.add_argument("--lr", type=float, default=3e-4)
    ap.add_argument("--epochs", type=int, default=10)
    ap.add_argument("--minibatches", type=int, default=8)
    ap.add_argument("--precision", default="f64")
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--target", type=float, default=31.5, help="SwingRacket-v0: the return to reach")
    ap.add_argument("--rollout-len", type=int, default=128, help="Tennisbot-v0: env steps per env per update")
    ap.add_argument("--curriculum", type=int, default=0, metavar="TOTAL",
                    help="Tennisbot-v0: train.py's racket-scale curriculum over TOTAL env steps (0: none)")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--eager-policy", action="store_true", help="torch policy in the rollout instead of tb_policy_rollout")
    ap.add_argument("--normalize", action="store_true", help="SB3 VecNormalize on the device rollout (tb_set_vecnorm)")
    ap.add_argument("--out", default="")
    ap.add_argument("--save", default="", help="npz of the trained policy (and the normaliser's record): GpuPPO.save")
    args = ap.parse_args()
    log = lambda s: print(s, flush=True)  # noqa: E731
    if args.env == "SwingRacket-v0":
        ppo = SwingPPO(args.envs, args.precision, args.seed, args.lr, args.epochs, args.minibatches, use_graph=not args.no_graph,
                       fused_policy=not args.eager_policy, normalize=args.normalize)
        summary = ppo.train(args.iters, args.target, log=log)
    else:
        ppo = HitPPO(args.envs, args.rollout_len, args.curriculum or None, args.precision, args.seed, args.lr, args.epochs,
                     args.minibatches, use_graph=not args.no_graph, fused_policy=not args.eager_policy, normalize=args.normalize)
        summary = ppo.train(args.iters, log=log)
    summary["normalize"] = args.normalize
    print(json.dumps({k: v for k, v in summary.items() if k != "history"}))
    if args.save:
        ppo.save(args.save)
    if args.out:
        Path(args.out).write_text(json.dumps(summary, indent=1))


if __name__ == "__main__":
    main()
