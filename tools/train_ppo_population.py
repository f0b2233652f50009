#!/usr/bin/env python3
"""CLI of tennisbot_rl_b200.population: a population of PPO agents in one env batch, optionally with PBT.

    python tools/train_ppo_population.py SwingRacket-v0 --agents 4 --envs-per-agent 4096 --iters 25
    python tools/train_ppo_population.py Tennisbot-v0 --agents 8 --envs-per-agent 16384 --rollout-len 128 --iters 60 --pbt 10
    python tools/train_ppo_population.py SwingRacket-v0 --throughput
    python tools/train_ppo_population.py Tennisbot-v0 --agents 8 --envs-per-agent 16384 --throughput --normalize

Prints the card's name and power limit, then per-agent curves (mean training return of the episodes that ended in each
rollout; raw returns with --normalize, which gives every agent its own VecNormalize record).  --throughput instead times, at
16 384 envs per agent, for P in 1, 4, 8:
  - the wall time of one population update (rollout + update, synchronised host clock) against P GpuPPO updates in turn;
  - the rollout time per env step (CUDA events) of P policies against one policy over the same P x 16 384 envs;
and the rollout time per step at 16 384 envs when agents straddle the 128-env CTAs of policy_kernel.
--throughput --normalize times the rollout per env step over --agents x --envs-per-agent envs with P policies and P training
records, with P policies and no normaliser, and with one policy and one training record; the same two normalised setups with
frozen records give the cost of the statistics pass per step (training minus frozen), segmented and with one record.
"""
import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
from tennisbot_rl_b200.batch import TennisBatch  # noqa: E402
from tennisbot_rl_b200.population import PopulationPPO  # noqa: E402
from tennisbot_rl_b200.ppo import ActorCritic, GpuPPO  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[torch.cuda.current_device()] if q else torch.cuda.get_device_name()


def wall_per_update(step, warm=2, reps=3):
    for _ in range(warm):  # the first update captures the graphs
        step()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(reps):
        step()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) / reps


def rollout_ms_per_step(env_id, N, agents_list, K, reps=5):
    """{key: ms per env step} of tb_policy_rollout over N envs; runs alternate.  agents_list: agents (0 meaning set_policy),
    or (key, agents, records, training) tuples that also attach a normaliser of `records` records (0: none)."""
    od, ad = (6, 6) if env_id == "SwingRacket-v0" else (12, 2)
    torch.manual_seed(0)
    row = ActorCritic(od, ad).packed().cuda()
    setups = {}
    for spec in agents_list:
        key, a, rec, training = spec if isinstance(spec, tuple) else (spec, spec, 0, True)
        b = TennisBatch(env_id, N, seed=1)
        if a:
            b.set_policies((row + 1e-3 * torch.randn(a, row.numel(), device="cuda")).contiguous())
        else:
            b.set_policy(row)
        if rec:
            b.set_vecnorm(training=training, agents=rec)
        z = lambda *s: torch.zeros(s, device="cuda")  # noqa: E731
        bufs = dict(obs=z(K, N, od), rew=z(K, N), done=torch.zeros((K, N), dtype=torch.uint8, device="cuda"), last=z(N, od),
                    act=z(K, N, ad), logp=z(K, N), val=z(K, N), lv=z(N))
        bufs["obs"][0].copy_(b.reset())
        setups[key] = (b, bufs)
    times = {a: [] for a in setups}
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    for r in range(reps + 1):
        for a, (b, q) in setups.items():
            ev[0].record()
            b.policy_rollout(q["obs"], q["rew"], q["done"], q["last"], actions=q["act"], logp=q["logp"], value=q["val"],
                             last_value=q["lv"], noise_seed=2)
            ev[1].record()
            q["obs"][0].copy_(q["last"])
            torch.cuda.synchronize()
            if r:  # the first round warms up
                times[a].append(ev[0].elapsed_time(ev[1]) / K)
    for b, _ in setups.values():
        b.close()
    return {a: sorted(t)[len(t) // 2] for a, t in times.items()}


def throughput(args, log):
    n, K = 16384, args.rollout_len
    out = {"card": card(), "env": args.env, "envs_per_agent": n, "rollout_len": K, "updates": [], "rollout": [], "straddle": {}}
    log(f"card: {out['card']}")
    for P in (1, 4, 8):
        pop = PopulationPPO(args.env, P, n, K, seeds=list(range(P)))
        t_pop = wall_per_update(lambda: (pop.rollout(), pop.update()))
        pop.env.close()
        del pop
        seq = [GpuPPO(args.env, n, K, seed=p) for p in range(P)]
        t_seq = wall_per_update(lambda: [(g.rollout(), g.update()) for g in seq])
        for g in seq:
            g.env.close()
        del seq
        torch.cuda.empty_cache()
        r = rollout_ms_per_step(args.env, P * n, [0, P] if P > 1 else [0], K)
        rec = {"agents": P, "population_update_s": t_pop, "sequential_updates_s": t_seq, "speedup": t_seq / t_pop}
        out["updates"].append(rec)
        out["rollout"].append({"agents": P, "envs": P * n, "one_policy_ms_per_step": r[0], "population_ms_per_step": r.get(P)})
        log(f"P={P}: population update {t_pop * 1e3:8.1f} ms, {P} GpuPPO updates {t_seq * 1e3:8.1f} ms ({t_seq / t_pop:.2f}x); "
            f"rollout per step one policy {r[0] * 1e3:7.1f} us, population {r.get(P, r[0]) * 1e3:7.1f} us")
    s = rollout_ms_per_step(args.env, n, [0, 128, 256, n], K)
    out["straddle"] = {"envs": n, "ms_per_step": {str(k): v for k, v in s.items()}}
    log("rollout per step at 16384 envs: " + ", ".join(f"{'one policy' if a == 0 else f'{a} agents ({n // a} envs each)'} "
                                                      f"{v * 1e3:.1f} us" for a, v in s.items()))
    return out


def throughput_normalize(args, log):
    P, n, K = args.agents, args.envs_per_agent, args.rollout_len
    out = {"card": card(), "env": args.env, "agents": P, "envs_per_agent": n, "rollout_len": K}
    log(f"card: {out['card']}")
    r = rollout_ms_per_step(args.env, P * n, [("records", P, P, True), ("none", P, 0, True), ("one", 0, 1, True),
                                              ("records_frozen", P, P, False), ("one_frozen", 0, 1, False)], K)
    out["ms_per_step"] = r
    out["stats_pass_ms_per_step"] = {"segmented": r["records"] - r["records_frozen"], "one_record": r["one"] - r["one_frozen"]}
    log(f"{P} x {n} envs, rollout per step: {P} policies with {P} records {r['records'] * 1e3:.1f} us, without a normaliser "
        f"{r['none'] * 1e3:.1f} us, one policy with one record {r['one'] * 1e3:.1f} us; statistics pass per step (training - "
        f"frozen): segmented {out['stats_pass_ms_per_step']['segmented'] * 1e3:.1f} us, one record "
        f"{out['stats_pass_ms_per_step']['one_record'] * 1e3:.1f} us")
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("env", choices=("SwingRacket-v0", "Tennisbot-v0"))
    ap.add_argument("--agents", type=int, default=4)
    ap.add_argument("--envs-per-agent", type=int, default=4096)
    ap.add_argument("--rollout-len", type=int, default=None, help="default: 26 (SwingRacket-v0's episode) / 128")
    ap.add_argument("--iters", type=int, default=25)
    ap.add_argument("--seed", type=int, default=1, help="agent p starts from GpuPPO(seed=seed + p)'s weights")
    ap.add_argument("--pbt", type=int, default=None, metavar="INTERVAL", help="a PBT round every INTERVAL updates")
    ap.add_argument("--pbt-seed", type=int, default=0)
    ap.add_argument("--precision", default="f64")
    ap.add_argument("--save", default=None, help="npz of PopulationPPO.state_dict()")
    ap.add_argument("--out", default=None, help="JSON of the result")
    ap.add_argument("--throughput", action="store_true")
    ap.add_argument("--normalize", action="store_true", help="one VecNormalize record per agent")
    args = ap.parse_args()
    if args.rollout_len is None:
        args.rollout_len = 26 if args.env == "SwingRacket-v0" else 128
    log = lambda m: print(m, flush=True)  # noqa: E731
    if args.throughput:
        res = throughput_normalize(args, log) if args.normalize else throughput(args, log)
    else:
        log(f"card: {card()}")
        pop = PopulationPPO(args.env, args.agents, args.envs_per_agent, args.rollout_len,
                            seeds=[args.seed + p for p in range(args.agents)], precision=args.precision, pbt_interval=args.pbt,
                            pbt_seed=args.pbt_seed, normalize=args.normalize)
        res = pop.train(args.iters, log=log)
        res["card"] = card()
        for a in res["per_agent"]:
            curve = " ".join("-" if h["mean_return"] is None else f"{h['mean_return']:.1f}" for h in a["history"])
            log(f"seed {a['seed']}: final {a['final_mean_return']} best {a['best_mean_return']}\n  {curve}")
        log(f"hyper-parameters: {json.dumps(res['hyper'])}")
        log(f"wall {res['wall_s']:.1f} s, rollouts {res['rollout_s']:.1f} s, {len(res['pbt_events'])} PBT events")
        if args.save:
            pop.save(args.save)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
