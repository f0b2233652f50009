#!/usr/bin/env python3
"""CLI of tennisbot_rl_b200.sac_population: a population of SAC agents in one env batch, optionally with PBT.

    python tools/train_sac_population.py SwingRacket-v0 --agents 4 --envs-per-agent 1024 --iters 5000
    python tools/train_sac_population.py SwingRacket-v0 --agents 8 --pbt-interval 500 --out pop.npz
    python tools/train_sac_population.py SwingRacket-v0 --throughput

Prints the card's name, power limit and SM clock, then per-agent curves (mean training return of the episodes that ended in
each collection), per-agent deterministic evaluations and the PBT events.  --out saves PopulationSAC.state_dict().
--throughput instead measures, in the same run:
  - the update graph's time per gradient step (CUDA events over replays) at P = 1, 2, 4, 8, 16 agents, batch 1 024 per agent,
    next to GpuSAC's at batch 1 024;
  - the collection time per env step (tb_sac_rollout in TB_SAC_SAMPLE, CUDA events) with P = --agents actors (16 by default
    here) against one actor over the same envs, at 16 384 and 65 536 envs: the cost of the per-agent image loads.  A CTA of
    sac_kernel reloads an image inside its loop only when its chunk of tiles spans two agents, which never happens when the
    tiles fit the SMs or when P divides the CTA count (4 on 148 SMs, for example); the output gives, per size, the CTAs
    that reload ("reloading_ctas"), so a comparison without reloads is visible as such.
"""
import argparse
import json
import subprocess
import sys
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
from tennisbot_rl_b200.batch import TennisBatch  # noqa: E402
from tennisbot_rl_b200.sac import GpuSAC, SacActor, pack_sac_actor  # noqa: E402
from tennisbot_rl_b200.sac_population import PopulationSAC  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[torch.cuda.current_device()] if q else torch.cuda.get_device_name()


def graph_ms(graph, reps=200, warm=20):
    for _ in range(warm):
        graph.replay()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ev[0].record()
    for _ in range(reps):
        graph.replay()
    ev[1].record()
    torch.cuda.synchronize()
    return ev[0].elapsed_time(ev[1]) / reps


def update_ms(env_id, agents_list):
    out = {}
    s = GpuSAC(env_id, num_envs=1024, slots=64)
    s.collect()
    s.update()
    out["GpuSAC"] = graph_ms(s.update_graph)
    s.env.close()
    del s
    for P in agents_list:
        pop = PopulationSAC(env_id, P, 1024, slots=64)
        pop.collect()
        pop.update()
        out[f"P={P}"] = graph_ms(pop.update_graph)
        pop.env.close()
        del pop
        torch.cuda.empty_cache()
    return out


def reloading_ctas(N, P):
    """CTAs of sac_kernel's grid (min(tiles, SMs), CTA b running tiles [tiles b / G, tiles (b + 1) / G)) whose chunk spans
    two agents of N / P envs: the ones that reload an image inside their loop."""
    tiles, per_agent = N // 128, N // P // 128
    G = min(tiles, torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count)
    return sum(1 for b in range(G) if (tiles * b // G) // per_agent != (tiles * (b + 1) // G - 1) // per_agent)


def collect_ms_per_step(env_id, N, P, K=8, reps=5):
    """ms per env step of tb_sac_rollout(K, SAMPLE) over N envs with P actors and with one; runs alternate."""
    od, ad = (6, 6) if env_id == "SwingRacket-v0" else (12, 2)
    torch.manual_seed(0)
    row = pack_sac_actor(SacActor(od, ad)).cuda()
    setups = {}
    for key in ("one actor", f"{P} actors"):
        b = TennisBatch(env_id, N, seed=1)
        if key == "one actor":
            b.set_sac_actor(row)
        else:
            b.set_sac_actors((row + 1e-3 * torch.randn(P, row.numel(), device="cuda")).contiguous())
        b.sac_begin()
        setups[key] = b
    times = {k: [] for k in setups}
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    for r in range(reps + 1):
        for k, b in setups.items():
            ev[0].record()
            b.sac_rollout(K, "sample", None, noise_seed=2)
            ev[1].record()
            torch.cuda.synchronize()
            if r:  # the first round warms up
                times[k].append(ev[0].elapsed_time(ev[1]) / K)
    for b in setups.values():
        b.close()
    out = {k: sorted(v)[len(v) // 2] for k, v in times.items()}
    out["reloading_ctas"] = reloading_ctas(N, P)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("env", nargs="?", default="SwingRacket-v0")
    ap.add_argument("--agents", type=int, default=None, help="4 for training, 16 for --throughput")
    ap.add_argument("--envs-per-agent", type=int, default=1024)
    ap.add_argument("--iters", type=int, default=5000)
    ap.add_argument("--pbt-interval", type=int, default=None)
    ap.add_argument("--eval-every", type=int, default=1000)
    ap.add_argument("--precision", default="f64")
    ap.add_argument("--throughput", action="store_true")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if a.agents is None:
        a.agents = 16 if a.throughput else 4
    print("card:", card(), flush=True)
    if a.throughput:
        res = {"card": card(), "update_ms_per_gradient_step": update_ms(a.env, (1, 2, 4, 8, 16))}
        print(json.dumps(res), flush=True)
        res["collect_ms_per_env_step"] = {str(N): collect_ms_per_step(a.env, N, a.agents) for N in (16384, 65536)}
        res["card_after"] = card()
        print(json.dumps(res), flush=True)
        return
    pop = PopulationSAC(a.env, a.agents, a.envs_per_agent, pbt_interval=a.pbt_interval, precision=a.precision)
    out = pop.train(a.iters, log=lambda m: print(m, flush=True), eval_every=a.eval_every)
    for p in out["per_agent"]:
        print(f"agent seed {p['seed']}: evaluations {[round(v, 2) for v in p['evaluations']]}")
    print(json.dumps({k: v for k, v in out.items() if k != "per_agent"} |
                     {"per_agent": [{k: v for k, v in p.items() if k != "history"} for p in out["per_agent"]]}))
    if a.out:
        pop.save(a.out)


if __name__ == "__main__":
    main()
