"""Where the time of a policy rollout goes at a given batch size.

SwingRacket-v0 (default): per-iteration time of the 26-step rollout while PPO trains (the workload changes as the policy
learns to hit the ball: longer flights, contact chains), and the per-kernel split of one rollout.
Tennisbot-v0: env-steps/s of the K-step rollout (CUDA graph replay, CUDA events) at each batch size, with the untrained
policy and with the weights of `iters` PPO updates at 16 384 envs, and the split: step_kernel time from the library's
per-step CUDA events (tb_set_kernel_timing, an eager run), the rest of the graph's time is policy_kernel and two copies.
--normalize: the cost of the device VecNormalize (tb_set_vecnorm): for both envs (SwingRacket-v0 K = 26, Tennisbot-v0
K = 128) and each batch size, the same policy rollout captured as two CUDA graphs, without and with a training normaliser,
replayed alternately in the same run (CUDA events); ms per rollout step of each and the difference.
usage: time_policy_rollout.py [n_envs] [iters]
       time_policy_rollout.py Tennisbot-v0 [iters] [K] [n_envs ...]      (default n_envs: 16384 1048576)
       time_policy_rollout.py --normalize [n_envs ...]                  (default n_envs: 16384 1048576)"""
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, ".")
from tennisbot_rl_b200.batch import TennisBatch  # noqa: E402
from tennisbot_rl_b200.ppo import EPISODE, ActorCritic, HitPPO, SwingPPO  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[torch.cuda.current_device()] if q else torch.cuda.get_device_name()


def time_hit(ppo, reps=10):
    """(env-steps/s of a graph replay, ms per rollout, of which step_kernel ms) - the rest is policy_kernel and two copies"""
    ppo.rollout()  # capture (and warm-up) outside the window
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(reps):
        ppo.graph.replay()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    # the same rollout issued eagerly with the library's per-step events around step_kernel (they synchronise every step,
    # so this run gives the step_kernel share, not the rate)
    ppo.env.set_kernel_timing(True)
    ppo.env.kernel_timing()
    with torch.no_grad():
        for _ in range(reps):
            ppo._rollout_body()
    torch.cuda.synchronize()
    step_ms, _, _ = ppo.env.kernel_timing()
    ppo.env.set_kernel_timing(False)
    return ppo.K * ppo.n / (ms * 1e-3), ms, step_ms / reps


def hit(argv):
    iters = int(argv[0]) if argv else 30
    K = int(argv[1]) if len(argv) > 1 else 128
    sizes = [int(a) for a in argv[2:]] or [16384, 1048576]
    print("card (name, power limit, max SM clock):", card(), flush=True)
    trainer = HitPPO(16384, rollout_len=K, seed=0)  # the "trained" weights: iters updates at 16 384 envs
    trainer.train(iters)
    trained = {k: v.clone() for k, v in trainer.ac.state_dict().items()}
    del trainer
    for n in sizes:
        ppo = HitPPO(n, rollout_len=K, seed=0)
        for label in ("untrained", f"after {iters} updates"):
            if label != "untrained":
                ppo.ac.load_state_dict(trained)  # in place: the captured graph packs the current weights on every replay
            rate, ms, step_ms = time_hit(ppo)
            st = ppo.rollout()
            eps = max(int(st[0]), 1)
            print(f"Tennisbot-v0 {n:8d} envs K={K} {label:>18s}: rollout {ms:8.3f} ms -> {rate:.3e} env-steps/s; per rollout "
                  f"step_kernel {step_ms:.3f} ms, policy_kernel + copies {ms - step_ms:.3f} ms; "
                  f"return {st[6] / 2 ** 20 / eps:.2f}, hits/ep {st[2] / eps:.3f}, episodes {int(st[0])}", flush=True)
        del ppo
        torch.cuda.empty_cache()


def swing(argv):
    n = int(argv[0]) if argv else 16384
    iters = int(argv[1]) if len(argv) > 1 else 100
    ppo = SwingPPO(num_envs=n, seed=0, use_graph=True, fused_policy=True)
    for it in range(iters):
        t0 = ppo.rollout_s
        st = ppo.rollout()
        dt = ppo.rollout_s - t0
        if it % 10 == 0 or it == iters - 1:
            eps = max(int(st[0]), 1)
            print("iter %3d rollout %.3f ms -> %.3e env-steps/s; return %.2f, mean episode length %.0f substeps, hits/ep %.2f" % (
                it, dt * 1e3, EPISODE * n / dt, st[6] / 2 ** 20 / eps, st[1] / eps, st[2] / eps), flush=True)
        ppo.update()
    # per-kernel split of one eager rollout with the trained policy (events inside the library, synchronised per step)
    ppo.env.set_kernel_timing(True)
    ppo.use_graph = False
    ppo.rollout()
    a, b, k = ppo.env.kernel_timing()
    print("trained policy, eager, timed per step: step_kernel %.3f ms + ff_kernel %.3f ms over %d steps" % (a, b, k))
    d = ppo.env.ff_diagnostics()
    print("last fast-forward: server visits %d, flights over after %.3f ms" % (d[1], d[2] * 1e-6))


def normalize_cost(argv, rounds=7, reps=5):
    sizes = [int(a) for a in argv] or [16384, 1048576]
    print("card (name, power limit, max SM clock):", card(), flush=True)
    for env_id, K in (("SwingRacket-v0", EPISODE), ("Tennisbot-v0", 128)):
        for n in sizes:
            torch.manual_seed(0)
            b = TennisBatch(env_id, n, seed=0)
            dev, od, ad = b.device, b.obs_dim, b.act_dim
            b.set_policy(ActorCritic(od, ad).to(dev).packed())
            z = lambda *s: torch.zeros(s, device=dev)  # noqa: E731
            obs, act, logp, val, rew, last, last_v = z(K, n, od), z(K, n, ad), z(K, n), z(K, n), z(K, n), z(n, od), z(n)
            done = torch.zeros((K, n), dtype=torch.uint8, device=dev)
            cur = b.reset().clone()

            def body():
                obs[0].copy_(cur)
                b.policy_rollout(obs, rew, done, last, actions=act, logp=logp, value=val, last_value=last_v, noise_seed=1)
                cur.copy_(last)

            graphs = {}
            for label in ("plain", "vecnorm"):  # a graph keeps the kernels it was captured with
                if label == "vecnorm":
                    b.set_vecnorm()
                s = torch.cuda.Stream(dev)
                s.wait_stream(torch.cuda.current_stream(dev))
                with torch.cuda.stream(s):
                    body()
                torch.cuda.current_stream(dev).wait_stream(s)
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    body()
                graphs[label] = g
            times = {k: [] for k in graphs}
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            for _ in range(rounds):
                for label, g in graphs.items():
                    g.replay()  # one untimed replay after the switch
                    e0.record()
                    for _ in range(reps):
                        g.replay()
                    e1.record()
                    torch.cuda.synchronize()
                    times[label].append(e0.elapsed_time(e1) / reps / K * 1e3)
            med = {k: statistics.median(v) for k, v in times.items()}
            spread = {k: (min(v), max(v)) for k, v in times.items()}
            print(f"{env_id} {n:8d} envs K={K}: per rollout step plain {med['plain']:9.2f} us "
                  f"[{spread['plain'][0]:.2f}, {spread['plain'][1]:.2f}], with vecnorm {med['vecnorm']:9.2f} us "
                  f"[{spread['vecnorm'][0]:.2f}, {spread['vecnorm'][1]:.2f}]: +{med['vecnorm'] - med['plain']:.2f} us "
                  f"({(med['vecnorm'] / med['plain'] - 1) * 100:+.1f} %); medians of {rounds} x {reps} replays", flush=True)
            del graphs
            b.close()
            torch.cuda.empty_cache()


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "--normalize":
        normalize_cost(sys.argv[2:])
    elif len(sys.argv) > 1 and sys.argv[1] in ("Tennisbot-v0", "hit"):
        hit(sys.argv[2:])
    else:
        swing(sys.argv[1:])
