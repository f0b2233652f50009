"""A population of SAC agents trained in one env batch, with population-based training (PBT).

PopulationSAC(env_id, P, n) holds one TennisBatch of P x n envs; env i acts with actor i // n (tb_set_sac_actors), so one
tb_sac_rollout collects the transitions of every agent into one replay ring, in which agent p owns columns [p n, (p + 1) n)
of every slot.  The learner is GpuSAC's gradient step, run for all agents at once: every tensor carries a leading agent
dimension and goes through batched matmuls, each agent samples its batch from its own columns, and every mean of the losses
is taken per agent, so agent p's update depends on agent p's transitions only.  lr, tau and gamma live in [P] device tensors
that the captured update graph reads, so PBT changes them in place.
"""
import math
import time

import numpy as np
import torch

from . import _lib
from .batch import TennisBatch
from .population import BatchedAdam, agent_values, episode_stats, exploit_explore
from .sac import LOG_STD_MAX, LOG_STD_MIN, SAC_FLOATS_BY_DIMS, SacActor, TwinCritic

HYPER_DEFAULTS = {"lr": 3e-4, "tau": 0.005, "gamma": 0.99}  # GpuSAC's
PBT_PERTURBED = ("lr", "tau")


def _linears(module):
    return [t for m in module.modules() if isinstance(m, torch.nn.Linear) for t in (m.weight, m.bias)]


def _stack(per_agent, device, grad):
    """[agent][tensor] -> one stacked tensor per position, with a leading agent dimension."""
    out = [torch.stack([a[i].detach() for a in per_agent]).to(device) for i in range(len(per_agent[0]))]
    return [t.requires_grad_() for t in out] if grad else out


def initial_agents(obs_dim, act_dim, seeds):
    """Per seed, the (actor, critic, critic target) GpuSAC(seed=s) starts from, built with its order of RNG draws: after
    torch.manual_seed(s), the actor, the critic, then the target (whose own draws are overwritten by the critic's weights)."""
    out = []
    for s in seeds:
        torch.manual_seed(int(s))
        actor, critic = SacActor(obs_dim, act_dim), TwinCritic(obs_dim, act_dim)
        target = TwinCritic(obs_dim, act_dim)
        target.load_state_dict(critic.state_dict())
        out.append((actor, critic, target))
    return out


def _linear(x, W, b):  # x [P, B, in], W [P, out, in], b [P, out] -> [P, B, out]
    return torch.baddbmm(b.unsqueeze(1), x, W.transpose(1, 2))


class BatchedSacActor:
    """P SacActors stacked: tensors in pack_sac_actor's order (latent_pi.0 W, b, latent_pi.2 W, b, mu W, b, log_std W, b),
    each [P, ...]."""

    def __init__(self, actors, device="cpu"):
        self.agents = len(actors)
        self.obs_dim, self.act_dim = actors[0].latent_pi[0].in_features, actors[0].mu.out_features
        self.params = _stack([_linears(a) for a in actors], device, grad=True)

    def dist(self, obs):  # obs [P, B, obs_dim] -> (mean, clamped log_std) [P, B, act_dim]
        W1, b1, W2, b2, Wm, bm, Wl, bl = self.params
        h = _linear(_linear(obs, W1, b1).relu(), W2, b2).relu()
        return _linear(h, Wm, bm), _linear(h, Wl, bl).clamp(LOG_STD_MIN, LOG_STD_MAX)

    def packed(self):
        """float32 [P, sac_floats]: row p is pack_sac_actor of agent p (tb_set_sac_actors' rows)."""
        rows = []
        for t in self.params:
            t = t.detach().reshape(self.agents, -1).to(torch.float32)
            r = (-t.shape[1]) % 4
            rows += [t] if r == 0 else [t, t.new_zeros(self.agents, r)]
        out = torch.cat(rows, 1)
        assert out.shape[1] == SAC_FLOATS_BY_DIMS[(self.obs_dim, self.act_dim)], out.shape
        return out


class BatchedTwinCritic:
    """P TwinCritics stacked: qf0's (W, b) x 3, then qf1's, each [P, ...].  grad=False: a target, updated by polyak()."""

    def __init__(self, critics, device="cpu", grad=True):
        self.agents = len(critics)
        self.params = _stack([_linears(c) for c in critics], device, grad=grad)

    def __call__(self, obs, act):  # -> (q0, q1), each [P, B, 1]
        x = torch.cat([obs, act], -1)
        out = []
        for q in range(2):
            W1, b1, W2, b2, W3, b3 = self.params[6 * q:6 * q + 6]
            out.append(_linear(_linear(_linear(x, W1, b1).relu(), W2, b2).relu(), W3, b3))
        return tuple(out)

    @torch.no_grad()
    def polyak(self, source, tau):
        """target <- (1 - tau[p]) target + tau[p] source, per agent (GpuSAC's lerp_ with agent p's tau)."""
        for tp, p in zip(self.params, source.params):
            tp.lerp_(p, tau.view((-1,) + (1,) * (p.dim() - 1)))


def batched_sac_losses(actor, critic, critic_target, log_alpha, batch, gamma, target_entropy, noise, next_noise):
    """sac.sac_losses for every agent: batch (obs, act, reward, next_obs, done) with a leading agent dimension [P, B, ...],
    log_alpha and gamma [P], noise [P, B, act_dim].  Returns (alpha_loss [P], critic_loss [P], pi, logp, alpha [P]), each loss
    a per-agent mean."""
    obs, act, rew, nxt, done = batch
    mu, ls = actor.dist(obs)
    u = mu + ls.exp() * noise
    pi, logp = torch.tanh(u), SacActor.log_prob(mu, ls, u)          # logp [P, B]
    alpha = log_alpha.detach().exp()
    alpha_loss = -(log_alpha.unsqueeze(1) * (logp + target_entropy).detach()).mean(1)
    with torch.no_grad():
        nmu, nls = actor.dist(nxt)
        nu = nmu + nls.exp() * next_noise
        nq = torch.min(*critic_target(nxt, torch.tanh(nu))) - alpha.view(-1, 1, 1) * SacActor.log_prob(nmu, nls, nu).unsqueeze(-1)
        target = rew.unsqueeze(-1) + (1.0 - done.unsqueeze(-1)) * gamma.view(-1, 1, 1) * nq
    q0, q1 = critic(obs, act)
    critic_loss = 0.5 * ((q0 - target).pow(2).mean((1, 2)) + (q1 - target).pow(2).mean((1, 2)))
    return alpha_loss, critic_loss, pi, logp, alpha


def batched_actor_loss(critic, obs, pi, logp, alpha):
    """sac.actor_loss for every agent: [P]."""
    return (alpha.unsqueeze(1) * logp - torch.min(*critic(obs, pi)).squeeze(-1)).mean(1)


class PopulationSAC:
    """agents SAC learners, each on its own envs_per_agent envs of one TennisBatch, updated together.  lr, tau and gamma are
    each a scalar for every agent or one value per agent.  Agent p starts from the actor, critic and target GpuSAC(seed=seeds[p])
    starts from and takes GpuSAC's gradient step on batch_size transitions drawn from its own filled ring rows: SB3's alpha,
    critic and actor losses, three Adams (eps 1e-8) stepped in SB3's order, and Polyak averaging with its own tau.  The context's
    env seed is seeds[0] and the actor noise seed seeds[0] + 1.  pbt_interval: run exploit_explore() after every pbt_interval
    iterations (None: never)."""

    def __init__(self, env_id="SwingRacket-v0", agents=4, envs_per_agent=1024, steps=1, batch_size=1024, gradient_steps=8,
                 slots=1024, seeds=None, lr=3e-4, tau=0.005, gamma=0.99, learning_starts=100, pbt_interval=None, pbt_seed=0,
                 eval_envs=1024, precision="f64", device=0):
        P = self.P = int(agents)
        if P < 1:
            raise ValueError(f"agents must be >= 1, got {agents}")
        self.seeds = list(range(P)) if seeds is None else [int(s) for s in agent_values("seeds", seeds, P)]
        values = {k: agent_values(k, v, P) for k, v in dict(lr=lr, tau=tau, gamma=gamma).items()}
        if pbt_interval is not None and (int(pbt_interval) < 1 or P < 2):
            raise ValueError("pbt_interval needs at least 2 agents and must be >= 1")
        n = int(envs_per_agent)
        if P > 1 and (n < 1 or n % 128):
            raise ValueError(f"envs_per_agent must be a multiple of 128 with more than one agent (a tile of the in-kernel actor "
                             f"holds one actor), got {n}")
        if P > 1 and int(eval_envs) % 128:
            raise ValueError(f"eval_envs must be a multiple of 128 with more than one agent, got {eval_envs}")
        self.pbt_interval, self.pbt_rng, self.pbt_log = pbt_interval, np.random.default_rng(pbt_seed), []
        self.env_id, self.dev = env_id, torch.device("cuda", device)
        self.n, self.K, self.B, self.G, self.slots = n, int(steps), int(batch_size), int(gradient_steps), int(slots)
        self.N = N = P * n
        self.env = TennisBatch(env_id, N, device=device, seed=self.seeds[0], precision=precision)
        self.od, self.ad = od, ad = self.env.obs_dim, self.env.act_dim
        self.hyper = {k: torch.tensor(v, dtype=torch.float32, device=self.dev) for k, v in values.items()}
        init = initial_agents(od, ad, self.seeds)
        self.actor = BatchedSacActor([a for a, _, _ in init], self.dev)
        self.critic = BatchedTwinCritic([c for _, c, _ in init], self.dev)
        self.critic_target = BatchedTwinCritic([t for _, _, t in init], self.dev, grad=False)
        self.log_alpha = torch.zeros(P, device=self.dev, requires_grad=True)  # initial alpha 1
        self.target_entropy = -float(ad)
        adam = lambda ps: BatchedAdam(ps, self.hyper["lr"], eps=1e-8)  # noqa: E731  (torch.optim.Adam's eps, as GpuSAC)
        self.actor_opt, self.critic_opt, self.alpha_opt = adam(self.actor.params), adam(self.critic.params), adam([self.log_alpha])
        z = lambda *s, dt=torch.float32: torch.zeros(s, dtype=dt, device=self.dev)  # noqa: E731
        S = self.slots
        self.ring = dict(obs=z(S, N, od), act=z(S, N, ad), reward=z(S, N), next_obs=z(S, N, od), done=z(S, N, dt=torch.uint8))
        self.flat = {k: v.view(S * N, *v.shape[2:]) for k, v in self.ring.items()}
        self.fill = z(1)           # filled rows of each agent's columns (a device scalar the update graph reads)
        self.steps_taken = 0       # env steps of every env since sac_begin
        self.ep_ret = torch.zeros(N, dtype=torch.float64, device=self.dev)  # return / length of each env's episode in progress
        self.ep_len = torch.zeros(N, dtype=torch.float64, device=self.dev)
        self.params = z(P, SAC_FLOATS_BY_DIMS[(od, ad)])
        self.params.copy_(self.actor.packed())
        self.env.set_sac_actors(self.params)  # (allocates the library's images outside the graph capture)
        self.env.sac_begin()
        warm = max(1, math.ceil(learning_starts / n))  # per agent, as GpuSAC(num_envs=n) counts it
        self.env.sac_rollout(warm, "uniform", self.ring, noise_seed=self.seeds[0] + 1)
        self.steps_taken += warm
        self._episode_stats(warm)  # the warm-up's episodes are not reported, but the ones in progress carry on
        self.collect_graph = self.update_graph = None
        self.losses = z(3, P)
        self.collect_s = self.update_s = 0.0
        self.eval_envs, self.precision = int(eval_envs), precision
        self._eval = None
        self._interval = np.zeros((2, P))  # return sum, episodes since the last PBT round
        self.iters = 0

    # ------------------------------------------------------------------ collection
    def _collect_body(self):
        self.params.copy_(self.actor.packed())
        self.env.set_sac_actors(self.params)
        self.env.sac_rollout(self.K, "sample", self.ring, noise_seed=self.seeds[0] + 1)

    def _episode_stats(self, k):
        """Per-agent episodes that ended in the last k env steps, read back from the ring slots they went to."""
        slots = torch.arange(self.steps_taken - k, self.steps_taken, device=self.dev) % self.slots
        return episode_stats(self.ring["reward"][slots], self.ring["done"][slots], self.ep_ret, self.ep_len, self.P)

    @torch.no_grad()
    def collect(self):
        """steps env steps of every env into the ring.  Returns (per-agent episodes int64 [P], return sums float64 [P], length
        sums float64 [P]) of the episodes that ended in it, as numpy."""
        if self.collect_graph is None:
            self.collect_graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.collect_graph):
                self._collect_body()
        self.collect_graph.replay()
        self.steps_taken += self.K
        return tuple(x.cpu().numpy() for x in self._episode_stats(self.K))

    # ------------------------------------------------------------------ update
    def sample(self):
        """batch_size ring rows per agent, uniform over agent p's filled rows slot * N + p n + j: int64 [P, batch_size]."""
        k = (torch.rand(self.P, self.B, device=self.dev) * self.fill).long()  # GpuSAC's draw, over n columns per slot
        agent = torch.arange(self.P, device=self.dev).unsqueeze(1) * self.n
        return (k // self.n) * self.N + agent + k % self.n

    def _gather(self, idx):
        f, shape = self.flat, idx.shape
        take = lambda x: x[idx.reshape(-1)].view(*shape, *x.shape[1:])  # noqa: E731
        return take(f["obs"]), take(f["act"]), take(f["reward"]), take(f["next_obs"]), take(f["done"]).float()

    def gradient_step(self, batch, noise, next_noise):
        """GpuSAC._grad_step for every agent on batch [P, B, ...] with the Gaussian draws given."""
        a_loss, c_loss, pi, logp, alpha = batched_sac_losses(self.actor, self.critic, self.critic_target, self.log_alpha, batch,
                                                             self.hyper["gamma"], self.target_entropy, noise, next_noise)
        # SB3's order: alpha, then the critics, then the actor (its loss reads the updated critics).  Agents share no
        # parameter, so the sum over agents gives each the gradient of its own loss.
        for opt, loss in ((self.alpha_opt, a_loss), (self.critic_opt, c_loss)):
            _zero_grads(opt.params)
            loss.sum().backward()
            opt.step()
        pi_loss = batched_actor_loss(self.critic, batch[0], pi, logp, alpha)
        _zero_grads(self.actor_opt.params)
        pi_loss.sum().backward()
        self.actor_opt.step()
        self.critic_target.polyak(self.critic, self.hyper["tau"])
        with torch.no_grad():
            self.losses.copy_(torch.stack([a_loss.detach(), c_loss.detach(), pi_loss.detach()]))

    def _grad_step(self):
        self.gradient_step(self._gather(self.sample()), torch.randn(self.P, self.B, self.ad, device=self.dev),
                           torch.randn(self.P, self.B, self.ad, device=self.dev))

    def _state(self):
        return (self.actor.params + self.critic.params + self.critic_target.params + [self.log_alpha] +
                self.actor_opt.state_tensors() + self.critic_opt.state_tensors() + self.alpha_opt.state_tensors())

    def update(self):
        self.fill.fill_(float(min(self.steps_taken, self.slots) * self.n))
        if self.update_graph is None:
            # warm-up steps are real updates: take them on a snapshot and put everything back, so the graph trains like the
            # eager path (capture itself executes nothing)
            state = self._state()
            snap = [t.detach().clone() for t in state]
            s = torch.cuda.Stream(self.dev)
            s.wait_stream(torch.cuda.current_stream(self.dev))
            with torch.cuda.stream(s):
                for _ in range(3):
                    self._grad_step()
            torch.cuda.current_stream(self.dev).wait_stream(s)
            self.update_graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.update_graph):
                self._grad_step()
            with torch.no_grad():
                for t, v in zip(state, snap):
                    t.copy_(v)
        for _ in range(self.G):
            self.update_graph.replay()

    # ------------------------------------------------------------------ PBT
    def exploit_explore(self, scores=None):
        """One PBT round (population.exploit_explore) on actor, critic, target, log_alpha, the moments and step counts of the
        three Adams, and lr / tau / gamma; lr and tau are perturbed.  Ring columns are not copied: the copy goes on learning
        off-policy from its own columns.  scores: None ranks by the mean training return since the previous round.  The events
        are appended to pbt_log as (iteration, destination, source, new hyper-parameters) and returned."""
        if scores is None:
            r, e = self._interval
            scores = [float(r[p] / e[p]) if e[p] else None for p in range(self.P)]
        ev = exploit_explore(scores, self._state(), self.hyper, self.pbt_rng, perturbed=PBT_PERTURBED)
        ev = [(self.iters, dst, src, hp) for dst, src, hp in ev]
        self.pbt_log += ev
        self._interval[:] = 0
        return ev

    # ------------------------------------------------------------------ training and evaluation
    def train(self, iters, log=None, eval_every=0, eval_episodes=1):
        """iters x (collection, gradient_steps gradient steps, and a PBT round every pbt_interval iterations).  Per agent and
        iteration: the episodes that ended in its collection and their mean return (None when none ended); per agent the
        deterministic evaluations taken every eval_every iterations and after the last."""
        P, t0 = self.P, time.time()
        hist, evals = [[] for _ in range(P)], []
        for it in range(iters):
            torch.cuda.synchronize()
            t1 = time.time()
            eps, rsum, _ = self.collect()
            torch.cuda.synchronize()
            t2 = time.time()
            self.update()
            torch.cuda.synchronize()
            self.collect_s += t2 - t1
            self.update_s += time.time() - t2
            self.iters += 1
            self._interval += np.stack([rsum, eps])
            if it % 50 == 0 or it == iters - 1:  # the per-agent curves, thinned to keep the history small
                for p in range(P):
                    e = int(eps[p])
                    hist[p].append({"iter": it, "env_steps": self.steps_taken * self.n, "episodes": e,
                                    "mean_return": float(rsum[p] / e) if e else None, "lr": float(self.hyper["lr"][p]),
                                    "tau": float(self.hyper["tau"][p])})
            if self.pbt_interval and self.iters % self.pbt_interval == 0:
                for ev in self.exploit_explore():
                    if log:
                        log(f"pbt iter {ev[0]}: agent {ev[1]} <- agent {ev[2]}, lr {ev[3]['lr']:.3g} tau {ev[3]['tau']:.3g}")
            if (eval_every and (it + 1) % eval_every == 0) or it == iters - 1:
                evals.append({"iter": it, "env_steps": self.steps_taken * self.n, "eval_mean_return": self.evaluate(eval_episodes)})
            if log and (it % 500 == 0 or it == iters - 1):
                rets = " ".join("   -   " if not eps[p] else f"{rsum[p] / eps[p]:7.2f}" for p in range(P))
                log(f"iter {it:5d} returns {rets} alpha {' '.join(f'{a:.4f}' for a in self.log_alpha.exp().tolist())} "
                    f"wall {time.time() - t0:6.1f}s")
        per_agent = []
        for p in range(P):
            per_agent.append({"seed": self.seeds[p], "evaluations": [e["eval_mean_return"][p] for e in evals],
                              "eval_mean_return": evals[-1]["eval_mean_return"][p] if evals else None, "history": hist[p]})
        return {"env": self.env_id, "agents": P, "envs_per_agent": self.n, "steps": self.K, "batch_size": self.B,
                "gradient_steps": self.G, "slots": self.slots, "iters": iters, "wall_s": time.time() - t0,
                "collect_s": self.collect_s, "update_s": self.update_s, "evaluations": evals,
                "hyper": {k: v.tolist() for k, v in self.hyper.items()},
                "pbt_events": [list(e[:3]) + [e[3]] for e in self.pbt_log], "per_agent": per_agent}

    @torch.no_grad()
    def evaluate(self, episodes=1):
        """Per agent, GpuSAC.evaluate: the mean return of `episodes` whole episodes per env of eval_envs envs with the
        deterministic action tanh(mu), on a context of its own of P x eval_envs envs (set_sac_actors), so training's envs and
        ring are untouched.  Episodes are counted per agent from a small ring of one chunk of steps.  Returns P floats."""
        P, M = self.P, self.P * self.eval_envs
        if self._eval is None:
            e = TennisBatch(self.env_id, M, device=self.dev.index, seed=self.seeds[0] + 1000, precision=self.precision)
            chunk = 26 if e.kind == _lib.ENV_SWING else 100
            z = lambda *s, dt=torch.float32: torch.zeros(s, dtype=dt, device=self.dev)  # noqa: E731
            ring = dict(obs=z(chunk, M, self.od), act=z(chunk, M, self.ad), reward=z(chunk, M), next_obs=z(chunk, M, self.od),
                        done=z(chunk, M, dt=torch.uint8))
            self._eval = (e, chunk, ring)
        e, chunk, ring = self._eval
        e.set_sac_actors(self.actor.packed().contiguous())
        e.sac_begin()
        carry = torch.zeros(2, M, dtype=torch.float64, device=self.dev)
        count, total = np.zeros(P, np.int64), np.zeros(P)
        while (count < episodes * self.eval_envs).any():  # sac_begin starts the ring at slot 0: each chunk fills it in order
            e.sac_rollout(chunk, "mean", ring, noise_seed=0)
            c, r, _ = episode_stats(ring["reward"], ring["done"], carry[0], carry[1], P)
            count += c.cpu().numpy()
            total += r.cpu().numpy()
        return [float(total[p] / count[p]) for p in range(P)]

    # ------------------------------------------------------------------ saving
    PBT_COLUMNS = ("iteration", "destination", "source") + tuple(HYPER_DEFAULTS)

    def state_dict(self):
        """numpy arrays: `actors` [P, sac_floats] (tb_set_sac_actors' rows), `seeds`, one [P] array per hyper-parameter, and
        `pbt_events` [E, len(PBT_COLUMNS)] float64 with the column names in `pbt_columns`."""
        out = {"actors": self.actor.packed().cpu().numpy(), "seeds": np.array(self.seeds)}
        out.update({k: v.cpu().numpy() for k, v in self.hyper.items()})
        out["pbt_events"] = np.array([[i, d, s] + [hp[k] for k in HYPER_DEFAULTS] for i, d, s, hp in self.pbt_log],
                                     np.float64).reshape(-1, len(self.PBT_COLUMNS))
        out["pbt_columns"] = np.array(self.PBT_COLUMNS)
        return out

    def save(self, path):
        np.savez(path, **self.state_dict())

    def agent_state_dict(self, p):
        """Agent p in GpuSAC.state_dict()'s layout ({"policy": tb_set_sac_actor's vector}): deploy it with set_sac_actor."""
        return {"policy": self.actor.packed()[p].cpu().numpy()}


def _zero_grads(params):
    for p in params:  # grads stay in place: the captured graph refers to their storage
        if p.grad is not None:
            p.grad.zero_()
