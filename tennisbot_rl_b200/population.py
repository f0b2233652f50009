"""A population of PPO agents trained in one env batch, with population-based training (PBT; Jaderberg et al. 2017).

PopulationPPO(env_id, P, n, K) holds one TennisBatch of P x n envs; env i acts with agent i // n (tb_set_policies), so one
tb_policy_rollout collects the rollouts of every agent.  The learner is GpuPPO's update, run for all agents at once: the
parameters carry a leading agent dimension and go through batched matmuls, and every reduction of the loss (advantage
normalisation, means, gradient norm) is taken per agent, so agent p's update depends on agent p's samples only.  The
hyper-parameters live in [P] device tensors that the captured minibatch graph reads, so PBT changes them in place.
With normalize=True every agent trains under its own SB3 VecNormalize record (tb_set_vecnorms), which PBT copies with the
weights.
"""
import math
import time

import numpy as np
import torch

from .batch import TennisBatch
from .ppo import POLICY_FLOATS_BY_DIMS, ActorCritic, vecnormalize_entries

# GpuPPO's hyper-parameters and their defaults (the reference's SB3 settings, train_swing.py:80-91, and lr 3e-4)
HYPER_DEFAULTS = {"lr": 3e-4, "ent_coef": 0.002, "clip": 0.2, "vf_coef": 0.5, "max_grad_norm": 0.5, "gamma": 0.99,
                  "gae_lambda": 0.95}
PBT_PERTURBED = ("lr", "ent_coef")
PBT_FACTORS = (0.8, 1.2)


def agent_values(name, value, agents):
    """A hyper-parameter as P floats: a scalar is broadcast, a sequence must have length P."""
    if np.ndim(value) == 0:
        return [float(value)] * agents
    vals = [float(v) for v in value]
    if len(vals) != agents:
        raise ValueError(f"{name}: expected a scalar or {agents} values (one per agent), got {len(vals)}")
    return vals


def agent_tensors(ac):
    """ActorCritic's tensors in pack_policy's order: the pi tower's (W, b) x 3, action head, the vf tower's, value head,
    log_std."""
    lin = [m for m in ac.pi if isinstance(m, torch.nn.Linear)] + [ac.mu] + \
          [m for m in ac.vf if isinstance(m, torch.nn.Linear)] + [ac.v]
    return [t for m in lin for t in (m.weight, m.bias)] + [ac.log_std]


class BatchedActorCritic:
    """P ActorCritics stacked: every tensor of agent_tensors() with a leading agent dimension.  Agent p starts bit-identical
    to ActorCritic(obs_dim, act_dim) built right after torch.manual_seed(seeds[p]), as GpuPPO(seed=seeds[p]) builds it."""

    def __init__(self, obs_dim, act_dim, seeds, device="cpu"):
        acs = []
        for s in seeds:
            torch.manual_seed(int(s))
            acs.append(agent_tensors(ActorCritic(obs_dim, act_dim)))
        self.agents, self.obs_dim, self.act_dim = len(acs), obs_dim, act_dim
        self.params = [torch.stack([a[i].detach() for a in acs]).to(device).requires_grad_() for i in range(len(acs[0]))]

    def _tower(self, x, first):  # x [P, B, in] -> [P, B, 32]
        for i in range(first, first + 6, 2):
            W, b = self.params[i], self.params[i + 1]
            x = torch.tanh(torch.baddbmm(b.unsqueeze(1), x, W.transpose(1, 2)))
        return x

    def mean(self, obs):  # [P, B, obs_dim] -> [P, B, act_dim]
        W, b = self.params[6], self.params[7]
        return torch.baddbmm(b.unsqueeze(1), self._tower(obs, 0), W.transpose(1, 2))

    def log_prob(self, obs, act):  # -> [P, B]
        mu, ls = self.mean(obs), self.params[16].unsqueeze(1)
        return (-0.5 * ((act - mu) / ls.exp()) ** 2 - ls - 0.5 * math.log(2 * math.pi)).sum(-1)

    def entropy(self):  # -> [P]
        return (0.5 + 0.5 * math.log(2 * math.pi) + self.params[16]).sum(-1)

    def value(self, obs):  # -> [P, B]
        W, b = self.params[14], self.params[15]
        return torch.baddbmm(b.unsqueeze(1), self._tower(obs, 8), W.transpose(1, 2)).squeeze(-1)

    def packed(self):
        """float32 [P, floats]: row p is pack_policy of agent p's towers (tb_set_policies' rows)."""
        rows = []
        for t in self.params:
            t = t.detach().reshape(self.agents, -1).to(torch.float32)
            r = (-t.shape[1]) % 4
            rows += [t] if r == 0 else [t, t.new_zeros(self.agents, r)]
        out = torch.cat(rows, 1)
        assert out.shape[1] == POLICY_FLOATS_BY_DIMS[(self.obs_dim, self.act_dim)], out.shape
        return out


class BatchedAdam:
    """Adam (eps 1e-5, betas 0.9 / 0.999) over stacked parameters with a per-agent learning rate lr [P], written out because
    torch.optim.Adam takes one lr per parameter group.  It follows torch.optim.Adam's formulas; the bias corrections are
    formed in float64 from a per-agent step count.  Every operation runs on the device, so a step can be captured."""

    def __init__(self, params, lr, betas=(0.9, 0.999), eps=1e-5):
        self.params, self.lr, self.betas, self.eps = params, lr, betas, eps
        self.m = [torch.zeros_like(p) for p in params]
        self.v = [torch.zeros_like(p) for p in params]
        self.steps = torch.zeros(lr.shape[0], dtype=torch.float64, device=lr.device)

    def state_tensors(self):
        return self.m + self.v + [self.steps]

    @torch.no_grad()
    def step(self):
        b1, b2 = self.betas
        self.steps += 1
        step_size = (self.lr.double() / (1 - b1 ** self.steps)).float()
        bc2_sqrt = (1 - b2 ** self.steps).sqrt().float()
        for p, m, v in zip(self.params, self.m, self.v):
            g, shape = p.grad, (-1,) + (1,) * (p.dim() - 1)
            m.lerp_(g, 1 - b1)
            v.mul_(b2).addcmul_(g, g, value=1 - b2)
            denom = (v.sqrt() / bc2_sqrt.view(shape)).add_(self.eps)
            p.sub_(step_size.view(shape) * (m / denom))


def clip_grad_norms(params, max_norm):
    """clip_grad_norm_ per agent: agent p's gradients are scaled by min(1, max_norm[p] / (norm_p + 1e-6))."""
    grads = [p.grad for p in params]
    P = grads[0].shape[0]
    norms = torch.stack([g.reshape(P, -1).norm(dim=1) for g in grads]).norm(dim=0)
    coef = (max_norm / (norms + 1e-6)).clamp(max=1.0)
    for g in grads:
        g.mul_(coef.view((-1,) + (1,) * (g.dim() - 1)))


def episode_stats(reward, done, carry_ret, carry_len, agents):
    """Episodes that ended in a rollout, per agent: (count int64 [P], return sum float64 [P], length sum float64 [P]).
    reward float32 [K, N], done [K, N]; carry_ret / carry_len float64 [N] hold the return and length of each env's episode
    in progress when the rollout began and are updated in place.  Env i belongs to agent i // (N // agents).  Vectorised over
    the K steps: the return of an episode ending at step t is the rewards after the env's previous done."""
    K, N = reward.shape
    d = done.bool()
    t = torch.arange(K, device=reward.device).unsqueeze(1).expand(K, N)
    last = torch.where(d, t, torch.full_like(t, -1)).cummax(0).values        # the latest done at or before t
    prev = torch.cat([torch.full_like(last[:1], -1), last[:-1]])             # the latest done before t
    cs = torch.cat([torch.zeros_like(carry_ret).unsqueeze(0), reward.double().cumsum(0)])  # cs[t + 1] = sum of r[0..t]
    began_before = prev < 0
    ret = cs[1:] - cs.gather(0, prev + 1) + torch.where(began_before, carry_ret, 0.0)
    length = (t - prev).double() + torch.where(began_before, carry_len, 0.0)
    per_agent = lambda x: x.sum(0).view(agents, -1).sum(1)  # noqa: E731
    out = (per_agent(d.long()), per_agent(torch.where(d, ret, 0.0)), per_agent(torch.where(d, length, 0.0)))
    lk = last[-1]
    none = lk < 0
    carry_ret.copy_(cs[K] - cs.gather(0, (lk + 1).unsqueeze(0))[0] + torch.where(none, carry_ret, 0.0))
    carry_len.copy_((K - 1 - lk).double() + torch.where(none, carry_len, 0.0))
    return out


@torch.no_grad()
def exploit_explore(scores, tensors, hyper, rng, perturbed=PBT_PERTURBED):
    """One PBT round.  scores: P floats, None for an agent that finished no episode (it ranks last).  Each of the bottom
    max(1, P // 4) agents copies an agent drawn from the top max(1, P // 4) with rng (numpy Generator): row dst of every
    tensor in `tensors` and of every [P] tensor in `hyper` takes row src; then its `perturbed` hyper-parameters (PPO's
    PBT_PERTURBED by default) are each multiplied by 0.8 or 1.2.  Returns [(dst, src, {name: new value})]."""
    P = len(scores)
    if P < 2:
        raise ValueError("exploit_explore needs at least 2 agents")
    q = max(1, P // 4)
    order = sorted(range(P), key=lambda p: (scores[p] is None, -(scores[p] if scores[p] is not None else 0.0), p))
    top, events = order[:q], []
    for dst in order[-q:]:
        src = top[int(rng.integers(q))]
        for t in tensors:
            t[dst] = t[src]
        for h in hyper.values():
            h[dst] = h[src]
        for name in perturbed:
            hyper[name][dst] = hyper[name][dst] * float(rng.choice(PBT_FACTORS))
        events.append((dst, src, {name: float(h[dst]) for name, h in hyper.items()}))
    return events


class PopulationPPO:
    """agents PPO learners, each on its own envs_per_agent envs of one TennisBatch, updated together.  Each hyper-parameter
    (HYPER_DEFAULTS: GpuPPO's) is a scalar for every agent or a sequence of one value per agent.  Agent p starts from the
    weights GpuPPO(seed=seeds[p]) starts from and takes exactly GpuPPO's update on its own samples: its own GAE, permutation,
    minibatches, advantage normalisation, loss coefficients, gradient-norm clipping and Adam learning rate.  The rollout is
    the fused one only (tb_set_policies + tb_policy_rollout in one CUDA graph).  The context's env seed is seeds[0] and the
    policy noise seed seeds[0] + 1.  pbt_interval: run exploit_explore() after every pbt_interval updates (None: never).
    normalize: each agent's envs run under that agent's own VecNormalize record (SB3's defaults, PPO's gamma, which must then
    be one value for every agent), as GpuPPO(normalize=True) runs its envs: the agent learns on normalised observations and
    rewards, while its episode statistics and PBT scores come from the raw rewards."""

    def __init__(self, env_id, agents, envs_per_agent, rollout_len, seeds=None, lr=3e-4, ent_coef=0.002, clip=0.2, vf_coef=0.5,
                 max_grad_norm=0.5, gamma=0.99, gae_lambda=0.95, epochs=10, minibatches=8, precision="f64", device=0,
                 use_graph=True, pbt_interval=None, pbt_seed=0, normalize=False):
        P = self.P = int(agents)
        if P < 1:
            raise ValueError(f"agents must be >= 1, got {agents}")
        self.seeds = list(range(P)) if seeds is None else [int(s) for s in agent_values("seeds", seeds, P)]
        given = dict(lr=lr, ent_coef=ent_coef, clip=clip, vf_coef=vf_coef, max_grad_norm=max_grad_norm, gamma=gamma,
                     gae_lambda=gae_lambda)
        values = {k: agent_values(k, v, P) for k, v in given.items()}
        self.normalize = bool(normalize)
        if self.normalize and len(set(values["gamma"])) != 1:
            raise ValueError(f"normalize=True needs one gamma for every agent (the records share one configuration, and PBT "
                             f"does not perturb gamma), got {values['gamma']}")
        if pbt_interval is not None and (int(pbt_interval) < 1 or P < 2):
            raise ValueError("pbt_interval needs at least 2 agents and must be >= 1")
        self.pbt_interval, self.pbt_rng, self.pbt_log = pbt_interval, np.random.default_rng(pbt_seed), []
        self.dev = torch.device("cuda", device)
        self.n, self.K = n, K = int(envs_per_agent), int(rollout_len)
        self.N = N = P * n
        self.env = TennisBatch(env_id, N, device=device, seed=self.seeds[0], precision=precision)
        self.od, self.ad = od, ad = self.env.obs_dim, self.env.act_dim
        self.hyper = {k: torch.tensor(v, dtype=torch.float32, device=self.dev) for k, v in values.items()}
        self.ac = BatchedActorCritic(od, ad, self.seeds, self.dev)
        self.opt = BatchedAdam(self.ac.params, self.hyper["lr"])
        self.gen = torch.Generator(self.dev)
        self.gen.manual_seed(self.seeds[0])
        self.epochs, self.minibatches, self.use_graph = epochs, minibatches, use_graph
        z = lambda *s: torch.zeros(s, device=self.dev)  # noqa: E731
        self.obs_buf, self.act_buf = z(K, N, od), z(K, N, ad)
        self.logp_buf, self.rew_buf, self.done_buf, self.val_buf = z(K, N), z(K, N), z(K, N), z(K + 1, N)
        self.done_u8 = torch.zeros((K, N), dtype=torch.uint8, device=self.dev)
        self.params = z(P, POLICY_FLOATS_BY_DIMS[(od, ad)])
        self.obs = self.env.reset().clone()  # raw: with normalize, obs_buf / rew_buf receive the normalised values
        self.vn_gamma = values["gamma"][0]  # the records' gamma (the [P] hyper tensor holds it rounded to float32)
        if self.normalize:  # one record per agent; the first rollout folds the reset observation
            self.env.set_vecnorm(gamma=self.vn_gamma, agents=P)
        self.raw_buf = z(K, N) if self.normalize else None  # the raw rewards the episode statistics are summed from
        self.ep_ret = torch.zeros(N, dtype=torch.float64, device=self.dev)  # return / length of each env's episode in progress
        self.ep_len = torch.zeros(N, dtype=torch.float64, device=self.dev)
        self.graph, self.upd_graph, self.warmed_up = None, None, False
        self.rollout_s, self.updates = 0.0, 0
        self.mb = K * n // minibatches  # samples per agent per minibatch
        self.mb_obs, self.mb_act = z(P, self.mb, od), z(P, self.mb, ad)
        self.mb_logp, self.mb_adv, self.mb_ret = z(P, self.mb), z(P, self.mb), z(P, self.mb)
        self._interval = np.zeros((2, P))  # return sum, episodes since the last PBT round

    # ------------------------------------------------------------------ rollout
    def _rollout_body(self):
        self.params.copy_(self.ac.packed())
        self.env.set_policies(self.params)
        self.obs_buf[0].copy_(self.obs)
        self.env.policy_rollout(self.obs_buf, self.rew_buf, self.done_u8, self.obs, actions=self.act_buf, logp=self.logp_buf,
                                value=self.val_buf[:self.K], last_value=self.val_buf[self.K], noise_seed=self.seeds[0] + 1,
                                raw_reward=self.raw_buf)
        self.done_buf.copy_(self.done_u8)

    def _episode_stats(self):
        return episode_stats(self.rew_buf if self.raw_buf is None else self.raw_buf, self.done_u8, self.ep_ret, self.ep_len, self.P)

    @torch.no_grad()
    def rollout(self):
        """rollout_len steps of every env into the buffers.  Returns (per-agent episodes int64 [P], return sums float64 [P],
        length sums float64 [P]) of the episodes that ended in it, as numpy, and the context's statistics vector."""
        self.env.read_stats(clear=True)
        torch.cuda.synchronize()
        t0 = time.time()
        if not self.use_graph:
            self._rollout_body()
        else:
            if self.graph is None:
                if not self.warmed_up:  # a real rollout on a side stream (library buffers, cuBLAS), then capture
                    s = torch.cuda.Stream(self.dev)
                    s.wait_stream(torch.cuda.current_stream(self.dev))
                    with torch.cuda.stream(s):
                        self._rollout_body()
                    torch.cuda.current_stream(self.dev).wait_stream(s)
                    self._episode_stats()  # its episodes are not reported, but the ones in progress carry on
                    torch.cuda.synchronize()
                    self.env.read_stats(clear=True)
                    self.warmed_up = True
                self.graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(self.graph):
                    self._rollout_body()
                torch.cuda.synchronize()
                t0 = time.time()
            self.graph.replay()
        torch.cuda.synchronize()
        self.rollout_s += time.time() - t0
        eps, ret, length = (x.cpu().numpy() for x in self._episode_stats())
        return eps, ret, length, self.env.read_stats()

    # ------------------------------------------------------------------ update
    def _agent_major(self, x):
        """[K, N, ...] rollout buffer -> [P * K * n, ...]: agent p's samples contiguous, in GpuPPO's order t * n + j."""
        K, P, n = self.K, self.P, self.n
        return x.view(K, P, n, *x.shape[2:]).transpose(0, 1).reshape(P * K * n, *x.shape[2:])

    def update(self):
        K, P, n, N = self.K, self.P, self.n, self.N
        gamma = self.hyper["gamma"].repeat_interleave(n)
        lam = self.hyper["gae_lambda"].repeat_interleave(n)
        adv = torch.zeros_like(self.rew_buf)
        last = torch.zeros(N, device=self.dev)
        for t in reversed(range(K)):
            nonterm = 1.0 - self.done_buf[t]
            delta = self.rew_buf[t] + gamma * self.val_buf[t + 1] * nonterm - self.val_buf[t]
            last = delta + gamma * lam * nonterm * last
            adv[t] = last
        ret = adv + self.val_buf[:K]
        B, mb = K * n, self.mb
        fo, fa, fl = self._agent_major(self.obs_buf), self._agent_major(self.act_buf), self._agent_major(self.logp_buf)
        fadv, fret = self._agent_major(adv), self._agent_major(ret)
        offs = (torch.arange(P, device=self.dev) * B).unsqueeze(1)
        outs = [(fo, self.mb_obs.view(P * mb, self.od)), (fa, self.mb_act.view(P * mb, self.ad)), (fl, self.mb_logp.view(-1)),
                (fadv, self.mb_adv.view(-1)), (fret, self.mb_ret.view(-1))]
        for _ in range(self.epochs):
            perm = torch.rand(P, B, device=self.dev, generator=self.gen).argsort(1) + offs  # one permutation per agent
            for k in range(self.minibatches):
                idx = perm[:, k * mb:(k + 1) * mb].reshape(-1)
                for src, dst in outs:
                    torch.index_select(src, 0, idx, out=dst)
                if not self.use_graph:
                    self._minibatch_step()
                    continue
                if self.upd_graph is None:
                    self._capture_update()
                self.upd_graph.replay()
        self.updates += 1

    def _capture_update(self):
        # warm-up steps are real Adam updates: take them on a snapshot and put parameters and Adam state back, so that the
        # graph path trains exactly like the eager one (GpuPPO.update does the same)
        state = self.ac.params + self.opt.state_tensors()
        snap = [t.detach().clone() for t in state]
        s = torch.cuda.Stream(self.dev)
        s.wait_stream(torch.cuda.current_stream(self.dev))
        with torch.cuda.stream(s):
            for _ in range(3):
                self._minibatch_step()
        torch.cuda.current_stream(self.dev).wait_stream(s)
        self.upd_graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.upd_graph):
            self._minibatch_step()
        with torch.no_grad():
            for t, v in zip(state, snap):
                t.copy_(v)

    def losses(self):
        """GpuPPO's minibatch loss for every agent, float32 [P], from the mb_* buffers."""
        ac, h = self.ac, self.hyper
        ratio = (ac.log_prob(self.mb_obs, self.mb_act) - self.mb_logp).exp()
        a_ = self.mb_adv
        a_ = (a_ - a_.mean(1, keepdim=True)) / (a_.std(1, keepdim=True) + 1e-8)
        clip = h["clip"].unsqueeze(1)
        pg = -torch.min(ratio * a_, ratio.clamp(1 - clip, 1 + clip) * a_).mean(1)
        vloss = 0.5 * (ac.value(self.mb_obs) - self.mb_ret).pow(2).mean(1)
        return pg + h["vf_coef"] * vloss - h["ent_coef"] * ac.entropy()

    def _minibatch_step(self):
        for p in self.ac.params:  # grads stay in place: the captured graph refers to their storage
            if p.grad is not None:
                p.grad.zero_()
        self.losses().sum().backward()  # agents share no parameter, so each gets the gradient of its own loss
        clip_grad_norms(self.ac.params, self.hyper["max_grad_norm"])
        self.opt.step()

    # ------------------------------------------------------------------ PBT
    def exploit_explore(self, scores=None):
        """One PBT round (module function exploit_explore) on parameters, Adam moments and step counts, hyper-parameters and,
        with normalize, the VecNormalize record the weights were trained against (a row copy in the library's buffer, which
        the next rollout reads); env state, the per-env discounted returns included, is not copied.  scores: None ranks by
        the mean training return since the previous round.  The events are appended to pbt_log as (update, destination,
        source, new hyper-parameters) and returned."""
        if scores is None:
            r, e = self._interval
            scores = [float(r[p] / e[p]) if e[p] else None for p in range(self.P)]
        rows = self.ac.params + self.opt.state_tensors() + ([self.env.vecnorm_records()] if self.normalize else [])
        ev = exploit_explore(scores, rows, self.hyper, self.pbt_rng)
        ev = [(self.updates, dst, src, hp) for dst, src, hp in ev]
        self.pbt_log += ev
        self._interval[:] = 0
        return ev

    # ------------------------------------------------------------------ training
    def train(self, iters, log=None):
        """iters x (rollout, update, and a PBT round every pbt_interval updates).  Per agent and iteration: the episodes
        that ended in the rollout, their mean return and length (None when none ended); per iteration the context-wide
        racket hits and goals per episode (tb_read_stats)."""
        P, t0 = self.P, time.time()
        hist, ctx = [[] for _ in range(P)], []
        for it in range(iters):
            eps, rsum, lsum, st = self.rollout()
            self._interval += np.stack([rsum, eps])
            for p in range(P):
                e = int(eps[p])
                hist[p].append({"iter": it, "env_steps": (it + 1) * self.K * self.n, "episodes": e,
                                "mean_return": float(rsum[p] / e) if e else None, "mean_length": float(lsum[p] / e) if e else None,
                                "lr": float(self.hyper["lr"][p]), "ent_coef": float(self.hyper["ent_coef"][p])})
            e = int(st[0])
            ctx.append({"iter": it, "episodes": e, "hits_per_episode": float(st[2] / e) if e else None,
                        "goal_fraction": float(st[3] / e) if e else None})
            self.update()
            if self.pbt_interval and self.updates % self.pbt_interval == 0:
                for ev in self.exploit_explore():
                    if log:
                        log(f"pbt update {ev[0]}: agent {ev[1]} <- agent {ev[2]}, lr {ev[3]['lr']:.3g} ent_coef {ev[3]['ent_coef']:.3g}")
            if log and (it % 10 == 0 or it == iters - 1):
                rets = " ".join("   -   " if h[-1]["mean_return"] is None else f"{h[-1]['mean_return']:7.2f}" for h in hist)
                log(f"iter {it:4d} returns {rets} wall {time.time() - t0:6.1f}s")
        per_agent = []
        for p in range(P):
            done = [h["mean_return"] for h in hist[p] if h["episodes"]]
            per_agent.append({"seed": self.seeds[p], "final_mean_return": done[-1] if done else None,
                              "best_mean_return": max(done) if done else None, "history": hist[p]})
        return {"agents": P, "envs_per_agent": self.n, "rollout_len": self.K, "iters": iters, "wall_s": time.time() - t0,
                "rollout_s": self.rollout_s, "hyper": {k: v.tolist() for k, v in self.hyper.items()},
                "pbt_events": [list(e[:3]) + [e[3]] for e in self.pbt_log], "per_agent": per_agent, "context": ctx}

    # ------------------------------------------------------------------ saving
    PBT_COLUMNS = ("update", "destination", "source") + tuple(HYPER_DEFAULTS)

    def state_dict(self):
        """numpy arrays: `policies` [P, floats] (tb_set_policies' rows), `seeds`, one [P] array per hyper-parameter, and
        `pbt_events` [E, len(PBT_COLUMNS)] float64 with the column names in `pbt_columns`.  With normalize also `vecnorm`
        [P, 2 obs_dim + 4] (tb_get_vecnorms' rows) and their configuration, `vecnorm_clip_obs`, `vecnorm_clip_reward`,
        `vecnorm_gamma` and `vecnorm_epsilon`: set_vecnorm(agents=P, stats=...) attaches them again."""
        out = {"policies": self.ac.packed().cpu().numpy(), "seeds": np.array(self.seeds)}
        if self.normalize:
            out.update(vecnorm=self.env.vecnorm_stats().cpu().numpy(), vecnorm_clip_obs=10.0, vecnorm_clip_reward=10.0,
                       vecnorm_gamma=self.vn_gamma, vecnorm_epsilon=1e-8)
        out.update({k: v.cpu().numpy() for k, v in self.hyper.items()})
        out["pbt_events"] = np.array([[u, d, s] + [hp[k] for k in HYPER_DEFAULTS] for u, d, s, hp in self.pbt_log],
                                     np.float64).reshape(-1, len(self.PBT_COLUMNS))
        out["pbt_columns"] = np.array(self.PBT_COLUMNS)
        return out

    def save(self, path):
        np.savez(path, **self.state_dict())

    def agent_state_dict(self, p):
        """Agent p in GpuPPO.state_dict()'s layout ({"policy": tb_set_policy's vector}, and with normalize agent p's record
        under load_vecnormalize_npz's keys): tools/record_episode.py plays it (--policy, and --vecnormalize with normalize)."""
        out = {"policy": self.ac.packed()[p].cpu().numpy()}
        if self.normalize:
            out.update(vecnormalize_entries(self.env.vecnorm_stats()[p], self.vn_gamma))
        return out

