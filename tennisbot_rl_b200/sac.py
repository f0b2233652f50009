"""GPU-resident SAC for SwingRacket-v0 and Tennisbot-v0 (SURVEY 8(f)-5): the actor runs in the library's sac_kernel, which
writes every transition into a replay ring in HBM; the learner around it is plain torch.

The reference offers SB3 SAC in train_swing.py and train.py.  SB3 is not installed here, so this is SB3 1.8 SAC's algorithm
with its defaults: MlpPolicy actor [256, 256] ReLU with mu / log_std heads, twin critics [256, 256] ReLU on cat(obs, act) with
Polyak targets (tau 0.005), gamma 0.99, automatic entropy tuning (target -act_dim, initial alpha 1), Adam 3e-4, and
learning_starts = 100 transitions taken with uniform actions.  Only the batch geometry is chosen here (num_envs, steps per
collection, batch size, gradient steps per collection, ring slots): SB3's one env step per gradient step at batch 256 does
not fit 16 k envs stepping in lock step.  DESIGN.md section 4.2 records the sweep the defaults come from.

One collection (pack the actor, tb_set_sac_actor, tb_sac_rollout of K steps) is captured once as a CUDA graph and replayed;
one gradient step (batch indices drawn on the device, uniform over the filled rows) is captured as another.

normalize=True is SB3's SAC on a VecNormalize env (its defaults, SAC's gamma): the in-kernel actor acts on normalised
observations and the statistics are folded on the device after every env step (TB_SAC_VECNORM); the ring stays raw, and each
gradient step normalises its sampled batch with the record as it stands (tb_vecnorm_apply), as SB3's ReplayBuffer.sample(env=...)
does.  Reported returns stay raw.
"""
import math
import time

import numpy as np

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import _lib
from .batch import TennisBatch
from .ppo import vecnormalize_entries

LOG_STD_MIN, LOG_STD_MAX = -20.0, 2.0  # SB3 sac/policies.py
HIDDEN = _lib.SAC_HIDDEN
SAC_FLOATS_BY_DIMS = {(6, 6): _lib.SAC_FLOATS, (12, 2): _lib.SAC_FLOATS_HIT}
ACTOR_KEYS = ("latent_pi.0.weight", "latent_pi.0.bias", "latent_pi.2.weight", "latent_pi.2.bias", "mu.weight", "mu.bias",
              "log_std.weight", "log_std.bias")


class SacActor(nn.Module):
    """SB3 SAC's Actor with its parameter names (latent_pi.0, latent_pi.2, mu, log_std): the float32 reference of sac_kernel."""

    def __init__(self, obs_dim=6, act_dim=6):
        super().__init__()
        self.latent_pi = nn.Sequential(nn.Linear(obs_dim, HIDDEN), nn.ReLU(), nn.Linear(HIDDEN, HIDDEN), nn.ReLU())
        self.mu = nn.Linear(HIDDEN, act_dim)
        self.log_std = nn.Linear(HIDDEN, act_dim)

    def dist(self, obs):
        """(mean, log_std) of the Gaussian before the squash, log_std clamped as SB3 does."""
        h = self.latent_pi(obs)
        return self.mu(h), self.log_std(h).clamp(LOG_STD_MIN, LOG_STD_MAX)

    def forward(self, obs, deterministic=False):
        mu, ls = self.dist(obs)
        return torch.tanh(mu if deterministic else mu + ls.exp() * torch.randn_like(mu))

    @staticmethod
    def log_prob(mu, log_std, u):
        """log-density of a = tanh(u), u ~ N(mu, exp(log_std)): the Gaussian's minus sum log(1 - tanh(u)^2 + 1e-6) (SB3's
        SquashedDiagGaussianDistribution)."""
        g = (-0.5 * ((u - mu) / log_std.exp()) ** 2 - log_std - 0.5 * math.log(2 * math.pi)).sum(-1)
        return g - torch.log(1.0 - torch.tanh(u) ** 2 + 1e-6).sum(-1)

    def action_log_prob(self, obs):
        mu, ls = self.dist(obs)
        u = mu + ls.exp() * torch.randn_like(mu)
        return torch.tanh(u), self.log_prob(mu, ls, u)

    def kernel_reference(self, obs, eps=None):
        """What sac_kernel computes, in torch: layer 1 float32 with each product and sum rounded in input order, ReLU, then
        activations and W2 rounded to BF16 with float32 accumulation, and float32 heads.  eps None: tanh(mu)."""
        W1, b1 = self.latent_pi[0].weight, self.latent_pi[0].bias
        acc = b1.expand(obs.shape[0], -1).clone()
        for c in range(obs.shape[1]):
            acc = acc + W1[:, c] * obs[:, c:c + 1]
        h1 = acc.clamp_min(0.0).to(torch.bfloat16).to(torch.float32)
        W2 = self.latent_pi[2].weight.to(torch.bfloat16).to(torch.float32)
        tf32 = torch.backends.cuda.matmul.allow_tf32
        torch.backends.cuda.matmul.allow_tf32 = False
        try:
            h2 = (h1 @ W2.t() + self.latent_pi[2].bias).clamp_min(0.0)
            mu, ls = self.mu(h2), self.log_std(h2).clamp(LOG_STD_MIN, LOG_STD_MAX)
        finally:
            torch.backends.cuda.matmul.allow_tf32 = tf32
        return torch.tanh(mu if eps is None else mu + ls.exp() * eps)


def pack_sac_actor(src):
    """Flat float32 vector in tb_set_sac_actor's layout from a SacActor, its state dict, or an SB3 SAC policy state dict (keys
    'actor.latent_pi.0.weight', ...; the critic's entries are ignored).  Each tensor row-major [out][in], padded to 4 floats."""
    sd = src.state_dict() if isinstance(src, nn.Module) else src
    if all(("actor." + k) in sd for k in ACTOR_KEYS):
        sd = {k: sd["actor." + k] for k in ACTOR_KEYS}
    missing = [k for k in ACTOR_KEYS if k not in sd]
    if missing:
        raise KeyError(f"pack_sac_actor: missing {missing} (expected SB3 SAC actor keys, optionally prefixed 'actor.')")

    def pad(t):
        t = t.detach().reshape(-1).to(torch.float32)
        r = (-t.numel()) % 4
        return t if r == 0 else torch.cat([t, t.new_zeros(r)])
    dims = (int(sd["latent_pi.0.weight"].shape[1]), int(sd["mu.weight"].shape[0]))
    if dims not in SAC_FLOATS_BY_DIMS:
        raise ValueError(f"no in-kernel SAC actor for (obs_dim, act_dim) = {dims}; there are {sorted(SAC_FLOATS_BY_DIMS)}")
    out = torch.cat([pad(sd[k]) for k in ACTOR_KEYS])
    assert out.numel() == SAC_FLOATS_BY_DIMS[dims], (out.numel(), dims)
    return out


def _mlp(inp, out):
    return nn.Sequential(nn.Linear(inp, HIDDEN), nn.ReLU(), nn.Linear(HIDDEN, HIDDEN), nn.ReLU(), nn.Linear(HIDDEN, out))


class TwinCritic(nn.Module):
    """SB3 SAC's ContinuousCritic with n_critics = 2: qf0, qf1 = [256, 256] ReLU on cat(obs, act)."""

    def __init__(self, obs_dim, act_dim):
        super().__init__()
        self.qf0, self.qf1 = _mlp(obs_dim + act_dim, 1), _mlp(obs_dim + act_dim, 1)

    def forward(self, obs, act):
        x = torch.cat([obs, act], -1)
        return self.qf0(x), self.qf1(x)


def sac_losses(actor, critic, critic_target, log_alpha, batch, gamma, target_entropy, noise, next_noise):
    """The entropy-coefficient and critic losses of SB3 SAC.train for one batch (obs, act, reward, next_obs, done) with the
    Gaussian draws given.  Returns (alpha_loss, critic_loss, pi, logp, alpha): pi and logp are the actor's squashed sample
    and its log-density on obs (for actor_loss), alpha = exp(log_alpha) before this step's alpha update, as in SB3."""
    obs, act, rew, nxt, done = batch
    mu, ls = actor.dist(obs)
    u = mu + ls.exp() * noise
    pi, logp = torch.tanh(u), SacActor.log_prob(mu, ls, u)
    alpha = log_alpha.detach().exp()
    alpha_loss = -(log_alpha * (logp + target_entropy).detach()).mean()
    with torch.no_grad():
        nmu, nls = actor.dist(nxt)
        nu = nmu + nls.exp() * next_noise
        nq = torch.min(*critic_target(nxt, torch.tanh(nu))) - alpha * SacActor.log_prob(nmu, nls, nu).unsqueeze(-1)
        target = rew.unsqueeze(-1) + (1.0 - done.unsqueeze(-1)) * gamma * nq
    q0, q1 = critic(obs, act)
    critic_loss = 0.5 * (F.mse_loss(q0, target) + F.mse_loss(q1, target))
    return alpha_loss, critic_loss, pi, logp, alpha


def actor_loss(critic, obs, pi, logp, alpha):
    """SB3's actor loss: mean(alpha logp - min(Q0, Q1)(obs, pi)), with the critics as they are after their update."""
    return (alpha * logp - torch.min(*critic(obs, pi)).squeeze(-1)).mean()


class GpuSAC:
    """SAC learner on a B200 env batch.  Per iteration: one collection of `steps` env steps of every env (in-kernel actor,
    transitions into the ring), then `gradient_steps` gradient steps on batches of `batch_size` drawn uniformly from the filled
    rows of the ring (slots x num_envs transitions)."""

    def __init__(self, env_id="SwingRacket-v0", num_envs=1024, steps=1, batch_size=1024, gradient_steps=8, slots=1024,
                 precision="f64", seed=0, lr=3e-4, gamma=0.99, tau=0.005, learning_starts=100, device=0, eval_envs=1024,
                 normalize=False):
        torch.manual_seed(seed)
        self.env_id, self.seed = env_id, seed
        self.dev = torch.device("cuda", device)
        self.n, self.K, self.B, self.G, self.slots = int(num_envs), int(steps), int(batch_size), int(gradient_steps), int(slots)
        self.env = TennisBatch(env_id, self.n, device=device, seed=seed, precision=precision)
        self.normalize = bool(normalize)
        if self.normalize:  # attached before any graph capture; the first rollout folds tb_sac_begin's reset observation
            self.env.set_vecnorm(gamma=gamma)
        self.od, self.ad = od, ad = self.env.obs_dim, self.env.act_dim
        self.actor = SacActor(od, ad).to(self.dev)
        self.critic = TwinCritic(od, ad).to(self.dev)
        self.critic_target = TwinCritic(od, ad).to(self.dev)
        self.critic_target.load_state_dict(self.critic.state_dict())
        self.critic_target.requires_grad_(False)
        self.log_alpha = torch.zeros(1, device=self.dev, requires_grad=True)  # initial alpha 1
        self.target_entropy = -float(ad)
        self.gamma, self.tau = gamma, tau
        opt = lambda p: torch.optim.Adam(p, lr=lr, capturable=True)  # noqa: E731
        self.actor_opt, self.critic_opt, self.alpha_opt = opt(self.actor.parameters()), opt(self.critic.parameters()), opt([self.log_alpha])
        z = lambda *s, dt=torch.float32: torch.zeros(s, dtype=dt, device=self.dev)  # noqa: E731
        S, n = self.slots, self.n
        self.ring = dict(obs=z(S, n, od), act=z(S, n, ad), reward=z(S, n), next_obs=z(S, n, od), done=z(S, n, dt=torch.uint8))
        self.flat = dict(obs=self.ring["obs"].view(S * n, od), act=self.ring["act"].view(S * n, ad),
                         reward=self.ring["reward"].view(S * n), next_obs=self.ring["next_obs"].view(S * n, od),
                         done=self.ring["done"].view(S * n))
        self.fill = z(1)           # filled rows of the ring (a device scalar: the graph's batch indices are drawn below it)
        self.steps_taken = 0       # env steps of every env since sac_begin
        self.params = z(SAC_FLOATS_BY_DIMS[(od, ad)])
        self.params.copy_(pack_sac_actor(self.actor))
        self.env.set_sac_actor(self.params)  # (allocates the library's image outside the graph capture)
        self.env.sac_begin()
        warm = max(1, math.ceil(learning_starts / n))  # SB3's learning_starts counts transitions of all envs
        self.env.sac_rollout(warm, "uniform", self.ring, noise_seed=seed + 1, normalize=self.normalize)
        self.steps_taken += warm
        self.collect_graph = self.update_graph = None
        self.losses = z(3)
        self.collect_s = self.update_s = 0.0
        self.eval_envs = int(eval_envs)
        self._eval = None

    # ------------------------------------------------------------------ collection
    def _collect_body(self):
        self.params.copy_(pack_sac_actor(self.actor))
        self.env.set_sac_actor(self.params)
        self.env.sac_rollout(self.K, "sample", self.ring, noise_seed=self.seed + 1, normalize=self.normalize)

    @torch.no_grad()
    def collect(self):
        if self.collect_graph is None:
            self.collect_graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.collect_graph):
                self._collect_body()
        self.collect_graph.replay()
        self.steps_taken += self.K

    # ------------------------------------------------------------------ update
    def _grad_step(self):
        idx = (torch.rand(self.B, device=self.dev) * self.fill).long()
        f = self.flat
        batch = (f["obs"][idx], f["act"][idx], f["reward"][idx], f["next_obs"][idx], f["done"][idx].float())
        if self.normalize:  # the gathered copies, in place, with the record at replay time
            for x, what in ((batch[0], "obs"), (batch[2], "reward"), (batch[3], "obs")):
                self.env.vecnorm_apply(x, what, out=x)
        noise = torch.randn(self.B, self.ad, device=self.dev)
        next_noise = torch.randn(self.B, self.ad, device=self.dev)
        a_loss, c_loss, pi, logp, alpha = sac_losses(self.actor, self.critic, self.critic_target, self.log_alpha, batch,
                                                     self.gamma, self.target_entropy, noise, next_noise)
        # SB3's order: alpha, then the critics, then the actor (its loss reads the updated critics)
        self.alpha_opt.zero_grad(set_to_none=False)
        a_loss.backward()
        self.alpha_opt.step()
        self.critic_opt.zero_grad(set_to_none=False)
        c_loss.backward()
        self.critic_opt.step()
        pi_loss = actor_loss(self.critic, batch[0], pi, logp, alpha)
        self.actor_opt.zero_grad(set_to_none=False)
        pi_loss.backward()
        self.actor_opt.step()
        with torch.no_grad():
            for p, tp in zip(self.critic.parameters(), self.critic_target.parameters()):
                tp.lerp_(p, self.tau)
            self.losses.copy_(torch.stack([a_loss.detach(), c_loss.detach(), pi_loss.detach()]))

    def update(self):
        self.fill.fill_(float(min(self.steps_taken, self.slots) * self.n))
        if self.update_graph is None:
            # warm-up steps are real updates: take them on a snapshot and put models, optimisers and alpha back, so the graph
            # trains like the eager path (capture itself executes nothing)
            mods = (self.actor, self.critic, self.critic_target)
            snap = [{k: v.clone() for k, v in m.state_dict().items()} for m in mods]
            la = self.log_alpha.detach().clone()
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
                for m, sd in zip(mods, snap):
                    for k, v in m.state_dict().items():
                        v.copy_(sd[k])
                self.log_alpha.copy_(la)
                for o in (self.actor_opt, self.critic_opt, self.alpha_opt):
                    for st in o.state.values():
                        for v in st.values():
                            if torch.is_tensor(v):
                                v.zero_()
        for _ in range(self.G):
            self.update_graph.replay()

    # ------------------------------------------------------------------ training and evaluation
    def train(self, iters, log=None, eval_every=0, eval_episodes=1):
        """iters x (collection, gradient_steps gradient steps).  The history holds, per iteration, the episodes that ended in
        its collection (mean return, goals, racket hits per episode), env steps so far and the losses; `evaluations` the
        deterministic evaluations taken every eval_every iterations (and after the last)."""
        history, evals, t0 = [], [], time.time()
        self.env.read_stats(clear=True)
        for it in range(iters):
            torch.cuda.synchronize()
            t1 = time.time()
            self.collect()
            torch.cuda.synchronize()
            t2 = time.time()
            self.update()
            torch.cuda.synchronize()
            t3 = time.time()
            self.collect_s += t2 - t1
            self.update_s += t3 - t2
            st = self.env.read_stats(clear=True)
            eps = int(st[0])
            h = {"iter": it, "env_steps": self.steps_taken * self.n, "episodes": eps,
                 "mean_return": float(st[6] / 2 ** 20 / eps) if eps else None, "goal_fraction": float(st[3] / eps) if eps else None,
                 "hits_per_episode": float(st[2] / eps) if eps else None}
            history.append(h)
            if (eval_every and (it + 1) % eval_every == 0) or it == iters - 1:
                evals.append({"iter": it, "env_steps": h["env_steps"], "eval_mean_return": self.evaluate(eval_episodes)})
            if log and (it % 500 == 0 or it == iters - 1):
                a, c, p = self.losses.tolist()
                log(f"iter {it:5d} env-steps {h['env_steps']:>10d} return {h['mean_return']} goals {h['goal_fraction']} "
                    f"alpha {float(self.log_alpha.exp()):.4f} critic {c:.4f} actor {p:.4f} wall {time.time() - t0:6.1f}s")
        done = [h for h in history if h["episodes"]]
        return {"env": self.env_id, "envs": self.n, "steps": self.K, "batch_size": self.B, "gradient_steps": self.G,
                "slots": self.slots, "iters": iters, "final_mean_return": done[-1]["mean_return"] if done else None,
                "eval_mean_return": evals[-1]["eval_mean_return"] if evals else None, "evaluations": evals,
                "wall_s": time.time() - t0, "collect_s": self.collect_s, "update_s": self.update_s, "history": history}

    def state_dict(self):
        """The trained actor as numpy arrays: `policy`, tb_set_sac_actor's vector, and with normalize the normaliser's record
        under load_vecnormalize_npz's keys."""
        out = {"policy": pack_sac_actor(self.actor).cpu().numpy()}
        if self.normalize:
            out.update(vecnormalize_entries(self.env.vecnorm_stats(), self.gamma))
        return out

    def save(self, path):
        """state_dict() as an npz.  Deploy: set_sac_actor(policy), and with normalize set_vecnorm(training=False, ...) from
        load_vecnormalize_npz, then sac_rollout(..., normalize=True)."""
        np.savez(path, **self.state_dict())

    @torch.no_grad()
    def evaluate(self, episodes=1):
        """Mean return of `episodes` whole episodes per env of eval_envs envs with the deterministic action tanh(mu), on a
        context of its own with ring = NULL (so training's envs and ring are untouched).  With normalize, that context gets a
        frozen copy of the training record first (SB3's sync_envs_normalization)."""
        if self._eval is None:
            self._eval = TennisBatch(self.env_id, self.eval_envs, device=self.dev.index, seed=self.seed + 1000,
                                     precision=self.env.precision)
        e = self._eval
        e.set_sac_actor(pack_sac_actor(self.actor).contiguous())
        if self.normalize:
            e.set_vecnorm(training=False, gamma=self.gamma, stats=self.env.vecnorm_stats())
        e.sac_begin()
        e.read_stats(clear=True)
        done = 0
        chunk = 26 if e.kind == _lib.ENV_SWING else 100
        # the statistics vector counts every episode that ends; stop once episodes x eval_envs of them have ended
        while done < episodes * self.eval_envs:
            e.sac_rollout(chunk, "mean", None, noise_seed=0, normalize=self.normalize)
            done = int(e.read_stats()[0])
        st = e.read_stats(clear=True)
        return float(st[6] / 2 ** 20 / max(int(st[0]), 1))
