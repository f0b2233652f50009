"""GPU-resident PPO on SwingRacket-v0 (BASELINE config 4: 16 384 envs on one B200) - SURVEY 8(f)-1 - and on Tennisbot-v0
with train.py's racket-scale curriculum (HitPPO).

The reference trains with SB3 PPO (`train_swing.py:80-91`: MlpPolicy, net_arch pi/vf [32,64,32], tanh, ent_coef
0.002, gamma .99, gae_lambda .95, clip .2, n_epochs 10, vf_coef .5, max_grad_norm .5) on ONE env, 1100 steps per
update.  SB3 is not installed here, so this is a plain-torch PPO with the same policy architecture and
hyper-parameters; only the batch geometry changes (N envs x 26 steps = one whole episode per env per update) and
the learning rate is the reference's 3e-4 default.  Observations and actions never leave HBM, and the rollout runs no
torch code at all: tb_policy_rollout evaluates the policy in a CUDA kernel of the library (forward, Philox Gaussian noise,
log-density, value), so the 26-step episode is 26 x (policy_kernel, step_kernel, ff_kernel) issued by one C call; the call
is captured once as a CUDA graph and replayed per update (nothing in it synchronises; the queue tags of ff_kernel advance
on the device).  `fused_policy=False` keeps the eager torch policy of round 1 for comparison.  Target: the mean episodic
return stored in backup_models/ppo_swing.zip, 31.5.  `normalize=True` puts SB3's VecNormalize on the device rollout
(tb_set_vecnorm): the policy learns on normalised observations and rewards, the reported returns stay raw.

HitPPO trains Tennisbot-v0 (train.py) the same way with the same hyper-parameters and the same towers on the env's 12
inputs and 2 outputs (train.py's net_arch is not recorded); its rollouts are K steps of episodes up to 1001 steps long.
"""
import math
import time

import numpy as np
import torch
import torch.nn as nn

from . import _lib
from .batch import TennisBatch
from .playground import curriculum_scale

EPISODE = 26  # agent steps per SwingRacket-v0 episode (swingracket_env.py:85-86: 25 control steps + the fast-forward step)


class ActorCritic(nn.Module):
    def __init__(self, obs_dim=6, act_dim=6):
        super().__init__()

        def mlp():
            return nn.Sequential(nn.Linear(obs_dim, 32), nn.Tanh(), nn.Linear(32, 64), nn.Tanh(), nn.Linear(64, 32), nn.Tanh())

        self.pi, self.vf = mlp(), mlp()
        self.mu = nn.Linear(32, act_dim)
        self.v = nn.Linear(32, 1)
        self.log_std = nn.Parameter(torch.zeros(act_dim))
        for m in list(self.pi) + list(self.vf):
            if isinstance(m, nn.Linear):
                nn.init.orthogonal_(m.weight, 2 ** 0.5)
                nn.init.zeros_(m.bias)
        nn.init.orthogonal_(self.mu.weight, 0.01)
        nn.init.orthogonal_(self.v.weight, 1.0)

    def mean(self, obs):
        return self.mu(self.pi(obs))

    def log_prob(self, obs, act):
        mu, ls = self.mean(obs), self.log_std
        return (-0.5 * ((act - mu) / ls.exp()) ** 2 - ls - 0.5 * math.log(2 * math.pi)).sum(-1)

    def entropy(self):
        return (0.5 + 0.5 * math.log(2 * math.pi) + self.log_std).sum()

    def value(self, obs):
        return self.v(self.vf(obs)).squeeze(-1)

    def packed(self):
        lin = lambda seq: [(m.weight, m.bias) for m in seq if isinstance(m, nn.Linear)]  # noqa: E731
        return pack_policy(lin(self.pi), (self.mu.weight, self.mu.bias), lin(self.vf), (self.v.weight, self.v.bias), self.log_std)


# (obs_dim, act_dim) -> floats of the in-kernel policy (TB_POLICY_FLOATS, TB_POLICY_FLOATS_HIT)
POLICY_FLOATS_BY_DIMS = {(6, 6): _lib.POLICY_FLOATS, (12, 2): _lib.POLICY_FLOATS_HIT}


def pack_policy(pi, mu, vf, v, log_std):
    """Flat float32 parameter vector in tb_set_policy's layout from (weight, bias) lists of the two towers: pi, vf = three
    (W [out, in], b) pairs each; mu, v = the heads; every tensor padded to a multiple of 4 floats.  The dimensions come from
    the first layer (obs_dim) and the action head (act_dim)."""
    def pad(t):
        t = t.detach().reshape(-1).to(torch.float32)
        r = (-t.numel()) % 4
        return t if r == 0 else torch.cat([t, t.new_zeros(r)])
    dims = (int(pi[0][0].shape[1]), int(mu[0].shape[0]))
    if dims not in POLICY_FLOATS_BY_DIMS:
        raise ValueError(f"no in-kernel policy for (obs_dim, act_dim) = {dims}; there are {sorted(POLICY_FLOATS_BY_DIMS)}")
    parts = []
    for tower, head in ((pi, mu), (vf, v)):
        for W, b in tower:
            parts += [pad(W), pad(b)]
        parts += [pad(head[0]), pad(head[1])]
    parts.append(pad(log_std))
    out = torch.cat(parts)
    assert out.numel() == POLICY_FLOATS_BY_DIMS[dims], (out.numel(), dims)
    return out


class GpuPPO:
    """PPO learner whose rollouts run on the B200 env batch: rollout_len steps of every env per update, collected by
    tb_policy_rollout (fused_policy) or by an eager torch policy.  use_graph: replay the rollout as one CUDA graph.
    GAE masks with the done flags and bootstraps from the value of the observation the rollout ends with, so a rollout
    need not hold whole episodes."""

    def __init__(self, env_id, num_envs, rollout_len, precision="f64", seed=0, lr=3e-4, epochs=10, minibatches=8, device=0,
                 use_graph=True, fused_policy=True, normalize=False):
        if normalize and not fused_policy:
            raise ValueError("normalize=True needs fused_policy=True: the normaliser runs inside tb_policy_rollout, and the eager "
                             "torch policy has none")
        torch.manual_seed(seed)
        self.normalize = bool(normalize)
        self.fused_policy = fused_policy
        self.seed = seed
        self.dev = torch.device("cuda", device)
        self.n = n = int(num_envs)
        self.K = K = int(rollout_len)
        self.env = TennisBatch(env_id, n, device=device, seed=seed, precision=precision)
        self.od, self.ad = od, ad = self.env.obs_dim, self.env.act_dim
        self.ac = ActorCritic(od, ad).to(self.dev)
        self.opt = torch.optim.Adam(self.ac.parameters(), lr=lr, eps=1e-5, capturable=use_graph)
        self.epochs, self.minibatches = epochs, minibatches
        self.gamma, self.lam, self.clip, self.ent_coef, self.vf_coef, self.max_norm = 0.99, 0.95, 0.2, 0.002, 0.5, 0.5
        z = lambda *s: torch.zeros(s, device=self.dev)  # noqa: E731
        self.obs_buf, self.act_buf = z(K, n, od), z(K, n, ad)
        self.logp_buf, self.rew_buf, self.done_buf, self.val_buf = z(K, n), z(K, n), z(K, n), z(K + 1, n)
        self.done_u8 = torch.zeros((K, n), dtype=torch.uint8, device=self.dev)
        self.params = z(POLICY_FLOATS_BY_DIMS[(od, ad)])
        self.obs = self.env.reset().clone()  # raw: with normalize, obs_buf / rew_buf receive the normalised values
        if self.normalize:  # SB3 VecNormalize's defaults, with PPO's gamma; the first rollout folds the reset observation
            self.env.set_vecnorm(gamma=self.gamma)
        self.graph = None
        self.warmed_up = False
        self.use_graph = use_graph
        self.rollout_s = 0.0
        # one minibatch update as a CUDA graph over static buffers (the update is ~40 small kernels, 80 times per iteration)
        self.mb = K * n // minibatches
        self.upd_graph = None
        self.mb_obs, self.mb_act = z(self.mb, od), z(self.mb, ad)
        self.mb_logp, self.mb_adv, self.mb_ret = z(self.mb), z(self.mb), z(self.mb)

    # ------------------------------------------------------------------ rollout
    def _rollout_body(self):
        ac, env, K = self.ac, self.env, self.K
        if self.fused_policy:
            # parameters -> the library's buffer (device to device, inside the graph: every replay sees the current weights)
            self.params.copy_(ac.packed())
            env.set_policy(self.params)
            self.obs_buf[0].copy_(self.obs)
            env.policy_rollout(self.obs_buf, self.rew_buf, self.done_u8, self.obs, actions=self.act_buf, logp=self.logp_buf,
                               value=self.val_buf[:K], last_value=self.val_buf[K], noise_seed=self.seed + 1)
            self.done_buf.copy_(self.done_u8)
            return
        for t in range(K):
            mu = ac.mean(self.obs)
            a = mu + ac.log_std.exp() * torch.randn_like(mu)
            self.obs_buf[t].copy_(self.obs)
            self.act_buf[t].copy_(a)
            self.logp_buf[t].copy_(ac.log_prob(self.obs, a))
            self.val_buf[t].copy_(ac.value(self.obs))
            o, r, dn, _, _ = env.step(a.clamp(-1, 1))  # SB3 clips to the Box before env.step
            self.rew_buf[t].copy_(r)
            self.done_buf[t].copy_(dn)
            self.obs.copy_(o)
        self.val_buf[K].copy_(ac.value(self.obs))

    @torch.no_grad()
    def rollout(self):
        """rollout_len steps of every env into the buffers; returns the statistics vector of the episodes that ended in them."""
        self.env.read_stats(clear=True)
        torch.cuda.synchronize()
        t0 = time.time()
        if not self.use_graph:
            self._rollout_body()
        else:
            if self.graph is None:
                if not self.warmed_up:  # warm up on a side stream (library state, cuBLAS handles), then capture
                    s = torch.cuda.Stream(self.dev)
                    s.wait_stream(torch.cuda.current_stream(self.dev))
                    with torch.cuda.stream(s):
                        self._rollout_body()
                    torch.cuda.current_stream(self.dev).wait_stream(s)
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
        return self.env.read_stats()

    # ------------------------------------------------------------------ update
    def update(self):
        n, ac, K = self.n, self.ac, self.K
        adv = torch.zeros_like(self.rew_buf)
        last = torch.zeros(n, device=self.dev)
        for t in reversed(range(K)):
            nonterm = 1.0 - self.done_buf[t]
            delta = self.rew_buf[t] + self.gamma * self.val_buf[t + 1] * nonterm - self.val_buf[t]
            last = delta + self.gamma * self.lam * nonterm * last
            adv[t] = last
        ret = adv + self.val_buf[:K]
        B = K * n
        fo, fa, fl = self.obs_buf.reshape(B, self.od), self.act_buf.reshape(B, self.ad), self.logp_buf.reshape(B)
        fadv, fret = adv.reshape(B), ret.reshape(B)
        mb = self.mb
        for _ in range(self.epochs):
            perm = torch.randperm(B, device=self.dev)
            for k in range(self.minibatches):
                idx = perm[k * mb:(k + 1) * mb]
                torch.index_select(fo, 0, idx, out=self.mb_obs)
                torch.index_select(fa, 0, idx, out=self.mb_act)
                torch.index_select(fl, 0, idx, out=self.mb_logp)
                torch.index_select(fadv, 0, idx, out=self.mb_adv)
                torch.index_select(fret, 0, idx, out=self.mb_ret)
                if not self.use_graph:
                    self._minibatch_step()
                    continue
                if self.upd_graph is None:
                    # warm-up steps are real Adam updates: take them on a snapshot and put model and optimiser back, so
                    # that the graph path trains exactly like the eager one (capture itself executes nothing)
                    snap_m = {k: v.clone() for k, v in self.ac.state_dict().items()}
                    s = torch.cuda.Stream(self.dev)
                    s.wait_stream(torch.cuda.current_stream(self.dev))
                    with torch.cuda.stream(s):
                        for _w in range(3):
                            self._minibatch_step()
                    torch.cuda.current_stream(self.dev).wait_stream(s)
                    self.upd_graph = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(self.upd_graph):
                        self._minibatch_step()
                    with torch.no_grad():  # back to "no update taken yet": weights, Adam moments and step counts
                        for k, v in self.ac.state_dict().items():
                            v.copy_(snap_m[k])
                        for st in self.opt.state.values():
                            for v in st.values():
                                if torch.is_tensor(v):
                                    v.zero_()
                self.upd_graph.replay()

    def state_dict(self):
        """The trained run as numpy arrays: `policy`, tb_set_policy's vector, and with normalize the normaliser's record
        under load_vecnormalize_npz's keys."""
        out = {"policy": self.ac.packed().cpu().numpy()}
        if self.normalize:
            out.update(vecnormalize_entries(self.env.vecnorm_stats(), self.gamma))
        return out

    def save(self, path):
        """state_dict() as an npz: tools/record_episode.py takes it as --policy (and as --vecnormalize with normalize)."""
        np.savez(path, **self.state_dict())

    def _minibatch_step(self):
        ac = self.ac
        ratio = (ac.log_prob(self.mb_obs, self.mb_act) - self.mb_logp).exp()
        a_ = self.mb_adv
        a_ = (a_ - a_.mean()) / (a_.std() + 1e-8)
        pg = -torch.min(ratio * a_, ratio.clamp(1 - self.clip, 1 + self.clip) * a_).mean()
        vloss = 0.5 * (ac.value(self.mb_obs) - self.mb_ret).pow(2).mean()
        loss = pg + self.vf_coef * vloss - self.ent_coef * ac.entropy()
        self.opt.zero_grad(set_to_none=False)  # grads stay in place: the captured graphs refer to their storage
        loss.backward()
        nn.utils.clip_grad_norm_(ac.parameters(), self.max_norm)
        self.opt.step()


class SwingPPO(GpuPPO):
    """PPO on SwingRacket-v0, one whole episode (26 steps) per env per update."""

    def __init__(self, num_envs=16384, precision="f64", seed=0, lr=3e-4, epochs=10, minibatches=8, device=0, use_graph=True,
                 fused_policy=True, normalize=False):
        super().__init__("SwingRacket-v0", num_envs, EPISODE, precision, seed, lr, epochs, minibatches, device, use_graph,
                         fused_policy, normalize)

    def train(self, iters=150, target=31.5, log=None):
        history, reached, t0 = [], None, time.time()
        for it in range(iters):
            st = self.rollout()
            eps = max(int(st[0]), 1)
            h = {"iter": it, "env_steps": (it + 1) * EPISODE * self.n, "mean_return": float(st[6] / 2 ** 20 / eps),
                 "goal_fraction": float(st[3] / eps), "hits_per_episode": float(st[2] / eps)}
            history.append(h)
            if reached is None and h["mean_return"] >= target:
                reached = h
            self.update()
            if log and (it % 10 == 0 or it == iters - 1):
                log(f"iter {it:4d} env-steps {h['env_steps']:>10d} return {h['mean_return']:7.2f} goals {h['goal_fraction']:5.3f} "
                    f"hits/ep {h['hits_per_episode']:.2f} wall {time.time() - t0:6.1f}s")
        wall = time.time() - t0
        return {"envs": self.n, "iters": iters, "cuda_graph_rollout": bool(self.use_graph),
                "final_mean_return": history[-1]["mean_return"], "best_mean_return": max(h["mean_return"] for h in history),
                "reference_target": target, "first_reached": reached, "wall_s": wall, "rollout_s": self.rollout_s,
                "rollout_env_steps_per_s": iters * EPISODE * self.n / max(self.rollout_s, 1e-9), "history": history}


class HitPPO(GpuPPO):
    """PPO on Tennisbot-v0 (train.py): rollouts of rollout_len steps per env, not aligned to episodes (up to 1001 steps).
    A time-out ends an episode like any other done, as in the reference (no bootstrap across it).

    curriculum_total_timesteps: train.py's ProgressCallback (train.py:155-176).  At each rollout start the racket scale is
    curriculum_scale(env_steps, total); when the stage changes, the library's racket_scale is set, every env is reset (an
    episode runs wholly at one scale) and the rollout graph is captured again: the scene constants are kernel arguments,
    which a captured graph holds by value.  None: the env's racket scale is left as it is."""

    def __init__(self, num_envs=16384, rollout_len=128, curriculum_total_timesteps=None, precision="f64", seed=0, lr=3e-4,
                 epochs=10, minibatches=8, device=0, use_graph=True, fused_policy=True, normalize=False):
        super().__init__("Tennisbot-v0", num_envs, rollout_len, precision, seed, lr, epochs, minibatches, device, use_graph,
                         fused_policy, normalize)
        self.curriculum_total = curriculum_total_timesteps
        self.env_steps = 0   # env steps of the rollouts taken so far (the curriculum's num_timesteps)
        self.scale = None    # racket scale set by the curriculum
        self.stages = []     # (env_steps, scale) of every stage change

    def apply_curriculum(self):
        """Set the curriculum's racket scale for the current env_steps; True when the stage changed (envs reset)."""
        if not self.curriculum_total:
            return False
        s = curriculum_scale(self.env_steps, self.curriculum_total)
        if s == self.scale:
            return False
        self.env.set_param("racket_scale", s)
        self.obs.copy_(self.env.reset())  # (a full reset: a normaliser zeroes its returns and folds this observation next)
        self.graph = None
        self.scale = s
        self.stages.append((self.env_steps, s))
        return True

    def rollout(self):
        self.apply_curriculum()
        st = super().rollout()
        self.env_steps += self.K * self.n
        return st

    def train(self, iters=100, log=None):
        """iters x (rollout, update).  Per iteration: the episodes that ended in the rollout, their mean return and
        racket-ball contact steps per episode (None when no episode ended), and the racket scale."""
        history, t0 = [], time.time()
        for it in range(iters):
            st = self.rollout()
            eps = int(st[0])
            h = {"iter": it, "env_steps": self.env_steps, "racket_scale": self.scale, "episodes": eps,
                 "mean_return": float(st[6] / 2 ** 20 / eps) if eps else None,
                 "hits_per_episode": float(st[2] / eps) if eps else None,
                 "mean_length": float(st[1] / eps) if eps else None}
            history.append(h)
            self.update()
            if log and (it % 10 == 0 or it == iters - 1):
                log(f"iter {it:4d} env-steps {h['env_steps']:>11d} scale {h['racket_scale']} episodes {eps:8d} "
                    f"return {h['mean_return']} hits/ep {h['hits_per_episode']} wall {time.time() - t0:6.1f}s")
        wall = time.time() - t0
        done = [h for h in history if h["episodes"]]
        return {"envs": self.n, "rollout_len": self.K, "iters": iters, "cuda_graph_rollout": bool(self.use_graph),
                "curriculum_total_timesteps": self.curriculum_total, "stages": self.stages,
                "final_mean_return": done[-1]["mean_return"] if done else None,
                "best_mean_return": max(h["mean_return"] for h in done) if done else None,
                "wall_s": wall, "rollout_s": self.rollout_s,
                "rollout_env_steps_per_s": iters * self.K * self.n / max(self.rollout_s, 1e-9), "history": history}


def load_sb3_policy_npz(path):
    """tb_set_policy's parameter vector from an npz of an SB3 MlpPolicy state dict with '.' written as '__' (the layout of
    tests/golden/ppo_swing_policy.npz: mlp_extractor__policy_net__0__weight, ..., action_net__weight, log_std)."""
    import numpy as np

    w = np.load(path)
    t = lambda key: torch.from_numpy(np.ascontiguousarray(w[key], np.float32))  # noqa: E731
    tower = lambda net: [(t(f"mlp_extractor__{net}__{i}__weight"), t(f"mlp_extractor__{net}__{i}__bias")) for i in (0, 2, 4)]  # noqa: E731
    return pack_policy(tower("policy_net"), (t("action_net__weight"), t("action_net__bias")), tower("value_net"),
                       (t("value_net__weight"), t("value_net__bias")), t("log_std"))


VECNORMALIZE_KEYS = ("obs_mean", "obs_var", "obs_count", "ret_mean", "ret_var", "ret_count", "clip_obs", "clip_reward", "gamma",
                     "epsilon")


def vecnormalize_entries(record, gamma):
    """A normaliser's record (float64 [2 obs_dim + 4], tb_get_vecnorm's layout, attached with SB3's VecNormalize defaults and
    this gamma) as numpy values under load_vecnormalize_npz's keys."""
    st = np.asarray(record.cpu() if torch.is_tensor(record) else record, np.float64)
    od = (st.size - 4) // 2
    return dict(obs_mean=st[:od], obs_var=st[od:2 * od], obs_count=st[2 * od], ret_mean=st[2 * od + 1], ret_var=st[2 * od + 2],
                ret_count=st[2 * od + 3], clip_obs=10.0, clip_reward=10.0, gamma=gamma, epsilon=1e-8)


def load_vecnormalize_npz(path, obs_dim=None):
    """(stats, config) of a saved VecNormalize: stats, float64 [2 obs_dim + 4] in tb_set_vecnorm's record layout; config, the
    keyword arguments of TennisBatch.set_vecnorm (clip_obs, clip_reward, gamma, epsilon).  The npz holds obs_mean, obs_var
    [obs_dim] and the scalars obs_count, ret_mean, ret_var, ret_count, clip_obs, clip_reward, gamma, epsilon (INTEGRATION.md
    section 2 writes one from SB3's vec_normalize.pkl).  Deploy with set_vecnorm(training=False, stats=..., **config)."""
    w = np.load(path)
    missing = [k for k in VECNORMALIZE_KEYS if k not in w]
    if missing:
        raise ValueError(f"{path}: missing VecNormalize keys {missing}")
    mean, var = np.asarray(w["obs_mean"], np.float64), np.asarray(w["obs_var"], np.float64)
    od = mean.size if obs_dim is None else int(obs_dim)
    if mean.shape != (od,) or var.shape != (od,):
        raise ValueError(f"{path}: obs_mean and obs_var must have shape ({od},), got {mean.shape} and {var.shape}")
    scalars = {k: np.asarray(w[k], np.float64) for k in VECNORMALIZE_KEYS[2:]}
    bad = [k for k, v in scalars.items() if v.shape != ()]
    if bad:
        raise ValueError(f"{path}: {bad} must be scalars")
    stats = np.concatenate([mean, var, [scalars["obs_count"], scalars["ret_mean"], scalars["ret_var"], scalars["ret_count"]]])
    config = {k: float(scalars[k]) for k in ("clip_obs", "clip_reward", "gamma", "epsilon")}
    return torch.from_numpy(stats), config
