"""Batched fitness evaluation for the reference's ES trainer (SURVEY 8(f)-2).

`tennisbot/ES/fitness_functions.py:18-158` evaluates ONE GatedCNN individual on ONE freshly made env per call and
`evolution_strategy_static.py:143-193` maps 2 x population x 10 such calls over a process pool.  Here every
(individual, repeat) pair is one env of a single CUDA batch: per-env GatedCNN weights (766 parameters for 6 -> 6,
`policies.py:59-128`), per-env running observation normaliser (`evolution_strategy_static.py:25-44`, each call
works on its own copy there as well), 8-step history, action clipped to the Box, reward summed until done.
Two implementations of that evaluation:
- `EsEvaluator`: the GatedCNN, the normalisers, the history and the returns live in HBM and are advanced by the library's
  es_kernel between env steps (tb_es_begin / tb_es_rollout); nothing between two env steps runs on the host.
- `batched_fitness_static`: the same semantics in plain torch around `TennisBatch.step`, kept as the reference.
"""
import torch

from .batch import TennisBatch

HISTORY_LEN = 8  # fitness_functions.py:16


def gated_cnn_sizes(input_c, action_dim):
    """(out, in, kernel) of conv_0, conv_gate_0, conv_1, conv_gate_1, conv_2 in parameters_to_vector order."""
    return [(8, input_c, 2), (8, input_c, 2), (12, 8, 2), (12, 8, 2), (action_dim, 12, 2)]


def num_params(input_c, action_dim):
    return sum(o * i * k + o for o, i, k in gated_cnn_sizes(input_c, action_dim))


def _split(weights, input_c, action_dim):
    out, off = [], 0
    for o, i, k in gated_cnn_sizes(input_c, action_dim):
        w = weights[:, off:off + o * i * k].reshape(-1, o, i, k)
        off += o * i * k
        b = weights[:, off:off + o]
        off += o
        out.append((w, b))
    return out


def _conv(x, w, b, dilation):
    """Per-sample Conv1d(kernel_size=2, dilation, padding='valid'): x [B,Cin,L], w [B,Cout,Cin,2], b [B,Cout]."""
    length = x.shape[2] - dilation
    return (torch.einsum("boc,bcl->bol", w[..., 0], x[:, :, :length]) +
            torch.einsum("boc,bcl->bol", w[..., 1], x[:, :, dilation:dilation + length]) + b[:, :, None])


def gated_cnn_forward(weights, hist, action_dim):
    """GatedCNN.forward (policies.py:96-125) for a batch with PER-ENV weights.
    weights [B, n_params] float32, hist [B, C, 8] (channels = obs dims, length = history) -> [B, action_dim]."""
    (w0, b0), (g0, c0), (w1, b1), (g1, c1), (w2, b2) = _split(weights, hist.shape[1], action_dim)
    h = torch.tanh(_conv(hist, w0, b0, 1)) * torch.sigmoid(_conv(hist, g0, c0, 1))
    h = torch.tanh(_conv(h, w1, b1, 2)) * torch.sigmoid(_conv(h, g1, c1, 2))
    return _conv(h, w2, b2, 4).squeeze(-1)


class BatchedNormalizer:
    """evolution_strategy_static.Normalizer (:25-44) with one independent running state per env."""

    def __init__(self, batch, dim, device, state=None):
        z = lambda: torch.zeros((batch, dim), dtype=torch.float64, device=device)  # noqa: E731
        self.n, self.mean, self.mean_diff, self.var = z(), z(), z(), z()
        if state is not None:  # (n, mean, mean_diff, var) of the trainer's master normaliser
            for dst, src in zip((self.n, self.mean, self.mean_diff, self.var), state):
                dst += torch.as_tensor(src, dtype=torch.float64, device=device).reshape(1, dim)

    def observe(self, x):
        x = x.double()
        self.n += 1.0
        last = self.mean.clone()
        self.mean += (x - self.mean) / self.n
        self.mean_diff += (x - last) * (x - self.mean)
        self.var = (self.mean_diff / self.n).clamp(min=1e-2)

    def normalize(self, x):
        return ((x.double() - self.mean) / self.var.sqrt()).float()


@torch.no_grad()
def batched_fitness_static(weights, env_id="SwingRacket-v0", repeats=10, normalizer_state=None, device=0, seed=0,
                           precision="f64", max_steps=1001):
    """Fitness of every individual = mean episodic return over `repeats` episodes (`_get_rewards`, :143-172).
    weights: [P, n_params].  Returns (fitness [P], returns [P, repeats]) as CUDA tensors."""
    dev = torch.device("cuda", device)
    w = torch.as_tensor(weights, dtype=torch.float32, device=dev)
    pop = w.shape[0]
    n = pop * repeats
    env = TennisBatch(env_id, n, device=device, seed=seed, precision=precision, auto_reset=True)
    if w.shape[1] != num_params(env.obs_dim, env.act_dim):
        raise ValueError(f"weight vectors must have {num_params(env.obs_dim, env.act_dim)} entries")
    wb = w.repeat_interleave(repeats, dim=0)                    # env e evaluates individual e // repeats
    low = torch.full((env.act_dim,), -1.0, device=dev)
    high = torch.full((env.act_dim,), 1.0, device=dev)
    norm = BatchedNormalizer(n, env.obs_dim, dev, normalizer_state)
    obs = env.reset().clone()
    norm.observe(obs)
    hist = norm.normalize(obs)[:, :, None].repeat(1, 1, HISTORY_LEN)   # the first observation repeated 8 times
    ret = torch.zeros(n, dtype=torch.float64, device=dev)
    alive = torch.ones(n, dtype=torch.bool, device=dev)
    for _ in range(max_steps):
        action = torch.minimum(torch.maximum(gated_cnn_forward(wb, hist, env.act_dim), low), high)
        o, r, d, term, _ = env.step(action.contiguous())
        done = d.bool()
        # a finished env's obs is already the next episode's reset obs: the episode's own last obs is the terminal one
        step_obs = torch.where(done[:, None], term, o)
        norm.observe(step_obs)
        hist = torch.cat([hist[:, :, 1:], norm.normalize(step_obs)[:, :, None]], dim=2)
        ret += torch.where(alive, r.double(), torch.zeros_like(ret))
        alive &= ~done
        if not bool(alive.any()):
            break
    env.close()
    per_episode = ret.reshape(pop, repeats)
    return per_episode.mean(dim=1), per_episode


class EsEvaluator:
    """batched_fitness_static on the device: the GatedCNN, the normalisers, the history and the returns live in HBM and are
    advanced by es_kernel between env steps (tb_es_begin / tb_es_rollout), so nothing between two env steps runs on the host.
    One context is kept across generations; each generation continues the envs' episode counters, so it gets fresh
    placements.  env_id_offset shards a population over contexts (env i of this one is global env env_id_offset + i)."""

    # env steps per tb_es_rollout call, with one 1-byte read of alive.any() after each: one whole SwingRacket-v0 episode
    # (every one takes 26 steps), so a SwingRacket-v0 generation is one call; a 1001-step Tennisbot-v0 one is 39
    CHUNK = 26

    def __init__(self, env_id, individuals, repeats, device=0, seed=0, precision="f64", env_id_offset=0):
        self.individuals, self.repeats = int(individuals), int(repeats)
        if self.individuals < 1 or self.repeats < 1:
            raise ValueError(f"EsEvaluator: individuals and repeats must be >= 1, got {individuals}, {repeats}")
        self.env = TennisBatch(env_id, self.individuals * self.repeats, device=device, seed=seed, precision=precision,
                               auto_reset=True, env_id_offset=env_id_offset)
        n, dev = self.env.num_envs, self.env.device
        self.num_params = num_params(self.env.obs_dim, self.env.act_dim)
        self.ret = torch.zeros(n, dtype=torch.float64, device=dev)
        self.alive = torch.zeros(n, dtype=torch.uint8, device=dev)
        self.steps_run = 0  # env steps the last evaluate() ran

    def close(self):
        self.env.close()

    def _normalizer(self, normalizer_state):
        if normalizer_state is None:
            return None
        dev, od = self.env.device, self.env.obs_dim
        return torch.stack([torch.as_tensor(x, dtype=torch.float64, device=dev).reshape(od) for x in normalizer_state[:3]])

    @torch.no_grad()
    def evaluate(self, weights, normalizer_state=None, max_steps=1001):
        """weights [individuals, num_params]; normalizer_state: the master's (n, mean, mean_diff, var) as BatchedNormalizer takes
        it (var is ignored: observe overwrites it).  Returns (fitness [individuals], returns [individuals, repeats]) like
        batched_fitness_static: the return of every env summed until its first done or max_steps."""
        if int(max_steps) < 1:
            raise ValueError(f"EsEvaluator.evaluate: max_steps must be >= 1, got {max_steps}")
        w = torch.as_tensor(weights, dtype=torch.float32, device=self.env.device).contiguous()
        if tuple(w.shape) != (self.individuals, self.num_params):
            raise ValueError(f"weights must have shape ({self.individuals}, {self.num_params}), got {tuple(w.shape)}")
        self.env.es_begin(w, self._normalizer(normalizer_state))
        return self.run(max_steps)

    @torch.no_grad()
    def evaluate_noise(self, theta, sigma, noise_seed, generation, normalizer_state=None, max_steps=1001):
        """evaluate() on the antithetic population the library draws around theta [num_params]: global individual
        g = env_id_offset // repeats + p is theta + sigma * eps_{g // 2} (g even) or theta - sigma * eps_{g // 2} (g odd), eps
        keyed by (noise_seed, direction, generation) as tb_es_begin_noise documents.  individuals must be even."""
        self.begin_noise(theta, sigma, noise_seed, generation, normalizer_state)
        return self.run(max_steps)

    def begin_noise(self, theta, sigma, noise_seed, generation, normalizer_state=None):
        """The first half of evaluate_noise: draw the population and start the generation (no synchronisation)."""
        th = torch.as_tensor(theta, dtype=torch.float32, device=self.env.device).reshape(-1).contiguous()
        if th.numel() != self.num_params:
            raise ValueError(f"theta must have {self.num_params} entries, got {th.numel()}")
        self.env.es_begin_noise(th, self.individuals, sigma, noise_seed, generation, self._normalizer(normalizer_state))

    @torch.no_grad()
    def run(self, max_steps=1001):
        """Roll the started generation out in CHUNK-step calls until every env is done or max_steps; returns
        (fitness [individuals], returns [individuals, repeats])."""
        if int(max_steps) < 1:
            raise ValueError(f"EsEvaluator.run: max_steps must be >= 1, got {max_steps}")
        steps = 0
        while steps < max_steps:
            k = min(self.CHUNK, int(max_steps) - steps)
            self.env.es_rollout(k, self.ret, self.alive)
            steps += k
            if not bool(self.alive.any()):
                break
        self.steps_run = steps
        per_episode = self.ret.reshape(self.individuals, self.repeats).clone()
        return per_episode.mean(dim=1), per_episode
