"""Device-resident ES trainer: ARS V2-t (Mania, Guy and Recht 2018) around the in-kernel fitness rollout, for both envs.

The reference's trainer (`evolution_strategy_static.py`, SURVEY row 10) is an ARS / OpenAI-ES hybrid with an antithetic
population, top-K = 66 directions and 10 repeats per individual; its sigma, step size, population size and master-normaliser
rule are not recorded.  One generation here:
- draw the population in the library: direction j's noise eps_j is regenerated from Philox on (noise_seed, generation, j),
  individual 2j is theta + sigma eps_j and 2j + 1 is theta - sigma eps_j (tb_es_begin_noise), so no [individuals x floats]
  matrix exists outside the library and every shard draws its own directions;
- evaluate it with es_kernel (EsEvaluator.run): r+_j, r-_j = mean return over `repeats` episodes;
- keep the b = top_k directions with the largest max(r+_j, r-_j), sigma_R = standard deviation of those 2b fitnesses,
  theta += lr / (b sigma_R) sum_kept (r+_j - r-_j) eps_j, the sum regenerated in the library (tb_es_noise_combine);
- merge every observation the generation's normalisers took into the master normaliser (tb_es_normalizer_stats, Chan's
  formula), which seeds every env's normaliser of the next generation.
With env_id_offset and `gather`, each process evaluates a contiguous shard of the directions; the gathered fitness and
normaliser moments are the same on every shard, so every shard applies an identical update.
"""
import numpy as np
import torch

from .es_eval import EsEvaluator


def ars_update(fit_plus, fit_minus, top_k):
    """The ARS V2-t step from the fitnesses of D antithetic pairs.  Returns (dirs int64 [b], coef float64 [b], sigma_R) with
    b = min(top_k, D): the kept directions in decreasing order of max(r+, r-) (ties keep the lower index first),
    coef_k = (r+ - r-) / (b sigma_R) for them, and sigma_R the standard deviation (population, ddof 0) of their 2b
    fitnesses; coef is 0 when sigma_R is 0.  theta moves by lr * sum_k coef_k eps_{dirs[k]}.  Pure torch, any device."""
    fp = torch.as_tensor(fit_plus, dtype=torch.float64).reshape(-1)
    fm = torch.as_tensor(fit_minus, dtype=torch.float64, device=fp.device).reshape(-1)
    if fp.numel() != fm.numel() or fp.numel() == 0:
        raise ValueError(f"ars_update: fit_plus and fit_minus must hold the same number (>= 1) of directions, "
                         f"got {fp.numel()} and {fm.numel()}")
    if int(top_k) < 1:
        raise ValueError(f"ars_update: top_k must be >= 1, got {top_k}")
    b = min(int(top_k), fp.numel())
    dirs = torch.sort(torch.maximum(fp, fm), descending=True, stable=True).indices[:b]
    kp, km = fp[dirs], fm[dirs]
    sigma_r = torch.cat([kp, km]).std(correction=0)
    coef = torch.where(sigma_r > 0, (kp - km) / (b * sigma_r), torch.zeros_like(kp))
    return dirs, coef, sigma_r


def merge_moments(a, b):
    """Chan's merge of two (count, mean, M2) float64 [3, dim] moment sets."""
    n = a[0] + b[0]
    frac = torch.where(n > 0, b[0] / torch.where(n > 0, n, torch.ones_like(n)), torch.zeros_like(n))
    delta = b[1] - a[1]
    return torch.stack([n, a[1] + delta * frac, a[2] + b[2] + delta * delta * (a[0] * frac)])


class EsTrainer:
    """ARS V2-t on the device (see the module docstring).

    directions: antithetic pairs this trainer evaluates (2 x directions individuals, 2 x directions x repeats envs); with
    env_id_offset (a multiple of 2 x repeats) they are global directions env_id_offset / (2 repeats) onwards, and `gather`
    assembles the whole population's tensors from this shard's along dim 0 (identity for one process;
    sharding.all_gather for torch.distributed).  top_k is clipped to the global number of directions.
    From the reference: the antithetic population, top_k = 66 and repeats = 10.  Not recorded there and chosen here:
    sigma = 0.05 and lr = 0.1 (the best of six (sigma, lr) pairs in 40-generation SwingRacket-v0 runs from theta = 0, DESIGN
    section 4.2), ARS V2-t's update rule
    and step normalisation by sigma_R, and the master normaliser as the union of every observation the envs' normalisers
    took.  theta: the starting parameters (default zeros), e.g. tests/golden/es_swing_weights.npz."""

    def __init__(self, env_id, directions, repeats=10, top_k=66, sigma=0.05, lr=0.1, seed=0, noise_seed=0, device=0,
                 precision="f64", env_id_offset=0, gather=None, theta=None, max_steps=1001):
        if int(directions) < 1 or int(top_k) < 1 or not (float(sigma) > 0) or not np.isfinite(float(sigma)):
            raise ValueError(f"EsTrainer: directions and top_k must be >= 1 and sigma a finite number above 0, "
                             f"got {directions}, {top_k}, {sigma}")
        self.env_id, self.directions, self.repeats, self.top_k = env_id, int(directions), int(repeats), int(top_k)
        self.sigma, self.lr, self.seed, self.noise_seed = float(sigma), float(lr), int(seed), int(noise_seed)
        self.max_steps = int(max_steps)
        self.gather = gather if gather is not None else (lambda t: t)
        self.ev = EsEvaluator(env_id, 2 * self.directions, self.repeats, device=device, seed=seed, precision=precision,
                              env_id_offset=env_id_offset)
        self.env, dev = self.ev.env, self.ev.env.device
        self.theta = torch.zeros(self.ev.num_params, dtype=torch.float32, device=dev)
        if theta is not None:
            self.set_theta(theta)
        self.normalizer = torch.zeros((3, self.env.obs_dim), dtype=torch.float64, device=dev)  # master (n, mean, M2)
        self.generation = 0
        self.fitness = None  # the last generation's fitness of the whole population (individual 2j: +, 2j + 1: -)

    def close(self):
        self.ev.close()

    def set_theta(self, theta):
        th = torch.as_tensor(theta, dtype=torch.float32).reshape(-1)
        if th.numel() != self.ev.num_params:
            raise ValueError(f"theta must have {self.ev.num_params} entries, got {th.numel()}")
        self.theta = th.to(self.env.device).contiguous()

    @torch.no_grad()
    def step(self, timings=None):
        """One generation.  Returns its statistics: mean and max fitness of the population, sigma_R, the master normaliser's
        count after the merge, and the env steps run.  timings: a dict that receives the wall time in seconds of each phase
        (draw, rollout, update, normalizer), with a device synchronisation at every boundary; None for no synchronisation."""
        clock = _Clock(timings)
        gen = self.generation
        self.ev.begin_noise(self.theta, self.sigma, self.noise_seed, gen, self.normalizer)
        clock.mark("draw")
        fit_local, _ = self.ev.run(self.max_steps)
        clock.mark("rollout")
        fit = self.fitness = self.gather(fit_local)
        dirs, coef, sigma_r = ars_update(fit[0::2], fit[1::2], self.top_k)
        step = self.env.es_noise_combine(dirs, (self.lr * coef).float(), self.noise_seed, gen)
        self.theta = self.theta + step
        clock.mark("update")
        for row in self.gather(self.env.es_normalizer_stats()[None]):
            self.normalizer = merge_moments(self.normalizer, row)
        clock.mark("normalizer")
        self.generation += 1
        return dict(generation=gen, fitness_mean=float(fit.mean()), fitness_max=float(fit.max()), sigma_r=float(sigma_r),
                    norm_count=float(self.normalizer[0, 0]), steps=self.ev.steps_run)

    def state_dict(self):
        """theta, the master normaliser (n, mean, M2), the next generation and the seeds, on the CPU."""
        return dict(env_id=self.env_id, theta=self.theta.cpu(), normalizer=self.normalizer.cpu(), generation=self.generation,
                    seed=self.seed, noise_seed=self.noise_seed)

    def load_state_dict(self, state):
        """Restore theta, the master normaliser, the generation and the noise seed.  The env seed is the context's and cannot
        change, so it must match; the envs' episode counters are not part of the state (placements differ after a restore)."""
        if state["env_id"] != self.env_id or int(state["seed"]) != self.seed:
            raise ValueError(f"state of {state['env_id']} seed {state['seed']} loaded into {self.env_id} seed {self.seed}")
        self.set_theta(state["theta"])
        self.normalizer = torch.as_tensor(state["normalizer"], dtype=torch.float64).to(self.env.device).reshape(3, -1).clone()
        self.generation, self.noise_seed = int(state["generation"]), int(state["noise_seed"])


class _Clock:
    def __init__(self, out):
        self.out = out
        if out is not None:
            import time

            self._now = time.perf_counter
            torch.cuda.synchronize()
            self.t = self._now()

    def mark(self, name):
        if self.out is not None:
            torch.cuda.synchronize()
            t = self._now()
            self.out[name] = self.out.get(name, 0.0) + t - self.t
            self.t = t
