"""The device-resident ES trainer: seeded population (tb_es_begin_noise), noise combination (tb_es_noise_combine), the
generation's normaliser moments (tb_es_normalizer_stats) and es_train.EsTrainer (ARS V2-t).

CPU tests restate ars_update in numpy and check the argument errors.  GPU tests (f64 contexts, both envs) restate the noise on
the host from oracle.binding.philox and the documented Box-Muller, feed a torch restatement of the population to tb_es_begin,
rebuild the normaliser moments from the traced observations in numpy, and join two shards with a concatenating gather.
"""
import ctypes as C
import re
import threading
from pathlib import Path

import numpy as np
import pytest
import torch

ROOT = Path(__file__).resolve().parent.parent
GOLD = Path(__file__).parent / "golden"
ENVS = {"SwingRacket-v0": (6, 6, 766), "Tennisbot-v0": (12, 2, 858)}


def _np_ars(fp, fm, top_k):
    """ARS V2-t selection and coefficients in numpy."""
    fp, fm = np.asarray(fp, np.float64), np.asarray(fm, np.float64)
    b = min(top_k, fp.size)
    dirs = np.argsort(-np.maximum(fp, fm), kind="stable")[:b]
    sr = np.concatenate([fp[dirs], fm[dirs]]).std()
    coef = (fp[dirs] - fm[dirs]) / (b * sr) if sr > 0 else np.zeros(b)
    return dirs, coef, sr


# ------------------------------------------------------------------------------------------------ CPU
@pytest.mark.parametrize("case", ["random", "ties", "top_k_above_directions", "all_equal"])
def test_ars_update_matches_numpy(case):
    from tennisbot_rl_b200.es_train import ars_update

    rng = np.random.default_rng(3)
    d, top_k = 200, 66
    fp, fm = rng.normal(10, 3, d), rng.normal(10, 3, d)
    if case == "ties":  # whole-number fitnesses: many equal max(r+, r-), ties across + and - and within one direction
        fp, fm = rng.integers(0, 12, d).astype(float), rng.integers(0, 12, d).astype(float)
        fm[:5] = fp[:5]
    elif case == "top_k_above_directions":
        d = 40
        fp, fm = fp[:d], fm[:d]
    elif case == "all_equal":
        fp, fm = np.full(d, 4.0), np.full(d, 4.0)
    dirs, coef, sr = ars_update(torch.from_numpy(fp), torch.from_numpy(fm), top_k)
    rd, rc, rs = _np_ars(fp, fm, top_k)
    np.testing.assert_array_equal(dirs.numpy(), rd)
    np.testing.assert_allclose(coef.numpy(), rc, rtol=1e-12, atol=0)
    assert abs(float(sr) - rs) <= 1e-12 * max(rs, 1.0)
    assert dirs.dtype == torch.int64 and coef.dtype == torch.float64
    assert len(dirs) == min(top_k, d)


def test_ars_update_rejects_mismatched_inputs():
    from tennisbot_rl_b200.es_train import ars_update

    with pytest.raises(ValueError, match="same number"):
        ars_update(torch.zeros(3), torch.zeros(4), 2)
    with pytest.raises(ValueError, match="top_k"):
        ars_update(torch.zeros(3), torch.zeros(3), 0)


def test_merge_moments_is_chan():
    from tennisbot_rl_b200.es_train import merge_moments

    rng = np.random.default_rng(1)
    a, b = rng.normal(3, 2, (57, 4)), rng.normal(-1, 0.5, (13, 4))
    mom = lambda x: torch.from_numpy(np.stack([np.full(4, len(x), float), x.mean(0), ((x - x.mean(0)) ** 2).sum(0)]))  # noqa: E731
    got = merge_moments(mom(a), mom(b)).numpy()
    np.testing.assert_allclose(got, mom(np.concatenate([a, b])).numpy(), rtol=1e-12)
    np.testing.assert_array_equal(merge_moments(torch.zeros(3, 4, dtype=torch.float64), mom(b)).numpy(), mom(b).numpy())


def test_es_noise_entry_points_reject_arguments_without_a_device():
    from tennisbot_rl_b200 import _lib, build

    build.build_library()
    L = _lib.load()
    fake = C.c_void_p(16)  # never dereferenced: every call below fails on its arguments first

    def err(rc):
        assert rc != 0
        return L.tb_last_error().decode()

    begin = lambda ind, sigma, theta=fake: L.tb_es_begin_noise(None, theta, ind, 766, sigma, 1, 0, None, None)  # noqa: E731
    assert "d_theta is NULL" in err(begin(4, 0.1, None))
    assert "individuals must be >= 1" in err(begin(0, 0.1))
    assert "individuals must be even" in err(begin(3, 0.1))
    for bad in (0.0, -0.5, float("nan"), float("inf")):
        assert "sigma must be a finite number above 0" in err(begin(4, bad))
    assert "context is NULL" in err(begin(4, 0.1))
    assert "count must be >= 0" in err(L.tb_es_noise_combine(None, fake, fake, -1, 0, 0, fake, None))
    assert "d_dirs and d_coef are required" in err(L.tb_es_noise_combine(None, None, fake, 2, 0, 0, fake, None))
    assert "d_dirs and d_coef are required" in err(L.tb_es_noise_combine(None, fake, None, 2, 0, 0, fake, None))
    assert "d_out is NULL" in err(L.tb_es_noise_combine(None, None, None, 0, 0, 0, None, None))
    assert "context is NULL" in err(L.tb_es_noise_combine(None, None, None, 0, 0, 0, fake, None))
    assert "d_out is NULL" in err(L.tb_es_normalizer_stats(None, None, None))
    assert "context is NULL" in err(L.tb_es_normalizer_stats(None, fake, None))


def test_es_floats_and_header_constants_still_agree():
    from tennisbot_rl_b200 import _lib, build, es_eval

    build.build_library()
    L = _lib.load()
    header = (ROOT / "include" / "tennisbot_b200.h").read_text()
    const = lambda name: int(re.search(rf"#define {name} (\d+)", header).group(1))  # noqa: E731
    for kind, od, ad, floats in ((_lib.ENV_SWING, 6, 6, "TB_ES_FLOATS"), (_lib.ENV_HIT, 12, 2, "TB_ES_FLOATS_HIT")):
        assert L.tb_es_floats(kind) == const(floats) == es_eval.num_params(od, ad)
    for name in ("tb_es_begin_noise", "tb_es_noise_combine", "tb_es_normalizer_stats"):
        assert name in _lib.EXPORTS and re.search(rf"\bint {name}\(", header)
    src = (ROOT / "tennisbot_rl_b200" / "csrc" / "tb_kernels.cu").read_text()
    assert re.search(r"constexpr uint32_t kStreamEsNoise = 3u;", src) and "(3 << 28)" in header  # the documented stream word


# ------------------------------------------------------------------------------------------------ GPU helpers
def _eps_host(binding, seed, j, gen, floats):
    """eps_j of generation gen, float64, as tb_es_begin_noise documents it."""
    out = np.empty(4 * ((floats + 3) // 4))
    for q in range(len(out) // 4):
        r = binding.philox(seed, j, gen, (3 << 28) | (q << 4)).astype(np.float64)
        for k in range(2):
            u1, u2 = (r[2 * k] + 0.5) / 2.0 ** 32, r[2 * k + 1] / 2.0 ** 32
            rho = np.sqrt(-2.0 * np.log(u1))
            out[4 * q + 2 * k], out[4 * q + 2 * k + 1] = rho * np.cos(2 * np.pi * u2), rho * np.sin(2 * np.pi * u2)
    return out[:floats]


def _eps_device(b, dirs, seed, gen):
    """eps_j for every j in dirs, read back through tb_es_noise_combine with one-hot coefficients: float32 [len(dirs), floats]."""
    one = torch.ones(1, dtype=torch.float32, device=b.device)
    rows = [b.es_noise_combine(torch.tensor([int(j)], dtype=torch.int64, device=b.device), one, seed, gen) for j in dirs]
    return torch.stack(rows)


def _master_data(od, n0, seed):
    rng = np.random.default_rng(seed)
    return rng.normal(rng.normal(0, 1, od), rng.uniform(0.2, 2.0, od), (n0, od))


def _moments(x):
    x = np.asarray(x, np.float64)
    m = x.mean(axis=0)
    return np.stack([np.full(x.shape[1], float(len(x))), m, ((x - m) ** 2).sum(axis=0)])


# ------------------------------------------------------------------------------------------------ GPU
@pytest.mark.gpu
@pytest.mark.parametrize("env_id", list(ENVS))
def test_noise_matches_host_restatement_and_is_standard_normal(oracle_lib, env_id):
    from tennisbot_rl_b200.batch import TennisBatch

    floats = ENVS[env_id][2]
    b = TennisBatch(env_id, 8, seed=0)
    seed = 0x1234_5678_9ABC
    dirs = [0, 1, 2, 65, 4097, 2 ** 33 + 5]
    worst = 0.0
    for gen in (0, 7):
        dev = _eps_device(b, dirs, seed, gen).cpu().numpy()
        for row, j in zip(dev, dirs):
            host = _eps_host(oracle_lib, seed, j, gen, floats)
            worst = max(worst, float(np.abs(row - host).max()))
    assert worst <= 1e-6, worst

    # >= 10^6 draws: two generations of 1400 directions
    nd = 1400
    e = np.stack([_eps_device(b, range(nd), seed, gen).cpu().numpy().astype(np.float64) for gen in (0, 1)])  # [2, nd, floats]
    x = e.reshape(-1)
    n = x.size
    assert n >= 10 ** 6
    se = 1.0 / np.sqrt(n)
    assert abs(x.mean()) < 4 * se, x.mean()
    assert abs(x.var() - 1.0) < 4 * np.sqrt(2.0) * se, x.var()
    corr = lambda a, c: float(np.corrcoef(a.reshape(-1), c.reshape(-1))[0, 1])  # noqa: E731
    pairs = {"parameter": (e[:, :, :-1], e[:, :, 1:]), "direction": (e[:, :-1], e[:, 1:]), "generation": (e[0], e[1])}
    for name, (a, c) in pairs.items():
        r = corr(a, c)
        assert abs(r) < 4 / np.sqrt(a.size), (name, r)
    print(f"{env_id}: worst |eps - host| {worst:.2e}; {n} draws mean {x.mean():.2e} var {x.var():.5f}; "
          + ", ".join(f"corr({k}) {corr(*v):.1e}" for k, v in pairs.items()))
    b.close()


@pytest.mark.gpu
@pytest.mark.parametrize("env_id,individuals,repeats", [("SwingRacket-v0", 96, 10), ("Tennisbot-v0", 64, 4)])
def test_population_is_the_documented_one(env_id, individuals, repeats):
    """Returns from tb_es_begin_noise equal, bit for bit, those of tb_es_begin fed theta +- float32(sigma * eps) (no FMA)."""
    from tennisbot_rl_b200 import es_eval

    od, _, floats = ENVS[env_id]
    rng = np.random.default_rng(5)
    theta = torch.from_numpy((0.2 * rng.standard_normal(floats)).astype(np.float32)).cuda()
    if env_id == "SwingRacket-v0":
        theta = torch.from_numpy(np.load(GOLD / "es_swing_weights.npz")["weights"].astype(np.float32)).cuda()
    master = _moments(_master_data(od, 300, 2))
    state = (master[0], master[1], master[2], master[2] / master[0])
    sigma, seed, gen = 0.07, 99, 3
    a = es_eval.EsEvaluator(env_id, individuals, repeats, seed=12)
    fit_a, ret_a = a.evaluate_noise(theta, sigma, seed, gen, state)
    eps = _eps_device(a.env, range(individuals // 2), seed, gen)
    d = torch.tensor(sigma, dtype=torch.float32, device=eps.device) * eps
    pop = torch.stack([theta + d, theta - d], dim=1).reshape(individuals, floats)
    b = es_eval.EsEvaluator(env_id, individuals, repeats, seed=12)
    fit_b, ret_b = b.evaluate(pop, state)
    assert torch.equal(ret_a, ret_b) and torch.equal(fit_a, fit_b)
    assert float(fit_a.std()) > 0  # the individuals differ
    print(f"{env_id}: {individuals * repeats} envs, {a.steps_run} steps, fitness {fit_a.min():.3f}..{fit_a.max():.3f}")
    a.close()
    b.close()


@pytest.mark.gpu
@pytest.mark.parametrize("env_id", list(ENVS))
def test_noise_combine_matches_float64_sum(env_id):
    from tennisbot_rl_b200.batch import TennisBatch

    floats = ENVS[env_id][2]
    b = TennisBatch(env_id, 8, seed=0)
    rng = np.random.default_rng(7)
    dirs = rng.choice(5000, 66, replace=False).astype(np.int64)
    coef = rng.normal(0, 1, 66).astype(np.float32)
    out = b.es_noise_combine(torch.from_numpy(dirs).cuda(), torch.from_numpy(coef).cuda(), 11, 4).cpu().numpy()
    eps = _eps_device(b, dirs, 11, 4).cpu().numpy().astype(np.float64)
    ref = coef.astype(np.float64) @ eps
    np.testing.assert_allclose(out, ref, rtol=1e-6, atol=1e-12)
    # count 0: zeros; and the result does not depend on the order the directions are drawn in beyond float64 rounding
    zero = b.es_noise_combine(torch.zeros(0, dtype=torch.int64, device="cuda"), torch.zeros(0, device="cuda"), 11, 4)
    assert not zero.any()
    b.close()


@pytest.mark.gpu
@pytest.mark.parametrize("env_id,individuals,repeats,k", [("SwingRacket-v0", 128, 10, 26), ("Tennisbot-v0", 64, 4, 1001)])
def test_normalizer_stats_match_numpy(env_id, individuals, repeats, k):
    """es_normalizer_stats merged with a master built from real data = numpy float64 moments of the master's data plus every
    observation the normalisers took: each env's traced observations 0 .. d (d = its first done step; 0 .. k if none)."""
    from tennisbot_rl_b200.batch import TennisBatch
    from tennisbot_rl_b200.es_train import merge_moments

    od, _, floats = ENVS[env_id]
    n = individuals * repeats
    b = TennisBatch(env_id, n, seed=21)
    x0 = _master_data(od, 400, 9)
    master = _moments(x0)
    theta = torch.from_numpy((0.2 * np.random.default_rng(1).standard_normal(floats)).astype(np.float32)).cuda()
    b.es_begin_noise(theta, individuals, 0.1, 5, 0, torch.from_numpy(master).cuda())
    obs = torch.zeros((k + 1, n, od), device="cuda")
    done = torch.zeros((k, n), dtype=torch.uint8, device="cuda")
    ret, alive = torch.zeros(n, dtype=torch.float64, device="cuda"), torch.zeros(n, dtype=torch.uint8, device="cuda")
    b.es_rollout(k, ret, alive, obs=obs, done=done)
    stats = b.es_normalizer_stats().cpu().numpy()
    obs, done = obs.cpu().numpy(), done.cpu().numpy()
    first = np.where(done.any(axis=0), done.argmax(axis=0), k)  # last consumed observation index per env
    taken = np.concatenate([obs[: first[e] + 1, e] for e in range(n)])
    np.testing.assert_array_equal(stats[0], np.full(od, float(len(taken))))
    merged = merge_moments(torch.from_numpy(master), torch.from_numpy(stats)).numpy()
    ref = _moments(np.concatenate([x0, taken]))
    np.testing.assert_allclose(merged, ref, rtol=1e-10, atol=1e-12)
    np.testing.assert_allclose(stats, _moments(taken), rtol=1e-9, atol=1e-9)
    if env_id == "SwingRacket-v0":
        assert (first == 25).all()  # every SwingRacket-v0 episode takes 26 steps: the last one ends it
    else:
        assert len(np.unique(first)) > 1  # Tennisbot-v0 envs die at different steps
    print(f"{env_id}: {n} envs x {k} steps, {len(taken)} observations taken, first done at steps "
          f"{first.min()}..{first.max()} ({len(np.unique(first))} distinct), alive at the end {int(alive.sum())}")
    b.close()


@pytest.mark.gpu
@pytest.mark.parametrize("env_id", list(ENVS))
def test_trainer_step_is_numpy_ars(env_id):
    from tennisbot_rl_b200.es_train import EsTrainer

    floats = ENVS[env_id][2]
    theta0 = (0.1 * np.random.default_rng(4).standard_normal(floats)).astype(np.float32)
    tr = EsTrainer(env_id, 48, repeats=4, top_k=20, sigma=0.05, lr=0.03, seed=3, noise_seed=17, theta=theta0)
    tr.generation = 2
    st = tr.step()
    fit = tr.fitness.cpu().numpy()
    dirs, coef, sr = _np_ars(fit[0::2], fit[1::2], 20)
    eps = _eps_device(tr.env, dirs, 17, 2).cpu().numpy().astype(np.float64)
    want = theta0.astype(np.float64) + (0.03 * coef).astype(np.float32).astype(np.float64) @ eps
    np.testing.assert_allclose(tr.theta.cpu().numpy(), want, rtol=0, atol=1e-6)
    assert sr > 0  # the kept fitnesses differ, so the update is not zero
    assert abs(st["sigma_r"] - sr) <= 1e-12 * max(sr, 1.0) and st["generation"] == 2 and tr.generation == 3
    assert float(np.abs(tr.theta.cpu().numpy() - theta0).max()) > 1e-4  # theta moved
    sd = tr.state_dict()
    tr2 = EsTrainer(env_id, 48, repeats=4, seed=3)
    tr2.load_state_dict(sd)
    assert torch.equal(tr2.theta, tr.theta) and torch.equal(tr2.normalizer, tr.normalizer) and tr2.generation == 3
    assert tr2.noise_seed == 17
    tr.close()
    tr2.close()


class _Join:
    """A concatenating gather for shards run in threads of one process."""

    def __init__(self, k):
        self.barrier, self.slots = threading.Barrier(k), [None] * k

    def gather(self, i):
        def g(t):
            self.slots[i] = t
            self.barrier.wait()
            out = torch.cat(self.slots)
            self.barrier.wait()
            return out
        return g


@pytest.mark.gpu
def test_two_shards_reproduce_the_full_trainer():
    from tennisbot_rl_b200.es_train import EsTrainer

    directions, repeats = 64, 10
    saved = np.load(GOLD / "es_swing_weights.npz")["weights"]
    master = torch.from_numpy(_moments(_master_data(6, 250, 3))).cuda()
    kw = dict(repeats=repeats, top_k=20, sigma=0.05, lr=0.05, seed=8, noise_seed=23, theta=saved)
    full = EsTrainer("SwingRacket-v0", directions, **kw)
    full.normalizer = master.clone()
    full.step()
    join = _Join(2)
    h = directions // 2
    shards = [EsTrainer("SwingRacket-v0", h, env_id_offset=i * 2 * h * repeats, gather=join.gather(i), **kw) for i in range(2)]
    errors = []

    def run(t):
        try:
            t.normalizer = master.clone()
            t.step()
        except Exception as e:  # noqa: BLE001  (reported below)
            errors.append(e)
            join.barrier.abort()

    threads = [threading.Thread(target=run, args=(t,)) for t in shards]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert not errors, errors
    for t in shards:
        assert torch.equal(t.fitness, full.fitness)
        assert torch.equal(t.theta, full.theta)
        np.testing.assert_allclose(t.normalizer.cpu().numpy(), full.normalizer.cpu().numpy(), rtol=1e-12, atol=0)
    assert torch.equal(shards[0].theta, shards[1].theta) and torch.equal(shards[0].normalizer, shards[1].normalizer)
    for t in shards + [full]:
        t.close()


# SwingRacket-v0 from theta = 0: 128 directions x 10 repeats (2560 envs), 40 generations, the trainer's defaults (sigma 0.05,
# lr 0.1), about 0.1 s on a B200.  Measured on an NVIDIA B200 (1000 W power limit): mean fitness 0.11 in the first generation,
# 20.7 by the 7th, 24.65 in the 40th (max of the last five).  The threshold leaves a quarter of that as margin; the saved ES
# policy of the reference scores 16.0 on the same evaluator with fresh normalisers.
SWING_LEARN = dict(directions=128, generations=40)
SWING_THRESHOLD = 18.0


@pytest.mark.gpu
def test_swing_learns_from_zero():
    from tennisbot_rl_b200.es_train import EsTrainer

    tr = EsTrainer("SwingRacket-v0", SWING_LEARN["directions"], seed=1, noise_seed=2)
    curve = [tr.step()["fitness_mean"] for _ in range(SWING_LEARN["generations"])]
    saved = np.load(GOLD / "es_swing_weights.npz")["weights"]
    saved_fit, _ = tr.ev.evaluate(np.tile(saved, (2 * SWING_LEARN["directions"], 1)))
    print("SwingRacket-v0 mean fitness per generation:", " ".join(f"{c:.2f}" for c in curve))
    print(f"saved ES policy on the same evaluator (fresh normalisers): {float(saved_fit.mean()):.2f}")
    assert max(curve[-5:]) > SWING_THRESHOLD and curve[-1] > curve[0]
    tr.close()


@pytest.mark.gpu
def test_hit_fitness_improves():
    from tennisbot_rl_b200.es_train import EsTrainer

    tr = EsTrainer("Tennisbot-v0", 64, repeats=4, top_k=32, seed=1, noise_seed=2)
    curve = [tr.step()["fitness_mean"] for _ in range(8)]
    print("Tennisbot-v0 mean fitness per generation:", " ".join(f"{c:.3f}" for c in curve))
    assert max(curve[1:]) > curve[0]
    tr.close()
