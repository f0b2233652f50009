"""The in-kernel ES fitness rollout (tb_es_begin / tb_es_rollout, es_eval.EsEvaluator, SURVEY 8(f)-2).

GPU tests compare the kernel's traces with the reference maths rebuilt on the host (float64 normaliser in numpy, the torch
GatedCNN of es_eval.gated_cnn_forward), with the CPU oracle stepped by the traced actions, and with the torch adapter
batched_fitness_static.  After an env's first done it acts 0 and its normaliser stops, so traces are compared while it is alive.
"""
import ctypes as C
import re
from pathlib import Path

import numpy as np
import pytest
import torch

ROOT = Path(__file__).resolve().parent.parent
GOLD = Path(__file__).parent / "golden"
ENVS = {"SwingRacket-v0": (6, 6), "Tennisbot-v0": (12, 2)}


# ------------------------------------------------------------------------------------------------ CPU
def test_es_floats_match_gated_cnn_and_header():
    from tennisbot_rl_b200 import _lib, build, es_eval

    build.build_library()
    L = _lib.load()
    header = (ROOT / "include" / "tennisbot_b200.h").read_text()
    const = lambda name: int(re.search(rf"#define {name} (\d+)", header).group(1))  # noqa: E731
    assert L.tb_es_floats(_lib.ENV_SWING) == es_eval.num_params(6, 6) == const("TB_ES_FLOATS") == _lib.ES_FLOATS == 766
    assert L.tb_es_floats(_lib.ENV_HIT) == es_eval.num_params(12, 2) == const("TB_ES_FLOATS_HIT") == _lib.ES_FLOATS_HIT == 858
    assert L.tb_es_floats(7) == -1
    assert const("TB_ES_HISTORY") == _lib.ES_HISTORY == es_eval.HISTORY_LEN


def test_es_argument_errors_without_a_device():
    from tennisbot_rl_b200 import _lib, build, es_eval

    build.build_library()
    L = _lib.load()
    fake = C.c_void_p(16)  # never dereferenced: every call below fails on its arguments first

    def err(rc):
        assert rc != 0
        return L.tb_last_error().decode()

    assert "d_weights is NULL" in err(L.tb_es_begin(None, None, 4, 766, None, None))
    assert "individuals must be >= 1" in err(L.tb_es_begin(None, fake, 0, 766, None, None))
    assert "context is NULL" in err(L.tb_es_begin(None, fake, 4, 766, None, None))
    assert "k_steps must be >= 1" in err(L.tb_es_rollout(None, 0, fake, fake, None, None, None, None, None))
    assert "d_return and d_alive are required" in err(L.tb_es_rollout(None, 3, None, fake, None, None, None, None, None))
    assert "d_return and d_alive are required" in err(L.tb_es_rollout(None, 3, fake, None, None, None, None, None, None))
    assert "context is NULL" in err(L.tb_es_rollout(None, 3, fake, fake, None, None, None, None, None))
    for ind, rep in ((0, 10), (4, 0)):
        with pytest.raises(ValueError, match="individuals and repeats"):
            es_eval.EsEvaluator("SwingRacket-v0", ind, rep)


# ------------------------------------------------------------------------------------------------ GPU helpers
def _master(od, seed):
    """A non-trivial master normaliser (n, mean, mean_diff) as a [3, od] float64 array."""
    rng = np.random.default_rng(seed)
    n = np.full(od, 57.0)
    return np.stack([n, rng.normal(0.0, 0.5, od), n * rng.uniform(0.05, 2.0, od)])


def _swing_population(individuals, seed):
    """The saved ES policy with antithetic perturbations, as the ES trainer samples them."""
    saved = np.load(GOLD / "es_swing_weights.npz")["weights"].astype(np.float32)
    eps = np.random.default_rng(seed).standard_normal((individuals // 2, saved.size)).astype(np.float32)
    return np.concatenate([saved + 0.05 * eps, saved - 0.05 * eps])


def _random_population(individuals, floats, seed):
    return (0.3 * np.random.default_rng(seed).standard_normal((individuals, floats))).astype(np.float32)


def _traced(env_id, individuals, repeats, weights, master, k, seed, precision="f64"):
    """One traced tb_es_rollout of k steps right after tb_es_begin on a fresh context."""
    from tennisbot_rl_b200.batch import TennisBatch

    od, ad = ENVS[env_id]
    n = individuals * repeats
    b = TennisBatch(env_id, n, seed=seed, precision=precision)
    dev = b.device
    b.es_begin(torch.from_numpy(np.ascontiguousarray(weights, np.float32)).to(dev),
               None if master is None else torch.from_numpy(master).to(dev))
    tr = dict(obs=torch.zeros((k + 1, n, od), device=dev), actions=torch.zeros((k, n, ad), device=dev),
              reward=torch.zeros((k, n), device=dev), done=torch.zeros((k, n), dtype=torch.uint8, device=dev))
    ret, alive = torch.zeros(n, dtype=torch.float64, device=dev), torch.zeros(n, dtype=torch.uint8, device=dev)
    b.es_rollout(k, ret, alive, **tr)
    torch.cuda.synchronize()
    out = {key: v.cpu().numpy() for key, v in tr.items()}
    out["ret"], out["alive"] = ret.cpu().numpy(), alive.cpu().numpy()
    b.close()
    # alive_before[t]: no done before step t
    alive_before = np.ones((k + 1, n), bool)
    for t in range(k):
        alive_before[t + 1] = alive_before[t] & (out["done"][t] == 0)
    out["alive_before"] = alive_before
    return out


def _check_actions(tr, weights, repeats, master, ad, bar=1e-5):
    """Rebuild every env's normaliser in float64 from the traced observations, run the torch GatedCNN on the rebuilt history
    and compare with the traced actions while the env is alive.  Returns the largest deviation."""
    from tennisbot_rl_b200 import es_eval

    obs = tr["obs"]
    k, n, od = obs.shape[0] - 1, obs.shape[1], obs.shape[2]
    wb = torch.from_numpy(np.repeat(weights, repeats, axis=0))
    cnt = np.zeros((n, od)) if master is None else np.broadcast_to(master[0], (n, od)).copy()
    mean = np.zeros((n, od)) if master is None else np.broadcast_to(master[1], (n, od)).copy()
    md = np.zeros((n, od)) if master is None else np.broadcast_to(master[2], (n, od)).copy()

    def observe(x):
        nonlocal mean, md
        x = x.astype(np.float64)
        cnt[:] += 1.0
        last = mean.copy()
        mean = mean + (x - mean) / cnt
        md = md + (x - last) * (x - mean)
        return ((x - mean) / np.sqrt(np.maximum(md / cnt, 1e-2))).astype(np.float32)

    hist = np.repeat(observe(obs[0])[:, :, None], 8, axis=2)
    worst = 0.0
    for t in range(k):
        live = tr["alive_before"][t]
        with torch.no_grad():
            ref = es_eval.gated_cnn_forward(wb, torch.from_numpy(hist), ad).clamp(-1, 1).numpy()
        dev = np.abs(tr["actions"][t][live] - ref[live]).max(initial=0.0)
        assert dev <= bar, (t, dev)
        worst = max(worst, dev)
        assert not tr["actions"][t][~live].any()  # a dead env acts 0
        hist = np.concatenate([hist[:, :, 1:], observe(obs[t + 1])[:, :, None]], axis=2)
    return worst


# ------------------------------------------------------------------------------------------------ GPU
@pytest.mark.gpu
@pytest.mark.parametrize("env_id,individuals,repeats,k", [("SwingRacket-v0", 256, 16, 26), ("Tennisbot-v0", 256, 8, 1001)])
def test_es_trace_matches_reference_and_oracle(oracle_lib, env_id, individuals, repeats, k):
    """f64: actions = the torch GatedCNN on the float64 normaliser rebuilt from the traced observations (1e-5); the oracle stepped
    with the traced actions reproduces done exactly, rewards to 2e-6 and the observations; returns are the traced rewards
    summed until the first done, and EsEvaluator's fitness is their mean over repeats."""
    from tennisbot_rl_b200 import es_eval

    od, ad = ENVS[env_id]
    n, seed = individuals * repeats, 31
    weights = _swing_population(individuals, 3) if od == 6 else _random_population(individuals, 858, 3)
    master = _master(od, 5)
    tr = _traced(env_id, individuals, repeats, weights, master, k, seed)
    worst = _check_actions(tr, weights, repeats, master, ad)

    o = oracle_lib.OracleEnv(env_id, n, seed=seed, threads=8)
    np.testing.assert_array_equal(tr["obs"][0], o.reset())
    obs_bar = 2e-6 if od == 6 else 2e-5
    for t in range(k):
        live = tr["alive_before"][t]
        if not live.any():
            break
        ref = o.step(tr["actions"][t])
        np.testing.assert_array_equal(tr["done"][t][live], ref["done"][live])
        np.testing.assert_allclose(tr["reward"][t][live], ref["reward"][live], atol=2e-6, rtol=0)
        step_obs = np.where(ref["done"][:, None] != 0, ref["terminal_obs"], ref["obs"])
        np.testing.assert_allclose(tr["obs"][t + 1][live], step_obs[live], atol=obs_bar, rtol=0)

    ret = np.zeros(n)
    for t in range(k):
        ret += np.where(tr["alive_before"][t], tr["reward"][t].astype(np.float64), 0.0)
    np.testing.assert_array_equal(tr["ret"], ret)
    np.testing.assert_array_equal(tr["alive"], tr["alive_before"][k].astype(np.uint8))

    ev = es_eval.EsEvaluator(env_id, individuals, repeats, seed=seed)
    fit, per_ep = ev.evaluate(weights, normalizer_state=(master[0], master[1], master[2], master[2] / master[0]), max_steps=k)
    np.testing.assert_array_equal(per_ep.cpu().numpy(), ret.reshape(individuals, repeats))
    np.testing.assert_array_equal(fit.cpu().numpy(), ret.reshape(individuals, repeats).mean(axis=1))
    done_steps = tr["alive_before"].sum(axis=0)
    print(f"{env_id}: {n} envs x {k} steps, worst action deviation {worst:.2e}, episode length min/mean/max "
          f"{done_steps.min()}/{done_steps.mean():.1f}/{done_steps.max()}, alive at the end {int(tr['alive'].sum())}")
    ev.close()


@pytest.mark.gpu
@pytest.mark.parametrize("env_id,k", [("SwingRacket-v0", 26), ("Tennisbot-v0", 200)])
def test_es_f32_context_actions_match_reference(env_id, k):
    od, ad = ENVS[env_id]
    weights = _swing_population(128, 4) if od == 6 else _random_population(128, 858, 4)
    master = _master(od, 6)
    tr = _traced(env_id, 128, 16, weights, master, k, seed=8, precision="f32")
    _check_actions(tr, weights, 16, master, ad)


@pytest.mark.gpu
@pytest.mark.parametrize("repeats", [1, 10, 33])
def test_es_each_env_uses_its_individual(repeats):
    """Individual p: all weights 0 but conv_2's bias c_p, so every env acts exactly clip(c_{i // repeats})."""
    individuals = 97
    c = np.random.default_rng(repeats).uniform(-1.5, 1.5, (individuals, 6)).astype(np.float32)
    w = np.zeros((individuals, 766), np.float32)
    w[:, 760:] = c
    tr = _traced("SwingRacket-v0", individuals, repeats, w, _master(6, 1), 3, seed=2)
    want = np.repeat(np.clip(c, -1, 1), repeats, axis=0)
    for t in range(3):
        np.testing.assert_array_equal(tr["actions"][t], want)


@pytest.mark.gpu
def test_es_evaluator_matches_torch_adapter():
    """The population and seed of test_batched_fitness_matches_sequential_oracle_evaluation: bit-equal reset observations,
    per-episode returns within 2e-3, the same fitness order."""
    from tennisbot_rl_b200 import es_eval
    from tennisbot_rl_b200.batch import TennisBatch

    saved = np.load(GOLD / "es_swing_weights.npz")["weights"]
    rng = np.random.default_rng(0)
    pop = np.stack([saved, saved + 0.05 * rng.standard_normal(766).astype(np.float32),
                    0.3 * rng.standard_normal(766).astype(np.float32)])
    repeats, seed = 4, 11
    tr = _traced("SwingRacket-v0", 3, repeats, pop, None, 1, seed)
    ref_env = TennisBatch("SwingRacket-v0", 3 * repeats, seed=seed)
    np.testing.assert_array_equal(tr["obs"][0], ref_env.reset().cpu().numpy())
    ref_env.close()
    fit_t, per_t = es_eval.batched_fitness_static(pop, "SwingRacket-v0", repeats=repeats, seed=seed)
    ev = es_eval.EsEvaluator("SwingRacket-v0", 3, repeats, seed=seed)
    fit, per = ev.evaluate(pop)
    np.testing.assert_allclose(per.cpu().numpy(), per_t.cpu().numpy(), atol=2e-3, rtol=0)
    np.testing.assert_array_equal(np.argsort(fit.cpu().numpy()), np.argsort(fit_t.cpu().numpy()))
    ev.close()


@pytest.mark.gpu
def test_es_sharded_evaluators_reproduce_the_full_batch():
    from tennisbot_rl_b200 import es_eval

    individuals, repeats = 64, 10
    pop = _swing_population(individuals, 9)
    m = _master(6, 2)
    state = (m[0], m[1], m[2], m[2] / m[0])
    _, full = es_eval.EsEvaluator("SwingRacket-v0", individuals, repeats, seed=4).evaluate(pop, state)
    h = individuals // 2
    _, lo = es_eval.EsEvaluator("SwingRacket-v0", h, repeats, seed=4).evaluate(pop[:h], state)
    _, hi = es_eval.EsEvaluator("SwingRacket-v0", h, repeats, seed=4, env_id_offset=h * repeats).evaluate(pop[h:], state)
    assert torch.equal(full, torch.cat([lo, hi]))


@pytest.mark.gpu
def test_es_rollout_replays_from_a_cuda_graph():
    """A rollout chunk captured in a CUDA graph and replayed is bit-identical to the same chunk issued eagerly."""
    from tennisbot_rl_b200.batch import TennisBatch

    individuals, repeats, k = 256, 8, 26
    n = individuals * repeats
    w = torch.from_numpy(_swing_population(individuals, 12)).cuda()
    m = torch.from_numpy(_master(6, 3)).cuda()
    runs = []
    for captured in (False, True):
        b = TennisBatch("SwingRacket-v0", n, seed=6)
        dev = b.device
        tr = dict(obs=torch.zeros((k + 1, n, 6), device=dev), actions=torch.zeros((k, n, 6), device=dev),
                  reward=torch.zeros((k, n), device=dev), done=torch.zeros((k, n), dtype=torch.uint8, device=dev))
        ret, alive = torch.zeros(n, dtype=torch.float64, device=dev), torch.zeros(n, dtype=torch.uint8, device=dev)
        b.es_begin(w, m)  # warm-up generation: the launch set-up of the env step happens outside the capture
        b.es_rollout(2, ret, alive)
        b.es_begin(w, m)
        torch.cuda.synchronize()
        if captured:
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                b.es_rollout(k, ret, alive, **tr)
            g.replay()
        else:
            b.es_rollout(k, ret, alive, **tr)
        torch.cuda.synchronize()
        runs.append({key: v.clone() for key, v in dict(tr, ret=ret, alive=alive).items()})
        b.close()
    for key in runs[0]:
        assert torch.equal(runs[0][key], runs[1][key]), key
    assert int(runs[0]["alive"].sum()) == 0


@pytest.mark.gpu
def test_es_second_generation_gets_new_placements():
    from tennisbot_rl_b200 import es_eval
    from tennisbot_rl_b200.batch import TennisBatch

    n = 512
    w = torch.from_numpy(_swing_population(64, 13)).cuda()
    b = TennisBatch("SwingRacket-v0", n, seed=17)
    ref = TennisBatch("SwingRacket-v0", n, seed=17)
    ret, alive = torch.zeros(n, dtype=torch.float64, device=b.device), torch.zeros(n, dtype=torch.uint8, device=b.device)
    firsts = []
    for _ in range(2):
        obs = torch.zeros((2, n, 6), device=b.device)
        b.es_begin(w)
        b.es_rollout(1, ret, alive, obs=obs)
        np.testing.assert_array_equal(obs[0].cpu().numpy(), ref.reset().cpu().numpy())
        firsts.append(obs[0].clone())
    assert not torch.equal(firsts[0], firsts[1])
    b.close()
    ref.close()
    ev = es_eval.EsEvaluator("SwingRacket-v0", 64, 8, seed=17)
    _, r1 = ev.evaluate(w)
    _, r2 = ev.evaluate(w)
    assert not torch.equal(r1, r2)
    ev.close()


@pytest.mark.gpu
def test_es_generation_termination():
    from tennisbot_rl_b200 import es_eval

    swing = es_eval.EsEvaluator("SwingRacket-v0", 64, 10, seed=1)
    pop = _swing_population(64, 14)
    swing.evaluate(pop)
    assert swing.steps_run == 26 and int(swing.alive.sum()) == 0  # one chunk holds the whole 26-step episode

    # max_steps shorter than the episodes truncates the returns, as the torch adapter does
    _, short = swing.evaluate(pop, max_steps=10)
    assert swing.steps_run == 10 and int(swing.alive.sum()) == 64 * 10
    _, short_t = es_eval.batched_fitness_static(pop, "SwingRacket-v0", repeats=10, seed=1, max_steps=10)
    swing.close()
    # (the adapter's fresh context places as the evaluator's first generation did, so compare with a fresh evaluator)
    fresh = es_eval.EsEvaluator("SwingRacket-v0", 64, 10, seed=1)
    _, short = fresh.evaluate(pop, max_steps=10)
    np.testing.assert_allclose(short.cpu().numpy(), short_t.cpu().numpy(), atol=2e-3, rtol=0)
    fresh.close()

    hit = es_eval.EsEvaluator("Tennisbot-v0", 64, 4, seed=1)
    hit.evaluate(_random_population(64, 858, 15))
    assert hit.steps_run <= 1001 and int(hit.alive.sum()) == 0
    print(f"Tennisbot-v0 generation: {hit.steps_run} steps")
    hit.close()
