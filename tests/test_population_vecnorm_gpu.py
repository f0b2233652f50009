"""Per-agent VecNormalize records in a population rollout on the B200 (tb_set_vecnorms, policy_kernel<OBS, ACT, true, true>,
the segmented statistics pass) and PopulationPPO(normalize=True).

- A context of P x n envs with P policies and P records gives, for every agent p, bit for bit what a one-policy context of n
  envs at env_id_offset = p n gives with that agent's policy and record (tb_set_vecnorm): outputs and records, training and
  frozen, through masked and full resets.
- Each record equals the numpy VecNormalize restatement driven with its agent's raw observations and rewards.
- One record through tb_set_vecnorms is tb_set_vecnorm; launch counts do not depend on the number of records; a replayed
  graph reads the records as they are at replay time; the rules reject what they must.
"""
import ctypes

import numpy as np
import pytest
import torch

from tennisbot_rl_b200 import _lib
from tennisbot_rl_b200.batch import TennisBatch
from tennisbot_rl_b200.population import PopulationPPO
from tennisbot_rl_b200.ppo import load_vecnormalize_npz

from .test_population_gpu import _policies
from .vecnorm_reference import VecNormalizeRef

pytestmark = pytest.mark.gpu
ENVS = ("SwingRacket-v0", "Tennisbot-v0")
KEYS = ("obs", "act", "logp", "value", "reward", "raw", "done", "last_obs", "last_value")
CONFIGS = {"default": {}, "no_norm_obs": dict(norm_obs=False), "no_norm_reward": dict(norm_reward=False),
           "tiny_clips": dict(clip_obs=0.3, clip_reward=0.01)}


def _records(od, P, seed=0):
    """P distinct valid records (float64 [P, 2 od + 4]) on the device."""
    rng = np.random.default_rng(seed)
    rows = [np.concatenate([rng.normal(0, 0.5, od), rng.uniform(0.2, 3.0, od), [50.0 + 7 * p, rng.normal(0, 0.1),
                                                                                rng.uniform(0.5, 2.0), 40.0 + 3 * p]])
            for p in range(P)]
    return torch.from_numpy(np.stack(rows)).cuda().contiguous()


def _buffers(b, K):
    n, od, ad = b.num_envs, b.obs_dim, b.act_dim
    z = lambda *s: torch.zeros(s, device="cuda")  # noqa: E731
    return dict(obs=z(K, n, od), act=z(K, n, ad), logp=z(K, n), value=z(K, n), reward=z(K, n), raw=z(K, n),
                done=torch.zeros((K, n), dtype=torch.uint8, device="cuda"), last_obs=z(n, od), last_value=z(n))


def _rollout(b, buf, seed=9):
    b.policy_rollout(buf["obs"], buf["reward"], buf["done"], buf["last_obs"], actions=buf["act"], logp=buf["logp"],
                     value=buf["value"], last_value=buf["last_value"], noise_seed=seed, raw_reward=buf["raw"])


def _slice(key, x, p, n):
    return x[p * n:(p + 1) * n] if key in ("last_obs", "last_value") else x[:, p * n:(p + 1) * n]


@pytest.mark.parametrize("config", tuple(CONFIGS))
@pytest.mark.parametrize("training", (True, False))
@pytest.mark.parametrize("P,n", ((2, 256), (3, 100), (7, 1)))
@pytest.mark.parametrize("precision", ("f64", "f32"))
@pytest.mark.parametrize("env_id", ENVS)
def test_population_with_records_equals_one_record_shards(env_id, precision, P, n, training, config):
    K = 30 if env_id == "SwingRacket-v0" else 24  # SwingRacket-v0: across an episode boundary
    kw = dict(CONFIGS[config], training=training)
    params = _policies(env_id, P)
    pop = TennisBatch(env_id, P * n, seed=5, precision=precision)
    rec = _records(pop.obs_dim, P)
    pop.set_policies(params)
    pop.set_vecnorm(agents=P, stats=rec, **kw)
    shards = [TennisBatch(env_id, n, seed=5, precision=precision, env_id_offset=p * n) for p in range(P)]
    for p, s in enumerate(shards):
        s.set_policy(params[p])
        s.set_vecnorm(stats=rec[p].clone(), **kw)
    got, ref = _buffers(pop, K), [_buffers(s, K) for s in shards]
    cur, cur_s = pop.reset().clone(), [s.reset().clone() for s in shards]
    mask = torch.from_numpy(np.random.default_rng(2).random(P * n) < 0.4).cuda()
    for rnd in range(3):
        if rnd == 1:  # masked reset: returns of those envs zeroed, nothing folded
            cur[mask] = pop.reset(mask=mask)[mask]
            for p, s in enumerate(shards):
                m = mask[p * n:(p + 1) * n].contiguous()
                cur_s[p][m] = s.reset(mask=m)[m]
        if rnd == 2:  # full reset: every return zeroed, the next rollout folds its observation
            cur.copy_(pop.reset())
            for p, s in enumerate(shards):
                cur_s[p].copy_(s.reset())
        got["obs"][0].copy_(cur)
        _rollout(pop, got)
        cur.copy_(got["last_obs"])
        for p, (s, r) in enumerate(zip(shards, ref)):
            r["obs"][0].copy_(cur_s[p])
            _rollout(s, r)
            cur_s[p].copy_(r["last_obs"])
        torch.cuda.synchronize()
        records = pop.vecnorm_stats()
        for p, (s, r) in enumerate(zip(shards, ref)):
            for k in KEYS:
                assert torch.equal(_slice(k, got[k], p, n), r[k]), (rnd, p, k)
            assert torch.equal(records[p], s.vecnorm_stats()), (rnd, p)
    if not training:
        assert torch.equal(pop.vecnorm_stats(), rec)


@pytest.mark.parametrize("env_id", ENVS)
def test_each_record_matches_the_numpy_restatement(env_id):
    """K = 1 per call, so every raw observation is seen: each agent's record equals VecNormalizeRef driven with its slice of
    the raw observations and raw_reward within 1e-10, and the normalised rewards within 1e-5 (the bar of
    test_statistics_match_the_numpy_restatement)."""
    P, n = 3, 512
    calls = 40 if env_id == "SwingRacket-v0" else 1010  # past an episode end (Tennisbot-v0's time-out: 1001 steps)
    b = TennisBatch(env_id, P * n, seed=4)
    od = b.obs_dim
    rec = _records(od, P, seed=3)
    b.set_policies(_policies(env_id, P, seed=2))
    b.set_vecnorm(agents=P, stats=rec)
    cur = b.reset().clone()
    refs = [VecNormalizeRef(n, od, record=rec[p].cpu().numpy()) for p in range(P)]
    for p, r in enumerate(refs):
        r.reset(cur[p * n:(p + 1) * n].cpu().numpy())
    ended = 0
    for _ in range(calls):
        buf = _buffers(b, 1)
        buf["obs"][0].copy_(cur)
        _rollout(b, buf)
        cur.copy_(buf["last_obs"])
        h = {k: v.cpu().numpy() for k, v in buf.items()}
        for p, r in enumerate(refs):
            sl = slice(p * n, (p + 1) * n)
            rhat = r.step(h["last_obs"][sl], h["raw"][0, sl], h["done"][0, sl])
            np.testing.assert_allclose(h["reward"][0, sl], rhat, rtol=1e-5, atol=1e-6)
        ended += int(h["done"].sum())
    got = b.vecnorm_stats().cpu().numpy()
    for p, r in enumerate(refs):
        want = r.record()
        err = np.abs(got[p] - want) / np.maximum(np.abs(want), 1e-300)
        assert err.max() <= 1e-10, (p, err.max())
    assert ended > 0


def _launches(b, call):
    before = b.launch_count()
    call()
    torch.cuda.synchronize()
    return b.launch_count() - before


@pytest.mark.parametrize("env_id", ENVS)
def test_one_record_equals_set_vecnorm_and_launch_counts_do_not_depend_on_records(env_id):
    P, n, K = 4, 256, 6
    s = 2 if env_id == "SwingRacket-v0" else 1
    params = _policies(env_id, P)
    a, c, d = (TennisBatch(env_id, P * n, seed=2) for _ in range(3))
    rec = _records(a.obs_dim, 1)
    # tb_set_vecnorms with one record against tb_set_vecnorm, through the C ABI
    a.set_policy(params[0])
    c.set_policy(params[0])
    cfg = _lib.TbVecNorm(ctypes.sizeof(_lib.TbVecNorm), 1, 1, 1, 10.0, 10.0, 0.99, 1e-8)
    assert _launches(a, lambda: _lib.check(a.lib.tb_set_vecnorm(a.h, ctypes.byref(cfg), ctypes.c_void_p(rec.data_ptr()),
                                                                a._stream()))) == 1
    assert _launches(c, lambda: _lib.check(c.lib.tb_set_vecnorms(c.h, ctypes.byref(cfg), 1, ctypes.c_void_p(rec.data_ptr()),
                                                                 c._stream()))) == 1
    # P policies with P records
    d.set_policies(params)
    assert _launches(d, lambda: d.set_vecnorm(agents=P, stats=_records(d.obs_dim, P))) == 1
    bufs = [_buffers(x, K) for x in (a, c, d)]
    for x, buf in zip((a, c, d), bufs):
        buf["obs"][0].copy_(x.reset())
    for rnd in range(2):
        counts = [_launches(x, lambda x=x, buf=buf: _rollout(x, buf)) for x, buf in zip((a, c, d), bufs)]
        assert counts == [K * (3 + s) + 3] * 3, (rnd, counts)
        for k in KEYS:
            assert torch.equal(bufs[0][k], bufs[1][k]), (rnd, k)
        assert torch.equal(a.vecnorm_stats(), c.vecnorm_stats())
        for buf in bufs:
            buf["obs"][0].copy_(buf["last_obs"])
    a.set_vecnorm(training=False, stats=a.vecnorm_stats().clone())
    d.set_vecnorm(training=False, agents=P, stats=d.vecnorm_stats().clone())
    assert _launches(a, lambda: _rollout(a, bufs[0])) == _launches(d, lambda: _rollout(d, bufs[2])) == K * (1 + s) + 2
    # without a normaliser the raw reward is the reward (raw starts as a sentinel no reward takes)
    d.clear_vecnorm()
    bufs[2]["raw"].fill_(-7.0)
    _rollout(d, bufs[2])
    torch.cuda.synchronize()
    assert torch.equal(bufs[2]["raw"], bufs[2]["reward"]) and not bool(bufs[2]["raw"].eq(-7.0).any())


@pytest.mark.parametrize("env_id", ENVS)
def test_graph_replay_reads_the_records_at_replay_time(env_id):
    """A captured set_policies + policy_rollout replays bit-identically to eager calls; an in-place edit of one row of
    vecnorm_records() between replays is seen by the next replay and changes only that agent's slice."""
    P, n, K = 3, 200, 8
    params = _policies(env_id, P, seed=1)
    graphed, eager, plain = (TennisBatch(env_id, P * n, seed=3) for _ in range(3))
    bufs = {}
    for x in (graphed, eager, plain):
        x.set_policies(params)
        x.set_vecnorm(agents=P, stats=_records(x.obs_dim, P, seed=5))
        buf = _buffers(x, K)
        buf["obs"][0].copy_(x.reset())
        bufs[x] = buf
    src = params.clone()

    def body(x, p):
        x.set_policies(p)
        _rollout(x, bufs[x])
        bufs[x]["obs"][0].copy_(bufs[x]["last_obs"])

    s = torch.cuda.Stream()  # an eager warm-up call on a side stream for each context
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for x in (graphed, eager, plain):
            body(x, params)
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        body(graphed, src)
    od = graphed.obs_dim
    for rep in range(4):
        if rep == 2:  # agent 1's record edited in place in two of the contexts
            for x in (graphed, eager):
                r = x.vecnorm_records()
                r[1, :od] += 0.5
                r[1, od:2 * od] *= 2.0
        g.replay()
        body(eager, params)
        body(plain, params)
        torch.cuda.synchronize()
        for k in KEYS:
            if k != "obs":
                assert torch.equal(bufs[graphed][k], bufs[eager][k]), (rep, k)
        assert torch.equal(graphed.vecnorm_stats(), eager.vecnorm_stats()), rep
        for p in range(P):
            same = all(torch.equal(_slice(k, bufs[graphed][k], p, n), _slice(k, bufs[plain][k], p, n))
                       for k in KEYS if k != "obs")
            assert same == (rep < 2 or p != 1), (rep, p)


def test_rejections():
    env_id, P, n = "Tennisbot-v0", 3, 128
    b = TennisBatch(env_id, P * n, seed=1)
    L, od = b.lib, b.obs_dim
    err = _lib.TennisbotLibraryError
    cfg = _lib.TbVecNorm(ctypes.sizeof(_lib.TbVecNorm), 1, 1, 1, 10.0, 10.0, 0.99, 1e-8)

    def fail(fn, *args):
        assert fn(b.h, *args) != 0
        return L.tb_last_error().decode()

    def nothing_attached():
        with pytest.raises(err, match="no normaliser"):
            b.vecnorm_stats()
        with pytest.raises(err, match="no normaliser"):
            b.vecnorm_records()

    nothing_attached()
    assert "divide" in fail(L.tb_set_vecnorms, ctypes.byref(cfg), 0, None, b._stream())
    assert "divide" in fail(L.tb_set_vecnorms, ctypes.byref(cfg), 5, None, b._stream())
    bad = _records(od, P)
    bad[2, 2 * od + 3] = -1.0
    assert f"stats[2][{2 * od + 3}]" in fail(L.tb_set_vecnorms, ctypes.byref(cfg), P, ctypes.c_void_p(bad.data_ptr()), b._stream())
    small = _lib.TbVecNorm(ctypes.sizeof(_lib.TbVecNorm) - 8, 1, 1, 1, 10.0, 10.0, 0.99, 1e-8)
    assert "struct_size" in fail(L.tb_set_vecnorms, ctypes.byref(small), P, None, b._stream())
    with pytest.raises(err, match="gamma"):
        b.set_vecnorm(agents=P, gamma=1.5)
    with pytest.raises(ValueError, match="stats"):
        b.set_vecnorm(agents=P, stats=_records(od, 1)[0])
    with pytest.raises(ValueError, match="divide"):
        b.set_vecnorm(agents=5)
    nothing_attached()  # no record is attached by the rejected calls

    b.set_vecnorm(agents=P)
    out = torch.empty((P, _lib.vecnorm_words(od)), dtype=torch.float64, device="cuda")
    assert "tb_get_vecnorms" in fail(L.tb_get_vecnorm, ctypes.c_void_p(out.data_ptr()), b._stream())
    assert "3 records" in fail(L.tb_get_vecnorms, ctypes.c_void_p(out.data_ptr()), 2, b._stream())
    with pytest.raises(err, match="tb_set_vecnorms"):
        b.vecnorm_apply(torch.zeros((4, od), device="cuda"))
    b.sac_begin()
    with pytest.raises(err, match="tb_set_vecnorms"):
        b.sac_rollout(1, mode="uniform", normalize=True)
    buf = _buffers(b, 4)
    buf["obs"][0].copy_(b.reset())
    params = _policies(env_id, P)
    b.set_policy(params[0])  # P = 1 with A = 3
    with pytest.raises(err, match="1 policies.*3 normaliser records"):
        _rollout(b, buf)
    b.set_policies(torch.cat([params, params]).contiguous())  # P = 6 with A = 3
    with pytest.raises(err, match="6 policies.*3 normaliser records"):
        _rollout(b, buf)
    b.set_policies(params)
    _rollout(b, buf)  # P = A = 3 runs
    b.set_vecnorm()  # A = 1 with P = 3: the one-record message, which points at tb_set_vecnorms
    with pytest.raises(err, match="tb_set_vecnorm.*tb_set_policies.*tb_set_vecnorms"):
        _rollout(b, buf)
    b.clear_vecnorm()
    nothing_attached()


# ------------------------------------------------------------------ PopulationPPO(normalize=True)
@pytest.mark.parametrize("env_id", ENVS)
def test_normalized_population_statistics_counts_and_saving(env_id, tmp_path):
    P, n = 4, 1024
    K = 26 if env_id == "SwingRacket-v0" else 128
    pop = PopulationPPO(env_id, P, n, K, seeds=[1, 2, 3, 4], normalize=True)
    iters, total_eps = 3, 0
    for it in range(iters):
        eps, rsum, lsum, st = pop.rollout()
        assert int(eps.sum()) == int(st[0]), it
        total_eps += int(st[0])
        if st[0]:
            np.testing.assert_allclose(rsum.sum(), st[6] / 2 ** 20, rtol=1e-4, atol=1e-3)
        pop.update()
    assert total_eps > 0
    od, words = pop.od, _lib.vecnorm_words(pop.od)
    rec = pop.env.vecnorm_stats().cpu().numpy()
    assert rec.shape == (P, words)
    want = 1e-4 + n + (1 + iters) * K * n  # the reset fold, then the eager warm-up rollout and `iters` replays
    np.testing.assert_allclose(rec[:, 2 * od], want, rtol=1e-12)
    assert np.abs(pop.obs_buf.cpu().numpy()).max() <= 10.0
    # a PBT round copies the record row with the weights, bit for bit, and leaves the other rows
    (upd, dst, src, _), = pop.exploit_explore(scores=[1.0, 4.0, 2.0, 3.0])
    after = pop.env.vecnorm_stats().cpu().numpy()
    np.testing.assert_array_equal(after[dst], rec[src])
    for p in range(P):
        if p != dst:
            np.testing.assert_array_equal(after[p], rec[p])
    # save / agent_state_dict
    pop.save(tmp_path / "pop.npz")
    w = np.load(tmp_path / "pop.npz")
    np.testing.assert_array_equal(w["vecnorm"], after)
    assert float(w["vecnorm_gamma"]) == 0.99 and float(w["vecnorm_clip_obs"]) == 10.0
    for p in (dst, 3):
        np.savez(tmp_path / f"a{p}.npz", **pop.agent_state_dict(p))
        stats, cfg = load_vecnormalize_npz(tmp_path / f"a{p}.npz", od)
        np.testing.assert_array_equal(stats.numpy(), after[p])
        assert cfg == {"clip_obs": 10.0, "clip_reward": 10.0, "gamma": 0.99, "epsilon": 1e-8}
        np.testing.assert_array_equal(np.load(tmp_path / f"a{p}.npz")["policy"], pop.ac.packed()[p].cpu().numpy())


def test_normalized_population_learns_swing():
    """4 agents x 4 096 SwingRacket-v0 envs, seeds 1-4, each with its own record, 25 updates: every agent's mean raw return
    over its last three updates is more than 2 above its first three."""
    pop = PopulationPPO("SwingRacket-v0", 4, 4096, 26, seeds=[1, 2, 3, 4], normalize=True)
    out = pop.train(25)
    for a in out["per_agent"]:
        rets = [h["mean_return"] for h in a["history"]]
        first, last = np.mean(rets[:3]), np.mean(rets[-3:])
        print(f"seed {a['seed']}: first three {first:.2f} last three {last:.2f} best {a['best_mean_return']:.2f}")
        assert last > first + 2.0, a["seed"]
