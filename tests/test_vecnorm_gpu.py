"""The device VecNormalize of tb_policy_rollout (tb_set_vecnorm / tb_get_vecnorm, policy_kernel<OBS, ACT, true>,
vecnorm_partial_kernel / vecnorm_final_kernel) against the float64 numpy restatement in tests/vecnorm_reference.py."""
import ctypes

import numpy as np
import pytest
import torch

from .vecnorm_reference import VecNormalizeRef, normalize, record_formula

pytestmark = pytest.mark.gpu

ENVS = ["SwingRacket-v0", "Tennisbot-v0"]


def _batch(env_id, n, precision="f64", seed=5):
    from tennisbot_rl_b200.batch import TennisBatch
    from tennisbot_rl_b200.ppo import ActorCritic

    b = TennisBatch(env_id, n, seed=seed, precision=precision)
    torch.manual_seed(11)
    b.set_policy(ActorCritic(b.obs_dim, b.act_dim).to(b.device).packed())
    return b


def _bufs(b, k):
    dev, n, od, ad = b.device, b.num_envs, b.obs_dim, b.act_dim
    z = lambda *s: torch.zeros(s, device=dev)  # noqa: E731
    return dict(obs=z(k, n, od), reward=z(k, n), done=torch.zeros((k, n), dtype=torch.uint8, device=dev), last_obs=z(n, od),
                actions=z(k, n, ad), logp=z(k, n), value=z(k, n), last_value=z(n))


def _roll(b, cur, k, seed=3):
    """One policy_rollout of k steps from the raw observation cur; returns the buffers on the host (cur becomes last_obs)."""
    buf = _bufs(b, k)
    buf["obs"][0].copy_(cur)
    b.policy_rollout(buf["obs"], buf["reward"], buf["done"], buf["last_obs"], actions=buf["actions"], logp=buf["logp"],
                     value=buf["value"], last_value=buf["last_value"], noise_seed=seed)
    cur.copy_(buf["last_obs"])
    torch.cuda.synchronize()
    return {k_: v.cpu().numpy() for k_, v in buf.items()}


def _rel_close(got, want, rtol):
    err = np.abs(got - want) / np.maximum(np.abs(want), 1e-300)
    assert err.max() <= rtol, (err.max(), int(err.argmax()), got, want)


@pytest.mark.parametrize("env_id", ENVS)
def test_statistics_match_the_numpy_restatement(env_id):
    """4096 envs (f64), episodes ending inside the calls, a masked and a full reset between calls: the record equals the
    numpy VecNormalize driven by the raw sequence of a twin stepped with tb_step on the traced actions within 1e-10."""
    n = 4096
    calls = (20, 30, 28) if env_id == "SwingRacket-v0" else (300, 400, 400)
    b, twin = _batch(env_id, n), _batch(env_id, n)
    od = b.obs_dim
    b.set_vecnorm()
    cur = b.reset().clone()
    tw_obs = twin.reset().clone()
    torch.testing.assert_close(cur, tw_obs, rtol=0, atol=0)
    ref = VecNormalizeRef(n, od)
    ref.reset(cur.cpu().numpy())
    rng = np.random.default_rng(0)
    ended = 0
    for i, k in enumerate(calls):
        if i == 1:  # masked reset: returns of those envs zeroed, nothing folded
            mask = torch.from_numpy(rng.random(n) < 0.3).to(b.device)
            cur[mask] = b.reset(mask=mask)[mask]  # (a masked reset writes the observations of the envs it resets)
            twin.reset(mask=mask)
            ref.reset(None, mask=mask.cpu().numpy())
        if i == 2:  # full reset: returns zeroed, the next rollout folds its observation
            cur.copy_(b.reset())
            ref.reset(twin.reset().cpu().numpy())
        h = _roll(b, cur, k)
        for t in range(k):
            o, r, d, _, _ = twin.step(torch.from_numpy(h["actions"][t]).to(b.device).clamp(-1, 1))
            o, r, d = o.cpu().numpy(), r.cpu().numpy(), d.cpu().numpy()
            np.testing.assert_array_equal(d, h["done"][t])
            rhat = ref.step(o, r, d)
            np.testing.assert_allclose(h["reward"][t], rhat, rtol=1e-5, atol=1e-6)
            ended += int(d.sum())
        np.testing.assert_array_equal(h["last_obs"], o)  # raw, and bit-identical to the twin's env
        _rel_close(b.vecnorm_stats().cpu().numpy(), ref.record(), 1e-10)
    assert ended > n // 4


@pytest.mark.parametrize("config", ["default", "tiny_clips", "no_norm_obs", "no_norm_reward"])
@pytest.mark.parametrize("env_id", ENVS)
def test_k1_values_bit_exact_and_the_policy_acts_on_them(env_id, config):
    """K = 1 per call: d_obs[0] and d_reward are the numpy float64 formula on the record read between calls, bit for bit; the
    actions, log-density and value equal a plain twin's given the normalised observation (same step counter), bit for bit."""
    n, steps = 2048, 40 if env_id == "SwingRacket-v0" else 60
    kw = {"default": {}, "tiny_clips": dict(clip_obs=0.3, clip_reward=0.01), "no_norm_obs": dict(norm_obs=False),
          "no_norm_reward": dict(norm_reward=False)}[config]
    b, twin = _batch(env_id, n), _batch(env_id, n)
    od = b.obs_dim
    b.set_vecnorm(**kw)
    clip_obs, clip_rew, eps = kw.get("clip_obs", 10.0), kw.get("clip_reward", 10.0), 1e-8
    cur = b.reset().clone()
    tw = twin.reset().clone()
    clipped_obs = clipped_rew = rewarded = 0
    prev_last_value = None
    for step in range(steps):
        raw = cur.cpu().numpy()
        before = b.vecnorm_stats().cpu().numpy()
        h = _roll(b, cur, 1)
        after = b.vecnorm_stats().cpu().numpy()
        tw.copy_(torch.from_numpy(h["obs"][0]).to(b.device))  # the twin acts on the normalised observation
        g = _roll(twin, tw, 1)
        for key in ("actions", "logp", "value", "done", "last_obs"):
            np.testing.assert_array_equal(h[key], g[key], err_msg=key)
        if prev_last_value is not None:  # the bootstrap value is the value of the next call's normalised observation
            np.testing.assert_array_equal(prev_last_value, g["value"][0])
        prev_last_value = h["last_value"]
        if kw.get("norm_obs", True):
            if step > 0:  # (the first call folds its observation before normalising it)
                np.testing.assert_array_equal(h["obs"][0], record_formula(before, od, raw, eps, clip_obs))
                clipped_obs += int((np.abs(h["obs"][0]) == np.float32(clip_obs)).sum())
        else:
            np.testing.assert_array_equal(h["obs"][0], raw)
        if kw.get("norm_reward", True):
            rewarded += int((g["reward"][0] != 0).sum())
            want = normalize(g["reward"][0], 0.0, after[2 * od + 2], eps, clip_rew)
            np.testing.assert_array_equal(h["reward"][0], want)
            clipped_rew += int((np.abs(h["reward"][0]) == np.float32(clip_rew)).sum())
        else:
            np.testing.assert_array_equal(h["reward"][0], g["reward"][0])
    if config == "tiny_clips":
        assert clipped_obs > 0 and (clipped_rew > 0 or rewarded == 0)


@pytest.mark.parametrize("env_id", ENVS)
def test_frozen_record_and_the_saved_record_round_trip(env_id, tmp_path):
    """training = 0 leaves the record bit-equal and normalises with it; a record saved and loaded through the npz of
    load_vecnormalize_npz, attached to a twin, rolls out bit for bit as the context it was read from."""
    from tennisbot_rl_b200.ppo import load_vecnormalize_npz

    n, k = 2048, 8
    a, b = _batch(env_id, n), _batch(env_id, n)
    od = a.obs_dim
    cur_a, cur_b = a.reset().clone(), b.reset().clone()
    for x, cur in ((a, cur_a), (b, cur_b)):
        x.set_vecnorm(gamma=0.95)
        _roll(x, cur, k)
    rec = a.vecnorm_stats().cpu().numpy()
    np.testing.assert_array_equal(rec, b.vecnorm_stats().cpu().numpy())
    path = tmp_path / "vn.npz"
    np.savez(path, obs_mean=rec[:od], obs_var=rec[od:2 * od], obs_count=rec[2 * od], ret_mean=rec[2 * od + 1],
             ret_var=rec[2 * od + 2], ret_count=rec[2 * od + 3], clip_obs=10.0, clip_reward=10.0, gamma=0.95, epsilon=1e-8)
    stats, cfg = load_vecnormalize_npz(path, od)
    a.set_vecnorm(training=False, gamma=0.95, stats=a.vecnorm_stats())
    b.set_vecnorm(training=False, stats=stats.to(b.device), **cfg)
    raw = cur_a.cpu().numpy()
    ha, hb = _roll(a, cur_a, k), _roll(b, cur_b, k)
    for key in ha:
        np.testing.assert_array_equal(ha[key], hb[key], err_msg=key)
    np.testing.assert_array_equal(a.vecnorm_stats().cpu().numpy(), rec)
    np.testing.assert_array_equal(b.vecnorm_stats().cpu().numpy(), rec)
    np.testing.assert_array_equal(ha["obs"][0], record_formula(rec, od, raw, 1e-8, 10.0))
    np.testing.assert_array_equal(a.get_state().cpu().numpy(), b.get_state().cpu().numpy())


@pytest.mark.parametrize("env_id", ENVS)
def test_attach_then_detach_changes_nothing(env_id):
    n, k = 2048, 12
    a, b = _batch(env_id, n), _batch(env_id, n)
    a.set_vecnorm()
    a.clear_vecnorm()
    cur_a, cur_b = a.reset().clone(), b.reset().clone()
    for _ in range(2):
        ha, hb = _roll(a, cur_a, k), _roll(b, cur_b, k)
        for key in ha:
            np.testing.assert_array_equal(ha[key], hb[key], err_msg=key)
    np.testing.assert_array_equal(a.get_state().cpu().numpy(), b.get_state().cpu().numpy())
    np.testing.assert_array_equal(a.read_stats(), b.read_stats())
    from tennisbot_rl_b200 import _lib

    with pytest.raises(_lib.TennisbotLibraryError, match="no normaliser"):
        a.vecnorm_stats()


@pytest.mark.parametrize("env_id", ENVS)
def test_graph_replays_equal_eager_calls(env_id):
    n, k = 2048, 6
    a, b = _batch(env_id, n), _batch(env_id, n)
    bufs = {}
    for x in (a, b):
        x.set_vecnorm()
        cur = x.reset().clone()
        buf = _bufs(x, k)

        def body(x=x, cur=cur, buf=buf):
            buf["obs"][0].copy_(cur)
            x.policy_rollout(buf["obs"], buf["reward"], buf["done"], buf["last_obs"], actions=buf["actions"], logp=buf["logp"],
                             value=buf["value"], last_value=buf["last_value"], noise_seed=9)
            cur.copy_(buf["last_obs"])

        bufs[id(x)] = (body, buf)
        s = torch.cuda.Stream(x.device)  # warm-up call (eager on both contexts)
        s.wait_stream(torch.cuda.current_stream(x.device))
        with torch.cuda.stream(s):
            body()
        torch.cuda.current_stream(x.device).wait_stream(s)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        bufs[id(a)][0]()
    for _ in range(3):
        g.replay()
        bufs[id(b)][0]()
        torch.cuda.synchronize()
        for key in bufs[id(a)][1]:
            np.testing.assert_array_equal(bufs[id(a)][1][key].cpu().numpy(), bufs[id(b)][1][key].cpu().numpy(), err_msg=key)
    np.testing.assert_array_equal(a.vecnorm_stats().cpu().numpy(), b.vecnorm_stats().cpu().numpy())
    np.testing.assert_array_equal(a.get_state().cpu().numpy(), b.get_state().cpu().numpy())
    np.testing.assert_array_equal(a.read_stats(), b.read_stats())


@pytest.mark.parametrize("precision", ["f32", "f64"])
@pytest.mark.parametrize("env_id", ENVS)
def test_launch_counts_and_fold_rules(env_id, precision):
    """Launches of tb_policy_rollout with a normaliser: K (3 + s) + 3 training, K (1 + s) + 2 frozen; tb_reset adds one while
    training.  The reset fold happens once after tb_set_vecnorm and after a full reset, not after a masked one (obs count)."""
    n, k = 256, 3
    b = _batch(env_id, n, precision)
    s = 2 if env_id == "SwingRacket-v0" else 1
    od = b.obs_dim
    cur = b.reset().clone()

    def launches(call):
        before = b.launch_count()
        call()
        torch.cuda.synchronize()
        return b.launch_count() - before

    counts = lambda: b.vecnorm_stats().cpu().numpy()[[2 * od, 2 * od + 3]]  # noqa: E731
    assert launches(lambda: b.set_vecnorm()) == 1
    assert launches(lambda: _roll(b, cur, k)) == k * (3 + s) + 3
    want = np.array([1e-4, 1e-4])
    want[0] += n
    for _ in range(k):
        want += n
    np.testing.assert_array_equal(counts(), want)
    assert launches(lambda: _roll(b, cur, k)) == k * (3 + s) + 3  # no fold of d_obs[0] this time
    for _ in range(k):
        want += n
    np.testing.assert_array_equal(counts(), want)
    mask = torch.zeros(n, dtype=torch.uint8, device=b.device)
    mask[::3] = 1
    assert launches(lambda: b.reset(mask=mask)) == 2
    cur[mask.bool()] = b.obs[mask.bool()]
    _roll(b, cur, k)
    for _ in range(k):
        want += n
    np.testing.assert_array_equal(counts(), want)
    assert launches(lambda: cur.copy_(b.reset())) == 2
    _roll(b, cur, k)
    want[0] += n
    for _ in range(k):
        want += n
    np.testing.assert_array_equal(counts(), want)
    b.set_vecnorm(training=False, stats=b.vecnorm_stats().clone())
    assert launches(lambda: _roll(b, cur, k)) == k * (1 + s) + 2
    assert launches(lambda: cur.copy_(b.reset())) == 1
    np.testing.assert_array_equal(counts(), want)
    b.clear_vecnorm()
    assert launches(lambda: _roll(b, cur, k)) == k * (1 + s) + 1


@pytest.mark.parametrize("env_id", ENVS)
def test_rejections(env_id):
    from tennisbot_rl_b200 import _lib

    b = _batch(env_id, 256)
    od = b.obs_dim
    err = _lib.TennisbotLibraryError
    with pytest.raises(err, match="no normaliser"):
        b.vecnorm_stats()
    cfg = _lib.TbVecNorm(ctypes.sizeof(_lib.TbVecNorm) - 8, 1, 1, 1, 10.0, 10.0, 0.99, 1e-8)
    with pytest.raises(err, match="struct_size"):
        _lib.check(b.lib.tb_set_vecnorm(b.h, ctypes.byref(cfg), None, b._stream()))
    for bad in (0.0, -1.0, float("inf"), float("nan")):
        with pytest.raises(err, match="clip_obs"):
            b.set_vecnorm(clip_obs=bad)
        with pytest.raises(err, match="clip_reward"):
            b.set_vecnorm(clip_reward=bad)
        with pytest.raises(err, match="epsilon"):
            b.set_vecnorm(epsilon=bad)
    for bad in (-0.01, 1.01, float("nan")):
        with pytest.raises(err, match="gamma"):
            b.set_vecnorm(gamma=bad)
    fresh = np.concatenate([np.zeros(od), np.ones(od), [1e-4, 0.0, 1.0, 1e-4]])
    for idx, val in ((2 * od, 0.0), (2 * od + 3, -1.0), (0, float("nan")), (od, -1e-12), (2 * od + 2, -1.0),
                     (2 * od + 1, float("inf"))):
        rec = fresh.copy()
        rec[idx] = val
        with pytest.raises(err, match="stats"):
            b.set_vecnorm(stats=torch.from_numpy(rec).to(b.device))
    with pytest.raises(ValueError, match="stats"):
        b.set_vecnorm(stats=torch.zeros(od, dtype=torch.float64, device=b.device))
    with pytest.raises(err, match="no normaliser"):  # nothing was attached by the rejected calls
        b.vecnorm_stats()
    b.set_vecnorm(gamma=0.0, clip_obs=1e-3)  # the edges are accepted
    b.set_vecnorm(gamma=1.0, stats=torch.from_numpy(fresh).to(b.device))
    np.testing.assert_array_equal(b.vecnorm_stats().cpu().numpy(), fresh)


@pytest.mark.parametrize("normalize", [False, True])
def test_hit_ppo_with_normalize_trains_and_saves(normalize, tmp_path):
    """HitPPO(normalize=...) through a racket-scale curriculum stage change (full reset, graph captured again): the episode
    statistics stay raw, the record's counts grow as the fold rules say, and save() writes what record_episode reads."""
    from tennisbot_rl_b200.ppo import HitPPO, load_vecnormalize_npz

    n, K = 1024, 16
    ppo = HitPPO(n, rollout_len=K, curriculum_total_timesteps=3 * n * K, seed=0, normalize=normalize)
    s = ppo.train(iters=4)
    assert s["iters"] == 4 and len(ppo.stages) >= 2
    path = tmp_path / "run.npz"
    ppo.save(path)
    w = np.load(path)
    np.testing.assert_array_equal(w["policy"], ppo.ac.packed().cpu().numpy())
    if normalize:
        stats, cfg = load_vecnormalize_npz(path, ppo.od)
        # one fold per stage change's full reset (the first stage is set before the first rollout, which also folds for
        # set_vecnorm), and K per rollout: 4 graph replays and the eager warm-up before the first capture
        count = stats.numpy()[2 * ppo.od]
        assert abs(count - (1e-4 + len(ppo.stages) * n + 5 * K * n)) < 1e-6 * count
        assert cfg["gamma"] == ppo.gamma
        assert np.abs(ppo.obs_buf.cpu().numpy()).max() <= 10.0
    else:
        assert "obs_mean" not in w


def test_swing_ppo_learns_with_normalize():
    """SwingPPO(normalize=True) at 4 096 envs: the raw mean return and the contact rate rise within 25 updates."""
    from tennisbot_rl_b200.ppo import SwingPPO

    ppo = SwingPPO(num_envs=4096, seed=1, use_graph=True, normalize=True)
    s = ppo.train(iters=25, target=31.5)
    first = np.mean([h["mean_return"] for h in s["history"][:3]])
    last = np.mean([h["mean_return"] for h in s["history"][-3:]])
    print(f"normalize: mean return {first:.2f} -> {last:.2f}, hits/ep {s['history'][0]['hits_per_episode']:.3f} -> "
          f"{s['history'][-1]['hits_per_episode']:.3f}")
    assert last > first + 2.0
