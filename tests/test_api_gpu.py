"""GPU tests of the reference-facing API (single-env gym classes, VecEnv adapter, shards) and of size-independent
properties at BASELINE.json's full sizes.  Everything goes through the C ABI."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def test_single_env_classes_match_oracle(oracle_lib):
    """gym.Env API of the reference, batch of one, replayed against the oracle with the same placement."""
    import tennisbot.envs as envs

    env = envs.SwingRacketEnv(use_gui=False, delay_mode=False, seed=4)
    assert env.action_space.shape == (6,) and env.observation_space.shape == (6,)
    obs = env.reset()
    assert isinstance(obs, tuple) and len(obs) == 6 and all(isinstance(x, float) for x in obs)
    st = env.state()
    o = oracle_lib.OracleEnv("SwingRacket-v0", 1, auto_reset=False)
    o.set_state(st[None])
    rng = np.random.default_rng(1)
    total = 0.0
    for k in range(26):
        a = rng.uniform(-1, 1, 6).astype(np.float32)
        ob, r, done, info = env.step(a)
        ref = o.step(a[None])
        assert info == {} and done == bool(ref["done"][0]) == (k == 25)
        assert r == pytest.approx(float(ref["reward"][0]), abs=1e-6)
        np.testing.assert_allclose(ob, ref["obs"][0], atol=2e-6)
        assert env.last_events == int(ref["events"][0])
        total += r
    assert env.step_count == int(o.get_state()[0, oracle_lib.S_STEP]) > 100
    assert env.seed(3) == [3]
    env.close()

    hit = envs.TennisbotEnv(seed=2)
    ob = hit.reset()
    assert ob.dtype == np.float32 and ob.shape == (12,) and np.all(ob[3:6] == 0) and np.all(ob[9:] == 0)
    hit.set_racket_scale(2.0)
    hit.reset()
    assert hit.state()[2] == pytest.approx(hit.state()[2])  # COM z = base z + 0.5 * scale
    assert 1.2 <= hit.state()[2] <= 1.21
    for k in range(6):
        ob, r, done, info = hit.step(np.zeros(2, np.float32))
        assert not done and r == 0
    hit.close()


def test_vecenv_on_gpu_matches_oracle(oracle_lib):
    from tennisbot_rl_b200.vec_env import TennisVecEnv

    n = 512
    env = TennisVecEnv("SwingRacket-v0", n, seed=9)
    o = oracle_lib.OracleEnv("SwingRacket-v0", n, seed=9, threads=4)
    obs = env.reset()
    np.testing.assert_array_equal(obs, o.reset())
    rng = np.random.default_rng(2)
    n_done = 0
    for t in range(55):
        a = rng.uniform(-1, 1, (n, 6)).astype(np.float32)
        obs, rew, dones, infos = env.step(a)
        ref = o.step(a)
        np.testing.assert_array_equal(dones, ref["done"].astype(bool))
        np.testing.assert_allclose(obs, ref["obs"], atol=2e-6)
        np.testing.assert_allclose(rew, ref["reward"], atol=2e-6)
        for i in np.nonzero(dones)[0]:
            np.testing.assert_allclose(infos[i]["terminal_observation"], ref["terminal_obs"][i], atol=2e-6)
            assert infos[i]["episode"]["l"] == 26 and infos[i]["events"] == ref["events"][i]
            n_done += 1
    assert n_done == 2 * n
    assert env.episode_statistics()["episodes"] == 2 * n
    env.close()


def test_shard_invariance():
    """(e): a batch sharded over G contexts with global-id offsets equals the single batch (here G = 2 on one GPU)."""
    from tennisbot_rl_b200.batch import TennisBatch
    from tennisbot_rl_b200.sharding import shard_range

    total, k = 6144, 40
    full = TennisBatch("SwingRacket-v0", total, seed=5)
    full.reset()
    fo, fr, fd = (x.cpu().numpy().copy() for x in full.rollout(k))
    parts, stats = [], np.zeros(10, np.int64)
    for g in range(2):
        lo, hi = shard_range(total, g, 2)
        b = TennisBatch("SwingRacket-v0", hi - lo, seed=5, env_id_offset=lo)
        b.reset()
        parts.append([x.cpu().numpy().copy() for x in b.rollout(k)])
        stats += b.read_stats()
    np.testing.assert_array_equal(np.concatenate([p[0] for p in parts]), fo)
    np.testing.assert_array_equal(np.concatenate([p[2] for p in parts]), fd)
    np.testing.assert_array_equal(stats, full.read_stats())


@pytest.mark.parametrize("env_id,n,steps", [("SwingRacket-v0", 1 << 20, 52), ("Tennisbot-v0", 65536, 1100)])
def test_full_size_properties(env_id, n, steps):
    """Size-independent properties at BASELINE.json's sizes (config 5 slice: 1 Mi envs; config 3: 65 536 envs):
    step accounting is conserved, episodes have the lengths the env logic dictates, every output is finite and
    inside physical bounds, and the run is bit-reproducible."""
    from tennisbot_rl_b200.batch import TennisBatch

    def run():
        b = TennisBatch(env_id, n, seed=1)
        b.reset()
        acts = [torch.empty((n, b.act_dim), device="cuda").uniform_(-1, 1, generator=torch.Generator("cuda").manual_seed(s))
                for s in range(3)]
        ndone = torch.zeros((), dtype=torch.int64, device="cuda")
        rsum = torch.zeros((), dtype=torch.float64, device="cuda")
        for t in range(steps):
            obs, rew, done, term, ev = b.step(acts[t % 3])
            ndone += done.sum()
            rsum += rew.double().sum()
            if t % 13 == 0:
                assert bool(torch.isfinite(obs).all()) and bool(torch.isfinite(rew).all())
        st = b.read_stats()
        state = b.get_state()
        return st, int(ndone), float(rsum), obs.clone(), state

    st, ndone, rsum, obs, state = run()
    assert st[9] == n * steps and st[0] == ndone               # env-step and episode accounting
    if env_id == "SwingRacket-v0":
        assert st[0] == 2 * n and st[8] >= st[9]                 # exactly 26 agent steps per episode
        assert st[1] == st[8]                                    # sum of episode lengths == physics steps taken
        assert abs(st[6] / 2 ** 20 - rsum) < 1e-3 * max(1.0, abs(rsum))  # fixed-point return sum == emitted rewards
        assert 100 < st[1] / st[0] < 200 and st[5] < 0.05 * st[0]
        q = state[:, 3:7]
        assert float((q.norm(dim=1) - 1).abs().max()) < 1e-9     # quaternions stay normalised
    else:
        assert st[8] == st[9]                                    # one physics step per env step
        assert 300 < st[1] / max(st[0], 1) <= 1001
        assert st[6] / 2 ** 20 <= rsum + 1e-3 * abs(rsum)         # returns of finished episodes <= all emitted rewards
    assert float(state[:, 7:22].abs().max()) <= 100.0            # Bullet's coordinate-velocity clamp
    st2, ndone2, rsum2, obs2, state2 = run()
    np.testing.assert_array_equal(st, st2)
    assert torch.equal(obs, obs2) and torch.equal(state, state2)  # bit-reproducible


@pytest.mark.parametrize("mode", ["zero_copy", "staging"])
def test_step_host_modes_match_oracle(oracle_lib, mode, monkeypatch):
    """tb_step_host's two transports (kernels addressing the pinned host buffers; plain staging) give the oracle's results,
    through SwingRacket's fast-forward step and the auto-resets."""
    from tennisbot_rl_b200.batch import TennisBatch

    monkeypatch.setenv("TB_HOST_MODE", mode)
    n = 5000  # not a multiple of the CTA size
    b = TennisBatch("SwingRacket-v0", n, seed=77)
    o = oracle_lib.OracleEnv("SwingRacket-v0", n, seed=77, threads=8)
    np.testing.assert_array_equal(b.reset_host(), o.reset())
    rng = np.random.default_rng(8)
    for t in range(54):
        a = rng.uniform(-1, 1, (n, 6)).astype(np.float32)
        hb = b.step_host(a)
        ref = o.step(a)
        np.testing.assert_array_equal(hb["done"], ref["done"])
        np.testing.assert_array_equal(hb["events"], ref["events"])
        np.testing.assert_allclose(hb["obs"], ref["obs"], atol=2e-6)
        np.testing.assert_allclose(hb["reward"], ref["reward"], atol=2e-6)
        d = ref["done"] != 0
        np.testing.assert_allclose(hb["terminal_obs"][d], ref["terminal_obs"][d], atol=2e-6)
    np.testing.assert_array_equal(b.read_stats(), o.read_stats())
    b.close()


def test_step_host_rejects_unknown_mode(monkeypatch):
    """A TB_HOST_MODE that names no transport (here the removed `pipeline`) fails the call instead of falling back."""
    from tennisbot_rl_b200 import _lib
    from tennisbot_rl_b200.batch import TennisBatch

    monkeypatch.setenv("TB_HOST_MODE", "pipeline")
    b = TennisBatch("SwingRacket-v0", 256, seed=1)
    b.reset_host()
    with pytest.raises(_lib.TennisbotLibraryError, match="pipeline") as err:
        b.step_host(np.zeros((256, 6), np.float32))
    assert "zero_copy" in str(err.value) and "staging" in str(err.value)
    b.close()
