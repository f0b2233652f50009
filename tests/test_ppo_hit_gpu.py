"""Tennisbot-v0's in-kernel policy rollout (policy_kernel<12, 2>) and HitPPO with train.py's racket-scale curriculum.

The first test runs without a GPU (it needs the built library only); the others are marked gpu."""
import re
from pathlib import Path

import numpy as np
import pytest
import torch

ROOT = Path(__file__).resolve().parent.parent
TOL_F64_OUT = 2e-6  # float32 rounding of the outputs at |x| <= 20 (as in test_parity_gpu.py)


def test_hit_policy_layout_matches_header():
    """pack_policy of an ActorCritic(12, 2) has tb_policy_floats(1) = POLICY_FLOATS_HIT = 9324 entries, every tensor at the
    offset the header's layout comment gives; tb_policy_floats(0) is SwingRacket-v0's 9076."""
    from tennisbot_rl_b200 import _lib, build
    from tennisbot_rl_b200.ppo import ActorCritic

    build.build_library()
    L = _lib.load()
    assert L.tb_policy_floats(0) == _lib.POLICY_FLOATS == 9076
    assert L.tb_policy_floats(1) == _lib.POLICY_FLOATS_HIT == 9324
    assert L.tb_policy_floats(7) == -1
    header = (ROOT / "include" / "tennisbot_b200.h").read_text()
    assert re.search(r"#define TB_POLICY_FLOATS_HIT 9324\b", header)
    hit = header[header.index("Tennisbot-v0 (obs_dim 12, act_dim 2)"):header.index("#define TB_POLICY_FLOATS ")]
    assert [int(x) for x in re.findall(r"\((\d+) floats\)", hit)] == [4676, 4644, 4]

    ac = ActorCritic(12, 2)
    with torch.no_grad():  # every tensor gets its own value, so the packed vector shows where each one went
        for i, p in enumerate(ac.parameters()):
            p.fill_(i + 1)
    flat = ac.packed().numpy()
    assert flat.size == 9324
    lin = lambda seq: [m for m in seq if isinstance(m, torch.nn.Linear)]  # noqa: E731
    tower = lambda seq: sum(([m.weight, m.bias] for m in lin(seq)), [])  # noqa: E731
    # (tensor, offset, floats, padded floats) in the header's order
    pi = list(zip(tower(ac.pi) + [ac.mu.weight, ac.mu.bias], (0, 384, 416, 2464, 2528, 4576, 4608, 4672), (384, 32, 2048, 64, 2048, 32, 64, 2)))
    vf = list(zip(tower(ac.vf) + [ac.v.weight, ac.v.bias], (4676 + o for o in (0, 384, 416, 2464, 2528, 4576, 4608, 4640)),
                  (384, 32, 2048, 64, 2048, 32, 32, 1)))
    for t, off, size in pi + vf + [(ac.log_std, 9320, 2)]:
        v = float(t.reshape(-1)[0])
        np.testing.assert_array_equal(flat[off:off + size], v)
        pad = (-size) % 4
        np.testing.assert_array_equal(flat[off + size:off + size + pad], 0.0)
    with pytest.raises(ValueError):
        ActorCritic(12, 6).packed()


def _random_policy(seed):
    """A seeded ActorCritic(12, 2) whose actions are not all near zero (the default action head is scaled by 0.01)."""
    from tennisbot_rl_b200.ppo import ActorCritic

    torch.manual_seed(seed)
    ac = ActorCritic(12, 2)
    with torch.no_grad():
        ac.mu.weight.normal_(0, 0.5)
        ac.mu.bias.uniform_(-0.3, 0.3)
        ac.log_std.copy_(torch.tensor([-0.4, -0.7]))
    return ac


def _forward(ac, obs):
    """float32 numpy forward of the policy: mean action and value."""
    def tower(seq, x):
        for m in seq:
            if isinstance(m, torch.nn.Linear):
                x = np.tanh(x @ m.weight.detach().numpy().T + m.bias.detach().numpy())
        return x
    obs = obs.astype(np.float32)
    mean = tower(ac.pi, obs) @ ac.mu.weight.detach().numpy().T + ac.mu.bias.detach().numpy()
    value = (tower(ac.vf, obs) @ ac.v.weight.detach().numpy().T + ac.v.bias.detach().numpy())[:, 0]
    return mean, value


def _buffers(b, K):
    n, dev = b.num_envs, b.device
    z = lambda *s: torch.zeros(s, device=dev)  # noqa: E731
    return dict(obs=z(K, n, 12), actions=z(K, n, 2), logp=z(K, n), value=z(K, n), reward=z(K, n),
                done=torch.zeros((K, n), dtype=torch.uint8, device=dev), last_obs=z(n, 12), last_value=z(n))


def _rollout(b, buf, **kw):
    b.policy_rollout(buf["obs"], buf["reward"], buf["done"], buf["last_obs"], actions=buf["actions"], logp=buf["logp"],
                     value=buf["value"], last_value=buf["last_value"], **kw)


@pytest.mark.gpu
@pytest.mark.parametrize("deterministic,racket_scale", [(False, None), (True, None), (False, 2.5)])
def test_hit_policy_rollout_matches_numpy_policy_and_oracle(oracle_lib, deterministic, racket_scale):
    """K = 600 steps of 4096 Tennisbot-v0 envs (f64) from tb_policy_rollout with a seeded random policy: the recorded
    value, log-density (and, deterministic, the mean) agree with a numpy forward on the recorded observations; the oracle
    stepped with the recorded clipped actions reproduces observations, rewards and done flags, and the statistics are
    equal.  Stochastic: the implied noise is N(0, 1), uncorrelated across the two components and between steps t and t+1
    (a noise counter that did not advance would repeat it)."""
    from tennisbot_rl_b200.batch import TennisBatch

    n, K = 4096, 600
    ac = _random_policy(3)
    b = TennisBatch("Tennisbot-v0", n, seed=21, precision="f64")
    o = oracle_lib.OracleEnv("Tennisbot-v0", n, seed=21, threads=8)
    if racket_scale is not None:
        b.set_param("racket_scale", racket_scale)
        o.set_param("racket_scale", racket_scale)
    b.set_policy(ac.packed().cuda())
    buf = _buffers(b, K)
    buf["obs"][0].copy_(b.reset())
    np.testing.assert_array_equal(buf["obs"][0].cpu().numpy(), o.reset())
    _rollout(b, buf, deterministic=deterministic, noise_seed=5)
    torch.cuda.synchronize()
    h = {k: v.cpu().numpy() for k, v in buf.items()}
    std = np.exp(ac.log_std.detach().numpy())
    eps_all = np.zeros((K, n, 2), np.float32)
    for t in range(K):
        mean, value = _forward(ac, h["obs"][t])
        np.testing.assert_allclose(h["value"][t], value, atol=2e-4, rtol=1e-4)
        eps = (h["actions"][t] - mean) / std
        if deterministic:
            assert np.abs(eps).max() < 1e-4
        eps_all[t] = eps
        ref_logp = (-0.5 * eps.astype(np.float64) ** 2 - ac.log_std.detach().numpy() - 0.5 * np.log(2 * np.pi)).sum(1)
        np.testing.assert_allclose(h["logp"][t], ref_logp, atol=2e-3)
        ref = o.step(np.clip(h["actions"][t], -1, 1).astype(np.float32))
        nxt = h["obs"][t + 1] if t + 1 < K else h["last_obs"]
        np.testing.assert_array_equal(h["done"][t], ref["done"])
        np.testing.assert_allclose(nxt, ref["obs"], atol=TOL_F64_OUT)
        np.testing.assert_allclose(h["reward"][t], ref["reward"], atol=TOL_F64_OUT)
    np.testing.assert_allclose(h["last_value"], _forward(ac, h["last_obs"])[1], atol=2e-4, rtol=1e-4)
    st = b.read_stats()
    np.testing.assert_array_equal(st, o.read_stats())
    assert st[0] > 0  # episodes ended inside the rollout (auto-reset crossed)
    if racket_scale is not None:
        assert st[2] > 0  # racket-ball contacts
    if not deterministic:
        e = eps_all.reshape(-1, 2)
        assert abs(e.mean()) < 0.01 and abs(e.std() - 1) < 0.01 and abs((e ** 3).mean()) < 0.03
        assert abs(np.corrcoef(e.T)[0, 1]) < 0.01
        for c in range(2):  # step t against step t + 1, per component
            assert abs(np.corrcoef(eps_all[:-1, :, c].ravel(), eps_all[1:, :, c].ravel())[0, 1]) < 0.01
    b.close()


@pytest.mark.gpu
def test_hit_policy_noise_advances_under_graph_replay():
    """The hit rollout captured once in a CUDA graph draws fresh noise on every replay: Tennisbot-v0 has no fast-forward
    kernel, so its noise counter is the context's own device word, advanced by step_kernel."""
    from tennisbot_rl_b200.batch import TennisBatch

    n, K = 2048, 16
    b = TennisBatch("Tennisbot-v0", n, seed=2)
    b.set_policy(_random_policy(4).packed().cuda())
    buf = _buffers(b, K)
    buf["obs"][0].copy_(b.reset())
    s = torch.cuda.Stream(b.device)
    s.wait_stream(torch.cuda.current_stream(b.device))
    with torch.cuda.stream(s):
        _rollout(b, buf, noise_seed=1)
    torch.cuda.current_stream(b.device).wait_stream(s)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        buf["obs"][0].copy_(buf["last_obs"])
        _rollout(b, buf, noise_seed=1)
    runs = []
    for _ in range(3):
        g.replay()
        torch.cuda.synchronize()
        runs.append(buf["actions"].clone())
    assert not torch.equal(runs[0], runs[1]) and not torch.equal(runs[1], runs[2]) and not torch.equal(runs[0], runs[2])
    assert not torch.equal(runs[0][0], runs[0][1])  # and within one rollout, step to step
    b.close()


@pytest.mark.gpu
def test_hit_policy_rollout_is_shard_invariant():
    """Two contexts covering envs [0, N/2) and [N/2, N) (env_id_offset) produce the full batch's rollout bit for bit: the
    noise is keyed by the global env id and the step counter, not by the context."""
    from tennisbot_rl_b200.batch import TennisBatch

    n, K = 4096, 200
    params = _random_policy(5).packed().cuda()
    out = []
    for lo, hi in ((0, n), (0, n // 2), (n // 2, n)):
        b = TennisBatch("Tennisbot-v0", hi - lo, seed=8, env_id_offset=lo)
        b.set_policy(params)
        buf = _buffers(b, K)
        buf["obs"][0].copy_(b.reset())
        _rollout(b, buf, noise_seed=9)
        torch.cuda.synchronize()
        out.append(({k: v.cpu().numpy() for k, v in buf.items()}, b.read_stats()))
        b.close()
    (full, st_full), (a, st_a), (c, st_c) = out
    for k in full:
        axis = 0 if k in ("last_obs", "last_value") else 1
        np.testing.assert_array_equal(full[k], np.concatenate([a[k], c[k]], axis=axis), err_msg=k)
    np.testing.assert_array_equal(st_full, st_a + st_c)


@pytest.mark.gpu
def test_hit_ppo_curriculum_stages_under_graph_replay():
    """HitPPO with a small curriculum_total_timesteps (each rollout is 5 % of it) crosses three stages in four rollouts.
    At each change every env starts a new episode and the library's racket_scale is curriculum_scale; the rollout graph,
    captured again, gives state and statistics bit-identical to the same rollouts issued eagerly."""
    from tennisbot_rl_b200.playground import curriculum_scale
    from tennisbot_rl_b200.ppo import HitPPO

    n, K = 2048, 64
    total = 20 * n * K
    g = HitPPO(n, rollout_len=K, curriculum_total_timesteps=total, seed=3, use_graph=True)
    e = HitPPO(n, rollout_len=K, curriculum_total_timesteps=total, seed=3, use_graph=False)
    changes = 0
    for it in range(4):
        steps0 = g.env_steps
        for ppo in (g, e):
            before = ppo.env.get_state().cpu().numpy()
            changed = ppo.apply_curriculum()
            if changed:
                after = ppo.env.get_state().cpu().numpy()
                assert (after[:, 31] == before[:, 31] + 1).all() and (after[:, 29] == 0).all()
            if ppo is e and it == 0:  # the graph path's first rollout() runs one rollout as its warm-up
                with torch.no_grad():
                    e._rollout_body()
        changes += changed
        scale = curriculum_scale(steps0, total)
        st_g, st_e = g.rollout(), e.rollout()
        assert g.env.get_param("racket_scale") == scale == e.env.get_param("racket_scale") == g.scale
        np.testing.assert_array_equal(st_g, st_e)
        np.testing.assert_array_equal(g.env.get_state().cpu().numpy(), e.env.get_state().cpu().numpy())
        torch.testing.assert_close(g.obs_buf, e.obs_buf, rtol=0, atol=0)
    assert changes == 4 and [s for _, s in g.stages] == [3.0, 2.3, 2.1, 1.9]


def _tracker_mean_return(n, seed, steps):
    """Mean episodic return of the scripted tracker (tb_rollout(TB_ACT_TRACK)) over the episodes that end in `steps`."""
    from tennisbot_rl_b200 import _lib
    from tennisbot_rl_b200.batch import TennisBatch

    b = TennisBatch("Tennisbot-v0", n, seed=seed)
    b.reset()
    b.read_stats(clear=True)
    b.rollout(steps, action_mode=_lib.ACT_TRACK, want_outputs=False)
    st = b.read_stats()
    b.close()
    return float(st[6] / 2 ** 20 / st[0]), float(st[2] / st[0])


@pytest.mark.gpu
def test_hit_ppo_learns_and_is_compared_with_the_scripted_tracker():
    """16 384 envs, 128-step rollouts, 60 updates (126 M env steps), seed 0, no curriculum.  Measured on a B200 (1000 W):
    the mean return of the episodes ending in a rollout rises from 4.7 (untrained) to 11.4 after 60 updates; the scripted
    tracker (tb_rollout(TB_ACT_TRACK), same envs and seed) reaches 14.7, so PPO does NOT reach it within this budget.
    Mean of the first three rollouts 4.9, of the last three 11.3.  With lr = 0 the return stays where it starts (4.6 in a
    4096-env run of 30 updates), below the bar of 8.  Racket-ball contact steps per episode are reported, not asserted: they
    are noisy at this budget (0.01 after 30 updates, 0.04 in the last rollout; tracker 0.07)."""
    from tennisbot_rl_b200.ppo import HitPPO

    n = 16384
    track_return, track_hits = _tracker_mean_return(n, 0, 2000)
    ppo = HitPPO(n, rollout_len=128, seed=0)
    s = ppo.train(iters=60)
    hist = [h for h in s["history"] if h["episodes"]]
    first = np.mean([h["mean_return"] for h in hist[:3]])
    last = np.mean([h["mean_return"] for h in hist[-3:]])
    print({"tracker_mean_return": track_return, "tracker_hits_per_episode": track_hits, "ppo_first3_mean_return": first,
           "ppo_last3_mean_return": last, "ppo_last_hits_per_episode": hist[-1]["hits_per_episode"],
           "rollout_env_steps_per_s": s["rollout_env_steps_per_s"]})
    assert first < 6 and last > 8


@pytest.mark.gpu
def test_policy_buffers_are_checked():
    """set_policy and policy_rollout refuse what the library would write through out of bounds: the other env's parameter
    vector, and buffers of the wrong shape, dtype, device or layout."""
    from tennisbot_rl_b200 import _lib
    from tennisbot_rl_b200.batch import TennisBatch

    n, K = 256, 4
    b = TennisBatch("Tennisbot-v0", n, seed=1)
    with pytest.raises(ValueError):
        b.set_policy(torch.zeros(_lib.POLICY_FLOATS, device=b.device))
    b.set_policy(_random_policy(6).packed().cuda())
    dev = b.device
    bad = {"obs": torch.zeros((K, n, 6), device=dev), "actions": torch.zeros((K, n, 6), device=dev),
           "logp": torch.zeros((K + 1, n), device=dev), "value": torch.zeros((K, n), dtype=torch.float64, device=dev),
           "reward": torch.zeros((K, n)), "done": torch.zeros((K, n), device=dev),
           "last_obs": torch.zeros((12, n), device=dev).t(), "last_value": torch.zeros(n + 1, device=dev)}
    for k, v in bad.items():
        buf = _buffers(b, K)
        buf[k] = v
        with pytest.raises(ValueError, match=k):
            _rollout(b, buf)
    buf = _buffers(b, K)
    buf["obs"][0].copy_(b.reset())
    _rollout(b, buf)
    torch.cuda.synchronize()
    b.close()
