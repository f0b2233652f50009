"""Population rollouts and the population PPO learner on the B200.

- A context of P x n envs with P policies (tb_set_policies) gives, for every agent p, bit for bit what a one-policy context of
  n envs with env_id_offset = p n gives with that agent's policy: eagerly, through a replayed CUDA graph, with n a multiple
  of 128 and with agents that straddle the 128-env CTAs (down to one env per agent).
- PopulationPPO's gradients equal GpuPPO's per agent, agents are independent, its per-agent episode statistics add up to
  tb_read_stats, it learns, and a PBT round is seen by the captured update graph.
"""
import numpy as np
import pytest
import torch

from tennisbot_rl_b200 import _lib
from tennisbot_rl_b200.batch import TennisBatch
from tennisbot_rl_b200.population import PopulationPPO, agent_tensors
from tennisbot_rl_b200.ppo import ActorCritic, GpuPPO

pytestmark = pytest.mark.gpu
ENVS = ("SwingRacket-v0", "Tennisbot-v0")
KEYS = ("obs", "act", "logp", "value", "reward", "done", "last_obs", "last_value")


def _policies(env_id, P, seed=0):
    """P distinct packed policies, with log_std spread so the noise matters."""
    od, ad = (6, 6) if env_id == "SwingRacket-v0" else (12, 2)
    rows = []
    for p in range(P):
        torch.manual_seed(seed * 1000 + p)
        ac = ActorCritic(od, ad)
        with torch.no_grad():
            ac.log_std.fill_(-1.0 + 0.1 * (p % 7))
            ac.mu.weight.mul_(50.0)  # a mean that depends on the observation
        rows.append(ac.packed())
    return torch.stack(rows).cuda().contiguous()


def _buffers(b, K):
    n, od, ad = b.num_envs, b.obs_dim, b.act_dim
    z = lambda *s: torch.zeros(s, device="cuda")  # noqa: E731
    return dict(obs=z(K, n, od), act=z(K, n, ad), logp=z(K, n), value=z(K, n), reward=z(K, n),
                done=torch.zeros((K, n), dtype=torch.uint8, device="cuda"), last_obs=z(n, od), last_value=z(n))


def _rollout(b, buf, det, seed=9):
    b.policy_rollout(buf["obs"], buf["reward"], buf["done"], buf["last_obs"], actions=buf["act"], logp=buf["logp"],
                     value=buf["value"], last_value=buf["last_value"], deterministic=det, noise_seed=seed)


def _start(b, buf, prev=None):
    buf["obs"][0].copy_(b.reset() if prev is None else prev)


def _agent_slice(key, x, p, n):
    return x[p * n:(p + 1) * n] if key in ("last_obs", "last_value") else x[:, p * n:(p + 1) * n]


@pytest.mark.parametrize("env_id", ENVS)
@pytest.mark.parametrize("precision", ("f64", "f32"))
@pytest.mark.parametrize("P,n", ((2, 256), (3, 100), (7, 1)))
def test_population_rollout_equals_one_policy_shards(env_id, precision, P, n):
    K = 30 if env_id == "SwingRacket-v0" else 24  # SwingRacket-v0: across an episode boundary
    params = _policies(env_id, P)
    pop = TennisBatch(env_id, P * n, seed=5, precision=precision)
    pop.set_policies(params)
    shards = [TennisBatch(env_id, n, seed=5, precision=precision, env_id_offset=p * n) for p in range(P)]
    for p, s in enumerate(shards):
        s.set_policy(params[p])
    for det in (False, True):
        got, ref = _buffers(pop, K), [_buffers(s, K) for s in shards]
        for rnd in range(2):  # the second rollout continues from the first's last observation
            _start(pop, got, None if rnd == 0 else got["last_obs"].clone())
            _rollout(pop, got, det)
            for s, r in zip(shards, ref):
                _start(s, r, None if rnd == 0 else r["last_obs"].clone())
                _rollout(s, r, det)
            torch.cuda.synchronize()
            for p, r in enumerate(ref):
                for k in KEYS:
                    assert torch.equal(_agent_slice(k, got[k], p, n), r[k]), (det, rnd, p, k)


@pytest.mark.parametrize("env_id", ENVS)
@pytest.mark.parametrize("P,n", ((4, 128), (3, 100)))
def test_population_rollout_through_a_graph_equals_eager_calls(env_id, P, n):
    K = 26 if env_id == "SwingRacket-v0" else 16
    params = _policies(env_id, P, seed=1)
    eager, graphed = (TennisBatch(env_id, P * n, seed=3) for _ in range(2))
    be, bg = _buffers(eager, K), _buffers(graphed, K)
    eager.set_policies(params)
    graphed.set_policies(params)  # sizes the library's buffer before the capture
    _start(eager, be)
    _start(graphed, bg)
    torch.cuda.synchronize()
    src = params.clone()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        graphed.set_policies(src)
        _rollout(graphed, bg, False)
        bg["obs"][0].copy_(bg["last_obs"])
    for rep in range(3):
        if rep == 2:  # a replay copies the weights src holds then
            params[1].mul_(0.5)
            src.copy_(params)
        eager.set_policies(params)
        _rollout(eager, be, False)
        g.replay()
        torch.cuda.synchronize()
        for k in KEYS:
            if k != "obs":
                assert torch.equal(bg[k], be[k]), (rep, k)
        assert torch.equal(bg["obs"][1:], be["obs"][1:])
        be["obs"][0].copy_(be["last_obs"])


@pytest.mark.parametrize("env_id", ENVS)
def test_one_agent_and_launch_counts_equal_set_policy(env_id):
    K = 20
    params = _policies(env_id, 4)
    a, b, c = (TennisBatch(env_id, 512, seed=2) for _ in range(3))
    a.set_policy(params[0])
    b.set_policies(params[:1].contiguous())
    c.set_policies(params)
    bufs = [_buffers(x, K) for x in (a, b, c)]
    counts = []
    for x, buf in zip((a, b, c), bufs):
        _start(x, buf)
        n0 = x.launch_count()
        _rollout(x, buf, False)
        counts.append(x.launch_count() - n0)
    torch.cuda.synchronize()
    for k in KEYS:
        assert torch.equal(bufs[0][k], bufs[1][k]), k
    assert counts[0] == counts[1] == counts[2]


def test_rejections_and_set_policy_restores_one_policy():
    env_id, n = "Tennisbot-v0", 384
    b = TennisBatch(env_id, n, seed=1)
    L, F = b.lib, _lib.POLICY_FLOATS_HIT
    params = _policies(env_id, 3)
    p = params.data_ptr()

    def err(*args):
        assert L.tb_set_policies(b.h, *args, b._stream()) != 0
        return L.tb_last_error().decode()

    assert "NULL" in err(None, 3, 3 * F)
    assert "divide" in err(p, 0, 0)
    assert "divide" in err(p, 5, 5 * F)
    assert "expected" in err(p, 3, 3 * F - 4)
    with pytest.raises(ValueError, match="set_policies"):
        b.set_policies(torch.zeros(5, F, device="cuda"))
    buf = _buffers(b, 8)
    b.set_policies(params)
    b.set_vecnorm()
    _start(b, buf)
    with pytest.raises(_lib.TennisbotLibraryError, match="tb_set_vecnorm.*tb_set_policies"):
        _rollout(b, buf, False)
    b.set_policy(params[0])  # one policy again: the normalised rollout runs
    _rollout(b, buf, False)
    b.clear_vecnorm()
    one = TennisBatch(env_id, n, seed=1)
    one.set_policy(params[0])
    ref = _buffers(one, 8)
    b.set_policies(params)
    b.set_policy(params[0])
    _start(one, ref)
    buf["obs"][0].copy_(ref["obs"][0])
    _rollout(b, buf, True)
    _rollout(one, ref, True)
    torch.cuda.synchronize()
    assert torch.equal(buf["act"][0], ref["act"][0])  # the same observation, one policy: the same deterministic action


# ------------------------------------------------------------------ learner
def _fill_minibatch(pop, gen):
    for t in (pop.mb_obs, pop.mb_act, pop.mb_logp, pop.mb_adv, pop.mb_ret):
        t.copy_(torch.randn(t.shape, device="cuda", generator=gen))
    pop.mb_logp.sub_(2.0)


@pytest.mark.parametrize("env_id", ENVS)
def test_population_gradients_equal_gpu_ppo_per_agent(env_id):
    seeds, n, K = [1, 2, 3], 256, 8
    pop = PopulationPPO(env_id, 3, n, K, seeds=seeds, use_graph=False, max_grad_norm=[0.5, 0.05, 10.0], ent_coef=[0.002, 0.01, 0.0])
    gen = torch.Generator("cuda").manual_seed(4)
    _fill_minibatch(pop, gen)
    pop.hyper["lr"].zero_()  # Adam with lr 0 leaves the weights: compare the clipped gradients
    pop._minibatch_step()
    for p, s in enumerate(seeds):
        ref = GpuPPO(env_id, n, K, seed=s, use_graph=False)
        ref.max_norm, ref.ent_coef = [0.5, 0.05, 10.0][p], [0.002, 0.01, 0.0][p]
        for dst, src in ((ref.mb_obs, pop.mb_obs), (ref.mb_act, pop.mb_act), (ref.mb_logp, pop.mb_logp), (ref.mb_adv, pop.mb_adv),
                         (ref.mb_ret, pop.mb_ret)):
            dst.copy_(src[p])
        for grp in ref.opt.param_groups:
            grp["lr"] = 0.0
        ref._minibatch_step()
        for t, r in zip(pop.ac.params, agent_tensors(ref.ac)):
            assert torch.equal(t[p].detach(), r.detach())
            rel = float((t.grad[p] - r.grad).norm() / r.grad.norm().clamp_min(1e-30))
            assert rel < 1e-5, (p, tuple(r.shape), rel)
        ref.env.close()


def _state(pop):
    return [t.detach().clone() for t in pop.ac.params + pop.opt.state_tensors() + list(pop.hyper.values())] + \
        [pop.gen.get_state()]


def _load(pop, st):
    with torch.no_grad():
        for t, v in zip(pop.ac.params + pop.opt.state_tensors() + list(pop.hyper.values()), st[:-1]):
            t.copy_(v)
    pop.gen.set_state(st[-1])


def test_agents_are_independent():
    n = 512
    pop = PopulationPPO("SwingRacket-v0", 2, n, 26, seeds=[1, 2], lr=[3e-4, 1e-3])
    pop.rollout()
    st = _state(pop)
    pop.update()
    a = [t.detach().clone() for t in pop.ac.params]
    _load(pop, st)
    pop.rew_buf[:, n:] += 1.0
    pop.obs_buf[:, n:] *= 0.5
    pop.update()
    for t, t0 in zip(pop.ac.params, a):
        assert torch.equal(t[0], t0[0])
    assert any(not torch.equal(t[1], t0[1]) for t, t0 in zip(pop.ac.params, a))


@pytest.mark.parametrize("env_id", ENVS)
def test_per_agent_statistics_add_up_to_read_stats(env_id):
    K = 26 if env_id == "SwingRacket-v0" else 128
    pop = PopulationPPO(env_id, 4, 1024, K, seeds=[1, 2, 3, 4])
    total_eps = 0
    for it in range(3):
        eps, rsum, lsum, st = pop.rollout()
        assert int(eps.sum()) == int(st[0]), it
        total_eps += int(st[0])
        if st[0]:
            np.testing.assert_allclose(rsum.sum(), st[6] / 2 ** 20, rtol=1e-4, atol=1e-3)
        pop.update()
    assert total_eps > 0


def test_population_learns_swing():
    """4 agents x 4 096 SwingRacket-v0 envs, seeds 1-4, 25 updates: each ends more than 2 above its first return (the bar of
    test_ppo_learns_on_the_gpu_env).  Measured on a B200 at 1000 W: first -> last 0.16 -> 24.84, 0.03 -> 24.66, 0.06 -> 24.83,
    0.10 -> 24.09."""
    pop = PopulationPPO("SwingRacket-v0", 4, 4096, 26, seeds=[1, 2, 3, 4])
    out = pop.train(25)
    for a in out["per_agent"]:
        first, last = a["history"][0]["mean_return"], a["history"][-1]["mean_return"]
        print(f"seed {a['seed']}: first {first:.2f} last {last:.2f} best {a['best_mean_return']:.2f}")
        assert last > first + 2.0, a["seed"]


def test_pbt_round_is_seen_by_the_captured_update_graph():
    pop = PopulationPPO("SwingRacket-v0", 4, 256, 26, seeds=[1, 2, 3, 4], pbt_seed=3)
    pop.train(2)  # captures the rollout and the update graphs
    assert pop.upd_graph is not None
    before = {k: v.clone() for k, v in pop.hyper.items()}
    ev = pop.exploit_explore(scores=[1.0, 4.0, 2.0, 3.0])
    (upd, dst, src, hp), = ev
    assert (dst, src) == (0, 1) and upd == 2 and not torch.equal(pop.hyper["lr"][dst], before["lr"][dst])
    pop.rollout()
    st = _state(pop)
    pop.update()  # the graph
    graph = [t.detach().clone() for t in pop.ac.params]
    _load(pop, st)
    pop.use_graph = False
    pop.update()  # eager, from the same state
    for t, g in zip(pop.ac.params, graph):
        torch.testing.assert_close(t.detach(), g, rtol=0, atol=0)
    _load(pop, st)  # the old hyper-parameters of the destination give another update
    with torch.no_grad():
        for k, v in pop.hyper.items():
            v[dst] = before[k][src]
    pop.update()
    assert any(not torch.equal(t[dst], g[dst]) for t, g in zip(pop.ac.params, graph))
