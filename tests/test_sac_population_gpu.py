"""A population of SAC actors in one context (tb_set_sac_actors, sac_kernel<.., POP>) and the PopulationSAC learner.

Every rollout comparison is bit for bit: agent p's envs of a P x n context against a context of n envs at env_id_offset = p n
with set_sac_actor(row p), which tests/test_sac_gpu.py ties to the float32 SacActor and the oracle.
"""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

ENVS = {"SwingRacket-v0": (6, 6), "Tennisbot-v0": (12, 2)}
KEYS = ("obs", "act", "reward", "next_obs", "done")


def _ring(slots, n, od, ad, dev):
    z = lambda *s, dt=torch.float32: torch.zeros(s, dtype=dt, device=dev)  # noqa: E731
    return dict(obs=z(slots, n, od), act=z(slots, n, ad), reward=z(slots, n), next_obs=z(slots, n, od),
                done=z(slots, n, dt=torch.uint8))


def _rows(env_id, seeds):
    """float32 [P, sac_floats] on the device: fresh SacActors, their log_std bias raised so the sampled noise matters."""
    from tennisbot_rl_b200.sac import SacActor, pack_sac_actor

    od, ad = ENVS[env_id]
    out = []
    for s in seeds:
        torch.manual_seed(s)
        a = SacActor(od, ad)
        with torch.no_grad():
            a.log_std.bias.add_(-1.0 + 0.1 * s)
        out.append(pack_sac_actor(a))
    return torch.stack(out).cuda().contiguous()


def _run(env_id, n, steps, mode, rows, precision="f64", offset=0, seed=9, single=False):
    """tb_sac_begin, a uniform warm-up step, then `steps` steps in `mode` on a fresh context of n envs; rows [P, floats] go
    through set_sac_actors (single: set_sac_actor(rows[0])).  Returns the ring and the last observation as numpy."""
    from tennisbot_rl_b200.batch import TennisBatch

    od, ad = ENVS[env_id]
    b = TennisBatch(env_id, n, seed=seed, precision=precision, env_id_offset=offset)
    if single:
        b.set_sac_actor(rows[0].contiguous())
    else:
        b.set_sac_actors(rows)
    b.sac_begin()
    ring = _ring(steps + 1, n, od, ad, b.device)
    last = torch.zeros(n, od, device=b.device)
    b.sac_rollout(1, "uniform", ring, noise_seed=5)
    b.sac_rollout(steps, mode, ring, noise_seed=5, last_obs=last)
    torch.cuda.synchronize()
    out = {k: v.cpu().numpy() for k, v in ring.items()}
    out["last_obs"] = last.cpu().numpy()
    b.close()
    return out


def _assert_shards(env_id, P, n, steps, mode, precision):
    rows = _rows(env_id, range(20, 20 + P))
    full = _run(env_id, P * n, steps, mode, rows, precision)
    for p in range(P):
        part = _run(env_id, n, steps, mode, rows[p:p + 1], precision, offset=p * n, single=True)
        for k in KEYS:
            np.testing.assert_array_equal(full[k][:, p * n:(p + 1) * n], part[k], err_msg=f"{k} agent {p}")
        np.testing.assert_array_equal(full["last_obs"][p * n:(p + 1) * n], part["last_obs"], err_msg=f"last_obs agent {p}")
    return full


@pytest.mark.parametrize("P,n", [(2, 128), (3, 256)])
@pytest.mark.parametrize("mode", ["sample", "mean"])
@pytest.mark.parametrize("precision", ["f32", "f64"])
@pytest.mark.parametrize("env_id", list(ENVS))
def test_agents_equal_one_actor_shards(env_id, precision, mode, P, n):
    steps = 30 if env_id == "SwingRacket-v0" else 12  # SwingRacket-v0: across the 26-step episode boundary
    full = _assert_shards(env_id, P, n, steps, mode, precision)
    if env_id == "SwingRacket-v0":
        assert full["done"].any()


def crossing_ctas(P, n, sms):
    """CTAs of sac_kernel's persistent grid (min(tiles, sms) CTAs, CTA b running tiles [tiles b / G, tiles (b + 1) / G)) whose
    chunk spans two agents, i.e. that reload the image inside their loop."""
    tiles, per_agent = P * n // 128, n // 128
    G = min(tiles, sms)
    return sum(1 for b in range(G) if (tiles * b // G) // per_agent != (tiles * (b + 1) // G - 1) // per_agent)


@pytest.mark.parametrize("env_id", list(ENVS))
def test_more_tiles_than_sms_reload_images_across_agent_boundaries(env_id):
    """More tiles than SMs with chunks that span two agents, so the reload branch inside the tile loop runs.  When P divides
    the CTA count every agent boundary falls on a chunk boundary and nothing reloads (4 x 8192 on 148 SMs), so the shape is
    the first of a few whose chunks cross on this card."""
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    P, n = next(((P, n) for P, n in ((16, 4096), (5, 8192), (3, 8192), (7, 4096)) if crossing_ctas(P, n, sms)), (0, 0))
    assert P, f"no candidate shape has a CTA whose chunk spans two agents on {sms} SMs"
    assert crossing_ctas(4, 8192, 148) == 0 and crossing_ctas(16, 4096, 148) == 8  # the count, checked on the B200's 148
    _assert_shards(env_id, P, n, 3, "sample", "f32")


@pytest.mark.parametrize("env_id", list(ENVS))
def test_one_agent_is_set_sac_actor_and_launch_counts(env_id):
    from tennisbot_rl_b200.batch import TennisBatch

    rows = _rows(env_id, (1, 2))
    a = _run(env_id, 256, 5, "sample", rows[:1])
    b = _run(env_id, 256, 5, "sample", rows[:1], single=True)
    for k in KEYS + ("last_obs",):
        np.testing.assert_array_equal(a[k], b[k], err_msg=k)
    od, ad = ENVS[env_id]
    s, K = (2 if env_id == "SwingRacket-v0" else 1), 3
    e = TennisBatch(env_id, 256, seed=3)
    ring = _ring(8, 256, od, ad, e.device)

    def launches(call):
        before = e.launch_count()
        call()
        torch.cuda.synchronize()
        return e.launch_count() - before

    assert launches(lambda: e.set_sac_actors(rows[:1].contiguous())) == 1
    assert launches(lambda: e.set_sac_actors(rows)) == 1
    assert launches(lambda: e.sac_begin()) == 1
    for mode in ("uniform", "sample", "mean"):
        assert launches(lambda: e.sac_rollout(K, mode, ring)) == (K + 1) + K * s
    e.close()
    # set_sac_actor after a population returns the context to one actor
    c = TennisBatch(env_id, 256, seed=9)
    c.set_sac_actors(rows)
    c.set_sac_actor(rows[1].contiguous())
    c.sac_begin()
    ring = _ring(6, 256, od, ad, c.device)
    last = torch.zeros(256, od, device=c.device)
    c.sac_rollout(1, "uniform", ring, noise_seed=5)
    c.sac_rollout(5, "sample", ring, noise_seed=5, last_obs=last)
    ref = _run(env_id, 256, 5, "sample", rows[1:2], single=True)
    for k in KEYS:
        np.testing.assert_array_equal(ring[k].cpu().numpy(), ref[k], err_msg=k)
    c.close()


@pytest.mark.parametrize("env_id", list(ENVS))
def test_captured_collection_equals_eager_calls_and_reads_weights_at_replay(env_id):
    from tennisbot_rl_b200.batch import TennisBatch

    od, ad = ENVS[env_id]
    P, n, K = 2, 256, 2
    rows, other = _rows(env_id, (3, 4)), _rows(env_id, (5, 6))
    outs = []
    for graphed, change in ((False, True), (True, True), (False, False)):
        b = TennisBatch(env_id, P * n, seed=4)
        params = rows.clone()
        b.set_sac_actors(params)  # grows the image buffer before any capture
        b.sac_begin()
        ring = _ring(3 * K + 1, P * n, od, ad, b.device)
        b.sac_rollout(1, "uniform", ring, noise_seed=2)

        def body():
            b.set_sac_actors(params)
            b.sac_rollout(K, "sample", ring, noise_seed=2)
        if graphed:
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                body()
            run = g.replay
        else:
            run = body
        for i in range(3):
            if i == 2 and change:
                params.copy_(other)  # written between replays: the third collection acts with these weights
            run()
        torch.cuda.synchronize()
        outs.append({k: v.cpu().numpy() for k, v in ring.items()})
        b.close()
    changed, graphed, unchanged = outs
    for k in KEYS:
        np.testing.assert_array_equal(changed[k], graphed[k], err_msg=k)
    # slot 0 is the warm-up, collection c fills slots 1 + c K .. (c + 1) K: the first two do not depend on the change, the
    # third acts with the new weights in every agent's columns
    third = slice(1 + 2 * K, 1 + 3 * K)
    for k in KEYS:
        np.testing.assert_array_equal(changed[k][:third.start], unchanged[k][:third.start], err_msg=k)
    for p in range(P):
        assert not np.array_equal(changed["act"][third, p * n:(p + 1) * n], unchanged["act"][third, p * n:(p + 1) * n])


@pytest.mark.parametrize("env_id", list(ENVS))
def test_rejections_leave_the_actors_in_place(env_id):
    from tennisbot_rl_b200 import _lib
    from tennisbot_rl_b200.batch import TennisBatch

    od, ad = ENVS[env_id]
    L = _lib.load()
    rows = _rows(env_id, (7, 8))
    n = 512
    b = TennisBatch(env_id, n, seed=9)
    b.set_sac_actors(rows)
    F = L.tb_sac_floats(b.kind)

    def err(rc):
        assert rc != 0
        return L.tb_last_error().decode()

    big = torch.zeros(8, F, device=b.device)
    p = big.data_ptr()
    assert "d_params is NULL" in err(L.tb_set_sac_actors(b.h, None, 2, 2 * F, None))
    assert "must be >= 1 and divide" in err(L.tb_set_sac_actors(b.h, p, 0, 0, None))
    assert "must be >= 1 and divide" in err(L.tb_set_sac_actors(b.h, p, 3, 3 * F, None))
    assert "expected agents x tb_sac_floats" in err(L.tb_set_sac_actors(b.h, p, 2, 2 * F + 4, None))
    msg = err(L.tb_set_sac_actors(b.h, p, 8, 8 * F, None))  # 64 envs per agent
    assert "multiple of 128" in msg and "two 128 KB images do not fit" in msg
    b.set_vecnorm(gamma=0.99)
    b.sac_begin()
    ring = _ring(6, n, od, ad, b.device)
    with pytest.raises(_lib.TennisbotLibraryError, match="2 actors are set"):
        b.sac_rollout(1, "sample", ring, normalize=True)
    last = torch.zeros(n, od, device=b.device)
    b.sac_rollout(1, "uniform", ring, noise_seed=5)
    b.sac_rollout(5, "sample", ring, noise_seed=5, last_obs=last)
    ref = _run(env_id, n, 5, "sample", rows)  # the actors of the last accepted call
    for k in KEYS:
        np.testing.assert_array_equal(ring[k].cpu().numpy(), ref[k], err_msg=k)
    b.close()


# ------------------------------------------------------------------------------------------------ the learner
def _small_pop(**kw):
    from tennisbot_rl_b200.sac_population import PopulationSAC

    args = dict(env_id="SwingRacket-v0", agents=2, envs_per_agent=128, batch_size=64, gradient_steps=2, slots=16,
                seeds=[0, 1], eval_envs=128, lr=[3e-4, 1e-3], tau=[0.005, 0.05], gamma=[0.99, 0.9])
    args.update(kw)
    return PopulationSAC(**args)


def test_gradient_step_equals_per_agent_gpusac_steps():
    from tennisbot_rl_b200.sac import SacActor, TwinCritic, actor_loss, sac_losses

    pop = _small_pop()
    for _ in range(3):
        pop.collect()
    P, B, ad = pop.P, pop.B, pop.ad
    torch.manual_seed(1)
    pop.fill.fill_(float(min(pop.steps_taken, pop.slots) * pop.n))
    batch = pop._gather(pop.sample())
    noise, next_noise = torch.randn(P, B, ad, device=pop.dev), torch.randn(P, B, ad, device=pop.dev)
    refs = []
    for p, s in enumerate(pop.seeds):  # GpuSAC(seed=s)'s starting modules, with torch.optim.Adam
        torch.manual_seed(s)
        actor, critic, target = SacActor(pop.od, ad).cuda(), TwinCritic(pop.od, ad).cuda(), TwinCritic(pop.od, ad).cuda()
        target.load_state_dict(critic.state_dict())
        la = torch.zeros(1, device=pop.dev, requires_grad=True)
        lr = float(pop.hyper["lr"][p])
        refs.append((actor, critic, target, la, [torch.optim.Adam(x, lr=lr) for x in (actor.parameters(), critic.parameters(), [la])]))
    pop.gradient_step(batch, noise, next_noise)
    for p, (actor, critic, target, la, (ao, co, lo)) in enumerate(refs):
        a_loss, c_loss, pi, logp, alpha = sac_losses(actor, critic, target, la, tuple(x[p] for x in batch),
                                                     float(pop.hyper["gamma"][p]), -float(ad), noise[p], next_noise[p])
        lo.zero_grad(); a_loss.backward(); lo.step()  # noqa: E702
        co.zero_grad(); c_loss.backward(); co.step()  # noqa: E702
        pl = actor_loss(critic, batch[0][p], pi, logp, alpha)
        ao.zero_grad(); pl.backward(); ao.step()  # noqa: E702
        with torch.no_grad():
            for q, tq in zip(critic.parameters(), target.parameters()):
                tq.lerp_(q, float(pop.hyper["tau"][p]))
        for mine, ref in ((pop.actor, actor), (pop.critic, critic), (pop.critic_target, target)):
            for t, r in zip(mine.params, ref.parameters()):
                torch.testing.assert_close(t[p].detach(), r.detach(), atol=1e-5, rtol=0)
        torch.testing.assert_close(pop.log_alpha[p].detach(), la[0].detach(), atol=1e-6, rtol=0)


def test_agents_are_independent():
    a, b = _small_pop(), _small_pop()
    with torch.no_grad():
        for t in b.actor.params + b.critic.params:
            t[1].add_(0.05 * torch.randn_like(t[1]))
    for pop in (a, b):
        pop.collect()
        pop.collect()
    torch.cuda.synchronize()
    n = a.n
    for k in KEYS:
        assert torch.equal(a.ring[k][:, :n], b.ring[k][:, :n]), k
    assert not torch.equal(a.ring["act"][:, n:], b.ring["act"][:, n:])
    torch.manual_seed(3)
    a.fill.fill_(float(min(a.steps_taken, a.slots) * n))
    idx = a.sample()
    g = torch.Generator(device=a.dev).manual_seed(4)
    noise = [torch.randn(a.P, a.B, a.ad, device=a.dev, generator=g) for _ in range(2)]
    for pop in (a, b):
        pop.gradient_step(pop._gather(idx), *noise)
    for mine, other in ((a.actor, b.actor), (a.critic, b.critic), (a.critic_target, b.critic_target)):
        for t, u in zip(mine.params, other.params):
            assert torch.equal(t[0], u[0])
            assert not torch.equal(t[1], u[1])
    assert torch.equal(a.log_alpha[0], b.log_alpha[0])


def test_pbt_round_is_seen_by_the_captured_update_graph():
    pop = _small_pop()
    pop.collect()
    pop.update()  # captures the graph
    ev = pop.exploit_explore([1.0, 0.0])
    assert [(e[1], e[2]) for e in ev] == [(1, 0)]
    for t in pop._state():
        assert torch.equal(t[1], t[0])
    assert float(pop.hyper["gamma"][1]) == float(pop.hyper["gamma"][0])
    with torch.no_grad():
        pop.hyper["lr"][1] = 0.0
        pop.hyper["tau"][1] = 0.0
    frozen = [t[1].clone() for t in pop.actor.params + pop.critic_target.params]
    moved = [t[0].clone() for t in pop.actor.params]
    pop.update()
    for t, f in zip(pop.actor.params + pop.critic_target.params, frozen):
        assert torch.equal(t[1], f)  # lr 0 and tau 0 for agent 1, read by the graph at replay
    assert any(not torch.equal(t[0], m) for t, m in zip(pop.actor.params, moved))
    sd = pop.state_dict()
    assert sd["actors"].shape == (2, pop.params.shape[1]) and sd["pbt_events"].shape == (1, 6)
    np.testing.assert_array_equal(pop.agent_state_dict(1)["policy"], sd["actors"][1])


# ------------------------------------------------------------------------------------------------ learning
SWING_BAR, SWING_ITERS = 22.0, 5000  # test_gpu_sac_learns_swing's bar and length


def test_population_sac_learns_swing():
    """4 agents x 1024 envs, seeds 0-3, GpuSAC's defaults: the mean of the agents' final deterministic evaluations must clear
    SWING_BAR, and every agent must end at least 10 above its first evaluation."""
    from tennisbot_rl_b200.sac_population import PopulationSAC

    pop = PopulationSAC("SwingRacket-v0", 4, 1024, seeds=[0, 1, 2, 3])
    out = pop.train(SWING_ITERS, log=print, eval_every=SWING_ITERS // 5)
    for a in out["per_agent"]:
        print(f"seed {a['seed']}: evaluations {[round(v, 2) for v in a['evaluations']]}")
    finals = [a["evaluations"][-1] for a in out["per_agent"]]
    print(f"SwingRacket-v0 PopulationSAC 4 x 1024: finals {[round(v, 2) for v in finals]} mean {np.mean(finals):.2f}, "
          f"collect {out['collect_s']:.1f}s update {out['update_s']:.1f}s wall {out['wall_s']:.1f}s")
    assert np.mean(finals) >= SWING_BAR
    for a in out["per_agent"]:
        assert a["evaluations"][-1] >= a["evaluations"][0] + 10, a["seed"]
