"""The population learner's host side, without a GPU: the stacked actor-critic against per-agent ActorCritics, the per-agent
Adam against torch.optim.Adam, per-agent gradient clipping, the vectorised episode statistics against a step loop, the PBT
round, and the argument checks of PopulationPPO and TennisBatch.set_policies."""
import numpy as np
import pytest
import torch
import torch.nn as nn

from tennisbot_rl_b200 import _lib
from tennisbot_rl_b200.batch import TennisBatch
from tennisbot_rl_b200.population import (BatchedActorCritic, BatchedAdam, PopulationPPO, agent_tensors, clip_grad_norms,
                                          episode_stats, exploit_explore)
from tennisbot_rl_b200.ppo import ActorCritic

DIMS = ((6, 6), (12, 2))
SEEDS = (3, 11, 5)


def _per_agent(od, ad, seeds=SEEDS):
    out = []
    for s in seeds:
        torch.manual_seed(s)
        out.append(ActorCritic(od, ad))
    return out


@pytest.mark.parametrize("od,ad", DIMS)
def test_initial_weights_and_packed_rows_equal_per_agent_actor_critics(od, ad):
    bac, acs = BatchedActorCritic(od, ad, SEEDS), _per_agent(od, ad)
    for p, ac in enumerate(acs):
        for t, ref in zip(bac.params, agent_tensors(ac)):
            assert torch.equal(t[p], ref.detach())
    packed = bac.packed()
    assert packed.shape == (len(SEEDS), _lib.POLICY_FLOATS if od == 6 else _lib.POLICY_FLOATS_HIT)
    for p, ac in enumerate(acs):
        assert torch.equal(packed[p], ac.packed())


@pytest.mark.parametrize("od,ad", DIMS)
def test_batched_log_prob_value_entropy_equal_per_agent(od, ad):
    bac, acs = BatchedActorCritic(od, ad, SEEDS), _per_agent(od, ad)
    g = torch.Generator().manual_seed(0)
    with torch.no_grad():  # distinct log_std per agent, so the entropy differs between them
        bac.params[16].copy_(torch.randn(bac.params[16].shape, generator=g) * 0.3)
        for p, ac in enumerate(acs):
            ac.log_std.copy_(bac.params[16][p])
    obs = torch.randn(len(SEEDS), 257, od, generator=g)
    act = torch.randn(len(SEEDS), 257, ad, generator=g)
    lp, v, ent = bac.log_prob(obs, act), bac.value(obs), bac.entropy()
    for p, ac in enumerate(acs):
        torch.testing.assert_close(lp[p], ac.log_prob(obs[p], act[p]), atol=1e-6, rtol=1e-6)
        torch.testing.assert_close(v[p], ac.value(obs[p]), atol=1e-6, rtol=1e-6)
        torch.testing.assert_close(ent[p], ac.entropy(), atol=1e-6, rtol=1e-6)


def test_per_agent_adam_and_clipping_equal_torch_per_agent():
    bac, acs = BatchedActorCritic(6, 6, SEEDS), _per_agent(6, 6)
    lr = torch.tensor([3e-4, 1e-3, 5e-5])
    max_norm = torch.tensor([0.5, 0.05, 10.0])
    opt = BatchedAdam(bac.params, lr)
    refs = [torch.optim.Adam(ac.parameters(), lr=float(lr[p]), eps=1e-5) for p, ac in enumerate(acs)]
    g = torch.Generator().manual_seed(1)
    for _ in range(6):
        obs, act = torch.randn(3, 64, 6, generator=g), torch.randn(3, 64, 6, generator=g)
        for t in bac.params:
            t.grad = None
        (bac.log_prob(obs, act).mean(1) + bac.value(obs).pow(2).mean(1)).sum().backward()
        clip_grad_norms(bac.params, max_norm)
        opt.step()
        for p, (ac, ref) in enumerate(zip(acs, refs)):
            ref.zero_grad()
            (ac.log_prob(obs[p], act[p]).mean() + ac.value(obs[p]).pow(2).mean()).backward()
            nn.utils.clip_grad_norm_(ac.parameters(), float(max_norm[p]))
            ref.step()
    for p, ac in enumerate(acs):
        for t, r in zip(bac.params, agent_tensors(ac)):
            torch.testing.assert_close(t[p].detach(), r.detach(), atol=1e-7, rtol=0)
    assert opt.steps.tolist() == [6.0] * 3


def test_episode_stats_equal_a_step_loop():
    g = torch.Generator().manual_seed(2)
    P, n, K = 3, 5, 9
    N = P * n
    carry_ret, carry_len = torch.rand(N, dtype=torch.float64, generator=g), torch.randint(0, 4, (N,), generator=g).double()
    ref_ret, ref_len = carry_ret.clone(), carry_len.clone()
    for _ in range(3):  # episodes that span rollouts
        reward = torch.randn(K, N, generator=g)
        done = (torch.rand(K, N, generator=g) < 0.25).to(torch.uint8)
        eps, rsum, lsum = episode_stats(reward, done, carry_ret, carry_len, P)
        e_ref, r_ref, l_ref = np.zeros(P, np.int64), np.zeros(P), np.zeros(P)
        for t in range(K):
            ref_ret += reward[t].double()
            ref_len += 1
            for i in range(N):
                if done[t, i]:
                    e_ref[i // n] += 1
                    r_ref[i // n] += ref_ret[i]
                    l_ref[i // n] += ref_len[i]
                    ref_ret[i] = 0
                    ref_len[i] = 0
        np.testing.assert_array_equal(eps.numpy(), e_ref)
        np.testing.assert_allclose(rsum.numpy(), r_ref, rtol=1e-12, atol=1e-12)
        np.testing.assert_array_equal(lsum.numpy(), l_ref)
        torch.testing.assert_close(carry_ret, ref_ret, rtol=1e-12, atol=1e-12)
        torch.testing.assert_close(carry_len, ref_len, rtol=0, atol=0)


def _pbt_setup(P=8):
    bac = BatchedActorCritic(6, 6, range(P))
    opt = BatchedAdam(bac.params, torch.full((P,), 3e-4))
    g = torch.Generator().manual_seed(3)
    with torch.no_grad():
        for t in opt.state_tensors():
            t.copy_(torch.rand(t.shape, generator=g, dtype=t.dtype))
    hyper = {k: torch.rand(P, generator=g) for k in ("lr", "ent_coef", "clip", "vf_coef", "max_grad_norm", "gamma", "gae_lambda")}
    return bac.params + opt.state_tensors(), hyper


def test_pbt_round_copies_the_top_into_the_bottom_and_perturbs_lr_and_ent_coef():
    P = 8
    scores = [5.0, None, 1.0, 7.0, -2.0, 3.0, 6.0, 0.5]  # ranking 3, 6, 0, 5, 2, 7, 4, 1 (no episode: last)
    tensors, hyper = _pbt_setup(P)
    before = [t.detach().clone() for t in tensors], {k: v.clone() for k, v in hyper.items()}
    events = exploit_explore(scores, tensors, hyper, np.random.default_rng(7))
    assert sorted(e[0] for e in events) == [1, 4]
    assert all(e[1] in (3, 6) for e in events)
    for dst, src, hp in events:
        for t, t0 in zip(tensors, before[0]):
            assert torch.equal(t[dst], t0[src])
        for k, v in hyper.items():
            if k in ("lr", "ent_coef"):
                assert any(torch.equal(v[dst], before[1][k][src] * f) for f in (0.8, 1.2))
            else:
                assert torch.equal(v[dst], before[1][k][src])
            assert hp[k] == float(v[dst])
    for p in range(P):  # every agent outside the bottom two is untouched
        if p in (1, 4):
            continue
        for t, t0 in zip(tensors, before[0]):
            assert torch.equal(t[p], t0[p])
        for k, v in hyper.items():
            assert torch.equal(v[p], before[1][k][p])
    again_t, again_h = _pbt_setup(P)
    assert exploit_explore(scores, again_t, again_h, np.random.default_rng(7)) == events
    with pytest.raises(ValueError, match="2 agents"):
        exploit_explore([1.0], tensors[:1], {}, np.random.default_rng(0))


def test_hyper_parameters_of_the_wrong_length_are_rejected():
    for kw in ({"lr": [3e-4, 1e-4]}, {"ent_coef": [0.0] * 4}, {"gamma": []}, {"seeds": [1, 2]}):
        with pytest.raises(ValueError, match="one per agent"):
            PopulationPPO("SwingRacket-v0", 3, 128, 26, **kw)
    with pytest.raises(ValueError, match="pbt_interval"):
        PopulationPPO("SwingRacket-v0", 1, 128, 26, pbt_interval=5)


def test_set_policies_argument_checks():
    b = TennisBatch.__new__(TennisBatch)  # only the checks that run before the library is called
    b.kind, b.num_envs, b.device, b.obs_dim, b.act_dim = _lib.ENV_SWING, 12, torch.device("cuda", 0), 6, 6
    F = _lib.POLICY_FLOATS
    for bad in (torch.zeros(F), torch.zeros(5, F), torch.zeros(0, F), torch.zeros(3, F + 4)):
        with pytest.raises(ValueError, match="set_policies"):
            b.set_policies(bad)
    with pytest.raises(ValueError, match="set_policies"):
        b.set_policies(torch.zeros(3, F, dtype=torch.float64))
    with pytest.raises(ValueError, match="set_policies"):  # not on the batch's device
        b.set_policies(torch.zeros(3, F))
