"""The SAC population learner's host side, without a GPU: initial weights against GpuSAC's, the batched losses against
sac_losses / actor_loss per agent, one full gradient step against per-agent torch steps, the per-agent sampling, the PBT
round, and the argument checks of TennisBatch.set_sac_actors."""
import re
from pathlib import Path

import numpy as np
import pytest
import torch

from tennisbot_rl_b200 import _lib
from tennisbot_rl_b200.batch import TennisBatch
from tennisbot_rl_b200.population import BatchedAdam
from tennisbot_rl_b200.sac import SacActor, TwinCritic, actor_loss, pack_sac_actor, sac_losses
from tennisbot_rl_b200.sac_population import (PBT_PERTURBED, BatchedSacActor, BatchedTwinCritic, PopulationSAC,
                                              batched_actor_loss, batched_sac_losses, initial_agents)

DIMS = ((6, 6), (12, 2))
SEEDS = (3, 11, 5)
ROOT = Path(__file__).resolve().parents[1]


def _gpusac_init(od, ad, seed):
    """GpuSAC.__init__'s draws, restated without a device: manual_seed, actor, critic, target loaded from the critic."""
    torch.manual_seed(seed)
    actor, critic, target = SacActor(od, ad), TwinCritic(od, ad), TwinCritic(od, ad)
    target.load_state_dict(critic.state_dict())
    return actor, critic, target


def _learner(od, ad, seeds=SEEDS, lr=(3e-4, 1e-3, 5e-5), tau=(0.005, 0.02, 0.1), gamma=(0.99, 0.9, 0.5)):
    """A PopulationSAC's learner state on the CPU (no context, no ring)."""
    L = PopulationSAC.__new__(PopulationSAC)
    L.P, L.dev, L.ad = len(seeds), torch.device("cpu"), ad
    L.hyper = {"lr": torch.tensor(lr), "tau": torch.tensor(tau), "gamma": torch.tensor(gamma)}
    init = initial_agents(od, ad, seeds)
    L.actor = BatchedSacActor([a for a, _, _ in init])
    L.critic = BatchedTwinCritic([c for _, c, _ in init])
    L.critic_target = BatchedTwinCritic([t for _, _, t in init], grad=False)
    L.log_alpha = torch.zeros(L.P, requires_grad=True)
    L.target_entropy = -float(ad)
    L.actor_opt, L.critic_opt, L.alpha_opt = (BatchedAdam(ps, L.hyper["lr"], eps=1e-8) for ps in
                                              (L.actor.params, L.critic.params, [L.log_alpha]))
    L.losses = torch.zeros(3, L.P)
    return L


def _batch(P, B, od, ad, g):
    return (torch.randn(P, B, od, generator=g), torch.rand(P, B, ad, generator=g) * 2 - 1, torch.randn(P, B, generator=g),
            torch.randn(P, B, od, generator=g), (torch.rand(P, B, generator=g) < 0.1).float())


@pytest.mark.parametrize("od,ad", DIMS)
def test_initial_weights_equal_gpusac_per_seed_and_packed_rows_equal_pack_sac_actor(od, ad):
    L = _learner(od, ad)
    for p, s in enumerate(SEEDS):
        actor, critic, target = _gpusac_init(od, ad, s)
        for t, ref in zip(L.actor.params, actor.parameters()):
            assert torch.equal(t[p], ref.detach())
        for t, ref in zip(L.critic.params, critic.parameters()):
            assert torch.equal(t[p], ref.detach())
        for t, ref in zip(L.critic_target.params, target.parameters()):
            assert torch.equal(t[p], ref.detach())
        assert torch.equal(L.actor.packed()[p], pack_sac_actor(actor))
    assert L.actor.packed().shape == (len(SEEDS), _lib.SAC_FLOATS if od == 6 else _lib.SAC_FLOATS_HIT)


@pytest.mark.parametrize("od,ad", DIMS)
def test_batched_losses_equal_sac_losses_per_agent(od, ad):
    L, P, B = _learner(od, ad), len(SEEDS), 64
    g = torch.Generator().manual_seed(0)
    with torch.no_grad():
        L.log_alpha.copy_(torch.tensor([0.0, -1.0, 0.5]))
    batch, noise, next_noise = _batch(P, B, od, ad, g), torch.randn(P, B, ad, generator=g), torch.randn(P, B, ad, generator=g)
    a, c, pi, logp, alpha = batched_sac_losses(L.actor, L.critic, L.critic_target, L.log_alpha, batch, L.hyper["gamma"],
                                               L.target_entropy, noise, next_noise)
    pl = batched_actor_loss(L.critic, batch[0], pi, logp, alpha)
    for p, s in enumerate(SEEDS):
        actor, critic, target = _gpusac_init(od, ad, s)
        la = L.log_alpha.detach()[p:p + 1].clone().requires_grad_()
        ra, rc, rpi, rlogp, ralpha = sac_losses(actor, critic, target, la, tuple(x[p] for x in batch), float(L.hyper["gamma"][p]),
                                                -float(ad), noise[p], next_noise[p])
        rpl = actor_loss(critic, batch[0][p], rpi, rlogp, ralpha)
        for got, ref in ((a[p], ra), (c[p], rc), (pl[p], rpl)):
            torch.testing.assert_close(got, ref.reshape(()), rtol=1e-5, atol=1e-6)


# float32 tolerance of one step: the batched matmuls and per-agent means sum in another order than the per-agent torch ops,
# and Adam's first step moves each weight by about lr whatever the gradient's size, so a last-bit difference in a
# near-zero gradient can flip it; 1e-6 absolute is far below every lr used (5e-5 .. 1e-3)
STEP_ATOL = 1e-6


def test_gradient_step_equals_independent_torch_steps():
    od, ad, P, B = 6, 6, len(SEEDS), 128
    L = _learner(od, ad)
    refs = []
    for p, s in enumerate(SEEDS):
        actor, critic, target = _gpusac_init(od, ad, s)
        la = torch.zeros(1, requires_grad=True)
        lr = float(L.hyper["lr"][p])
        opts = [torch.optim.Adam(ps, lr=lr) for ps in (actor.parameters(), critic.parameters(), [la])]
        refs.append((actor, critic, target, la, opts))
    g = torch.Generator().manual_seed(4)
    for _ in range(3):
        batch, noise, next_noise = _batch(P, B, od, ad, g), torch.randn(P, B, ad, generator=g), torch.randn(P, B, ad, generator=g)
        L.gradient_step(batch, noise, next_noise)
        for p, (actor, critic, target, la, (a_opt, c_opt, al_opt)) in enumerate(refs):  # GpuSAC._grad_step
            a_loss, c_loss, pi, logp, alpha = sac_losses(actor, critic, target, la, tuple(x[p] for x in batch),
                                                         float(L.hyper["gamma"][p]), -float(ad), noise[p], next_noise[p])
            al_opt.zero_grad()
            a_loss.backward()
            al_opt.step()
            c_opt.zero_grad()
            c_loss.backward()
            c_opt.step()
            pi_loss = actor_loss(critic, batch[0][p], pi, logp, alpha)
            a_opt.zero_grad()
            pi_loss.backward()
            a_opt.step()
            with torch.no_grad():
                for q, tq in zip(critic.parameters(), target.parameters()):
                    tq.lerp_(q, float(L.hyper["tau"][p]))
    for p, (actor, critic, target, la, _) in enumerate(refs):
        for mine, ref in ((L.actor, actor), (L.critic, critic), (L.critic_target, target)):
            for t, r in zip(mine.params, ref.parameters()):
                torch.testing.assert_close(t[p].detach(), r.detach(), atol=STEP_ATOL, rtol=0)
        torch.testing.assert_close(L.log_alpha[p].detach(), la[0].detach(), atol=STEP_ATOL, rtol=0)
    assert L.actor_opt.steps.tolist() == [3.0] * P


def test_sampled_rows_stay_in_the_agents_columns_and_filled_slots():
    L = PopulationSAC.__new__(PopulationSAC)
    L.P, L.n, L.B, L.dev = 3, 256, 4096, torch.device("cpu")
    L.N, filled = 3 * 256, 5
    L.fill = torch.tensor([float(filled * L.n)])
    torch.manual_seed(0)
    idx = L.sample()
    assert idx.shape == (L.P, L.B)
    slot, col = idx // L.N, idx % L.N
    for p in range(L.P):
        assert bool(((col[p] >= p * L.n) & (col[p] < (p + 1) * L.n)).all())
        assert set(slot[p].tolist()) == set(range(filled))  # every filled slot is drawn, and nothing else
    assert len(set(col[0].tolist())) == L.n


def test_pbt_round_copies_every_row_and_perturbs_lr_and_tau():
    P = 8
    L = _learner(6, 6, seeds=range(P), lr=[3e-4] * P, tau=[0.005] * P, gamma=[0.99] * P)
    L.pbt_rng, L.pbt_log, L.iters, L._interval = np.random.default_rng(7), [], 12, np.zeros((2, P))
    g = torch.Generator().manual_seed(3)
    with torch.no_grad():
        for t in L._state():
            t.copy_(torch.rand(t.shape, generator=g, dtype=t.dtype))
        for v in L.hyper.values():
            v.copy_(torch.rand(P, generator=g))
    rows = L._state()
    before, hyper0 = [t.detach().clone() for t in rows], {k: v.clone() for k, v in L.hyper.items()}
    assert len(rows) == 8 + 12 + 12 + 1 + (2 * 8 + 1) + (2 * 12 + 1) + (2 * 1 + 1)  # weights, log_alpha, Adam m, v, steps
    scores = [5.0, None, 1.0, 7.0, -2.0, 3.0, 6.0, 0.5]
    events = L.exploit_explore(scores)
    assert sorted(e[1] for e in events) == [1, 4] and all(e[2] in (3, 6) for e in events) and all(e[0] == 12 for e in events)
    for _, dst, src, hp in events:
        for t, t0 in zip(rows, before):
            assert torch.equal(t[dst], t0[src])
        for k, v in L.hyper.items():
            if k in PBT_PERTURBED:
                assert any(torch.equal(v[dst], hyper0[k][src] * f) for f in (0.8, 1.2))
            else:
                assert torch.equal(v[dst], hyper0[k][src])
            assert hp[k] == float(v[dst])
    assert PBT_PERTURBED == ("lr", "tau")
    for p in set(range(P)) - {1, 4}:
        for t, t0 in zip(rows, before):
            assert torch.equal(t[p], t0[p])
    assert L.actor_opt.lr is L.hyper["lr"] and L.critic_opt.lr is L.hyper["lr"]  # the Adams read the perturbed lr


def test_set_sac_actors_argument_checks():
    b = TennisBatch.__new__(TennisBatch)  # only the checks that run before the library is called
    b.kind, b.num_envs, b.device, b.obs_dim, b.act_dim = _lib.ENV_SWING, 768, torch.device("cuda", 0), 6, 6
    F = _lib.SAC_FLOATS
    for bad in (torch.zeros(F), torch.zeros(5, F), torch.zeros(0, F), torch.zeros(3, F + 4)):
        with pytest.raises(ValueError, match="set_sac_actors"):
            b.set_sac_actors(bad)
    with pytest.raises(ValueError, match="multiple of 128"):  # 768 / 4 = 192 envs per agent
        b.set_sac_actors(torch.zeros(4, F))
    with pytest.raises(ValueError, match="set_sac_actors"):
        b.set_sac_actors(torch.zeros(3, F, dtype=torch.float64))
    with pytest.raises(ValueError, match="set_sac_actors"):  # not on the batch's device
        b.set_sac_actors(torch.zeros(3, F))
    with pytest.raises(ValueError, match="multiple of 128"):
        PopulationSAC("SwingRacket-v0", 2, 192)
    with pytest.raises(ValueError, match="one per agent"):
        PopulationSAC("SwingRacket-v0", 3, 128, tau=[0.1, 0.2])


def test_header_declares_tb_set_sac_actors_as_the_binding_does():
    h = (ROOT / "include" / "tennisbot_b200.h").read_text()
    m = re.search(r"int tb_set_sac_actors\(([^)]*)\);", h)
    assert m is not None
    assert [a.strip() for a in m.group(1).split(",")] == \
        ["tb_ctx *ctx", "const float *d_params", "int64_t agents", "int64_t count", "void *stream"]
    assert len(_lib.SIGNATURES["tb_set_sac_actors"]) == 5
    assert "tb_set_sac_actors" in _lib.EXPORTS
    assert re.search(r"#define TB_SAC_FLOATS (\d+)", h).group(1) == str(_lib.SAC_FLOATS)
    assert re.search(r"#define TB_SAC_FLOATS_HIT (\d+)", h).group(1) == str(_lib.SAC_FLOATS_HIT)
