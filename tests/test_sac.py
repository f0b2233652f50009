"""CPU checks of the SAC actor layout and learner: header constants, pack_sac_actor's order, SacActor.log_prob and the losses of
one gradient step, each against a numpy restatement; the SAC entry points' argument rejections that need no device."""
import ctypes as C
import math
import re
from pathlib import Path

import numpy as np
import pytest
import torch

ROOT = Path(__file__).resolve().parent.parent
DIMS = {"SwingRacket-v0": (0, 6, 6), "Tennisbot-v0": (1, 12, 2)}


def _pad4(x):
    return (x + 3) // 4 * 4


def test_header_constants_equal_the_layout_sizes():
    from tennisbot_rl_b200 import _lib, build

    header = (ROOT / "include" / "tennisbot_b200.h").read_text()
    const = lambda name: int(re.search(rf"#define {name} (\d+)", header).group(1))  # noqa: E731
    build.build_library()
    L = _lib.load()
    for kind, od, ad in DIMS.values():
        want = 256 * od + 256 + 256 * 256 + 256 + 2 * (256 * ad + _pad4(ad))
        name = "TB_SAC_FLOATS" if kind == 0 else "TB_SAC_FLOATS_HIT"
        assert const(name) == want == L.tb_sac_floats(kind) == (_lib.SAC_FLOATS if kind == 0 else _lib.SAC_FLOATS_HIT)
    assert L.tb_sac_floats(7) == -1
    assert const("TB_SAC_HIDDEN") == _lib.SAC_HIDDEN == 256
    assert (const("TB_SAC_SAMPLE"), const("TB_SAC_MEAN"), const("TB_SAC_UNIFORM")) == (_lib.SAC_SAMPLE, _lib.SAC_MEAN, _lib.SAC_UNIFORM)


@pytest.mark.parametrize("env_id", list(DIMS))
def test_pack_follows_the_sb3_state_dict_order(env_id):
    from tennisbot_rl_b200.sac import SacActor, pack_sac_actor

    _, od, ad = DIMS[env_id]
    torch.manual_seed(1)
    actor = SacActor(od, ad)
    # a synthetic SB3 SAC policy state dict: actor entries (in SB3's order) among critic and target entries
    sb3 = {"critic.qf0.0.weight": torch.ones(3, 3)}
    sb3.update({"actor." + k: v.clone() for k, v in actor.state_dict().items()})
    sb3["critic_target.qf0.0.weight"] = torch.ones(3, 3)
    assert list(actor.state_dict()) == ["latent_pi.0.weight", "latent_pi.0.bias", "latent_pi.2.weight", "latent_pi.2.bias",
                                        "mu.weight", "mu.bias", "log_std.weight", "log_std.bias"]
    v = pack_sac_actor(sb3)
    assert torch.equal(v, pack_sac_actor(actor)) and torch.equal(v, pack_sac_actor(actor.state_dict()))
    parts, at = [], 0
    for key, t in actor.state_dict().items():
        parts.append((key, at))
        flat = t.detach().reshape(-1).numpy()
        np.testing.assert_array_equal(v[at:at + flat.size].numpy(), flat)
        np.testing.assert_array_equal(v[at + flat.size:at + _pad4(flat.size)].numpy(), 0)
        at += _pad4(flat.size)
    assert at == v.numel()
    with pytest.raises(KeyError):
        pack_sac_actor({"actor.mu.weight": torch.zeros(ad, 256)})
    with pytest.raises(ValueError):
        pack_sac_actor(SacActor(5, 3))


def test_log_prob_is_sb3s_squashed_gaussian():
    from tennisbot_rl_b200.sac import SacActor

    rng = np.random.default_rng(2)
    mu, ls, u = rng.normal(0, 1, (64, 6)), rng.uniform(-3, 1, (64, 6)), rng.normal(0, 2, (64, 6))
    got = SacActor.log_prob(*(torch.from_numpy(x) for x in (mu, ls, u))).numpy()
    ref = (-0.5 * ((u - mu) / np.exp(ls)) ** 2 - ls - 0.5 * np.log(2 * np.pi)).sum(-1) - np.log(1 - np.tanh(u) ** 2 + 1e-6).sum(-1)
    np.testing.assert_allclose(got, ref, rtol=1e-12, atol=1e-12)


def _np_mlp(layers, x):
    for i, (W, b) in enumerate(layers):
        x = x @ W.T + b
        if i < len(layers) - 1:
            x = np.maximum(x, 0.0)
    return x


def test_losses_of_one_gradient_step_match_numpy():
    from tennisbot_rl_b200.sac import SacActor, TwinCritic, actor_loss, sac_losses

    torch.manual_seed(4)
    od, ad, B, gamma = 6, 6, 16, 0.99
    actor, critic, target = SacActor(od, ad).double(), TwinCritic(od, ad).double(), TwinCritic(od, ad).double()
    log_alpha = torch.tensor([0.3], dtype=torch.float64, requires_grad=True)
    rng = np.random.default_rng(5)
    obs, nxt = rng.normal(0, 1, (B, od)), rng.normal(0, 1, (B, od))
    act, rew = rng.uniform(-1, 1, (B, ad)), rng.normal(0, 1, B)
    done = (rng.uniform(0, 1, B) < 0.3).astype(np.float64)
    noise, next_noise = rng.normal(0, 1, (B, ad)), rng.normal(0, 1, (B, ad))
    T = torch.from_numpy
    a_loss, c_loss, pi, logp, alpha = sac_losses(actor, critic, target, log_alpha, (T(obs), T(act), T(rew), T(nxt), T(done)), gamma,
                                                 -float(ad), T(noise), T(next_noise))
    p_loss = actor_loss(critic, T(obs), pi, logp, alpha)

    lin = lambda seq: [(m.weight.detach().numpy(), m.bias.detach().numpy()) for m in seq if isinstance(m, torch.nn.Linear)]  # noqa: E731
    lat = lin(actor.latent_pi)

    def dist(x):
        h = _np_mlp(lat + [(np.eye(256), np.zeros(256))], x)
        h = np.maximum(h, 0.0)
        m = h @ actor.mu.weight.detach().numpy().T + actor.mu.bias.detach().numpy()
        s = np.clip(h @ actor.log_std.weight.detach().numpy().T + actor.log_std.bias.detach().numpy(), -20, 2)
        return m, s

    def logprob(m, s, u):
        return (-0.5 * ((u - m) / np.exp(s)) ** 2 - s - 0.5 * math.log(2 * math.pi)).sum(-1) - np.log(1 - np.tanh(u) ** 2 + 1e-6).sum(-1)

    def q(c, x, a):
        z = np.concatenate([x, a], -1)
        return _np_mlp(lin(c.qf0), z)[:, 0], _np_mlp(lin(c.qf1), z)[:, 0]

    al = math.exp(0.3)
    m, s = dist(obs)
    u = m + np.exp(s) * noise
    lp = logprob(m, s, u)
    nm, ns = dist(nxt)
    nu = nm + np.exp(ns) * next_noise
    tq = rew + (1 - done) * gamma * (np.minimum(*q(target, nxt, np.tanh(nu))) - al * logprob(nm, ns, nu))
    q0, q1 = q(critic, obs, act)
    np.testing.assert_allclose(a_loss.item(), -(0.3 * (lp - ad)).mean(), rtol=1e-10)
    np.testing.assert_allclose(c_loss.item(), 0.5 * (((q0 - tq) ** 2).mean() + ((q1 - tq) ** 2).mean()), rtol=1e-10)
    np.testing.assert_allclose(p_loss.item(), (al * lp - np.minimum(*q(critic, obs, np.tanh(u)))).mean(), rtol=1e-10)
    np.testing.assert_allclose(float(alpha), al, rtol=1e-12)


def test_sac_entry_points_reject_arguments_without_a_device():
    from tennisbot_rl_b200 import _lib, build

    build.build_library()
    L = _lib.load()
    fake = C.c_void_p(16)  # never dereferenced: every call below fails on its arguments first

    def err(rc):
        assert rc != 0
        return L.tb_last_error().decode()

    ring = _lib.TbSacRing(C.sizeof(_lib.TbSacRing), 0, 4, 16, 16, 16, 16, 16)
    assert "k_steps must be >= 1" in err(L.tb_sac_rollout(fake, 0, 0, 0, C.byref(ring), None, None))
    assert "unknown mode" in err(L.tb_sac_rollout(fake, 1, 5, 0, C.byref(ring), None, None))
    ring.slots = 0
    assert "slots must be >= 1" in err(L.tb_sac_rollout(fake, 1, 0, 0, C.byref(ring), None, None))
    ring.slots, ring.done = 4, None
    assert "every ring array" in err(L.tb_sac_rollout(fake, 1, 0, 0, C.byref(ring), None, None))
    assert "context is NULL" in err(L.tb_sac_rollout(None, 1, 0, 0, None, None, None))
    assert "context is NULL" in err(L.tb_sac_begin(None, None))
    assert "context is NULL" in err(L.tb_set_sac_actor(None, fake, _lib.SAC_FLOATS, None))
