"""GPU parity tests: CUDA path (through the C ABI) vs the CPU oracle on identical seeded inputs.

Bars (north star): contact / hit events and done flags exact; poses and rewards within a float tolerance.
  f64 path: every event and done flag identical over the whole horizon; state within 1e-9, float32 outputs 2e-6.
  f32 path: identical except for near-threshold flips, i.e. discrete mismatches where the oracle's own margin
            |quantity - threshold| is below BAND_F32; envs that flipped are dropped from then on and counted.
"""
import numpy as np
import pytest
import torch

from tests.harness import reference_reset_params, run_parity

pytestmark = pytest.mark.gpu

TOL_F64_STATE = 5e-8   # absolute, on a state record whose spin entries reach ~50 rad/s after a bounce
TOL_F64_OUT = 2e-6      # float32 rounding of the outputs at |x| <= 20
BAND_F32 = 2e-4         # metres: fp32 position drift over an 800-substep flight stays below this
TOL_F32_OUT = 2e-3


def _make(env, n, precision, seed, oracle_lib):
    from tennisbot_rl_b200.batch import TennisBatch

    b = TennisBatch(env, n, device=0, seed=seed, precision=precision)
    o = oracle_lib.OracleEnv(env, n, seed=seed, threads=8)
    return b, o


@pytest.mark.parametrize("env,steps", [("SwingRacket-v0", 80), ("Tennisbot-v0", 1200)])
def test_f64_parity_random_actions(oracle_lib, env, steps):
    """config 2 shape: 4096 envs, random actions, explicit initial states, horizon > 3 episodes (swing) /
    beyond the 1000-step time-out (hit); crosses in-kernel auto-resets (Philox placement parity)."""
    n = 4096
    b, o = _make(env, n, "f64", 11, oracle_lib)
    rng = np.random.default_rng(5)
    init = reference_reset_params(o.kind, n, rng)
    g0 = b.reset(init=init).cpu().numpy()
    o0 = o.reset(init=init)
    np.testing.assert_array_equal(g0, o0)
    rep, valid = run_parity(b, o, steps, lambda t, _obs: rng.uniform(-1, 1, (n, o.act_dim)), band=0.0, check_state_every=20)
    print(rep)
    assert rep.event_mismatch_hard == 0 and rep.event_mismatch_near == 0
    assert rep.max_state_err < TOL_F64_STATE
    assert rep.max_obs_err < TOL_F64_OUT and rep.max_reward_err < TOL_F64_OUT
    np.testing.assert_array_equal(b.read_stats(), o.read_stats())


def test_f64_parity_trained_policy(oracle_lib):
    """Saved PPO policy (tests/golden/ppo_swing_policy.npz): ~100 % of episodes hit the ball, exercising the
    racket-ball contact solve and deep-penetration path that random actions rarely reach."""
    from pathlib import Path

    n = 2048
    w = np.load(Path(__file__).parent / "golden" / "ppo_swing_policy.npz")
    b, o = _make("SwingRacket-v0", n, "f64", 3, oracle_lib)
    rng = np.random.default_rng(9)
    obs0 = o.reset()
    np.testing.assert_array_equal(b.reset().cpu().numpy(), obs0)
    std = np.exp(w["log_std"])

    def policy(t, obs):
        h = obs
        for l in (0, 2, 4):
            h = np.tanh(h @ w[f"mlp_extractor__policy_net__{l}__weight"].T + w[f"mlp_extractor__policy_net__{l}__bias"])
        mean = h @ w["action_net__weight"].T + w["action_net__bias"]
        return np.clip(mean + std * rng.standard_normal((n, 6)), -1, 1)

    rep, valid = run_parity(b, o, 52, policy, band=0.0, check_state_every=13, obs0=obs0)
    print(rep)
    assert rep.event_mismatch_hard == 0 and rep.event_mismatch_near == 0
    assert rep.max_state_err < TOL_F64_STATE and rep.max_obs_err < TOL_F64_OUT and rep.max_reward_err < TOL_F64_OUT
    st = b.read_stats()
    np.testing.assert_array_equal(st, o.read_stats())
    assert st[2] > 0.8 * st[0]  # racket hits in most episodes


@pytest.mark.parametrize("params", [{"racket_scale": 2.5}, {"gravity_z": -3.0, "racket_scale": 1.6},
                                    {"lin_damping": 0.0, "ang_damping": 0.0}])
def test_f64_parity_fast_forward_paths(oracle_lib, params):
    """Scenes that push many flights through every path of ff_kernel: a larger racket (contacts and near misses in
    the fast-forward: server warps, repeated visits, flights finished by the servers), weak gravity (long flights,
    800-step time-outs), no damping (balls leave the court: floor-edge contacts, time-outs).  Same bars as the
    random-action test; the diagnostics must show that the generic full-substep path was actually used."""
    n = 4096
    b, o = _make("SwingRacket-v0", n, "f64", 17, oracle_lib)
    for k, v in params.items():
        b.set_param(k, v)
        o.set_param(k, v)
    np.testing.assert_array_equal(b.reset().cpu().numpy(), o.reset())
    rng = np.random.default_rng(12)
    rep, valid = run_parity(b, o, 52, lambda t, _obs: rng.uniform(-1, 1, (n, 6)), band=0.0, check_state_every=13)
    print(rep, b.ff_diagnostics()[:3])
    assert rep.event_mismatch_hard == 0 and rep.event_mismatch_near == 0
    assert rep.max_state_err < TOL_F64_STATE and rep.max_obs_err < TOL_F64_OUT and rep.max_reward_err < TOL_F64_OUT
    np.testing.assert_array_equal(b.read_stats(), o.read_stats())
    d = b.ff_diagnostics()
    assert d[15] == 0 and d[1] > 0  # no queue time-out; envs went through the server path in the last fast-forward


@pytest.mark.parametrize("params", [{}, {"racket_scale": 2.5}, {"gravity_z": -3.0, "racket_scale": 1.6}])
def test_f64_fast_forward_final_state(oracle_lib, params):
    """Without auto-reset the state a fast-forward ends with stays in place: compare the whole record (racket pose and
    spin after up to 775 substeps in ff_kernel's body-frame formulation, ball velocity and spin after the landing
    impulse) with the oracle's, and the done flag of the record."""
    from tennisbot_rl_b200.batch import TennisBatch

    n = 4096
    b = TennisBatch("SwingRacket-v0", n, device=0, seed=23, precision="f64", auto_reset=False)
    o = oracle_lib.OracleEnv("SwingRacket-v0", n, seed=23, threads=8, auto_reset=False)
    for k, v in params.items():
        b.set_param(k, v)
        o.set_param(k, v)
    np.testing.assert_array_equal(b.reset().cpu().numpy(), o.reset())
    rng = np.random.default_rng(31)
    rep, valid = run_parity(b, o, 26, lambda t, _obs: rng.uniform(-1, 1, (n, 6)), band=0.0, check_state_every=26)
    print(rep)
    assert rep.event_mismatch_hard == 0 and rep.max_obs_err < TOL_F64_OUT and rep.max_reward_err < TOL_F64_OUT
    gs, os_ = b.get_state().cpu().numpy(), o.get_state()
    assert (gs[:, 30] == 1).all() and (os_[:, 30] == 1).all()  # every episode is over after 26 steps
    assert np.abs(gs - os_).max() < TOL_F64_STATE


def test_f64_parity_hit_env_tracking_policy(oracle_lib):
    """Config 3 shape (incoming-ball env *with racket-ball contact*): random actions almost never meet the ball, so the
    racket is steered towards the ball's y (a scripted policy on the oracle's observation).  A few hundred episodes then
    contain racket-ball contact steps (asserted), which exercises the dynamic two-body solve and the hit rewards
    (tennisbot_env.py:170-180)."""
    n = 4096
    b, o = _make("Tennisbot-v0", n, "f64", 31, oracle_lib)
    obs0 = o.reset()
    np.testing.assert_array_equal(b.reset().cpu().numpy(), obs0)
    rng = np.random.default_rng(2)

    def policy(t, obs):
        a = np.zeros((n, 2))
        a[:, 0] = rng.uniform(-0.2, 0.2, n)
        a[:, 1] = np.clip(4.0 * (obs[:, 7] - obs[:, 1]) - 1.5 * obs[:, 4], -1, 1)  # PD on ball y - racket y
        return a

    rep, valid = run_parity(b, o, 900, policy, band=0.0, check_state_every=50, obs0=obs0)
    print(rep, b.read_stats().tolist())
    assert rep.event_mismatch_hard == 0 and rep.event_mismatch_near == 0
    assert rep.max_state_err < TOL_F64_STATE and rep.max_obs_err < TOL_F64_OUT and rep.max_reward_err < TOL_F64_OUT
    st = b.read_stats()
    np.testing.assert_array_equal(st, o.read_stats())
    assert st[0] > 0 and st[2] > 0.05 * st[0]  # several times the hit rate of random actions (the racket cannot choose its height)


@pytest.mark.parametrize("params,tol_state,tol_out", [
    ({"racket_scale": 2.5}, TOL_F64_STATE, TOL_F64_OUT),
    ({"lin_damping": 0.0, "ang_damping": 0.0}, TOL_F64_STATE, TOL_F64_OUT),
    # balls come to rest and roll on the court here: hundreds of consecutive contact steps, each turning position
    # rounding into velocity at 1/dt = 240.  Measured 3.2e-6 (3.8e-6 with the generic step in line instead of hit_fast):
    # the amplification is the contact model's, not the straight line's, hence the wider bar for this scene only
    ({"gravity_z": -25.0, "racket_scale": 1.6}, 2e-5, 2e-5)])
def test_f64_parity_hit_env_paths(oracle_lib, params, tol_state, tol_out):
    """Scenes that push Tennisbot-v0 through every branch of its substep (hit_fast / the generic step out of line): a
    larger racket steered at the ball (many contacts, then a spinning racket on the straight line for the rest of the
    episode), no damping (fast balls: net and floor-edge contacts, balls leaving the court), strong gravity (many
    bounces per episode on the closed-form floor contact).  Same bars as the random-action test."""
    n = 4096
    b, o = _make("Tennisbot-v0", n, "f64", 37, oracle_lib)
    for k, v in params.items():
        b.set_param(k, v)
        o.set_param(k, v)
    obs0 = o.reset()
    np.testing.assert_array_equal(b.reset().cpu().numpy(), obs0)
    rng = np.random.default_rng(3)

    def policy(t, obs):
        a = np.zeros((n, 2))
        a[:, 0] = rng.uniform(-0.5, 0.5, n)
        a[:, 1] = np.clip(4.0 * (obs[:, 7] - obs[:, 1]) - 1.5 * obs[:, 4], -1, 1)
        return a

    rep, valid = run_parity(b, o, 700, policy, band=0.0, check_state_every=50, obs0=obs0)
    st = b.read_stats()
    print(rep, st.tolist())
    assert rep.event_mismatch_hard == 0 and rep.event_mismatch_near == 0
    assert rep.max_state_err < tol_state and rep.max_obs_err < tol_out and rep.max_reward_err < tol_out
    np.testing.assert_array_equal(st, o.read_stats())
    assert st[0] > 0


@pytest.mark.parametrize("env,steps", [("SwingRacket-v0", 52), ("Tennisbot-v0", 700)])
def test_f32_parity_with_band(oracle_lib, env, steps):
    """float32 path: every contact / done decision equals the oracle's unless the oracle's own margin to the
    threshold is inside BAND_F32; poses and rewards within TOL_F32_OUT.  TB_EV_RACKET_LOW (a diagnostic, no env
    logic depends on it) is not compared.  Tennisbot-v0 envs leave the per-step comparison at their first impact
    (racket or floor, see harness.run_parity); past that point the float32 path is checked statistically."""
    n = 4096
    b, o = _make(env, n, "f32", 21, oracle_lib)
    rng = np.random.default_rng(6)
    init = reference_reset_params(o.kind, n, rng)
    b.reset(init=init)
    o.reset(init=init)
    hit = env == "Tennisbot-v0"
    rep, valid = run_parity(b, o, steps, lambda t, _obs: rng.uniform(-1, 1, (n, o.act_dim)), band=BAND_F32,
                            event_mask=0xff & ~oracle_lib.EV_RACKET_LOW,
                            drop_after={oracle_lib.EV_RACKET_BALL: 0, oracle_lib.EV_COURT_BALL: 0} if hit else None)
    print(rep)
    assert rep.event_mismatch_hard == 0
    assert rep.compared > 0.3 * n * steps
    assert rep.max_obs_err < TOL_F32_OUT and rep.max_reward_err < 10 * TOL_F32_OUT
    # whole-horizon statistics of the two paths (episodes, lengths, contact counts) agree closely
    gs, os_ = b.read_stats().astype(np.float64), o.read_stats().astype(np.float64)
    assert gs[9] == os_[9] and gs[8] == os_[8] or not hit  # same env / physics step counts in the hit env
    for k in (0, 1, 2, 4):
        assert abs(gs[k] - os_[k]) <= 0.02 * max(os_[k], 50.0), (k, gs, os_)


@pytest.mark.parametrize("env", ["SwingRacket-v0", "Tennisbot-v0"])
def test_fused_rollout_matches_stepwise(oracle_lib, env):
    """tb_rollout (K fused env steps, in-kernel Philox actions) == oracle rollout with the same streams."""
    n = 2048
    b, o = _make(env, n, "f64", 77, oracle_lib)
    b.reset()
    o.reset()
    k = 60 if env == "SwingRacket-v0" else 300
    gobs, grs, gdc = (x.cpu().numpy() for x in b.rollout(k))
    r = o.rollout(k)
    np.testing.assert_array_equal(gdc, r["done_count"])
    assert np.abs(gobs.astype(np.float64) - r["obs"]).max() < TOL_F64_OUT
    assert np.abs(grs - r["reward_sum"]).max() < 1e-3
    np.testing.assert_array_equal(b.read_stats(), o.read_stats())
    assert np.abs(b.get_state().cpu().numpy() - o.get_state()).max() < TOL_F64_STATE


@pytest.mark.parametrize("env", ["SwingRacket-v0", "Tennisbot-v0"])
def test_pid_control_mode_parity(oracle_lib, env):
    """A9 (TB_CONTROL_PID): actions are target positions, three in-kernel simple_pid controllers; f64 parity with the
    oracle over a horizon that crosses auto-resets (controller memory is cleared by reset)."""
    n = 1024
    b, o = _make(env, n, "f64", 5, oracle_lib)
    b.set_control_mode("pid")
    o.set_control_mode("pid")
    np.testing.assert_array_equal(b.reset().cpu().numpy(), o.reset())
    rng = np.random.default_rng(3)
    lo, hi = (np.array([5, -4, 0.5, 0, 0, 0]), np.array([12, 4, 2.0, 0, 0, 0])) if o.act_dim == 6 else (np.array([7, -5]), np.array([13, 5]))
    steps = 60 if env == "SwingRacket-v0" else 700
    rep, valid = run_parity(b, o, steps, lambda t, _obs: rng.uniform(lo, hi, (n, o.act_dim)), band=0.0, check_state_every=15)
    print(rep)
    assert rep.event_mismatch_hard == 0 and rep.event_mismatch_near == 0
    assert rep.max_state_err < TOL_F64_STATE and rep.max_obs_err < TOL_F64_OUT
    np.testing.assert_array_equal(b.read_stats(), o.read_stats())


@pytest.mark.parametrize("n", [1, 31, 33, 127, 129, 1000])
@pytest.mark.parametrize("env", ["SwingRacket-v0", "Tennisbot-v0"])
def test_ragged_batch_sizes(oracle_lib, env, n):
    """Batch sizes that do not fill a warp / a CTA / the staging tiles: same bars as the full-size f64 test, through
    both the device-pointer entry point and the host-buffer one (zero-copy tiles with partial rows)."""
    b, o = _make(env, n, "f64", 2, oracle_lib)
    np.testing.assert_array_equal(b.reset().cpu().numpy(), o.reset())
    rng = np.random.default_rng(n)
    steps = 30 if env == "SwingRacket-v0" else 40
    rep, valid = run_parity(b, o, steps, lambda t, _obs: rng.uniform(-1, 1, (n, o.act_dim)), band=0.0, check_state_every=10)
    assert rep.event_mismatch_hard == 0 and rep.max_state_err < TOL_F64_STATE and rep.max_obs_err < TOL_F64_OUT
    for t in range(30):  # host-buffer path, crossing the swing env's fast-forward step again
        a = rng.uniform(-1, 1, (n, o.act_dim)).astype(np.float32)
        hb = b.step_host(a)
        ref = o.step(a)
        np.testing.assert_array_equal(hb["done"], ref["done"])
        np.testing.assert_array_equal(hb["events"], ref["events"])
        np.testing.assert_allclose(hb["obs"], ref["obs"], atol=TOL_F64_OUT)
        np.testing.assert_allclose(hb["reward"], ref["reward"], atol=TOL_F64_OUT)
        d = ref["done"] != 0
        np.testing.assert_allclose(hb["terminal_obs"][d], ref["terminal_obs"][d], atol=TOL_F64_OUT)
    np.testing.assert_array_equal(b.read_stats(), o.read_stats())


def test_host_staging_fallback_matches(oracle_lib):
    """tb_step_host with PAGEABLE numpy buffers takes the staged-copy path; results equal the zero-copy path's."""
    import ctypes as C

    from tennisbot_rl_b200 import _lib

    n = 300
    b, o = _make("SwingRacket-v0", n, "f64", 8, oracle_lib)
    b.reset()
    o.reset()
    rng = np.random.default_rng(4)
    obs, rew, done = np.zeros((n, 6), np.float32), np.zeros(n, np.float32), np.zeros(n, np.uint8)
    vp = C.c_void_p
    for t in range(30):
        a = rng.uniform(-1, 1, (n, 6)).astype(np.float32)
        _lib.check(b.lib.tb_step_host(b.h, a.ctypes.data_as(vp), obs.ctypes.data_as(vp), rew.ctypes.data_as(vp),
                                      done.ctypes.data_as(vp), None, None))
        ref = o.step(a)
        np.testing.assert_array_equal(done, ref["done"])
        np.testing.assert_allclose(obs, ref["obs"], atol=TOL_F64_OUT)
        np.testing.assert_allclose(rew, ref["reward"], atol=TOL_F64_OUT)


@pytest.mark.parametrize("env,n,steps,every,tol_state", [("SwingRacket-v0", 262144, 78, 13, TOL_F64_STATE),
                                                         ("Tennisbot-v0", 65536, 1100, 100, 1e-6)])
def test_f64_parity_at_config_sizes(oracle_lib, env, n, steps, every, tol_state):
    """BASELINE.json's batch sizes against the oracle step by step (config 3: 65 536 incoming-ball envs over whole episodes
    incl. the 1000-step time-out; SwingRacket: 262 144 envs x 3 episodes = 786 k episodes): every event byte and done flag
    identical, statistics identical.  State bar: the 4096-env tests' 5e-8 for SwingRacket (observed 5e-15 on mid-episode
    records); 1e-6 for Tennisbot-v0 - the maximum over 7e7 env steps sits in a ball-spin entry (rad/s, values up to ~50)
    right after a bounce on the closed-form floor contact and has been seen at 2e-7 to 3e-7."""
    b, o = _make(env, n, "f64", 101, oracle_lib)
    o.close() if hasattr(o, "close") else None
    o = oracle_lib.OracleEnv(env, n, seed=101, threads=16)
    rng = np.random.default_rng(77)
    init = reference_reset_params(o.kind, n, rng)
    np.testing.assert_array_equal(b.reset(init=init).cpu().numpy(), o.reset(init=init))
    rep, valid = run_parity(b, o, steps, lambda t, _obs: rng.uniform(-1, 1, (n, o.act_dim)), band=0.0, check_state_every=every)
    print(env, n, steps, rep)
    assert rep.event_mismatch_hard == 0 and rep.event_mismatch_near == 0 and rep.dropped == 0
    assert rep.max_state_err < tol_state and rep.max_obs_err < TOL_F64_OUT and rep.max_reward_err < TOL_F64_OUT
    np.testing.assert_array_equal(b.read_stats(), o.read_stats())


@pytest.mark.parametrize("policy", ["random", "zero"])
def test_f64_parity_racket_court_contact(oracle_lib, policy):
    """A12 with racket_court_contact = 1: the racket's contact with the court's floor box (up to four support corners of the
    hull's bounding box, PGS rows together with the ball's contacts) on the generic path.  With zero actions every racket
    drops onto the court during the fast-forward (SURVEY 7: handle tip on the floor at physics step 118, ball lands at 133);
    with random actions about two thirds do.  Nothing is masked: every event byte incl. TB_EV_RACKET_LOW, done flag, reward
    and step count must agree for every env, and so must the whole final state record (racket pose and velocities after its
    bounces on the court included) - to 1e-6 for episodes of up to 300 physics steps (observed: 6e-14 with zero actions,
    median 2e-14 with random ones).  A racket that lies on the court while the ball has come to rest ON it tumbles for the
    775 substeps up to the time-out; such chaotic contact sequences amplify rounding without bound and are only counted
    (a handful in 4096 envs)."""
    from tennisbot_rl_b200.batch import TennisBatch

    n = 4096
    b = TennisBatch("SwingRacket-v0", n, device=0, seed=19, precision="f64", auto_reset=False)
    o = oracle_lib.OracleEnv("SwingRacket-v0", n, seed=19, threads=8, auto_reset=False)
    b.set_param("racket_court_contact", 1.0)
    o.set_param("racket_court_contact", 1.0)
    np.testing.assert_array_equal(b.reset().cpu().numpy(), o.reset())
    rng = np.random.default_rng(6)
    act = (lambda t, _obs: rng.uniform(-1, 1, (n, 6))) if policy == "random" else (lambda t, _obs: np.zeros((n, 6)))
    rep, valid = run_parity(b, o, 25, act, band=0.0, check_state_every=5)
    assert rep.event_mismatch_hard == 0 and rep.max_state_err < TOL_F64_STATE and rep.max_obs_err < TOL_F64_OUT
    a = act(25, None).astype(np.float32)
    g_obs, g_rew, g_done, g_term, g_ev = (x.cpu().numpy() for x in b.step(torch.from_numpy(a).cuda()))
    ref = o.step(a)
    np.testing.assert_array_equal(g_done, ref["done"])
    np.testing.assert_array_equal(g_ev, ref["events"])           # TB_EV_RACKET_LOW included
    gs, os_ = b.get_state().cpu().numpy(), o.get_state()
    np.testing.assert_array_equal(gs[:, 29], os_[:, 29])         # every episode ended on the same physics step
    short = os_[:, 29] <= 300
    low = (ref["events"] & 64) != 0
    err = np.abs(gs - os_).max(1)
    print(policy, "racket on the court in %.1f %% of the episodes; state error: max over short episodes %.2e, long episodes %d, of them "
          "beyond 1e-6: %d" % (100 * low.mean(), err[short].max(), (~short).sum(), (err[~short] > 1e-6).sum()))
    assert low.mean() > (0.99 if policy == "zero" else 0.5)
    assert err[short].max() < 1e-6 and short.mean() > 0.98
    np.testing.assert_allclose(g_rew[short], ref["reward"][short], atol=1e-5)
    np.testing.assert_allclose(g_term[short], ref["terminal_obs"][short], atol=1e-5)   # racket x, y compared for every env
    np.testing.assert_allclose(gs[:, 13:16], os_[:, 13:16], atol=1e-5)                  # the ball lands where the oracle's does
    np.testing.assert_array_equal(b.read_stats()[:6], o.read_stats()[:6])


def test_racket_rests_on_the_court_when_contact_is_modelled(oracle_lib):
    """Final states of a no-auto-reset episode with racket_court_contact = 1: no hull corner is below the floor by more than
    the penetration a contact allows, where without the contact most rackets have fallen through."""
    from tennisbot_rl_b200.batch import TennisBatch

    n = 2048
    out = {}
    for mode in (0.0, 1.0):
        b = TennisBatch("SwingRacket-v0", n, seed=5, precision="f64", auto_reset=False)
        b.set_param("racket_court_contact", mode)
        b.reset()
        ev_all = torch.zeros(n, dtype=torch.uint8, device="cuda")
        for t in range(26):
            _, _, _, _, ev = b.step(torch.zeros((n, 6), device="cuda"))
            ev_all |= ev
        out[mode] = (b.get_state().cpu().numpy(), ev_all.cpu().numpy())
        b.close()
    low = (out[1.0][1] & 64) != 0
    assert low.mean() > 0.9                       # zero actions: the racket always reaches the court before the ball lands
    # zero actions: the handle tip meets the court 15 physics steps before the ball lands.  Without the contact the racket keeps
    # falling (COM at 0.249 m when the episode ends), with it the tip is held up and the racket starts to topple (COM 0.314 m)
    assert (out[1.0][0][low, 2] > out[0.0][0][low, 2] + 0.03).all()
    assert out[1.0][0][low, 9].mean() > out[0.0][0][low, 9].mean() + 1.0   # ... its COM no longer falls at free-fall speed
