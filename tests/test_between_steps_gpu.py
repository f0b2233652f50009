"""GPU tests of what happens to the CUDA path's per-env shortcuts when envs do not run in lock step, or when their state is
changed between two steps.

step_kernel skips loads and stores per env under conditions that one entry point establishes and another must undo
(tb_device.cuh, kStDerived / kStSpin / kStPristine): the goal of an RNG-placed episode is re-derived instead of loaded, the ball
spin's y/z half is loaded only when non-zero, and a ball that has only fallen from rest takes its velocity from the
`ball_vz` table.  Each shortcut is valid for a state produced by one entry point only.  The tests here reach the same state
through other entry points - masked resets, explicit placements, injected state records, parameter changes mid-episode,
stepping past `done` - and with envs in different phases of their episodes, so that one launch mixes control steps,
fast-forward entrants and deferred envs.  They compare against the oracle at the float64 bars of test_parity_gpu.py, or,
where no tolerance would be tight enough, against a twin context stepped without the operation, bit for bit.

Every test also checks that its workload is the one it claims (phases, mixed tiles, spin share, done counts) and prints it.
"""
import numpy as np
import pytest
import torch

from tests.harness import reference_reset_params, run_parity

pytestmark = pytest.mark.gpu

TOL_STATE = 5e-8   # the f64 bars of test_parity_gpu.py
TOL_OUT = 2e-6
EPISODE = 26       # SwingRacket-v0: agent steps per episode, every episode
GROUP = 128        # bench.py --stagger: envs per phase group
N = 4096
SWING, HIT = "SwingRacket-v0", "Tennisbot-v0"
SWING_KIND = 0   # TB_ENV_SWING: the env with a fast-forward step
S_STEP = 29      # physics step word of the state record
OUTPUTS = ("obs", "reward", "done", "terminal_obs", "events")


# ---------------------------------------------------------------------------------------------------- helpers
class _Recorded:
    """OracleEnv whose step() keeps the done flags of every step (run_parity does not return them)."""

    def __init__(self, o):
        self.o = o
        self.dones = []

    def __getattr__(self, name):
        return getattr(self.o, name)

    def step(self, actions, **kw):
        out = self.o.step(actions, **kw)
        self.dones.append(out["done"].astype(bool))
        return out


def _pair(oracle_lib, env, n, seed, auto_reset=True, batch=None):
    from tennisbot_rl_b200.batch import TennisBatch

    b = batch or TennisBatch(env, n, device=0, seed=seed, precision="f64", auto_reset=auto_reset)
    o = _Recorded(oracle_lib.OracleEnv(env, n, seed=seed, threads=8, auto_reset=auto_reset))
    return b, o


def _state_err(b, o):
    return float(np.abs(b.get_state().cpu().numpy() - o.get_state()).max())


def _step(b, o, a, via="device"):
    """One env step on both sides at the f64 bars, the whole state record compared after it.  via: 'device' (tb_step, through
    run_parity), 'host' (tb_step_host, the transport TB_HOST_MODE selects).  Returns the oracle's done flags."""
    a = np.asarray(a, np.float32)
    if via == "device":
        rep, _ = run_parity(b, o, 1, lambda t, _obs: a, band=0.0, check_state_every=1)
        assert rep.event_mismatch_hard == 0 and rep.dropped == 0, rep
        assert rep.max_state_err < TOL_STATE and rep.max_obs_err < TOL_OUT and rep.max_reward_err < TOL_OUT, rep
    else:
        hb = b.step_host(a)
        ref = o.step(a)
        np.testing.assert_array_equal(hb["done"], ref["done"])
        np.testing.assert_array_equal(hb["events"], ref["events"])
        np.testing.assert_allclose(hb["obs"], ref["obs"], atol=TOL_OUT, rtol=0)
        np.testing.assert_allclose(hb["reward"], ref["reward"], atol=TOL_OUT, rtol=0)
        d = ref["done"] != 0
        np.testing.assert_allclose(hb["terminal_obs"][d], ref["terminal_obs"][d], atol=TOL_OUT, rtol=0)
        assert _state_err(b, o) < TOL_STATE
    if b.kind == SWING_KIND:
        assert b.ff_diagnostics()[15] == 0  # the fast-forward of this step ended without a queue time-out or fault
    return o.dones[-1]


def _reset(b, o, mask=None, init=None, via="device"):
    """The same (masked) reset on both sides; the observations of the envs it restarted must be equal."""
    ref = o.reset(mask=mask, init=init)
    if via == "device":
        g = b.reset(mask=mask, init=init).cpu().numpy()
    else:
        assert init is None
        g = b.reset_host(mask)
    rows = slice(None) if mask is None else np.asarray(mask, bool)
    np.testing.assert_array_equal(g[rows], ref[rows])


def bench_phase(n):
    """bench.py --stagger: group g of 128 envs starts g mod 26 steps late."""
    return np.arange(n) // GROUP % EPISODE


def random_phase(n, seed):
    """An independent phase per env: phases differ inside nearly every warp."""
    return np.random.default_rng(seed).integers(0, EPISODE, n)


def mixed_tile_share(phase):
    tiles = [phase[i:i + 32] for i in range(0, len(phase), 32)]
    return float(np.mean([len(np.unique(t)) > 1 for t in tiles]))


def _stagger(b, o, phase, act, via="device"):
    """Start every env, then for p = 1 .. 25: one step, and a masked reset of the envs of phase p on both sides.  Afterwards
    an env of phase p is 25 - p steps into its episode, so (SwingRacket-v0) it ends episodes on the steps t = p mod 26 that
    follow (t counted from 0)."""
    _reset(b, o, via=via)
    for p in range(1, EPISODE):
        _step(b, o, act(), via)
        _reset(b, o, mask=phase == p, via=via)


def _swing_schedule_holds(dones, phase):
    """The done flags of the steps after _stagger are exactly the phase schedule."""
    return all(np.array_equal(d, phase == t % EPISODE) for t, d in enumerate(dones))


# ---------------------------------------------------------------------------------------------------- A: staggered phases
def _staggered_run(oracle_lib, phase, via, act, pid=False, seed=41):
    n = len(phase)
    b, o = _pair(oracle_lib, SWING, n, seed)
    if pid:
        b.set_control_mode("pid")
        o.set_control_mode("pid")
    _stagger(b, o, phase, act, via)
    assert not any(d.any() for d in o.dones)  # no episode ended during the set-up
    o.dones.clear()
    steps = 3 * EPISODE
    for t in range(steps):
        _step(b, o, act(), via)
    counts = [int(d.sum()) for d in o.dones]
    print(f"n={n} via={via} pid={pid}: {len(np.unique(phase))} phases, mixed 32-env tiles {100 * mixed_tile_share(phase):.1f} %, "
          f"done per step {counts[:EPISODE]}")
    assert _swing_schedule_holds(o.dones, phase)
    np.testing.assert_array_equal(b.read_stats(), o.read_stats())
    if pid:  # tb_rollout's in-kernel random actions are forces: it has no PID mode
        return counts
    # fused rollout from the staggered states (bars of test_fused_rollout_matches_stepwise)
    k = 60
    gobs, grs, gdc = (x.cpu().numpy() for x in b.rollout(k))
    r = o.rollout(k)
    np.testing.assert_array_equal(gdc, r["done_count"])
    assert np.abs(gobs.astype(np.float64) - r["obs"]).max() < TOL_OUT
    assert np.abs(grs - r["reward_sum"]).max() < 1e-3
    np.testing.assert_array_equal(b.read_stats(), o.read_stats())
    assert _state_err(b, o) < TOL_STATE
    assert b.ff_diagnostics()[15] == 0
    return counts


@pytest.mark.parametrize("n", [N, 1000])
@pytest.mark.parametrize("pattern,via", [("bench", "device"), ("random", "device"), ("random", "zero_copy"), ("random", "staging")])
def test_staggered_phases_match_oracle(oracle_lib, monkeypatch, pattern, via, n):
    """Envs in different phases of their episodes (SwingRacket-v0, f64): every step some envs enter the fast-forward while
    the others take control steps, so ff_kernel mixes deferred control substeps with flights and its finishing pass sees tiles
    of landed and already finished envs.  'bench' is bench.py --stagger's grouping, 'random' mixes phases inside warps; the
    random pattern also runs through tb_step_host's two transports (zero copy: the staged step_kernel leaves deferred rows
    to ff_kernel in the caller's pinned buffer)."""
    if via != "device":
        monkeypatch.setenv("TB_HOST_MODE", via)
    phase = bench_phase(n) if pattern == "bench" else random_phase(n, 3)
    rng = np.random.default_rng(n)
    counts = _staggered_run(oracle_lib, phase, "device" if via == "device" else "host", lambda: rng.uniform(-1, 1, (n, 6)))
    if pattern == "bench":
        assert sum(c > 0 for c in counts[:EPISODE]) == len(np.unique(phase)) == (26 if n == N else 8)
    else:
        assert all(0 < c < n for c in counts)
        assert mixed_tile_share(phase) >= 0.9


@pytest.mark.parametrize("via", ["device", "zero_copy", "staging"])
def test_staggered_pid_mode_match_oracle(oracle_lib, monkeypatch, via):
    """PID control mode (every control substep deferred to ff_kernel's prologue) with random phases: a masked reset clears
    the controller memory of the envs it restarts and leaves the others' alone, or the next steps differ from the oracle."""
    if via != "device":
        monkeypatch.setenv("TB_HOST_MODE", via)
    phase = random_phase(N, 4)
    rng = np.random.default_rng(8)
    lo, hi = np.array([5, -4, 0.5, 0, 0, 0]), np.array([12, 4, 2.0, 0, 0, 0])  # test_pid_control_mode_parity's targets
    counts = _staggered_run(oracle_lib, phase, "device" if via == "device" else "host", lambda: rng.uniform(lo, hi, (N, 6)),
                            pid=True)
    assert all(0 < c < N for c in counts) and mixed_tile_share(phase) >= 0.9


# ---------------------------------------------------------------------------------------------------- B: placements mid-episode
@pytest.mark.parametrize("env", [SWING, HIT])
def test_masked_resets_mid_episode_match_oracle(oracle_lib, env):
    """Mid-episode, a random ~30 % of the envs get an explicit placement (tb_reset_from with a mask: no kStDerived, goal and
    spawn from the record), later another ~30 % a plain masked reset.  Their next auto-resets must return them to the RNG
    placement, keyed by their own env id and episode."""
    n = N
    swing = env == SWING
    b, o = _pair(oracle_lib, env, n, 13)
    rng = np.random.default_rng(21)
    t_init, t_plain, steps = (10, 18, 90) if swing else (40, 100, 1110)
    m_init, m_plain = rng.random(n) < 0.3, rng.random(n) < 0.3
    _reset(b, o)
    last = np.zeros(n, np.int64)
    for t in range(1, steps + 1):
        _step(b, o, rng.uniform(-1, 1, (n, o.act_dim)))
        if t == t_init:
            _reset(b, o, mask=m_init, init=reference_reset_params(o.kind, n, rng))
            last[m_init] = t
        if t == t_plain:
            _reset(b, o, mask=m_plain)
            last[m_plain] = t
    dones = np.array(o.dones)
    ended_after = np.array([dones[last[i]:, i].any() for i in range(n)])  # step index last[i] is step last[i] + 1
    print(f"{env}: explicit placements {m_init.sum()}, plain masked resets {m_plain.sum()}, done per step "
          f"{dones.sum(1)[:EPISODE].tolist()} ..., masked envs that ended an episode since: {ended_after[last > 0].mean():.3f}")
    assert ended_after[last > 0].all()  # every masked env went through its next auto-reset
    if swing:
        t = np.arange(1, steps + 1)[:, None]
        np.testing.assert_array_equal(dones, (t > last) & ((t - last) % EPISODE == 0))
    np.testing.assert_array_equal(b.read_stats(), o.read_stats())


# ---------------------------------------------------------------------------------------------------- C: injected records
def _inject(b, o, records):
    b.set_state(records)
    o.set_state(records)
    np.testing.assert_array_equal(b.get_state().cpu().numpy(), records)


@pytest.mark.parametrize("case", ["swing_control", "swing_mixed", "hit_shoot", "hit_bounced"])
def test_set_state_permuted_records_match_oracle(oracle_lib, case):
    """tb_set_state with the oracle's records permuted across envs: env i then holds env j's goal, spawn, shoot force and
    episode number, which only the loaded packs give (kStDerived must be clear; a kept bit re-derives env i's own goal).
    Stepping continues past every env's next auto-reset, which sets the bit again."""
    from oracle.binding import S_BW

    n = N
    env = SWING if case.startswith("swing") else HIT
    b, o = _pair(oracle_lib, env, n, 29)
    rng = np.random.default_rng(17)
    act = lambda: rng.uniform(-1, 1, (n, o.act_dim))  # noqa: E731
    _reset(b, o)
    if case == "swing_control":        # all envs at physics step 10 of the control phase
        for _ in range(10):
            _step(b, o, act())
        rec = o.get_state()[rng.permutation(n)]
    elif case == "swing_mixed":        # half at step 25 (the next step enters the fast-forward), half at step 10
        for t in range(25):
            _step(b, o, act())
            if t == 9:
                s10 = o.get_state()
        s25 = o.get_state()
        late = rng.random(n) < 0.5
        rec = np.where(late[:, None], s25[rng.permutation(n)], s10[rng.permutation(n)])
    elif case == "hit_shoot":          # inside the shoot window (defaults: frames 0..4), where pack 5's shoot force is read
        for _ in range(3):
            _step(b, o, act())
        rec = o.get_state()[rng.permutation(n)]
        assert o.get_param("shoot_start") <= 3 < o.get_param("shoot_start") + o.get_param("shoot_frames")
    else:                              # after the first floor bounces (step ~390): most balls spin about y or z (kStSpin)
        for _ in range(420):
            _step(b, o, act())
        rec = o.get_state()[rng.permutation(n)]
    _inject(b, o, rec)
    spin = (rec[:, S_BW + 1:S_BW + 3] != 0).any(1)
    print(f"{case}: injected at physics steps {np.unique(rec[:, S_STEP]).astype(int).tolist()[:8]}, records with y/z spin "
          f"{100 * spin.mean():.1f} %")
    if case == "hit_bounced":
        assert spin.mean() >= 0.5
    o.dones.clear()
    steps = 60 if env == SWING else 1010
    for _ in range(steps):
        _step(b, o, act())
    dones = np.array(o.dones)
    assert dones.any(0).all()  # every env passed its next auto-reset
    if case == "swing_mixed":
        assert 0.4 < late.mean() < 0.6 and np.array_equal(dones[0], late)  # one launch: fast-forward entrants and control steps
    np.testing.assert_array_equal(b.read_stats(), o.read_stats())


# ---------------------------------------------------------------------------------------------------- D: parameters mid-episode
@pytest.mark.parametrize("change", ["gravity_damping", "racket_scale"])
@pytest.mark.parametrize("env", [SWING, HIT])
def test_set_param_mid_episode_matches_oracle(oracle_lib, env, change):
    """Scene parameters changed between two steps take effect at once on both sides (tbo_set_param rebuilds its shapes).
    In SwingRacket-v0 the envs in the control phase keep their ball velocity in the free-fall table, indexed by their step:
    tb_set_param must write it out under the old parameters before the table changes.  Random phases use every table
    index.  racket_scale goes through TennisVecEnv.set_racket_scale(apply_now=True)."""
    from tennisbot_rl_b200.vec_env import TennisVecEnv

    n = N
    venv = TennisVecEnv(env, n, seed=33) if change == "racket_scale" else None
    b, o = _pair(oracle_lib, env, n, 33, batch=venv.batch if venv else None)
    rng = np.random.default_rng(5)
    act = lambda: rng.uniform(-1, 1, (n, o.act_dim))  # noqa: E731
    phase = random_phase(n, 6)
    _stagger(b, o, phase, act)
    o.dones.clear()
    changes = {5: ("gravity_z", -7.5), 14: ("lin_damping", 0.2)} if change == "gravity_damping" else {5: ("racket_scale", 1.6)}
    steps = 3 * EPISODE if env == SWING else 400
    for t in range(steps):
        if t in changes:
            name, v = changes[t]
            if env == SWING:  # every ball_vz index 0..25 is in use by control-phase envs
                st = o.get_state()[:, S_STEP]
                print(f"{name} -> {v} before step {t}: envs per physics step {np.bincount(st.astype(int)).tolist()}")
                assert np.array_equal(np.unique(st), np.arange(EPISODE))
            if name == "racket_scale":
                venv.set_racket_scale(v, apply_now=True)
            else:
                b.set_param(name, v)
            o.set_param(name, v)
            assert b.get_param(name) == v
        _step(b, o, act())
    if env == SWING:
        assert _swing_schedule_holds(o.dones, phase)
    print(f"{env} {change}: done per step {[int(d.sum()) for d in o.dones][:EPISODE]} ...")
    np.testing.assert_array_equal(b.read_stats(), o.read_stats())


# ---------------------------------------------------------------------------------------------------- E: bit-exact twins
def _assert_same(t, xs, ys, names=OUTPUTS):
    for name, x, y in zip(names, xs, ys):
        if not torch.equal(x, y):
            bad = (x != y).reshape(x.shape[0], -1).any(1).nonzero().flatten()
            raise AssertionError(f"step {t}: {name} differs in {len(bad)} envs, first {bad[:8].tolist()}")


TWIN_CASES = [(op, env, prec) for op in ("set_state", "set_param", "zero_mask_reset") for env in (SWING, HIT) for prec in ("f64", "f32")]
TWIN_CASES += [("init_from_record", SWING, prec) for prec in ("f64", "f32")]


@pytest.mark.parametrize("op,env,precision", TWIN_CASES)
def test_twin_unchanged_by_state_operations(op, env, precision):
    """Twin contexts stepped with the same seed, phases and actions, where B also undergoes an operation that must change
    nothing: every output of every step, the state records and the statistics must be bit-identical.
      set_state         B.set_state(B.get_state()) every 3 steps.  Pack 4 is written from the ball_vz table and the kStPristine /
                        kStDerived bits are cleared, so B steps its falling ball with ctl_fast's arithmetic where A reads
                        the next table entry: equal only if ball_vz_kernel rounds exactly as ctl_fast does
      set_param         B.set_param(name, current value) every 9 steps (gravity_z, lin_damping): materialise_kernel and the
                        table rebuild
      zero_mask_reset   B.reset with an all-zero mask every 5 steps, with and without placements
      init_from_record  (SwingRacket-v0, whose spawn and goal are stored as drawn) B starts every episode of the set-up from
                        the placement read back from A's record (trajectory.init_from_reset_state): B loads what A derives,
                        through the episode and the auto-resets that follow"""
    from tennisbot_rl_b200 import trajectory
    from tennisbot_rl_b200.batch import TennisBatch

    n = N
    A, B = (TennisBatch(env, n, device=0, seed=47, precision=precision) for _ in range(2))
    gen = torch.Generator(device="cuda").manual_seed(11)
    phase = random_phase(n, 9)
    steps = 4 * EPISODE if env == SWING else 1100
    ops = 0

    def reset_both(mask=None):
        nonlocal ops
        oa = A.reset(mask=mask).clone()
        if op == "init_from_record":
            ops += 1
            rec = A.get_state().cpu().numpy()
            ob = B.reset(mask=mask, init=np.stack([trajectory.init_from_reset_state(env, r) for r in rec]))
        else:
            ob = B.reset(mask=mask)
        rows = slice(None) if mask is None else torch.as_tensor(mask, device="cuda")
        assert torch.equal(oa[rows], ob[rows])

    def step_both(t):
        a = torch.empty((n, A.act_dim), device="cuda").uniform_(-1, 1, generator=gen)
        ya = [x.clone() for x in A.step(a)]
        _assert_same(t, ya, B.step(a))
        return ya[2]

    reset_both()
    for p in range(1, EPISODE):
        step_both(p - EPISODE)
        reset_both(phase == p)
    ndone = []
    for t in range(steps):
        if op == "set_state" and t % 3 == 0:
            B.set_state(B.get_state())
            ops += 1
        elif op == "set_param" and t % 9 == 0:
            name = ("gravity_z", "lin_damping")[(t // 9) % 2]
            B.set_param(name, B.get_param(name))
            ops += 1
        elif op == "zero_mask_reset" and t % 5 == 0:
            zero = np.zeros(n, np.uint8)
            B.reset(mask=zero, init=None if t % 10 else np.ones((n, 8)))
            ops += 1
        ndone.append(int(step_both(t).sum()))
        if t % 13 == 12:
            assert torch.equal(A.get_state(), B.get_state()), f"state after step {t}"
    assert torch.equal(A.get_state(), B.get_state())
    np.testing.assert_array_equal(A.read_stats(), B.read_stats())
    print(f"{op} {env} {precision}: {ops} operations, mixed 32-env tiles {100 * mixed_tile_share(phase):.1f} %, "
          f"done per step {ndone[:EPISODE]} ..., episodes {A.read_stats()[0]}")
    if env == SWING:
        assert all(0 < c < n for c in ndone) and mixed_tile_share(phase) >= 0.9


@pytest.mark.parametrize("precision", ["f64", "f32"])
def test_twin_shards_with_offset(precision):
    """Two SwingRacket-v0 shards with env_id_offset (split at 1000: not a multiple of a warp), stepped through tb_step with
    random phases applied by global env id: step_kernel re-derives each goal and ff_kernel auto-resets each env by its global
    id, so the union of the shards equals the full batch bit for bit and the statistics add up."""
    from tennisbot_rl_b200.batch import TennisBatch

    n, split = N, 1000
    full = TennisBatch(SWING, n, device=0, seed=53, precision=precision)
    shards = [TennisBatch(SWING, hi - lo, device=0, seed=53, precision=precision, env_id_offset=lo)
              for lo, hi in ((0, split), (split, n))]
    gen = torch.Generator(device="cuda").manual_seed(12)
    phase = random_phase(n, 10)

    bounds = ((0, split), (split, n))

    def reset_all(mask=None):
        of = full.reset(mask=mask).clone()
        parts = torch.cat([s.reset(mask=None if mask is None else mask[lo:hi]).clone() for s, (lo, hi) in zip(shards, bounds)])
        rows = slice(None) if mask is None else torch.as_tensor(mask, device="cuda")
        assert torch.equal(of[rows], parts[rows])

    def step_all(t):
        a = torch.empty((n, 6), device="cuda").uniform_(-1, 1, generator=gen)
        yf = full.step(a)
        ys = [s.step(a[lo:hi].contiguous()) for s, (lo, hi) in zip(shards, bounds)]
        _assert_same(t, yf, [torch.cat([y[k] for y in ys]) for k in range(len(OUTPUTS))])
        return int(yf[2].sum())

    reset_all()
    for p in range(1, EPISODE):
        step_all(p - EPISODE)
        reset_all(phase == p)
    ndone = [step_all(t) for t in range(3 * EPISODE)]
    assert torch.equal(full.get_state(), torch.cat([s.get_state() for s in shards]))
    np.testing.assert_array_equal(full.read_stats(), sum(s.read_stats() for s in shards))
    print(f"shards {precision}: done per step {ndone[:EPISODE]}, episodes {full.read_stats()[0]}")
    assert all(0 < c < n for c in ndone)


# ---------------------------------------------------------------------------------------------------- F: stepping after done
@pytest.mark.parametrize("env", [SWING, HIT])
def test_steps_after_done_without_auto_reset(oracle_lib, env):
    """auto_reset = 0: an env whose episode is over keeps being stepped (the oracle runs the physics step with the action and
    reports done again; the CUDA path defers a done SwingRacket-v0 env to the generic path every step).  Four steps past the
    end of every episode, outputs and the final state records must agree."""
    n = N
    b, o = _pair(oracle_lib, env, n, 59, auto_reset=False)
    rng = np.random.default_rng(23)
    _reset(b, o)
    last = EPISODE if env == SWING else 1001  # the step on which the last episode ends (fast-forward / time-out)
    for _ in range(last + 4):
        _step(b, o, rng.uniform(-1, 1, (n, o.act_dim)))
    dones = np.array(o.dones)
    first = dones.argmax(0)
    after = (dones.shape[0] - first - 1)
    print(f"{env}: episodes end on steps {first.min() + 1}..{first.max() + 1}, steps taken after done: "
          f"{after.min()}..{after.max()}")
    assert dones[-5:].all()  # every env was done on the last five steps
    assert _state_err(b, o) < TOL_STATE
    np.testing.assert_array_equal(b.read_stats(), o.read_stats())
