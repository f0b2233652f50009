"""tb_trace_step on the B200: the traced step against tb_step, each substep against the oracle's physics step, padding and
truncation, the time-out bound, no side effects, determinism and graph capture, the rejections, and the recorder's flight
frames."""
import ctypes as C
import re
import struct
import subprocess
import sys
import zlib
from pathlib import Path

import numpy as np
import pytest
import torch

from oracle import binding as ob
from tennisbot_rl_b200 import _lib
from tennisbot_rl_b200.batch import TennisBatch
from tennisbot_rl_b200.render import default_camera

pytestmark = pytest.mark.gpu

ROOT = Path(__file__).resolve().parent.parent
GOLDEN = ROOT / "tests" / "golden" / "ppo_swing_policy.npz"
SWING, HIT = "SwingRacket-v0", "Tennisbot-v0"
PHYS = _lib.STAT_NAMES.index("physics_steps")


def episode(env_id, precision, n, source, seed=3):
    """Every env step of one whole episode with auto_reset = 0 (a swing episode: 26 steps; Tennisbot-v0: 450 steps), stepped
    by tb_step.  Yields, per step, the batch and a dict: `before` (get_state() before the step), `act` (the actions tb_step
    received), reward / done / events / `after` (get_state() after it) and `phys` (the TB_STAT_PHYSICS_STEPS it added).
    source 'policy': swing, the saved PPO policy (deterministic; a twin batch runs tb_policy_rollout and hands its clipped
    actions over); hit, a torch restatement of the scripted tracker's law on the observation.  'random': uniform actions."""
    from tennisbot_rl_b200.ppo import load_sb3_policy_npz

    swing = env_id == SWING
    b = TennisBatch(env_id, n, seed=seed, precision=precision, auto_reset=False)
    obs = b.reset().clone()
    g = torch.Generator("cuda").manual_seed(seed + 11)
    twin = None
    if swing and source == "policy":
        twin = TennisBatch(env_id, n, seed=seed, precision=precision, auto_reset=False)
        twin.set_policy(load_sb3_policy_npz(GOLDEN).cuda())
        pobs, last = torch.zeros((1, n, 6), device="cuda"), torch.zeros((n, 6), device="cuda")
        rew, done = torch.zeros((1, n), device="cuda"), torch.zeros((1, n), dtype=torch.uint8, device="cuda")
        act = torch.zeros((1, n, 6), device="cuda")
        pobs[0].copy_(twin.reset())
    for _ in range(26 if swing else 450):
        before = b.get_state()
        if twin is not None:
            twin.policy_rollout(pobs, rew, done, last, actions=act, deterministic=True)
            pobs[0].copy_(last)
            taken = act[0].clamp(-1, 1).contiguous()
        else:
            taken = torch.empty((n, b.act_dim), device="cuda").uniform_(-1, 1, generator=g)
            if source == "policy":  # rollout_action's TB_ACT_TRACK law, in float32 on the observation
                u = 4.0 * (obs[:, 7] - obs[:, 1]) - 1.5 * obs[:, 4]
                taken = torch.stack([0.2 * taken[:, 0], u.clamp(-1.0, 1.0)], 1).contiguous()
        p0 = int(b.read_stats()[PHYS])
        o, r, d, _, e = b.step(taken)
        obs = o.clone()
        if twin is not None:
            assert torch.equal(last, obs)  # the twin and this batch step the same envs with the same actions
        step = dict(before=before, act=taken, reward=r.clone(), done=d.clone(), events=e.clone(), after=b.get_state(),
                    phys=int(b.read_stats()[PHYS]) - p0)
        yield b, step
    b.close()
    if twin is not None:
        twin.close()


def np_(*xs):
    return [x.cpu().numpy() for x in xs]


# ------------------------------------------------------------------------------------------------ 1. against tb_step
@pytest.mark.parametrize("precision", ["f64", "f32"])
@pytest.mark.parametrize("env_id,source", [(SWING, "policy"), (SWING, "random"), (HIT, "policy"), (HIT, "random")])
def test_trace_ends_where_tb_step_ends(env_id, source, precision):
    near = contacts = flights = 0
    for b, st in episode(env_id, precision, 4096, source):
        trace, bits, sub, rew, done, ev = b.trace_step(st["act"], st["before"])
        final, sub, rew, done, ev = np_(trace[-1], sub, rew, done, ev)
        want_rew, want_done, want_ev, after = np_(st["reward"], st["done"], st["events"], st["after"])
        contacts += int((ev & _lib.EV_RACKET_BALL != 0).sum())
        flights += int((sub > 1).sum())
        if precision == "f64":
            np.testing.assert_array_equal(rew, want_rew)
            np.testing.assert_array_equal(done, want_done)
            np.testing.assert_array_equal(ev, want_ev)
            assert int(sub.sum()) == st["phys"]
            np.testing.assert_allclose(final[:, :28], after[:, :28], rtol=0, atol=5e-8)
            np.testing.assert_array_equal(final[:, 28:], after[:, 28:])
        else:  # float32: a decision may flip where the oracle's margin to its threshold is below 2e-4 m
            bad = np.flatnonzero((done != want_done) | (ev != want_ev))
            if bad.size:
                o = ob.OracleEnv(env_id, bad.size, auto_reset=False)
                o.set_state(st["before"].cpu().numpy()[bad])
                margin = o.step(st["act"].cpu().numpy()[bad], want_margin=True)["margin"]
                o.close()
                assert (margin < 2e-4).all(), (bad[margin >= 2e-4][:5], margin)
                near += bad.size
    print(f"{env_id} {source} {precision}: {flights} flights, {contacts} racket contacts, {near} near-threshold flips (f32)")
    if env_id == SWING:
        assert flights > 0
    elif source == "policy":
        assert contacts > 0


# ------------------------------------------------------------------------------------------------ 2. against the oracle
def substep_forces(kind, k, prev, a, shoot):
    """The forces of substep k (0-based) of an env step, restated from env_substep: (racket force, racket torque, ball force).
    prev: the record before the substep; a: the float32 action."""
    z = np.zeros(3)
    a = a.astype(np.float64)
    if kind == _lib.ENV_SWING:
        if k == 0:  # phase 0: the action
            return np.array([a[0] * 400, a[1] * 400, a[2] * 400 + 4 * 9.81]), a[3:6] * 5, z
        if k == 1:  # phase 1: the forces were cleared
            return z, z, z
        # phase 2: the hold force queued from the pose before this substep
        return np.array([-50 * (prev[0] - prev[22]), -2 * (prev[1] - prev[23]), -2 * (prev[2] - prev[24] - 4)]), z, z
    s0, sn = shoot
    fb = prev[22:25].copy() if s0 <= prev[29] < s0 + sn else z
    return np.array([a[0] * 10, a[1] * 10, 4 * 9.81]), z, fb


@pytest.mark.parametrize("env_id,source,n", [(SWING, "policy", 512), (SWING, "random", 512), (HIT, "policy", 256)])
def test_each_substep_matches_the_oracle(env_id, source, n):
    worst_a = worst_b = 0.0
    for b, st in episode(env_id, "f64", n, source):
        shoot = (b.get_param("shoot_start"), b.get_param("shoot_frames"))
        trace, bits, sub, rew, done, ev = np_(*b.trace_step(st["act"], st["before"]))
        before, act = np_(st["before"], st["act"])
        o = ob.OracleEnv(env_id, 1, auto_reset=False)
        for i in range(n):
            chain = before[i]
            for k in range(sub[i]):
                prev = before[i] if k == 0 else trace[k - 1, i]
                got, got_bits = o.physics_step(prev, *substep_forces(b.kind, k, prev, act[i], shoot))  # (a) one substep
                err = np.abs(got[:22] - trace[k, i, :22]).max()
                assert err <= 5e-8 and got_bits == bits[k, i], (i, k, err, got_bits, bits[k, i])
                worst_a = max(worst_a, err)
                chain, chain_bits = o.physics_step(chain, *substep_forces(b.kind, k, chain, act[i], shoot))  # (b) free chain
                err = np.abs(chain[:22] - trace[k, i, :22]).max()
                assert err <= 5e-8 and chain_bits == bits[k, i], (i, k, err, chain_bits, bits[k, i])
                worst_b = max(worst_b, err)
        o.close()
        o = ob.OracleEnv(env_id, n, auto_reset=False)  # the flight's end against the oracle's whole step
        o.set_state(before)
        ref = o.step(act)
        o.close()
        np.testing.assert_array_equal(done, ref["done"])
        np.testing.assert_allclose(rew, ref["reward"], rtol=0, atol=2e-6)
    print(f"{env_id} {source}: worst pose error per substep {worst_a:.2e}, along a free oracle chain {worst_b:.2e}")


# ------------------------------------------------------------------------------------------------ 3. padding and truncation
@pytest.mark.parametrize("precision", ["f64", "f32"])
@pytest.mark.parametrize("source", ["policy", "random"])
def test_padding_and_truncation(source, precision):
    truncated = False
    for b, st in episode(SWING, precision, 512, source):
        trace, bits, sub, rew, done, ev = b.trace_step(st["act"], st["before"])
        s = sub.long()
        idx = torch.arange(trace.shape[0], device="cuda")[:, None]
        pad = idx >= s[None, :]
        final = trace[s - 1, torch.arange(512, device="cuda")]
        assert torch.equal(trace[pad], final[None].expand_as(trace)[pad])
        assert not bits[pad].any()
        if int(s.max()) > 40:  # the flight: keep 40 records only
            t2, b2, s2, r2, d2, e2 = b.trace_step(st["act"], st["before"], max_substeps=40)
            assert torch.equal(t2, trace[:40]) and torch.equal(b2, bits[:40])
            for x, y in ((s2, sub), (r2, rew), (d2, done), (e2, ev)):
                assert torch.equal(x, y)
            truncated = True
    assert truncated


# ------------------------------------------------------------------------------------------------ 4. time-out bound
@pytest.mark.parametrize("precision", ["f64", "f32"])
def test_a_flight_that_cannot_land_takes_the_bound(precision):
    b = TennisBatch(SWING, 4, seed=1, precision=precision, auto_reset=False)
    b.set_param("gravity_z", 0.0)
    b.reset()
    rec = b.get_state()
    rec[:, 13:16] = torch.tensor([-20.0, 0.0, 30.0], dtype=torch.float64)  # the ball, at rest, far from every shape
    rec[:, 16:22] = 0
    rec[:, _lib.STATE_WORDS - 3] = 25  # the step counter before the 26th step
    b.set_state(rec)
    act = torch.zeros((4, 6), device="cuda")
    trace, bits, sub, rew, done, ev = b.trace_step(act)
    assert (sub == _lib.TRACE_MAX_SUBSTEPS).all() and (done == 1).all() and (rew == 0).all()
    assert ((ev & _lib.EV_TIMEOUT) != 0).all()
    assert (trace[-1, :, 29] == 801).all() and (trace[-1, :, 30] == 1).all()
    assert ((ev & (_lib.EV_COURT_BALL | _lib.EV_GOAL_BALL | _lib.EV_RACKET_BALL)) == 0).all()
    b.close()


# ------------------------------------------------------------------------------------------------ 5. no side effects
@pytest.mark.parametrize("precision", ["f64", "f32"])
@pytest.mark.parametrize("env_id", [SWING, HIT])
def test_tracing_leaves_the_context_alone(env_id, precision):
    n = 512
    a, b = (TennisBatch(env_id, n, seed=5, precision=precision) for _ in range(2))
    a.reset(), b.reset()
    g = torch.Generator("cuda").manual_seed(2)
    perm = torch.randperm(n, generator=torch.Generator().manual_seed(0))[:300].cuda()
    for t in range(30):
        act = torch.empty((n, a.act_dim), device="cuda").uniform_(-1, 1, generator=g)
        st = a.get_state()
        before = a.launch_count()
        full = a.trace_step(act, st)
        assert a.launch_count() - before == 1
        part = a.trace_step(act[perm].contiguous(), st[perm].contiguous())  # count != N, rows permuted
        assert torch.equal(part[0], full[0][:, perm]) and torch.equal(part[1], full[1][:, perm])
        for x, y in zip(part[2:], full[2:]):
            assert torch.equal(x, y[perm])
        ra = [x.clone() for x in a.step(act)]
        rb = [x.clone() for x in b.step(act)]
        for x, y in zip(ra, rb):
            assert torch.equal(x, y), t
    assert torch.equal(a.get_state(), b.get_state())
    np.testing.assert_array_equal(a.read_stats(), b.read_stats())


# ------------------------------------------------------------------------------------------------ 6. determinism, graphs
@pytest.mark.parametrize("precision", ["f64", "f32"])
def test_trace_is_deterministic_and_capturable(precision):
    n = 512
    b = TennisBatch(SWING, n, seed=9, precision=precision, auto_reset=False)
    b.reset()
    g = torch.Generator("cuda").manual_seed(4)
    states, acts = [], []
    for _ in range(26):
        acts.append(torch.empty((n, 6), device="cuda").uniform_(-1, 1, generator=g))
        states.append(b.get_state())
        b.step(acts[-1])
    eager = b.trace_step(acts[25], states[25])
    again = b.trace_step(acts[25], states[25])
    for x, y in zip(eager, again):
        assert torch.equal(x, y)
    st_buf, act_buf = states[24].clone(), acts[24].clone()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        b.trace_step(act_buf, st_buf)
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = b.trace_step(act_buf, st_buf)
    st_buf.copy_(states[25]), act_buf.copy_(acts[25])  # replay on the 26th step's records: the flight
    graph.replay()
    torch.cuda.synchronize()
    for x, y in zip(out, eager):
        assert torch.equal(x, y)
    b.close()


# ------------------------------------------------------------------------------------------------ 7. rejections
def test_rejections():
    b = TennisBatch(SWING, 4, seed=0)
    L = b.lib
    st = b.get_state()
    act = torch.zeros((4, 6), device="cuda")
    trace = torch.empty((8, 4, 32), dtype=torch.float64, device="cuda")
    sub = torch.empty(4, dtype=torch.int32, device="cuda")

    def call(batch=b, states=st, actions=act, count=4, max_substeps=8, out=trace, substeps=sub):
        p = [None if x is None else C.c_void_p(x.data_ptr()) for x in (states, actions, out, substeps)]
        before = batch.launch_count()
        rc = L.tb_trace_step(batch.h, p[0], p[1], count, max_substeps, p[2], None, p[3], None, None, None, batch._stream())
        torch.cuda.synchronize()
        assert batch.launch_count() - before == (1 if rc == 0 else 0)
        return rc, L.tb_last_error().decode()

    assert call()[0] == 0
    for kwargs, msg in [
        (dict(states=None), "required"),
        (dict(actions=None), "required"),
        (dict(out=None), "required"),
        (dict(substeps=None), "required"),
        (dict(count=0), "count"),
        (dict(count=-2), "count"),
        (dict(max_substeps=0), "max_substeps"),
        (dict(max_substeps=-1), "max_substeps"),
        (dict(max_substeps=777), "max_substeps"),
        (dict(count=2 ** 60, max_substeps=776), "overflow"),
    ]:
        rc, err = call(**kwargs)
        assert rc != 0 and msg in err and "tb_trace_step" in err, (kwargs, err)
    h = TennisBatch(HIT, 4, seed=0)
    rc, err = call(batch=h, states=h.get_state(), actions=torch.zeros((4, 2), device="cuda"), max_substeps=2)
    assert rc != 0 and "max_substeps" in err
    assert call(batch=h, states=h.get_state(), actions=torch.zeros((4, 2), device="cuda"), max_substeps=1)[0] == 0
    p = TennisBatch(SWING, 4, seed=0)
    p.set_control_mode("pid")
    rc, err = call(batch=p)
    assert rc != 0 and "TB_CONTROL_PID" in err
    assert L.tb_trace_step(None, C.c_void_p(st.data_ptr()), C.c_void_p(act.data_ptr()), 4, 8, C.c_void_p(trace.data_ptr()),
                           None, C.c_void_p(sub.data_ptr()), None, None, None, None) != 0
    for kwargs in (dict(actions=act[:3]), dict(actions=act.double()), dict(actions=act, states=st.float()),
                   dict(actions=act, states=st[:, :16].contiguous()), dict(actions=act, max_substeps=0),
                   dict(actions=act, max_substeps=777)):
        with pytest.raises(ValueError):
            b.trace_step(**kwargs)


# ------------------------------------------------------------------------------------------------ 8. frames end to end
def read_png(path):
    data = Path(path).read_bytes()
    pos, idat, w, h = 8, b"", 0, 0
    while pos < len(data):
        n, tag = struct.unpack(">I4s", data[pos:pos + 8])
        body = data[pos + 8:pos + 8 + n]
        if tag == b"IHDR":
            w, h = struct.unpack(">II", body[:8])
        elif tag == b"IDAT":
            idat += body
        pos += 12 + n
    rows = np.frombuffer(zlib.decompress(idat), np.uint8).reshape(h, 1 + 3 * w)
    assert (rows[:, 0] == 0).all()
    return rows[:, 1:].reshape(h, w, 3)


def test_recorder_draws_the_flight(tmp_path):
    from tennisbot_rl_b200.ppo import load_sb3_policy_npz

    k, m = 4, 2
    res = subprocess.run([sys.executable, str(ROOT / "tools" / "record_episode.py"), SWING, "--policy", str(GOLDEN),
                          "--flight-every", str(k), "--envs", str(m), "--out", str(tmp_path)],
                         capture_output=True, text=True, cwd=ROOT)
    assert res.returncode == 0, res.stderr
    # the same episode here: the tool's seed 0, f64, deterministic policy, without auto-reset
    b = TennisBatch(SWING, m, seed=0, precision="f64", auto_reset=False)
    b.set_policy(load_sb3_policy_npz(GOLDEN).cuda())
    obs, last = torch.zeros((1, m, 6), device="cuda"), torch.zeros((m, 6), device="cuda")
    rew, done = torch.zeros((1, m), device="cuda"), torch.zeros((1, m), dtype=torch.uint8, device="cuda")
    act = torch.zeros((1, m, 6), device="cuda")
    obs[0].copy_(b.reset())
    for _ in range(26):
        before = b.get_state()
        b.policy_rollout(obs, rew, done, last, actions=act, deterministic=True)
        obs[0].copy_(last)
    trace, _, sub = b.trace_step(act[0].clamp(-1, 1), before)[:3]
    last_k = int(sub.max()) - 1
    ks = list(range(k - 1, last_k, k)) + [last_k]
    assert f"{len(ks)} of the frames show flight substeps" in res.stdout, res.stdout
    pngs = sorted(tmp_path.glob("env*_frame*.png"))
    assert len(pngs) == m * (27 + len(ks))
    cam = default_camera(SWING)
    rgb, _, body = b.render(cam, trace[ks].reshape(-1, 32), body=True)
    rgb = rgb.reshape(len(ks), m, *rgb.shape[1:]).cpu().numpy()
    body = body.reshape(len(ks), m, *body.shape[1:]).cpu().numpy()
    moved = False
    for i in range(m):
        for j in range(len(ks)):
            np.testing.assert_array_equal(read_png(tmp_path / f"env{i:03d}_frame{26 + j:04d}.png"), rgb[j, i])
        # the last flight frame is the landed state the episode's final frame shows
        np.testing.assert_array_equal(read_png(tmp_path / f"env{i:03d}_frame{26 + len(ks) - 1:04d}.png"),
                                      read_png(tmp_path / f"env{i:03d}_frame{26 + len(ks):04d}.png"))
        centres = {tuple(np.argwhere(body[j, i] == _lib.BODY_BALL).mean(0).round(1)) for j in range(len(ks))
                   if (body[j, i] == _lib.BODY_BALL).any()}
        moved |= len(centres) > 1
    assert moved  # the ball is drawn in flight, not only where it lands
    assert (tmp_path / "contact_sheet.png").exists()
    b.close()
