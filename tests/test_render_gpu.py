"""tb_render on the B200: frames of states from real rollouts against the float64 numpy reference (tests/render_reference.py),
determinism, no side effects on the env, CUDA-graph capture, records from outside the batch, the rejections, and the gym /
VecEnv frames."""
import ctypes as C
import math
from pathlib import Path

import numpy as np
import pytest
import torch

from tennisbot_rl_b200 import _lib
from tennisbot_rl_b200.batch import TennisBatch
from tennisbot_rl_b200.render import Camera, default_camera, tile_images
from tests import render_reference as rr

pytestmark = pytest.mark.gpu

GOLDEN = Path(__file__).parent / "golden" / "ppo_swing_policy.npz"
W, H = 160, 120


def _policy_states(env_id, precision, n=16, scale=None):
    """get_state() after every env step of one swing episode of the saved PPO policy (deterministic), or of 450 steps of the
    scripted tracker (hit: the shot ball takes about 400 steps to reach the racket): [T, n, 32]; and the same for uniform
    random actions."""
    from tennisbot_rl_b200.ppo import load_sb3_policy_npz

    out = []
    for source in ("policy", "random"):
        # (a swing episode is exactly 26 steps: without auto-reset the last state is the episode's own)
        b = TennisBatch(env_id, n, seed=3, precision=precision, auto_reset=env_id != "SwingRacket-v0")
        if scale is not None:
            b.set_param("racket_scale", scale)
        b.reset()
        states = []
        if env_id == "SwingRacket-v0" and source == "policy":
            b.set_policy(load_sb3_policy_npz(GOLDEN).cuda())
            obs, last = torch.zeros((1, n, 6), device="cuda"), torch.zeros((n, 6), device="cuda")
            rew, done = torch.zeros((1, n), device="cuda"), torch.zeros((1, n), dtype=torch.uint8, device="cuda")
            obs[0].copy_(b.obs)
            for _ in range(26):
                b.policy_rollout(obs, rew, done, last, deterministic=True)
                obs[0].copy_(last)
                states.append(b.get_state())
        else:
            g = torch.Generator("cuda").manual_seed(7)
            for _ in range(26 if env_id == "SwingRacket-v0" else 450):
                if source == "policy":
                    b.rollout(1, _lib.ACT_TRACK)
                else:
                    b.step(torch.empty((n, b.act_dim), device="cuda").uniform_(-1, 1, generator=g))
                states.append(b.get_state())
        out.append(torch.stack(states))
        b.close()
    return out


def _cameras(env_id):
    if env_id == "SwingRacket-v0":  # default; close to the racket's start region; from above the goal region
        return [default_camera(env_id, W, H), Camera(W, H, eye=(13.0, -4.0, 1.8), target=(8.0, 0.0, 0.8), fov_y_deg=45.0),
                Camera(W, H, eye=(-7.0, 0.0, 16.0), target=(-7.5, 0.0, 0.0), up=(1.0, 0.0, 0.0), fov_y_deg=60.0)]
    return [default_camera(env_id, W, H), Camera(W, H, eye=(15.0, -3.0, 1.2), target=(9.0, 0.0, 0.6), fov_y_deg=45.0),
            Camera(W, H, eye=(10.0, 0.0, 14.0), target=(9.5, 0.0, 0.0), up=(1.0, 0.0, 0.0), fov_y_deg=60.0)]


def _pick(states, hit_step):
    """A few frames of a [T, n, 32] trajectory: early, middle, `hit_step` and the last."""
    T = states.shape[0]
    steps = sorted({1, T // 2, hit_step, T - 1})
    return torch.cat([states[t, :2] for t in steps])


def _compare(got, ref, label):
    rgb, depth, body = got
    amb = ref["ambiguous"]
    assert amb.mean() < 0.02, (label, amb.mean())
    same = body == ref["body"]
    bad = ~same & ~amb
    assert not bad.any(), (label, np.argwhere(bad)[:5], body[bad][:5], ref["body"][bad][:5])
    hit = same & (ref["body"] != 0) & (np.abs(ref["ndotd"]) > 0.02)
    rel = np.abs(depth[hit].astype(np.float64) - ref["depth"][hit]) / ref["depth"][hit]
    assert rel.size == 0 or rel.max() <= 1e-4, (label, rel.max())
    assert np.isinf(depth[same & (ref["body"] == 0)]).all(), label
    shade = same & ~ref["shade_ambiguous"]
    diff = np.abs(rgb.astype(int) - ref["rgb"].astype(int)).max(-1)
    assert diff[shade].max(initial=0) <= 1, (label, np.argwhere(shade & (diff > 1))[:5])


@pytest.mark.parametrize("precision", ["f64", "f32"])
@pytest.mark.parametrize("env_id,scale", [("SwingRacket-v0", None), ("Tennisbot-v0", None), ("Tennisbot-v0", 2.5)])
def test_frames_match_the_reference(env_id, scale, precision):
    policy, random = _policy_states(env_id, precision, scale=scale)
    b = TennisBatch(env_id, 4, seed=0, precision=precision)
    if scale is not None:
        b.set_param("racket_scale", scale)
    scene = rr.Scene(b.kind, b.get_param("racket_scale"))
    # the step where the racket of env 0 comes closest to the ball
    st = policy[:, 0].cpu().numpy()
    hit_step = int(np.argmin(np.linalg.norm(st[:, 0:3] - st[:, 13:16], axis=1)))
    recs = torch.cat([_pick(policy, hit_step), _pick(random, random.shape[0] // 3)]).contiguous()
    goals_seen, near = 0, False
    for ci, cam in enumerate(_cameras(env_id)):
        rgb, depth, body = (t.cpu().numpy() for t in b.render(cam, recs, depth=True, body=True))
        for i, rec in enumerate(recs.cpu().numpy()):
            ref = rr.render(scene, cam, rec)
            _compare((rgb[i], depth[i], body[i]), ref, f"{env_id} x{scale} {precision} camera {ci} frame {i}")
            goals_seen += int((ref["body"] == _lib.BODY_GOAL).any())
            near |= bool((body[i] == _lib.BODY_RACKET).any() and (body[i] == _lib.BODY_BALL).any())
    if env_id == "SwingRacket-v0":
        assert goals_seen > 0
    assert near  # some frame shows the racket and the ball together
    b.close()


def _twins(env_id, precision, n=256):
    return [TennisBatch(env_id, n, seed=5, precision=precision) for _ in range(2)]


@pytest.mark.parametrize("precision", ["f64", "f32"])
@pytest.mark.parametrize("env_id", ["SwingRacket-v0", "Tennisbot-v0"])
def test_rendering_is_deterministic_and_leaves_the_env_alone(env_id, precision):
    a, b = _twins(env_id, precision)
    cam = default_camera(env_id, 96, 64)
    a.reset(), b.reset()
    g = torch.Generator("cuda").manual_seed(1)
    for t in range(30):
        act = torch.empty((a.num_envs, a.act_dim), device="cuda").uniform_(-1, 1, generator=g)
        before = a.launch_count()
        f1 = a.render(cam, depth=True, body=True)  # (get_state + render)
        f2 = a.render(cam, a.get_state(), depth=True, body=True)
        assert a.launch_count() - before == 4
        for x, y in zip(f1, f2):
            assert torch.equal(x, y)
        ra = [x.clone() for x in a.step(act)]
        rb = [x.clone() for x in b.step(act)]
        for x, y in zip(ra, rb):
            assert torch.equal(x, y)
    assert torch.equal(a.get_state(), b.get_state())
    np.testing.assert_array_equal(a.read_stats(), b.read_stats())


@pytest.mark.parametrize("precision", ["f64", "f32"])
def test_graph_of_policy_rollout_state_and_render(precision):
    from tennisbot_rl_b200.ppo import load_sb3_policy_npz

    n, cam = 512, default_camera("SwingRacket-v0", 80, 60)
    params = load_sb3_policy_npz(GOLDEN).cuda()

    def setup():
        b = TennisBatch("SwingRacket-v0", n, seed=13, precision=precision)
        b.set_policy(params)
        bufs = dict(obs=torch.zeros((1, n, 6), device="cuda"), rew=torch.zeros((1, n), device="cuda"),
                    done=torch.zeros((1, n), dtype=torch.uint8, device="cuda"), last=torch.zeros((n, 6), device="cuda"))
        bufs["obs"][0].copy_(b.reset())
        return b, bufs

    def iteration(b, bufs):
        b.policy_rollout(bufs["obs"], bufs["rew"], bufs["done"], bufs["last"], noise_seed=3)
        bufs["obs"][0].copy_(bufs["last"])
        return b.render(cam, b.get_state(), depth=True, body=True)

    e, ebufs = setup()
    eager = [[x.clone() for x in iteration(e, ebufs)] for _ in range(4)]
    g_b, gbufs = setup()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):  # warm-up outside the graph = eager iteration 0
        iteration(g_b, gbufs)
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = iteration(g_b, gbufs)
    for k in range(1, 4):
        graph.replay()
        torch.cuda.synchronize()
        for x, y in zip(out, eager[k]):
            assert torch.equal(x, y), k


@pytest.mark.parametrize("env_id", ["SwingRacket-v0", "Tennisbot-v0"])
def test_rows_of_the_state_render_like_the_batch(env_id):
    b = TennisBatch(env_id, 64, seed=2)
    b.reset()
    b.rollout(7)
    cam = default_camera(env_id, 64, 48)
    whole = b.render(cam, depth=True, body=True)
    st = b.get_state()
    m, k = 17, 9
    part = b.render(cam, st[m:m + k].contiguous(), depth=True, body=True)
    for x, y in zip(whole, part):
        assert torch.equal(x[m:m + k], y)


def test_rejections():
    b = TennisBatch("SwingRacket-v0", 4, seed=0)
    L = b.lib
    st = b.get_state()
    rgb = torch.empty((4, 8, 8, 3), dtype=torch.uint8, device="cuda")
    good = Camera(8, 8)

    def call(cam=good, states=st, count=4, out=rgb, raw=None):
        c = raw if raw is not None else cam.to_c()
        before = b.launch_count()
        rc = L.tb_render(b.h, None if c is False else C.byref(c), None if states is None else C.c_void_p(states.data_ptr()),
                         count, None if out is None else C.c_void_p(out.data_ptr()), None, None, b._stream())
        torch.cuda.synchronize()
        assert b.launch_count() - before == (1 if rc == 0 else 0)
        return rc, L.tb_last_error().decode()

    assert call()[0] == 0
    for kwargs, msg in [
        (dict(raw=False), "required"),
        (dict(states=None), "required"),
        (dict(out=None), "required"),
        (dict(count=0), "count"),
        (dict(count=-3), "count"),
        (dict(cam=Camera(0, 8)), "width and height"),
        (dict(cam=Camera(8, 0)), "width and height"),
        (dict(cam=Camera(4097, 8)), "width and height"),
        (dict(cam=Camera(8, 4097)), "width and height"),
        (dict(cam=Camera(8, 8, fov_y_deg=0.0)), "fov_y_deg"),
        (dict(cam=Camera(8, 8, fov_y_deg=180.0)), "fov_y_deg"),
        (dict(cam=Camera(8, 8, fov_y_deg=-10.0)), "fov_y_deg"),
        (dict(cam=Camera(8, 8, fov_y_deg=math.nan)), "fov_y_deg"),
        (dict(cam=Camera(8, 8, fov_y_deg=math.inf)), "fov_y_deg"),
        (dict(cam=Camera(8, 8, eye=(1.0, 2.0, 3.0), target=(1.0, 2.0, 3.0))), "coincide"),
        (dict(cam=Camera(8, 8, eye=(0.0, 0.0, 5.0), target=(0.0, 0.0, 0.0), up=(0.0, 0.0, 1.0))), "parallel"),
        (dict(cam=Camera(8, 8, up=(0.0, 0.0, 0.0))), "parallel"),
        (dict(cam=Camera(4096, 4096), count=2 ** 40), "overflow"),
    ]:
        rc, err = call(**kwargs)
        assert rc != 0 and msg in err and "tb_render" in err, (kwargs, err)
    bad = good.to_c()
    bad.struct_size = 8
    rc, err = call(raw=bad)
    assert rc != 0 and "struct_size" in err
    assert L.tb_render(None, C.byref(good.to_c()), C.c_void_p(st.data_ptr()), 4, C.c_void_p(rgb.data_ptr()), None, None, None) != 0
    with pytest.raises(ValueError):
        b.render(good, st[:, :16].contiguous())
    with pytest.raises(ValueError):
        b.render(good, st.float())


def test_gym_env_frames():
    from tennisbot_rl_b200.envs import SwingRacketEnv, TennisbotEnv

    for cls, env_id in ((SwingRacketEnv, "SwingRacket-v0"), (TennisbotEnv, "Tennisbot-v0")):
        env = cls(seed=4)
        for _ in range(5):
            env.step(env.action_space.sample())
        frame = env.render("rgb_array")
        assert frame.shape == (240, 320, 3) and frame.dtype == np.uint8
        ref, _, _ = env._batch.render(default_camera(env_id), env._batch.get_state())
        np.testing.assert_array_equal(frame, ref[0].cpu().numpy())
        assert env.render() is None and env.render("human") is None
        env.close()


def test_vec_env_frames():
    from tennisbot_rl_b200.vec_env import TennisVecEnv

    cam = Camera(48, 32)
    env = TennisVecEnv("Tennisbot-v0", num_envs=7, seed=1, camera=cam)
    env.reset()
    for _ in range(12):
        env.step(np.random.default_rng(0).uniform(-1, 1, (7, 2)).astype(np.float32))
    imgs = env.get_images()
    ref, _, _ = env.batch.render(cam)
    assert len(imgs) == 7
    for i in range(7):
        np.testing.assert_array_equal(imgs[i], ref[i].cpu().numpy())
    np.testing.assert_array_equal(env.render("rgb_array"), tile_images(imgs))
    assert env.render("human") is None
    env.close()
