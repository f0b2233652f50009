"""SAC under the device VecNormalize: tb_sac_rollout with TB_SAC_VECNORM (sac_kernel<OBS, ACT, true>, the statistics pass after
every step, the entry fold of tb_sac_begin's reset), tb_vecnorm_apply, and GpuSAC(normalize=True), against the float64 numpy
restatement in tests/vecnorm_reference.py, SacActor.kernel_reference and twins stepped with tb_step."""
import numpy as np
import pytest
import torch

from .test_sac_gpu import _ring, host_noise
from .vecnorm_reference import VecNormalizeRef, normalize, record_formula

pytestmark = pytest.mark.gpu

ENVS = ["SwingRacket-v0", "Tennisbot-v0"]
KEYS = ("obs", "act", "reward", "next_obs", "done")


def _ctx(env_id, n, precision="f64", seed=5, actor_seed=3):
    from tennisbot_rl_b200.batch import TennisBatch
    from tennisbot_rl_b200.sac import SacActor, pack_sac_actor

    b = TennisBatch(env_id, n, seed=seed, precision=precision)
    torch.manual_seed(actor_seed)
    actor = SacActor(b.obs_dim, b.act_dim).to(b.device)
    b.set_sac_actor(pack_sac_actor(actor).to(b.device))
    return b, actor


def _host(ring):
    return {k: v.cpu().numpy() for k, v in ring.items()}


def _record(b):
    return b.vecnorm_stats().cpu().numpy()


def _rel_close(got, want, rtol):
    err = np.abs(got - want) / np.maximum(np.abs(want), 1e-300)
    assert err.max() <= rtol, (err.max(), int(err.argmax()), got, want)


def _synthetic_record(od, seed=0):
    """A record far from the fresh one (means of the observations' scale, variances both above and below 1)."""
    rng = np.random.default_rng(seed)
    return np.concatenate([rng.normal(0, 2, od), rng.uniform(0.01, 4, od), [1234.5, 0.7, rng.uniform(0.05, 3), 987.0]])


# ------------------------------------------------------------------------------------------------ statistics and the raw ring
@pytest.mark.parametrize("precision", ["f64", "f32"])
@pytest.mark.parametrize("env_id", ENVS)
def test_record_matches_the_restatement_and_the_ring_is_raw(env_id, precision):
    """4096 envs in three calls (uniform warm-up, sample; tb_sac_begin; sample), episodes ending inside calls: the record after
    each call equals VecNormalizeRef driven by the raw sequence read from the ring within 1e-10 relative, and a twin stepped
    with tb_step on the ring's actions reproduces obs, reward, done and next_obs bit for bit."""
    n = 4096
    calls = [(10, "uniform"), (30, "sample"), (38, "sample")] if env_id == "SwingRacket-v0" else \
        [(100, "uniform"), (500, "sample"), (500, "sample")]
    b, _ = _ctx(env_id, n, precision)
    twin, _ = _ctx(env_id, n, precision)
    od = b.obs_dim
    b.set_vecnorm()
    ref = VecNormalizeRef(n, od)
    ended = 0
    segments = [calls[:2], calls[2:]]  # tb_sac_begin before each: the ring restarts at slot 0
    for seg in segments:
        b.sac_begin()
        ring = _ring(sum(k for k, _ in seg), n, od, b.act_dim, b.device)
        lasts, records = [], []
        for k, mode in seg:
            last = torch.zeros((n, od), device=b.device)
            b.sac_rollout(k, mode, ring, noise_seed=7, last_obs=last, normalize=True)
            lasts.append(last.cpu().numpy())
            records.append(_record(b))
        h = _host(ring)
        tw = twin.reset().cpu().numpy()
        np.testing.assert_array_equal(h["obs"][0], tw)  # raw: the reset observation the first action was computed from
        ref.reset(h["obs"][0])
        j = 0
        for (k, _), last, rec in zip(seg, lasts, records):
            for t in range(k):
                o, r, d, term, _ = twin.step(torch.from_numpy(h["act"][j]).to(b.device))
                o, r, d, term = o.cpu().numpy(), r.cpu().numpy(), d.cpu().numpy(), term.cpu().numpy()
                folded = h["obs"][j + 1] if t + 1 < k else last
                np.testing.assert_array_equal(folded, o)
                np.testing.assert_array_equal(h["reward"][j], r)
                np.testing.assert_array_equal(h["done"][j], d)
                np.testing.assert_array_equal(h["next_obs"][j], np.where(d[:, None] != 0, term, o))
                ref.step(folded, h["reward"][j], h["done"][j])
                ended += int(d.sum())
                j += 1
            _rel_close(rec, ref.record(), 1e-10)
    assert ended > 0
    np.testing.assert_array_equal(b.read_stats(), twin.read_stats())  # the episode statistics stay raw


# ------------------------------------------------------------------------------------------------ the actor's input
@pytest.mark.parametrize("config", ["default", "tiny_clips", "no_norm_obs", "frozen"])
@pytest.mark.parametrize("env_id", ENVS)
def test_actions_act_on_the_normalised_observation(env_id, config):
    """K = 1 per call: the actions equal SacActor.kernel_reference of numpy's normalisation of the raw current observation
    with the record read before the call (bar 1e-4, as test_sac_gpu), for TB_SAC_SAMPLE and TB_SAC_MEAN.  A frozen record
    stays bit-equal."""
    from tennisbot_rl_b200 import _lib

    n, steps = 2048, 30 if env_id == "SwingRacket-v0" else 40
    kw = {"default": {}, "tiny_clips": dict(clip_obs=0.3, clip_reward=0.01), "no_norm_obs": dict(norm_obs=False),
          "frozen": dict(training=False)}[config]
    b, actor = _ctx(env_id, n)
    od, ad = b.obs_dim, b.act_dim
    stats = torch.from_numpy(_synthetic_record(od)).to(b.device) if config == "frozen" else None
    b.set_vecnorm(stats=stats, **kw)
    clip_obs = kw.get("clip_obs", 10.0)
    b.sac_begin()
    ring = _ring(steps + 1, n, od, ad, b.device)
    b.sac_rollout(1, "uniform", ring, noise_seed=5, normalize=True)  # folds the reset observation and the first step
    clipped = 0
    for j in range(1, steps + 1):
        mode = _lib.SAC_SAMPLE if j % 2 else _lib.SAC_MEAN
        before = _record(b)
        b.sac_rollout(1, mode, ring, noise_seed=5, normalize=True)
        raw = ring["obs"][j].cpu().numpy()
        x = record_formula(before, od, raw, 1e-8, clip_obs) if kw.get("norm_obs", True) else raw
        clipped += int((np.abs(x) == np.float32(clip_obs)).sum())
        eps = torch.from_numpy(host_noise(5, np.arange(n), j, ad, True)).cuda() if mode == _lib.SAC_SAMPLE else None
        with torch.no_grad():
            want = actor.kernel_reference(torch.from_numpy(x).cuda(), eps).cpu().numpy()
        got = ring["act"][j].cpu().numpy()
        assert np.abs(got - want).max() <= 1e-4, (j, mode, float(np.abs(got - want).max()))
    if config == "tiny_clips":
        assert clipped > 0
    if config == "frozen":
        np.testing.assert_array_equal(_record(b), stats.cpu().numpy())


# ------------------------------------------------------------------------------------------------ tb_vecnorm_apply
@pytest.mark.parametrize("config", ["default", "tiny_clips", "off"])
@pytest.mark.parametrize("env_id", ENVS)
def test_vecnorm_apply_is_the_formula_bit_for_bit(env_id, config):
    """Observations and rewards equal the numpy float64 formula on the record bit for bit, in place too; norm_* = 0 copies;
    a captured call reads the record as it stands at replay."""
    kw = {"default": {}, "tiny_clips": dict(clip_obs=0.3, clip_reward=0.01), "off": dict(norm_obs=False, norm_reward=False)}[config]
    b, _ = _ctx(env_id, 256)
    od = b.obs_dim
    rec = _synthetic_record(od, 1)
    b.set_vecnorm(stats=torch.from_numpy(rec).to(b.device), **kw)
    clip_obs, clip_rew = kw.get("clip_obs", 10.0), kw.get("clip_reward", 10.0)
    rng = np.random.default_rng(2)
    rows = 5000
    x = (rng.normal(0, 1, (rows, od)) * rng.choice([0.01, 1.0, 100.0], (rows, od))).astype(np.float32)
    r = (rng.normal(0, 1, rows) * rng.choice([0.001, 1.0, 50.0], rows)).astype(np.float32)

    def want(rec):
        if config == "off":
            return x, r
        return normalize(x, rec[:od], rec[od:2 * od], 1e-8, clip_obs), normalize(r, 0.0, rec[2 * od + 2], 1e-8, clip_rew)
    wo, wr = want(rec)
    xd, rd = torch.from_numpy(x).to(b.device), torch.from_numpy(r).to(b.device)
    np.testing.assert_array_equal(b.vecnorm_apply(xd, "obs").cpu().numpy(), wo)
    np.testing.assert_array_equal(b.vecnorm_apply(rd, "reward").cpu().numpy(), wr)
    if config != "off":
        assert (np.abs(wo) == np.float32(clip_obs)).any() and (np.abs(wr) == np.float32(clip_rew)).any()
    xi, ri = xd.clone(), rd.clone()
    b.vecnorm_apply(xi, "obs", out=xi)
    b.vecnorm_apply(ri, "reward", out=ri)
    np.testing.assert_array_equal(xi.cpu().numpy(), wo)
    np.testing.assert_array_equal(ri.cpu().numpy(), wr)
    b.vecnorm_apply(torch.zeros((0, od), device=b.device), "obs")  # zero rows: accepted
    # graph: captured with one record, replayed after the record changed in place
    outs = (torch.empty_like(xd), torch.empty_like(rd))
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        b.vecnorm_apply(xd, "obs", out=outs[0])
        b.vecnorm_apply(rd, "reward", out=outs[1])
    rec2 = _synthetic_record(od, 3)
    b.set_vecnorm(stats=torch.from_numpy(rec2).to(b.device), **kw)
    g.replay()
    torch.cuda.synchronize()
    wo2, wr2 = want(rec2)
    np.testing.assert_array_equal(outs[0].cpu().numpy(), wo2)
    np.testing.assert_array_equal(outs[1].cpu().numpy(), wr2)


# ------------------------------------------------------------------------------------------------ without the flag, graphs
@pytest.mark.parametrize("env_id", ENVS)
def test_without_the_flag_nothing_changes(env_id):
    """A context with a training normaliser attached, rolled out without TB_SAC_VECNORM, is bit-equal to one that never had a
    normaliser (ring, state, statistics), and its record stays the fresh one."""
    n, od = 2048, 6 if env_id == "SwingRacket-v0" else 12
    fresh = np.concatenate([np.zeros(od), np.ones(od), [1e-4, 0.0, 1.0, 1e-4]])
    outs = []
    for attach in (True, False):
        b, _ = _ctx(env_id, n)
        if attach:
            b.set_vecnorm()
        b.sac_begin()
        ring = _ring(40, n, od, b.act_dim, b.device)
        last = torch.zeros((n, od), device=b.device)
        for k, mode in ((5, "uniform"), (15, "sample"), (20, "mean")):
            b.sac_rollout(k, mode, ring, noise_seed=2, last_obs=last)
        torch.cuda.synchronize()
        outs.append((_host(ring), last.cpu().numpy(), b.get_state().cpu().numpy(), b.read_stats()))
        if attach:
            np.testing.assert_array_equal(_record(b), fresh)
    (ra, la, sa, sta), (rb, lb, sb, stb) = outs
    for key in KEYS:
        np.testing.assert_array_equal(ra[key], rb[key], err_msg=key)
    np.testing.assert_array_equal(la, lb)
    np.testing.assert_array_equal(sa, sb)
    np.testing.assert_array_equal(sta, stb)


@pytest.mark.parametrize("env_id", ENVS)
def test_graph_replays_equal_eager_calls(env_id):
    """A captured flagged rollout (the first after tb_sac_begin, so replay 1 folds the reset) replayed 3 times equals 3 eager
    calls bit for bit: ring, record, state, statistics."""
    n, K = 2048, 4
    outs = []
    for graph in (False, True):
        b, _ = _ctx(env_id, n)
        b.set_vecnorm()
        b.sac_begin()
        ring = _ring(3 * K, n, b.obs_dim, b.act_dim, b.device)
        torch.cuda.synchronize()
        if graph:
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                b.sac_rollout(K, "sample", ring, noise_seed=3, normalize=True)
            for _ in range(3):
                g.replay()
        else:
            for _ in range(3):
                b.sac_rollout(K, "sample", ring, noise_seed=3, normalize=True)
        torch.cuda.synchronize()
        outs.append((_host(ring), _record(b), b.get_state().cpu().numpy(), b.read_stats()))
    (r0, v0, s0, st0), (r1, v1, s1, st1) = outs
    for key in KEYS:
        np.testing.assert_array_equal(r1[key], r0[key], err_msg=key)
    np.testing.assert_array_equal(v1, v0)
    np.testing.assert_array_equal(s1, s0)
    np.testing.assert_array_equal(st1, st0)


# ------------------------------------------------------------------------------------------------ launch counts, rejections
@pytest.mark.parametrize("precision", ["f32", "f64"])
@pytest.mark.parametrize("env_id", ENVS)
def test_launch_counts_and_the_entry_fold(env_id, precision):
    """(K + 1) + K s launches frozen or without the flag, + 2 K + 3 training; tb_sac_begin 1; tb_vecnorm_apply 1.  The reset is
    folded once after each tb_sac_begin (obs count), every step folds N observations and N returns."""
    n, K = 256, 3
    s = 2 if env_id == "SwingRacket-v0" else 1
    b, _ = _ctx(env_id, n, precision)
    od = b.obs_dim
    ring = _ring(8, n, od, b.act_dim, b.device)

    def launches(call):
        before = b.launch_count()
        call()
        torch.cuda.synchronize()
        return b.launch_count() - before

    counts = lambda: _record(b)[[2 * od, 2 * od + 3]]  # noqa: E731
    b.set_vecnorm()
    assert launches(lambda: b.sac_begin()) == 1
    want = np.array([1e-4, 1e-4])
    for first, mode in ((True, "uniform"), (False, "sample"), (False, "mean")):
        assert launches(lambda: b.sac_rollout(K, mode, ring, normalize=True)) == (K + 1) + K * s + 2 * K + 3
        want += [(n if first else 0) + K * n, K * n]
        np.testing.assert_array_equal(counts(), want)
    assert launches(lambda: b.sac_rollout(K, "sample", None)) == (K + 1) + K * s  # no flag: the record does not move
    np.testing.assert_array_equal(counts(), want)
    assert launches(lambda: b.sac_begin()) == 1
    assert launches(lambda: b.sac_rollout(K, "sample", None, normalize=True)) == (K + 1) + K * s + 2 * K + 3
    want += [n + K * n, K * n]
    np.testing.assert_array_equal(counts(), want)
    assert launches(lambda: b.vecnorm_apply(torch.zeros((5, od), device=b.device), "obs")) == 1
    assert launches(lambda: b.vecnorm_apply(torch.zeros(0, device=b.device), "reward")) == 1
    frozen = b.vecnorm_stats().clone()
    b.set_vecnorm(training=False, stats=frozen)
    b.sac_begin()
    for mode in ("uniform", "sample", "mean"):
        assert launches(lambda: b.sac_rollout(K, mode, ring, normalize=True)) == (K + 1) + K * s
    np.testing.assert_array_equal(_record(b), frozen.cpu().numpy())


@pytest.mark.parametrize("env_id", ENVS)
def test_rejections(env_id):
    from tennisbot_rl_b200 import _lib

    b, _ = _ctx(env_id, 256)
    od = b.obs_dim
    L = _lib.load()
    err = _lib.TennisbotLibraryError
    x = torch.zeros((4, od), device=b.device)
    b.sac_begin()
    with pytest.raises(err, match="tb_set_vecnorm"):
        b.sac_rollout(1, "sample", None, normalize=True)
    with pytest.raises(err, match="no normaliser"):
        b.vecnorm_apply(x, "obs")
    b.set_vecnorm()
    b.sac_rollout(1, "sample", None, normalize=True)
    for mode in (3 | _lib.SAC_VECNORM, 0x200, _lib.SAC_VECNORM | 0x200):
        with pytest.raises(err, match="unknown mode"):
            b.sac_rollout(1, mode, None)

    def msg(rc):
        assert rc != 0
        return L.tb_last_error().decode()
    s = b._stream()
    assert "d_in and d_out" in msg(L.tb_vecnorm_apply(b.h, None, 4, _lib.VECNORM_OBS, x.data_ptr(), s))
    assert "d_in and d_out" in msg(L.tb_vecnorm_apply(b.h, x.data_ptr(), 4, _lib.VECNORM_OBS, None, s))
    assert "rows" in msg(L.tb_vecnorm_apply(b.h, x.data_ptr(), -1, _lib.VECNORM_OBS, x.data_ptr(), s))
    assert "rows" in msg(L.tb_vecnorm_apply(b.h, x.data_ptr(), 2 ** 62, _lib.VECNORM_REWARD, x.data_ptr(), s))
    assert "unknown what" in msg(L.tb_vecnorm_apply(b.h, x.data_ptr(), 4, 2, x.data_ptr(), s))
    assert "context is NULL" in msg(L.tb_vecnorm_apply(None, x.data_ptr(), 4, _lib.VECNORM_OBS, x.data_ptr(), s))
    b.clear_vecnorm()
    with pytest.raises(err, match="tb_set_vecnorm"):
        b.sac_rollout(1, "uniform", None, normalize=True)
    assert "no normaliser" in msg(L.tb_vecnorm_apply(b.h, x.data_ptr(), 4, _lib.VECNORM_OBS, x.data_ptr(), s))


# ------------------------------------------------------------------------------------------------ GpuSAC
def test_save_deploys_as_the_evaluation_context(tmp_path):
    """GpuSAC(normalize=True).save -> load_vecnormalize_npz -> a frozen TB_SAC_MEAN rollout on a fresh context reproduces the
    evaluation context's episode (its raw return sum over 512 envs, exactly), and both records stay the training record."""
    from tennisbot_rl_b200.batch import TennisBatch
    from tennisbot_rl_b200.ppo import load_vecnormalize_npz
    from tennisbot_rl_b200.sac import GpuSAC, pack_sac_actor

    s = GpuSAC("SwingRacket-v0", num_envs=1024, batch_size=256, gradient_steps=2, slots=64, seed=3, eval_envs=512,
               normalize=True)
    out = s.train(20)  # ends with an evaluation: the evaluation context's first episode of every env (26 steps)
    path = tmp_path / "sac.npz"
    s.save(path)
    w = np.load(path)
    np.testing.assert_array_equal(w["policy"], pack_sac_actor(s.actor).cpu().numpy())
    stats, cfg = load_vecnormalize_npz(path, 6)
    rec = _record(s.env)
    np.testing.assert_array_equal(stats.numpy(), rec)
    assert cfg["gamma"] == s.gamma and rec[12] > 1024 * 21  # the reset and every step folded
    t = TennisBatch("SwingRacket-v0", 512, seed=s.seed + 1000, precision="f64")
    t.set_sac_actor(torch.from_numpy(w["policy"]).to(t.device))
    t.set_vecnorm(training=False, stats=stats.to(t.device), **cfg)
    t.sac_begin()
    t.read_stats(clear=True)
    t.sac_rollout(26, "mean", None, normalize=True)
    st = t.read_stats()
    assert int(st[0]) == 512
    assert float(st[6] / 2 ** 20 / st[0]) == out["eval_mean_return"]
    np.testing.assert_array_equal(_record(t), rec)
    np.testing.assert_array_equal(_record(s._eval), rec)


# measured on a B200: DESIGN.md section 4.2.  The bars are those of the unnormalised runs' tests (18: the ES bar).
SWING_BAR, SWING_ITERS = 18.0, 5000
HIT_ITERS = 4000


def test_gpu_sac_learns_swing_with_normalize():
    from tennisbot_rl_b200.sac import GpuSAC

    s = GpuSAC("SwingRacket-v0", seed=0, normalize=True)
    out = s.train(SWING_ITERS, log=print, eval_every=SWING_ITERS // 5)
    curve = [(e["env_steps"], round(e["eval_mean_return"], 2)) for e in out["evaluations"]]
    print(f"SwingRacket-v0 SAC normalize: evaluations {curve}, collect {out['collect_s']:.1f}s update {out['update_s']:.1f}s "
          f"wall {out['wall_s']:.1f}s (unnormalised 28.5, ES bar 18)")
    assert out["eval_mean_return"] >= SWING_BAR


def test_gpu_sac_improves_tennisbot_with_normalize():
    from tennisbot_rl_b200.sac import GpuSAC

    s = GpuSAC("Tennisbot-v0", num_envs=256, slots=4096, seed=0, eval_envs=512, normalize=True)
    first = s.evaluate()
    out = s.train(HIT_ITERS, log=print, eval_every=HIT_ITERS // 4)
    ev = [first] + [e["eval_mean_return"] for e in out["evaluations"]]
    print(f"Tennisbot-v0 SAC normalize: evaluations {[round(v, 2) for v in ev]}")
    assert ev[-1] > first, ev
