"""The kernel launches each entry point adds to tb_launch_count (bench.py's gpu_launches), for both envs and both precisions.
An env step is s launches: step_kernel, and for SwingRacket-v0 also ff_kernel (s = 2, Tennisbot-v0 s = 1)."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

N, INDIVIDUALS, K = 256, 8, 3


@pytest.mark.parametrize("precision", ["f32", "f64"])
@pytest.mark.parametrize("env_id", ["SwingRacket-v0", "Tennisbot-v0"])
def test_launches_per_entry_point(env_id, precision, monkeypatch):
    from tennisbot_rl_b200 import _lib
    from tennisbot_rl_b200.batch import TennisBatch

    b = TennisBatch(env_id, N, seed=3, precision=precision)
    s = 2 if env_id == "SwingRacket-v0" else 1
    od, ad = b.obs_dim, b.act_dim
    floats = _lib.ES_FLOATS if b.kind == _lib.ENV_SWING else _lib.ES_FLOATS_HIT
    pol_floats = _lib.POLICY_FLOATS if b.kind == _lib.ENV_SWING else _lib.POLICY_FLOATS_HIT
    dev = b.device
    rng = np.random.default_rng(0)
    f32 = lambda *shape: torch.from_numpy(rng.uniform(-0.1, 0.1, shape).astype(np.float32)).to(dev)  # noqa: E731

    def launches(call):
        before = b.launch_count()
        call()
        torch.cuda.synchronize()
        return b.launch_count() - before

    assert launches(lambda: b.reset()) == 1
    assert launches(lambda: b.reset_host()) == 1
    actions = f32(N, ad)
    assert launches(lambda: b.step(actions)) == s
    for mode in ("zero_copy", "staging"):
        monkeypatch.setenv("TB_HOST_MODE", mode)
        assert launches(lambda: b.step_host(rng.uniform(-1, 1, (N, ad)))) == s, mode
    monkeypatch.delenv("TB_HOST_MODE")
    assert launches(lambda: b.rollout(K)) == 1
    state = b.get_state()
    assert launches(lambda: b.get_state()) == 1
    assert launches(lambda: b.set_state(state)) == 1

    assert launches(lambda: b.set_policy(f32(pol_floats))) == 0
    obs = torch.zeros((K, N, od), dtype=torch.float32, device=dev)
    obs[0] = b.reset()
    out = dict(reward=torch.zeros((K, N), device=dev), done=torch.zeros((K, N), dtype=torch.uint8, device=dev),
               last_obs=torch.zeros((N, od), device=dev))
    assert launches(lambda: b.policy_rollout(obs, **out)) == K * (1 + s)
    obs[0] = out["last_obs"]
    last_value = torch.zeros(N, device=dev)
    assert launches(lambda: b.policy_rollout(obs, **out, last_value=last_value)) == K * (1 + s) + 1

    assert launches(lambda: b.es_begin(f32(INDIVIDUALS, floats))) == 3
    assert launches(lambda: b.es_begin_noise(f32(floats), INDIVIDUALS, 0.05, 1, 0)) == 3
    ret, alive = torch.zeros(N, dtype=torch.float64, device=dev), torch.zeros(N, dtype=torch.uint8, device=dev)
    assert launches(lambda: b.es_rollout(K, ret, alive)) == (K + 1) + K * s
    dirs, coef = torch.arange(4, dtype=torch.int64, device=dev), f32(4)
    assert launches(lambda: b.es_noise_combine(dirs, coef, 1, 0)) == 1
    assert launches(lambda: b.es_normalizer_stats()) == 2
    b.close()
