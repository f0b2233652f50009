"""The device VecNormalize's host side, without a GPU: tb_vecnorm against the header, load_vecnormalize_npz, GpuPPO's refusal
of the eager arm, and the numpy restatement (tests/vecnorm_reference.py) against a hand-computed two-batch Chan merge."""
import ctypes
import re
import shutil
import subprocess
from pathlib import Path

import numpy as np
import pytest

from tennisbot_rl_b200 import _lib
from tennisbot_rl_b200.ppo import VECNORMALIZE_KEYS, load_vecnormalize_npz

from .vecnorm_reference import RunningMeanStd, VecNormalizeRef, normalize

ROOT = Path(__file__).resolve().parent.parent
FIELDS = ("struct_size", "training", "norm_obs", "norm_reward", "clip_obs", "clip_reward", "gamma", "epsilon")


def test_vecnorm_struct_matches_the_header(tmp_path):
    cc = shutil.which("gcc") or shutil.which("cc")
    if cc is None:
        pytest.skip("no C compiler")
    src = tmp_path / "vn.c"
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "tennisbot_b200.h"\n'
                   'int main(void) { printf("%zu %d %d", sizeof(tb_vecnorm), TB_VECNORM_WORDS(6), TB_VECNORM_WORDS(12));\n'
                   + "".join(f'printf(" %zu", offsetof(tb_vecnorm, {f}));\n' for f in FIELDS) + "return 0; }\n")
    exe = tmp_path / "vn"
    subprocess.run([cc, "-I", str(ROOT / "include"), str(src), "-o", str(exe)], check=True)
    got = [int(x) for x in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    T = _lib.TbVecNorm
    assert got == [ctypes.sizeof(T), _lib.vecnorm_words(6), _lib.vecnorm_words(12)] + [getattr(T, f).offset for f in FIELDS]
    assert got[1:3] == [16, 28]
    text = (ROOT / "include" / "tennisbot_b200.h").read_text()
    assert re.search(r"int tb_set_vecnorm\(tb_ctx \*ctx, const tb_vecnorm \*cfg, const double \*d_stats, void \*stream\);", text)
    assert re.search(r"int tb_get_vecnorm\(tb_ctx \*ctx, double \*d_stats, void \*stream\);", text)


def _write(path, **over):
    rec = dict(obs_mean=np.arange(6.0), obs_var=np.full(6, 2.0), obs_count=100.0, ret_mean=0.5, ret_var=3.0, ret_count=99.0,
               clip_obs=10.0, clip_reward=5.0, gamma=0.95, epsilon=1e-8)
    rec.update(over)
    np.savez(path, **{k: v for k, v in rec.items() if v is not None})
    return path


def test_load_vecnormalize_npz(tmp_path):
    stats, cfg = load_vecnormalize_npz(_write(tmp_path / "ok.npz"), obs_dim=6)
    assert stats.dtype.is_floating_point and stats.numpy().dtype == np.float64
    np.testing.assert_array_equal(stats.numpy(), np.concatenate([np.arange(6.0), np.full(6, 2.0), [100.0, 0.5, 3.0, 99.0]]))
    assert cfg == {"clip_obs": 10.0, "clip_reward": 5.0, "gamma": 0.95, "epsilon": 1e-8}
    for key in VECNORMALIZE_KEYS:
        with pytest.raises(ValueError, match="missing"):
            load_vecnormalize_npz(_write(tmp_path / f"no_{key}.npz", **{key: None}))
    with pytest.raises(ValueError, match="shape"):
        load_vecnormalize_npz(_write(tmp_path / "od.npz"), obs_dim=12)
    with pytest.raises(ValueError, match="shape"):
        load_vecnormalize_npz(_write(tmp_path / "var.npz", obs_var=np.ones(5)))
    with pytest.raises(ValueError, match="scalars"):
        load_vecnormalize_npz(_write(tmp_path / "cnt.npz", obs_count=np.ones(2)))


def test_normalize_needs_the_fused_policy():
    from tennisbot_rl_b200.ppo import GpuPPO

    with pytest.raises(ValueError, match="fused_policy"):
        GpuPPO("SwingRacket-v0", 8, 4, fused_policy=False, normalize=True)


def test_restatement_against_a_hand_computed_chan_merge():
    a = np.array([[1.0, -2.0], [3.0, 0.0], [5.0, 4.0]], np.float32)
    b = np.array([[0.5, 1.0], [-1.5, 7.0]], np.float32)
    rms = RunningMeanStd((2,))
    rms.update(a)
    rms.update(b)
    # by hand: the fresh record (mean 0, var 1, count 1e-4) merged with a, then with b
    c0, n1 = 1e-4, 3.0
    m1 = a.mean(0, dtype=np.float64)
    t1 = c0 + n1
    mean1 = m1 * n1 / t1
    var1 = (1.0 * c0 + a.var(0, dtype=np.float64) * n1 + m1 ** 2 * c0 * n1 / t1) / t1
    n2 = 2.0
    d2 = b.mean(0, dtype=np.float64) - mean1
    t2 = t1 + n2
    np.testing.assert_allclose(rms.mean, mean1 + d2 * n2 / t2, rtol=1e-15)
    np.testing.assert_allclose(rms.var, (var1 * t1 + b.var(0, dtype=np.float64) * n2 + d2 ** 2 * t1 * n2 / t2) / t2, rtol=1e-15)
    assert rms.count == t2
    # with tiny counts the merge is the statistics of all five rows
    allrows = np.concatenate([a, b]).astype(np.float64)
    np.testing.assert_allclose(rms.mean, allrows.mean(0), rtol=1e-4)
    np.testing.assert_allclose(rms.var, allrows.var(0), rtol=1e-4)


def test_restatement_returns_and_formulas():
    ref = VecNormalizeRef(3, 2, gamma=0.5, clip_reward=0.75)
    ref.reset(np.zeros((3, 2), np.float32))
    r1 = ref.step(np.ones((3, 2), np.float32), np.array([1.0, 2.0, 4.0], np.float32), np.array([0, 1, 0], np.uint8))
    np.testing.assert_array_equal(ref.returns, [1.0, 0.0, 4.0])  # done envs' returns are zeroed after the fold
    assert ref.ret_rms.count == 1e-4 + 3
    np.testing.assert_array_equal(r1, normalize([1.0, 2.0, 4.0], 0.0, ref.ret_rms.var, 1e-8, 0.75))
    assert np.abs(r1).max() == np.float32(0.75)
    ref.step(np.ones((3, 2), np.float32), np.array([2.0, 2.0, 2.0], np.float32), np.zeros(3, np.uint8))
    np.testing.assert_array_equal(ref.returns, [2.5, 2.0, 4.0])
    ref.reset(None, mask=[1, 0, 0])
    np.testing.assert_array_equal(ref.returns, [0.0, 2.0, 4.0])
    frozen = VecNormalizeRef(3, 2, training=False, record=ref.record())
    before = frozen.record().copy()
    frozen.step(np.ones((3, 2), np.float32), np.ones(3, np.float32), np.zeros(3, np.uint8))
    np.testing.assert_array_equal(frozen.record(), before)
