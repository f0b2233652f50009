"""SAC under the device VecNormalize, without a GPU: TB_SAC_VECNORM, TB_VECNORM_OBS / TB_VECNORM_REWARD and tb_vecnorm_apply's
declaration against _lib, and TennisBatch's argument checks that run before the library is called."""
import re
import shutil
import subprocess
from pathlib import Path

import pytest
import torch

from tennisbot_rl_b200 import _lib

ROOT = Path(__file__).resolve().parent.parent


def test_constants_match_the_header(tmp_path):
    cc = shutil.which("gcc") or shutil.which("cc")
    if cc is None:
        pytest.skip("no C compiler")
    src = tmp_path / "sv.c"
    src.write_text('#include <stdio.h>\n#include "tennisbot_b200.h"\n'
                   'int main(void) { printf("%d %d %d %d %d %d", TB_SAC_VECNORM, TB_VECNORM_OBS, TB_VECNORM_REWARD, TB_SAC_SAMPLE, '
                   'TB_SAC_MEAN, TB_SAC_UNIFORM); return 0; }\n')
    exe = tmp_path / "sv"
    subprocess.run([cc, "-I", str(ROOT / "include"), str(src), "-o", str(exe)], check=True)
    got = [int(x) for x in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    assert got == [_lib.SAC_VECNORM, _lib.VECNORM_OBS, _lib.VECNORM_REWARD, _lib.SAC_SAMPLE, _lib.SAC_MEAN, _lib.SAC_UNIFORM]
    assert got[0] == 0x100
    for m in (_lib.SAC_SAMPLE, _lib.SAC_MEAN, _lib.SAC_UNIFORM):  # a flag bit: OR'd into any mode, it leaves the mode readable
        assert m & _lib.SAC_VECNORM == 0 and (m | _lib.SAC_VECNORM) & ~_lib.SAC_VECNORM == m
    text = (ROOT / "include" / "tennisbot_b200.h").read_text()
    assert re.search(r"int tb_vecnorm_apply\(tb_ctx \*ctx, const float \*d_in, int64_t rows, int what, float \*d_out, "
                     r"void \*stream\);", text)
    assert _lib.SIGNATURES["tb_vecnorm_apply"] == [_lib._vp, _lib._vp, _lib._i64, _lib._i32, _lib._vp, _lib._vp]


class _Stub:
    """A TennisBatch without a context: the host-side checks run, and a call that reaches the library records its arguments."""

    def __init__(self, obs_dim=6, act_dim=6, n=8):
        from tennisbot_rl_b200.batch import TennisBatch

        self.b = TennisBatch.__new__(TennisBatch)
        self.calls = []
        b = self.b
        b.h, b.obs_dim, b.act_dim, b.num_envs, b.device = None, obs_dim, act_dim, n, torch.device("cpu")
        b._stream = lambda: None
        stub = self

        class Lib:
            def tb_vecnorm_apply(self, *a):
                stub.calls.append(("tb_vecnorm_apply", a))
                return 0

            def tb_sac_rollout(self, *a):
                stub.calls.append(("tb_sac_rollout", a))
                return 0
        b.lib = Lib()


def test_vecnorm_apply_checks_its_buffers():
    s = _Stub()
    b = s.b
    x = torch.zeros(5, 6)
    with pytest.raises(ValueError, match="what"):
        b.vecnorm_apply(x, "action")
    with pytest.raises(ValueError, match="shape"):
        b.vecnorm_apply(torch.zeros(5, 4), "obs")
    with pytest.raises(ValueError, match="shape"):
        b.vecnorm_apply(torch.zeros(5, 6), "reward")
    with pytest.raises(ValueError, match="float32"):
        b.vecnorm_apply(torch.zeros(5, 6, dtype=torch.float64), "obs")
    with pytest.raises(ValueError, match="out"):
        b.vecnorm_apply(x, "obs", out=torch.zeros(4, 6))
    with pytest.raises(ValueError, match="contiguous"):
        b.vecnorm_apply(torch.zeros(6, 5).t(), "obs")
    assert s.calls == []
    assert b.vecnorm_apply(x, "obs", out=x) is x
    r = torch.zeros(7)
    out = b.vecnorm_apply(r, _lib.VECNORM_REWARD)
    assert out.shape == (7,) and out is not r
    (n0, a0), (n1, a1) = s.calls
    assert n0 == n1 == "tb_vecnorm_apply"
    assert (a0[2], a0[3]) == (5, _lib.VECNORM_OBS) and a0[1].value == a0[4].value == x.data_ptr()
    assert (a1[2], a1[3]) == (7, _lib.VECNORM_REWARD)


def test_sac_rollout_ors_the_flag_into_the_mode():
    s = _Stub()
    for mode, normalize, want in (("sample", False, _lib.SAC_SAMPLE), ("mean", True, _lib.SAC_MEAN | _lib.SAC_VECNORM),
                                  ("uniform", True, _lib.SAC_UNIFORM | _lib.SAC_VECNORM)):
        s.calls.clear()
        s.b.sac_rollout(3, mode, None, normalize=normalize)
        assert s.calls[0][1][1:3] == (3, want)
