"""tb_trace_step without a GPU: the substep bound the header states, against a walk of env_substep's step-counter rule, and
the recorder's flight option."""
import re
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent


@pytest.fixture(scope="module")
def lib():
    from tennisbot_rl_b200 import _lib, build

    build.build_library()
    return _lib.load()


def substeps_without_landing(s0, done):
    """Substeps of one SwingRacket-v0 env step from step counters s0 when the ball never lands (the longest case):
    env_substep's phase 0 ends the step when its counter k = s0 + 1 is <= 25 or the env is done; the fast-forward substeps
    after it end the step at the time-out, the first k > 800."""
    s0 = np.asarray(s0, np.int64)
    k = s0 + 1
    n = np.ones_like(s0)
    flying = (k > 25) & ~np.asarray(done, bool)
    while flying.any():
        k = np.where(flying, k + 1, k)
        n = np.where(flying, n + 1, n)
        flying &= ~(k > 800)
    return n


def test_bound_of_the_flight(lib):
    from tennisbot_rl_b200 import _lib

    s0 = np.arange(-50, 1200)
    longest = max(int(substeps_without_landing(s0, False).max()), int(substeps_without_landing(s0, True).max()))
    assert longest == 776 == _lib.TRACE_MAX_SUBSTEPS
    assert int(np.argmax(substeps_without_landing(s0, False))) == 50 + 25  # the 26th step of an episode
    assert lib.tb_trace_max_substeps(_lib.ENV_SWING) == 776
    assert lib.tb_trace_max_substeps(_lib.ENV_HIT) == 1
    assert lib.tb_trace_max_substeps(7) == -1 and lib.tb_trace_max_substeps(-1) == -1
    header = (ROOT / "include" / "tennisbot_b200.h").read_text()
    assert int(re.search(r"#define TB_TRACE_MAX_SUBSTEPS (\d+)", header).group(1)) == 776


def test_recorder_offers_flight_frames():
    out = subprocess.run([sys.executable, str(ROOT / "tools" / "record_episode.py"), "--help"], capture_output=True, text=True,
                         check=True).stdout
    assert "--flight-every" in out
