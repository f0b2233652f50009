"""Per-agent VecNormalize records of a PPO population, host side (no GPU): the C ABI's new entry points, PopulationPPO's
argument check, the record's npz entries and the PBT row copy of a record buffer."""
import re
from pathlib import Path

import numpy as np
import pytest
import torch

from tennisbot_rl_b200 import _lib
from tennisbot_rl_b200.population import PopulationPPO, exploit_explore
from tennisbot_rl_b200.ppo import VECNORMALIZE_KEYS, load_vecnormalize_npz, vecnormalize_entries

HEADER = (Path(__file__).resolve().parent.parent / "include" / "tennisbot_b200.h").read_text()


@pytest.mark.parametrize("name,params", [
    ("tb_set_vecnorms", "tb_ctx *ctx, const tb_vecnorm *cfg, int64_t agents, const double *d_stats, void *stream"),
    ("tb_get_vecnorms", "tb_ctx *ctx, double *d_stats, int64_t agents, void *stream"),
    ("tb_vecnorm_device_ptr", "tb_ctx *ctx, double **d_records, int64_t *agents"),
])
def test_header_declares_the_record_entry_points(name, params):
    m = re.search(r"int " + name + r"\(([^)]*)\);", HEADER)
    assert m and " ".join(m.group(1).split()) == params
    assert len(_lib.SIGNATURES[name]) == params.count(",") + 1


def test_policy_rollout_raw_is_policy_rollout_plus_the_raw_reward():
    def args(name):
        m = re.search(r"int " + name + r"\(([^)]*)\);", HEADER)
        return [a.split()[-1].lstrip("*") for a in " ".join(m.group(1).split()).split(", ")]

    base, raw = args("tb_policy_rollout"), args("tb_policy_rollout_raw")
    assert raw == base[:9] + ["d_raw_reward"] + base[9:]
    assert len(_lib.SIGNATURES["tb_policy_rollout_raw"]) == len(_lib.SIGNATURES["tb_policy_rollout"]) + 1


def test_mixed_gammas_are_refused_with_normalize():
    with pytest.raises(ValueError, match="one gamma"):
        PopulationPPO("SwingRacket-v0", 2, 4, 4, gamma=[0.99, 0.95], normalize=True)


@pytest.mark.parametrize("od", (6, 12))
def test_record_entries_round_trip_through_the_npz(tmp_path, od):
    rng = np.random.default_rng(od)
    rec = np.concatenate([rng.normal(size=od), rng.uniform(0.1, 2, od), [123.0001, 0.3, 4.5, 77.0001]])
    for record in (rec, torch.from_numpy(rec)):
        e = vecnormalize_entries(record, 0.97)
        assert set(e) == set(VECNORMALIZE_KEYS)
        np.savez(tmp_path / "a.npz", **e)
        stats, cfg = load_vecnormalize_npz(tmp_path / "a.npz", od)
        np.testing.assert_array_equal(stats.numpy(), rec)
        assert cfg == {"clip_obs": 10.0, "clip_reward": 10.0, "gamma": 0.97, "epsilon": 1e-8}


def test_pbt_copies_a_record_row_bit_for_bit():
    P, words = 4, _lib.vecnorm_words(12)
    rec = torch.from_numpy(np.random.default_rng(1).normal(size=(P, words)))
    before = rec.clone()
    hyper = {"lr": torch.full((P,), 3e-4), "ent_coef": torch.full((P,), 0.002)}
    (dst, src, _), = exploit_explore([1.0, 4.0, 2.0, 3.0], [rec], hyper, np.random.default_rng(0))
    assert (dst, src) == (0, 1)
    assert torch.equal(rec[dst], before[src])
    assert torch.equal(rec[1:], before[1:])
