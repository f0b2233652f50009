"""Batched VecEnv adapter: N lock-step envs on one B200 behind the stable-baselines3 `VecEnv` contract.

SB3 is not a dependency (it is absent from this image): when it is importable the class derives from
`stable_baselines3.common.vec_env.VecEnv`, otherwise from a small stand-in with the same abstract surface, so
`PPO("MlpPolicy", TennisVecEnv(...))` works wherever SB3 exists and the contract is testable where it does not.

Contract kept (SB3 1.8, the version recorded in backup_models/ppo_swing.zip):
  reset() -> float32 [N, obs];  step_async(actions[N, act]);  step_wait() -> (obs, rewards f32[N], dones bool[N], infos)
  auto-reset on done with infos[i]["terminal_observation"], infos[i]["episode"] = {"r", "l", "t"} (VecMonitor
  semantics).  The reference registers both envs WITHOUT max_episode_steps and returns an empty info dict, so SB3 treats
  the 800 / 1000-step time-outs as terminations (no bootstrap from the terminal value); infos[i]["TimeLimit.truncated"] is
  therefore only emitted on request (report_truncation=True).  infos[i]["events"] always carries the event bits.
Returned arrays are fresh copies (SB3 keeps `_last_obs` across the next step).
Frames: get_images() renders every env on the device through the `camera` constructor keyword (default:
render.default_camera(env_id), 320 x 240) and copies them to the host, so its cost grows with N; render("rgb_array") tiles
them as SB3's VecEnv.render does, which is what VecVideoRecorder records.
"""
import time

import numpy as np

from . import _lib
from .batch import TennisBatch
from .render import default_camera, tile_images
from .spaces import spaces_for

try:
    from stable_baselines3.common.vec_env import VecEnv as _VecEnvBase

    _HAVE_SB3 = True
except Exception:
    _HAVE_SB3 = False

    class _VecEnvBase:  # the subset of VecEnv's constructor / helpers SB3 algorithms rely on
        def __init__(self, num_envs, observation_space, action_space):
            self.num_envs = num_envs
            self.observation_space = observation_space
            self.action_space = action_space
            self.render_mode = None

        def step(self, actions):
            self.step_async(actions)
            return self.step_wait()

        def _get_indices(self, indices):
            if indices is None:
                return list(range(self.num_envs))
            if isinstance(indices, int):
                return [indices]
            return list(indices)

        @property
        def unwrapped(self):
            return self


class TennisVecEnv(_VecEnvBase):
    def __init__(self, env_id="SwingRacket-v0", num_envs=4096, device=0, seed=0, precision="f64", env_id_offset=0,
                 report_truncation=False, camera=None):
        obs_space, act_space = spaces_for(env_id)
        self.report_truncation = bool(report_truncation)
        self._pending_scale = None
        super().__init__(num_envs, obs_space, act_space)
        self.env_id = env_id
        self.batch = TennisBatch(env_id, num_envs, device=device, seed=seed, precision=precision, auto_reset=True,
                                 env_id_offset=env_id_offset)
        self._actions = None
        self._ep_ret = np.zeros(num_envs, np.float64)
        self._ep_len = np.zeros(num_envs, np.int64)
        self._t0 = time.time()
        self.racket_scale = 1.0
        self.metadata = {"render.modes": ["human", "rgb_array"]}
        self.camera = camera or default_camera(env_id)

    # ---------------------------------------------------------------- VecEnv API
    def reset(self):
        if self._pending_scale is not None:
            self.batch.set_param("racket_scale", self._pending_scale)
            self._pending_scale = None
        obs = self.batch.reset_host()
        self._ep_ret[:] = 0
        self._ep_len[:] = 0
        return obs.copy()

    def step_async(self, actions):
        a = np.asarray(actions, dtype=np.float32)
        if a.shape != (self.num_envs, self.batch.act_dim):
            raise ValueError(f"actions must have shape ({self.num_envs}, {self.batch.act_dim}), got {a.shape}")
        self._actions = a

    def step_wait(self):
        hb = self.batch.step_host(self._actions)
        obs, rew = hb["obs"].copy(), hb["reward"].copy()
        dones = hb["done"].astype(bool)
        self._ep_ret += rew
        self._ep_len += 1
        infos = [{} for _ in range(self.num_envs)]
        idx = np.nonzero(dones)[0]
        if idx.size:
            ev = hb["events"]
            term = hb["terminal_obs"]
            now = round(time.time() - self._t0, 6)
            ended_by_env = _lib.EV_COURT_BALL | _lib.EV_GOAL_BALL | _lib.EV_BALL_PASSED
            # (one bulk conversion per column: in lock-step SwingRacket every env ends on the same step, and a Python-level
            # numpy scalar access per field costs more than the env step itself at 16 384 envs)
            evs = ev[idx].astype(np.int64)
            trunc = (((evs & _lib.EV_TIMEOUT) != 0) & ((evs & ended_by_env) == 0)).tolist()
            rows = term[idx].copy()
            for k, (i, r, l, e, t) in enumerate(zip(idx.tolist(), self._ep_ret[idx].tolist(), self._ep_len[idx].tolist(),
                                                    evs.tolist(), trunc)):
                infos[i] = {"terminal_observation": rows[k], "episode": {"r": r, "l": l, "t": now}, "events": e}
                if self.report_truncation:
                    infos[i]["TimeLimit.truncated"] = t
            self._ep_ret[idx] = 0
            self._ep_len[idx] = 0
        return obs, rew, dones, infos

    def close(self):
        self.batch.close()

    def seed(self, seed=None):
        """Placement streams are keyed by (seed, global env id, episode) at construction; returns the per-env seeds."""
        return [seed] * self.num_envs

    def get_attr(self, attr_name, indices=None):
        n = len(self._get_indices(indices))
        return [getattr(self, attr_name)] * n

    def set_attr(self, attr_name, value, indices=None):
        setattr(self, attr_name, value)

    def env_method(self, method_name, *method_args, indices=None, **method_kwargs):
        n = len(self._get_indices(indices))
        return [getattr(self, method_name)(*method_args, **method_kwargs)] * n

    def env_is_wrapped(self, wrapper_class, indices=None):
        return [False] * len(self._get_indices(indices))

    def get_images(self):
        """N uint8 [H, W, 3] frames of the envs' current states, rendered on the device (one launch for all N) and copied to
        the host once."""
        rgb, _, _ = self.batch.render(self.camera)
        return list(rgb.cpu().numpy())

    def render(self, mode="human"):
        """mode "rgb_array": get_images() tiled into one image (SB3's VecEnv.render); "human" returns None (no GUI)."""
        if mode != "rgb_array":
            return None
        return tile_images(self.get_images())

    # ---------------------------------------------------------------- reference-specific hooks
    def set_racket_scale(self, scale, apply_now=False):
        """TennisbotEnv.set_racket_scale for the whole batch (train.py:155-176 calls it through the env).  As in the reference
        (tennisbot_env.py:213-215,234) the scale is only stored here and takes effect at the next reset(): the hull, its
        inertia and the COM offset are scene-wide in the kernels, so applying it at once would change the geometry under
        every episode in flight (apply_now=True does exactly that, for scripted use)."""
        self.racket_scale = float(scale)
        if apply_now:
            self.batch.set_param("racket_scale", self.racket_scale)
            self._pending_scale = None
        else:
            self._pending_scale = self.racket_scale

    def episode_statistics(self, clear=False):
        return stats_dict(self.batch.read_stats(clear=clear))


def stats_dict(vec):
    """Readable view of the int64[10] statistics vector (include/tennisbot_b200.h TB_STAT_*)."""
    v = [int(x) for x in vec]
    eps = max(v[0], 1)
    mean = v[6] / 1048576.0 / eps
    return {
        "episodes": v[0], "mean_length": v[1] / eps, "racket_hits": v[2], "goals": v[3], "court": v[4],
        "timeouts": v[5], "mean_return": mean, "std_return": max(v[7] / 1024.0 / eps - mean * mean, 0.0) ** 0.5,
        "physics_steps": v[8], "env_steps": v[9],
    }
