"""Single-env classes with the reference's gym 0.21 API, backed by a CUDA batch of one.

Mirrors `tennisbot/envs/swingracket_env.py` and `tennisbot/envs/tennisbot_env.py` of the reference: same class
names, constructor kwargs, spaces, `reset()` -> obs, `step(a)` -> (obs, reward, done, {}), `seed`, `close`,
`render`, `metadata`, and `TennisbotEnv.set_racket_scale`.  `render("rgb_array")` returns a frame drawn on the device
(tb_render); `render()` / `render("human")` return None, since there is no GUI.  Every number comes from the sm_100a
kernel through the C ABI; without the compiled library or a B200 the constructor raises.
"""
import numpy as np

from . import _lib
from .spaces import hit_spaces, swing_spaces

try:  # subclass the real gym.Env when it exists so isinstance checks in SB3 / wrappers pass
    import gym as _gym

    _EnvBase = _gym.Env
except Exception:  # gym is not in this image
    try:
        import gymnasium as _gym

        _EnvBase = _gym.Env
    except Exception:
        _EnvBase = object


class _SingleEnv(_EnvBase):
    metadata = {"render.modes": ["human"]}
    _env_id = None

    def __init__(self, device=0, precision="f64", seed=None):
        from .batch import TennisBatch

        self._batch = TennisBatch(self._env_id, 1, device=device, seed=0, precision=precision, auto_reset=False)
        self._rng = np.random.default_rng(seed)
        self.done = False
        self.last_events = 0

    # -- gym API
    def seed(self, seed=None):
        """The reference's seed() only re-creates an unused np_random (swingracket_env.py:147-149); here it seeds the
        generator that draws the reset placement, which is what a caller expects it to do."""
        self._rng = np.random.default_rng(seed)
        return [seed]

    def close(self):
        if getattr(self, "_batch", None) is not None:
            self._batch.close()
            self._batch = None

    def render(self, mode="human", camera=None):
        """mode "rgb_array": uint8 [H, W, 3] of the current state through `camera` (default: render.default_camera of this env,
        320 x 240), drawn on the device.  Any other mode returns None: the env is headless."""
        if mode != "rgb_array":
            return None
        from .render import default_camera

        rgb, _, _ = self._batch.render(camera or default_camera(self._env_id))
        return rgb[0].cpu().numpy()

    @property
    def step_count(self):
        """Physics steps since reset (the reference's self.step_count), read from the device state."""
        return int(self._batch.get_state()[0, _S_STEP].item())

    def state(self):
        """Canonical 32-word state record (include/tennisbot_b200.h TB_S_*) of this env."""
        return self._batch.get_state()[0].cpu().numpy()

    def _draw_placement(self):
        raise NotImplementedError

    def _format_obs(self, row):
        raise NotImplementedError

    def reset(self):
        init = np.zeros((1, _lib.INIT_WORDS))
        init[0] = self._draw_placement()
        obs = self._batch.reset(init=init).cpu().numpy()[0]
        self.done = False
        return self._format_obs(obs)

    def step(self, action):
        a = np.asarray(action, dtype=np.float32).reshape(1, self._batch.act_dim)
        hb = self._batch.step_host(a)
        reward = float(hb["reward"][0])
        self.done = bool(hb["done"][0])
        self.last_events = int(hb["events"][0])
        return self._format_obs(hb["obs"][0].copy()), reward, self.done, dict()


_S_STEP = 29  # TB_S_STEP of the canonical state record


class SwingRacketEnv(_SingleEnv):
    """`gym.make('SwingRacket-v0', use_gui=False, delay_mode=False)` (swingracket_env.py:25-61)."""
    _env_id = "SwingRacket-v0"

    def __init__(self, use_gui=False, delay_mode=False, device=0, precision="f64", seed=None):
        if use_gui:
            raise NotImplementedError("use_gui=True needs the PyBullet GUI; the CUDA env is headless")
        self.observation_space, self.action_space = swing_spaces()
        self.delay_mode = delay_mode
        super().__init__(device=device, precision=precision, seed=seed)
        self.reset()  # the reference constructor resets itself (:61)

    def _draw_placement(self):
        r = self._rng
        # swingracket_env.py:161-173: racket base, goal = (uniform(-3,-12), uniform(-5,5))
        return [r.uniform(5.5, 11), r.uniform(-4, 4), 0.6, -3.0 - 9.0 * r.uniform(0, 1), r.uniform(-5, 5), 0, 0, 0]

    def _format_obs(self, row):
        self.goal = (float(row[4]), float(row[5]))
        return tuple(float(x) for x in row)  # the reference returns a 6-tuple of Python floats (:143-144)


class TennisbotEnv(_SingleEnv):
    """`gym.make('Tennisbot-v0', use_gui=False, is_sparse_reward=False)` (tennisbot_env.py:33-88)."""
    _env_id = "Tennisbot-v0"

    def __init__(self, use_gui=False, is_sparse_reward=False, device=0, precision="f64", seed=None):
        if use_gui:
            raise NotImplementedError("use_gui=True needs the PyBullet GUI; the CUDA env is headless")
        self.observation_space, self.action_space = hit_spaces()
        self.is_sparse_reward = is_sparse_reward
        self.racket_scale = 1.0
        super().__init__(device=device, precision=precision, seed=seed)
        self.reset()

    def set_racket_scale(self, scale):
        """Curriculum hook of train.py:155-176; takes effect at the next reset like the reference's (:213-215,234)."""
        self.racket_scale = float(scale)

    def reset(self):
        if self._batch.get_param("racket_scale") != self.racket_scale:
            self._batch.set_param("racket_scale", self.racket_scale)
        return super().reset()

    def _draw_placement(self):
        r = self._rng
        # tennisbot_env.py:227-246
        return [r.uniform(7.5, 12.5), r.uniform(-5, 5), r.uniform(0.2, 0.21), r.uniform(25, 37.5), r.uniform(-10, 10),
                r.uniform(-12, -6), r.uniform(-1, 1), r.uniform(1, 1.5)]

    def _format_obs(self, row):
        return np.asarray(row, dtype=np.float32)


ENV_CLASSES = {"SwingRacket-v0": SwingRacketEnv, "Tennisbot-v0": TennisbotEnv}


def make(env_id, **kwargs):
    """gym.make for the two ids, usable without gym installed."""
    return ENV_CLASSES[env_id](**kwargs)
