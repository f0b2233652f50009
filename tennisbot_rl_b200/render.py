"""Cameras for tb_render (TennisBatch.render) and the tiling SB3's VecEnv.render applies to get_images().

The reference's PyBullet camera (tennisbot_env.py:269-279) is not recorded in this repository, so the default cameras
below are chosen here: each looks across the court at the region where its env places the racket.
"""
from dataclasses import dataclass

import numpy as np

from . import _lib


@dataclass(frozen=True)
class Camera:
    """A pinhole camera in the world frame (metres); see tb_render in include/tennisbot_b200.h for the ray of each pixel."""
    width: int = 320
    height: int = 240
    eye: tuple = (16.0, -10.0, 5.0)
    target: tuple = (4.0, 0.0, 0.5)
    up: tuple = (0.0, 0.0, 1.0)
    fov_y_deg: float = 50.0

    def to_c(self):
        c = _lib.TbCamera()
        c.struct_size = _lib.C.sizeof(_lib.TbCamera)
        c.width, c.height, c.reserved = int(self.width), int(self.height), 0
        c.eye[:], c.target[:], c.up[:] = (tuple(float(x) for x in v) for v in (self.eye, self.target, self.up))
        c.fov_y_deg = float(self.fov_y_deg)
        return c


# SwingRacket-v0 places the racket at x in [5.5, 11], y in [-4, 4] and the goal at x in [-12, -3] (swingracket_env.py:161-173):
# from beside the racket's half of the court, the swing in front and the goal beyond the net.  Tennisbot-v0 places the racket
# at x in [7.5, 12.5], y in [-5, 5] and shoots the ball from x in [-12, -6] (tennisbot_env.py:227-246): a lower view of the
# racket's half, the ball coming over the net.
_DEFAULTS = {
    _lib.ENV_SWING: dict(eye=(16.5, -7.5, 3.5), target=(6.0, 0.0, 0.5), fov_y_deg=55.0),
    _lib.ENV_HIT: dict(eye=(16.0, -7.0, 2.5), target=(8.0, 0.0, 0.6), fov_y_deg=55.0),
}


def default_camera(env_id, width=320, height=240):
    """The default camera of an env id ('SwingRacket-v0' / 'Tennisbot-v0', or the TB_ENV_* value)."""
    from .batch import ENV_IDS

    kind = ENV_IDS[env_id] if isinstance(env_id, str) else int(env_id)
    return Camera(width=int(width), height=int(height), **_DEFAULTS[kind])


def tile_images(images):
    """N images [H, W, C] -> one image: a grid of ceil(sqrt(N)) rows and ceil(N / rows) columns, filled row by row, empty
    cells black (what SB3's VecEnv.render shows)."""
    imgs = np.asarray(images)
    n, h, w, c = imgs.shape
    rows = int(np.ceil(np.sqrt(n)))
    cols = int(np.ceil(n / rows))
    grid = np.zeros((rows * cols, h, w, c), imgs.dtype)
    grid[:n] = imgs
    return grid.reshape(rows, cols, h, w, c).transpose(0, 2, 1, 3, 4).reshape(rows * h, cols * w, c)
