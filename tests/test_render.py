"""tb_render's contract without a GPU: the numpy reference against closed forms, the ctypes camera struct against the header,
and the host side of the gym / VecEnv frames (tiling, get_images) through a fake batch."""
import ctypes
import math
import shutil
import subprocess
from pathlib import Path

import numpy as np
import pytest
import torch

from tennisbot_rl_b200 import _lib, vec_env
from tennisbot_rl_b200.render import Camera, default_camera, tile_images
from tests import render_reference as rr

ROOT = Path(__file__).resolve().parent.parent


@pytest.fixture(scope="module")
def scene(lib):
    return rr.Scene(_lib.ENV_SWING)


@pytest.fixture(scope="module")
def lib():
    from tennisbot_rl_b200 import build

    build.build_library()
    return _lib.load()


def test_depth_of_the_empty_court_from_above(scene):
    h = 7.0
    cam = Camera(width=33, height=21, eye=(5.0, 2.0, h), target=(5.0, 2.0, 0.0), up=(0.0, 1.0, 0.0), fov_y_deg=40.0)
    f = rr.render(scene, cam, rr.record())
    assert f["body"][10, 16] == _lib.BODY_COURT
    assert f["depth"][10, 16] == pytest.approx(h - scene.floor_h[2], rel=1e-12)
    assert (f["body"] == _lib.BODY_COURT).all()


def test_ball_on_the_view_axis(scene):
    d, fov, size = 3.0, 30.0, 201
    eye = np.array([4.0, -2.0, 1.5])
    cam = Camera(width=size, height=size, eye=tuple(eye), target=(4.0, 5.0, 1.5), up=(0.0, 0.0, 1.0), fov_y_deg=fov)
    f = rr.render(scene, cam, rr.record(ball_pos=eye + [0.0, d, 0.0]))
    c = size // 2
    assert f["body"][c, c] == _lib.BODY_BALL
    assert f["depth"][c, c] == pytest.approx(d - scene.ball_r, rel=1e-12)
    radius = (size / 2) * math.tan(math.asin(scene.ball_r / d)) / math.tan(math.radians(fov) / 2)
    row = f["body"][c] == _lib.BODY_BALL
    assert abs(row.sum() / 2 - radius) <= 1
    assert np.nonzero(row)[0].mean() == pytest.approx(c, abs=0.5)


def test_net_seen_face_on(scene):
    e, fov, size = 20.0, 60.0, 301
    cam = Camera(width=size, height=size, eye=(e, 0.0, 0.3), target=(0.0, 0.0, 0.3), up=(0.0, 0.0, 1.0), fov_y_deg=fov)
    f = rr.render(scene, cam, rr.record())
    t = math.tan(math.radians(fov) / 2)
    c = size // 2
    half = (size / 2) * scene.net_h[1] / ((e - scene.net_h[0]) * t)
    row = f["body"][c] == _lib.BODY_NET
    assert abs(row.sum() / 2 - half) <= 1
    assert f["depth"][c, c] == pytest.approx(e - scene.net_h[0], rel=1e-12)
    above = (size / 2) * (scene.net_h[2] - 0.3) / ((e - scene.net_h[0]) * t)  # rows of net above the centre row
    col = f["body"][:c, c] == _lib.BODY_NET
    assert abs(col.sum() - above) <= 1
    assert (f["rgb"][0, 0] == _lib.RENDER_SKY).all() and not f["ambiguous"][c, c]


def test_racket_scale_grows_the_racket(scene):
    cam = default_camera("Tennisbot-v0", 96, 72)
    rec = rr.record(racket_pos=(9.0, 0.0, 0.7))
    small = (rr.render(rr.Scene(_lib.ENV_HIT, 1.0), cam, rec)["body"] == _lib.BODY_RACKET).sum()
    big = (rr.render(rr.Scene(_lib.ENV_HIT, 2.5), cam, rec)["body"] == _lib.BODY_RACKET).sum()
    assert 0 < small and big > 4 * small


def test_camera_struct_matches_the_header(tmp_path):
    cc = shutil.which("gcc") or shutil.which("cc")
    if cc is None:
        pytest.skip("no C compiler")
    src = tmp_path / "cam.c"
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "tennisbot_b200.h"\n'
                   'int main(void) { printf("%zu", sizeof(tb_camera));\n'
                   + "".join(f'printf(" %zu", offsetof(tb_camera, {f}));\n' for f in
                             ("struct_size", "width", "height", "reserved", "eye", "target", "up", "fov_y_deg"))
                   + "return 0; }\n")
    exe = tmp_path / "cam"
    subprocess.run([cc, "-I", str(ROOT / "include"), str(src), "-o", str(exe)], check=True)
    got = [int(x) for x in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    T = _lib.TbCamera
    assert got == [ctypes.sizeof(T)] + [getattr(T, f).offset for f in
                                        ("struct_size", "width", "height", "reserved", "eye", "target", "up", "fov_y_deg")]


def test_tile_images():
    imgs = [np.full((3, 4, 3), i + 1, np.uint8) for i in range(5)]
    big = tile_images(imgs)
    assert big.shape == (3 * 3, 2 * 4, 3)  # ceil(sqrt(5)) = 3 rows, 2 columns
    assert (big[0:3, 0:4] == 1).all() and (big[0:3, 4:8] == 2).all() and (big[3:6, 0:4] == 3).all()
    assert (big[6:9, 0:4] == 5).all() and (big[6:9, 4:8] == 0).all()
    assert tile_images(imgs[:1]).shape == (3, 4, 3)


class _FrameBatch:
    """Stands in for TennisBatch in TennisVecEnv: frames whose pixels carry the env index."""

    def __init__(self, env_id, num_envs, **kwargs):
        self.num_envs, self.act_dim = num_envs, 6
        self.cameras = []

    def render(self, camera, states=None, depth=False, body=False):
        self.cameras.append(camera)
        rgb = torch.arange(self.num_envs, dtype=torch.uint8).reshape(-1, 1, 1, 1).expand(-1, camera.height, camera.width, 3)
        return rgb.contiguous(), None, None


def test_vec_env_frames(monkeypatch):
    monkeypatch.setattr(vec_env, "TennisBatch", _FrameBatch)
    env = vec_env.TennisVecEnv("SwingRacket-v0", num_envs=6)
    assert "rgb_array" in env.metadata["render.modes"]
    assert env.camera == default_camera("SwingRacket-v0")
    imgs = env.get_images()
    assert len(imgs) == 6 and all(im.shape == (240, 320, 3) and im.dtype == np.uint8 for im in imgs)
    assert [int(im[0, 0, 0]) for im in imgs] == list(range(6))
    big = env.render("rgb_array")
    np.testing.assert_array_equal(big, tile_images(imgs))
    assert big.shape == (3 * 240, 2 * 320, 3)
    assert env.render() is None and env.render("human") is None
    cam = Camera(width=16, height=8)
    env = vec_env.TennisVecEnv("Tennisbot-v0", num_envs=2, camera=cam)
    assert env.get_images()[1].shape == (8, 16, 3) and env.batch.cameras == [cam]
