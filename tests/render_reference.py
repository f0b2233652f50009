"""Float64 numpy restatement of tb_render (include/tennisbot_b200.h): the shapes, the camera, the shading.

The scene comes from tb_scene_constant and racket_scale (tb_get_param), so it follows the same parameter the kernel reads.
Every pixel is cast three times: as specified, with every shape grown by delta and with every shape shrunk by delta,
delta = 1e-4 x the distance along the ray (for a plane: where the ray crosses it, i.e. c + s n.d <= +-1e-4 s; for the
sphere: 1e-4 x the distance of its centre).  A pixel whose grown and shrunk casts see different bodies is ambiguous: float32
rounding in the kernel may land it on either side.
"""
import numpy as np

from tennisbot_rl_b200 import _lib

REL = 1e-4
S_RACKET_POS, S_RACKET_QUAT, S_BALL_POS, S_GOAL = 0, 3, 13, 25


def _outward_planes(poly):
    """CCW polygon [K, 2] -> unit outward edge normals [K, 2] and offsets h (n.p <= h inside)."""
    e = np.roll(poly, -1, axis=0) - poly
    n = np.stack([e[:, 1], -e[:, 0]], 1) / np.hypot(e[:, 0], e[:, 1])[:, None]
    return n, np.einsum("ij,ij->i", n, poly)


class Scene:
    def __init__(self, env_kind, racket_scale=1.0):
        sc = _lib.scene_constant
        s = float(racket_scale)
        k = int(sc("racket_outline_n"))
        poly = np.array([[sc("racket_outline_y", i), sc("racket_outline_z", i)] for i in range(k)])
        self.racket_n, self.racket_h = _outward_planes(s * (poly - [0.0, sc("racket_com_z")]))
        self.racket_ht = s * sc("racket_half_x")
        g = int(sc("goal_sides"))
        self.goal_n, self.goal_h = _outward_planes(np.array([[sc("goal_vertex_x", i), sc("goal_vertex_y", i)] for i in range(g)]))
        self.goal_hz = sc("goal_half_z")
        self.with_goal = env_kind == _lib.ENV_SWING
        self.floor_h = np.array([sc("floor_hx"), sc("floor_hy"), sc("floor_hz")])
        self.net_h = np.array([sc("net_hx"), sc("net_hy"), sc("net_hz")])
        self.ball_r = sc("ball_radius")


def ray_directions(cam):
    """[H, W, 3] unit ray directions of camera `cam` (render.Camera)."""
    eye, target, up = (np.asarray(v, np.float64) for v in (cam.eye, cam.target, cam.up))
    f = target - eye
    f /= np.linalg.norm(f)
    r = np.cross(f, up)
    r /= np.linalg.norm(r)
    u = np.cross(r, f)
    t = np.tan(np.radians(cam.fov_y_deg) / 2)
    w, h = cam.width, cam.height
    a = (2 * (np.arange(w) + 0.5) / w - 1) * t * w / h
    b = (1 - 2 * (np.arange(h) + 0.5) / h) * t
    d = f + a[None, :, None] * r + b[:, None, None] * u
    return d / np.linalg.norm(d, axis=-1, keepdims=True)


def quat_to_mat(q):
    x, y, z, w = q
    return np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w)],
                     [2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w)],
                     [2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)]])


def _clip(c, m, d, eps):
    """Entry distance [R] and entry-plane normal [R, 3] of the convex body {p : m_i.(p - eye) + c_i <= 0 along the ray} for rays
    d [R, 3]; planes grown by eps x the crossing distance."""
    den = d @ m.T - eps
    with np.errstate(divide="ignore", invalid="ignore"):
        s = -c[None, :] / den
    enter = np.where(den < 0, s, -np.inf)
    leave = np.where(den > 0, s, np.inf)
    s0, face = enter.max(1), enter.argmax(1)
    s1 = leave.min(1)
    s1 = np.where(((den == 0) & (c[None, :] > 0)).any(1), -np.inf, s1)
    return np.where((s0 > 0) & (s0 < s1), s0, np.inf), m[face]


def _box(h, eye, d, eps):
    m = np.concatenate([np.eye(3), -np.eye(3)])
    c = np.concatenate([eye - h, -eye - h])
    return _clip(c, m, d, eps)


def _shapes(scene, rec, eye, d, eps):
    """Entry distance and normal of every body, in TB_BODY_* order (court, net, goal, racket, ball)."""
    out = [_box(scene.floor_h, eye, d, eps), _box(scene.net_h, eye, d, eps)]
    if scene.with_goal:
        gx, gy = rec[S_GOAL], rec[S_GOAL + 1]
        m = np.concatenate([[[0, 0, 1.0], [0, 0, -1.0]], np.c_[scene.goal_n, np.zeros(len(scene.goal_h))]])
        c = np.concatenate([[eye[2] - scene.goal_hz, -eye[2] - scene.goal_hz], scene.goal_n @ (eye[:2] - [gx, gy]) - scene.goal_h])
        out.append(_clip(c, m, d, eps))
    else:
        out.append((np.full(len(d), np.inf), np.zeros((len(d), 3))))
    R = quat_to_mat(rec[S_RACKET_QUAT:S_RACKET_QUAT + 4])
    ol = R.T @ (eye - rec[S_RACKET_POS:S_RACKET_POS + 3])
    ml = np.concatenate([[[1.0, 0, 0], [-1.0, 0, 0]], np.c_[np.zeros(len(scene.racket_h)), scene.racket_n]])
    c = np.concatenate([[ol[0] - scene.racket_ht, -ol[0] - scene.racket_ht], scene.racket_n @ ol[1:] - scene.racket_h])
    out.append(_clip(c, ml @ R.T, d, eps))
    cb = rec[S_BALL_POS:S_BALL_POS + 3] - eye
    r = scene.ball_r + eps * np.linalg.norm(cb)
    b = d @ cb
    q2 = np.sum((cb[None, :] - b[:, None] * d) ** 2, 1)
    with np.errstate(invalid="ignore"):
        s = b - np.sqrt(r * r - q2)
    s = np.where((q2 <= r * r) & (s > 0), s, np.inf)
    out.append((s, (np.where(np.isfinite(s), s, 0)[:, None] * d - cb) / r))
    return out


def _cast(scene, rec, eye, d, eps):
    shapes = _shapes(scene, rec, eye, d, eps)
    dist = np.stack([s for s, _ in shapes])  # [5, R]
    k = dist.argmin(0)  # first minimum: equal distances go to the lower body id
    depth = dist[k, np.arange(len(d))]
    body = np.where(np.isfinite(depth), k + 1, _lib.BODY_NONE)
    normal = np.stack([n for _, n in shapes])[k, np.arange(len(d))]
    return body, depth, normal


def render(scene, cam, rec):
    """One frame of the record `rec` (float64 [32]): dict of rgb uint8 [H, W, 3], depth float64 [H, W], body uint8 [H, W],
    ndotd float64 [H, W] (n.d of the surface hit; 0 for sky), ambiguous bool [H, W] and shade_ambiguous bool [H, W] (also where
    the grown and shrunk casts enter the same body through different faces: next to a box's or a prism's edge)."""
    rec = np.asarray(rec, np.float64)
    eye = np.asarray(cam.eye, np.float64)
    d = ray_directions(cam).reshape(-1, 3)
    body, depth, n = _cast(scene, rec, eye, d, 0.0)
    grown, _, n_grown = _cast(scene, rec, eye, d, REL)
    shrunk, _, n_shrunk = _cast(scene, rec, eye, d, -REL)
    nd = np.einsum("ij,ij->i", n, d)
    n = np.where(nd[:, None] > 0, -n, n)
    light = np.asarray(_lib.RENDER_LIGHT, np.float64)
    light /= np.linalg.norm(light)
    k = 0.35 + 0.65 * np.maximum(0.0, n @ light)
    colors = np.asarray(_lib.RENDER_COLORS, np.float64)
    rgb = np.floor(colors[body] * k[:, None] + 0.5)
    rgb[body == _lib.BODY_NONE] = _lib.RENDER_SKY
    shape = (cam.height, cam.width)
    return dict(rgb=rgb.astype(np.uint8).reshape(*shape, 3), depth=depth.reshape(shape), body=body.astype(np.uint8).reshape(shape),
                ndotd=np.where(body == 0, 0.0, nd).reshape(shape), ambiguous=(grown != shrunk).reshape(shape),
                shade_ambiguous=((grown != shrunk) | ((grown != _lib.BODY_BALL) &  # (a sphere's normal moves smoothly)
                                             (np.abs(n_grown - n_shrunk).max(1) > 1e-3))).reshape(shape))


def record(racket_pos=(0, 0, -100), racket_quat=(0, 0, 0, 1), ball_pos=(0, 0, -100), goal=(-100, 0)):
    """A canonical state record with the given racket pose, ball position and goal (every other word 0)."""
    rec = np.zeros(_lib.STATE_WORDS)
    rec[S_RACKET_POS:S_RACKET_POS + 3] = racket_pos
    rec[S_RACKET_QUAT:S_RACKET_QUAT + 4] = racket_quat
    rec[S_BALL_POS:S_BALL_POS + 3] = ball_pos
    rec[S_GOAL:S_GOAL + 2] = goal
    return rec
