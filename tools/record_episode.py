"""Record episodes as PNG frames: M envs stepped for E episodes, every env step rendered on the device (tb_render) into one
[T, M, H, W, 3] buffer that is copied to the host once, then written as frames and a contact sheet.

Action sources: uniform random (default); the scripted ball tracker (--tracker, Tennisbot-v0); or a policy in tb_set_policy's
layout, rolled by tb_policy_rollout with K = 1 (--policy: a .npy flat vector, or an .npz of an SB3 MlpPolicy state dict such
as the reference's trained policy tests/golden/ppo_swing_policy.npz, or GpuPPO.save's npz).  A policy trained under VecNormalize
acts on normalised observations: --vecnormalize FILE attaches that record, frozen (ppo.load_vecnormalize_npz's keys; a
GpuPPO.save npz of a normalize=True run holds them too).  Frames exist per env step: a SwingRacket-v0 episode is
26 frames, and its 26th step fast-forwards the ball's whole flight (about 106 physics substeps, at most 776).  With
--flight-every K that step is also traced substep by substep (tb_trace_step, from the states saved before it and the actions
it took), and every K-th flight substep plus the last is drawn between frame 25 and the episode's final frame.

  python tools/record_episode.py SwingRacket-v0 --policy tests/golden/ppo_swing_policy.npz --out frames/swing
  python tools/record_episode.py SwingRacket-v0 --policy tests/golden/ppo_swing_policy.npz --flight-every 4 --out frames/shot
  python tools/record_episode.py Tennisbot-v0 --tracker --out frames/hit
  python tools/record_episode.py Tennisbot-v0 --policy run.npz --vecnormalize run.npz --out frames/hit_norm
"""
import argparse
import struct
import sys
import zlib
from pathlib import Path

import numpy as np
import torch

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
from tennisbot_rl_b200 import _lib  # noqa: E402
from tennisbot_rl_b200.batch import TennisBatch  # noqa: E402
from tennisbot_rl_b200.render import default_camera  # noqa: E402

SWING_STEPS = 26  # env steps of a SwingRacket-v0 episode (25 control steps + the fast-forward)


def write_png(path, rgb):
    """uint8 [H, W, 3] -> an 8-bit RGB PNG (stdlib zlib; filter type 0 on every row)."""
    h, w, _ = rgb.shape
    raw = b"".join(b"\x00" + rgb[y].tobytes() for y in range(h))

    def chunk(tag, data):
        return struct.pack(">I", len(data)) + tag + data + struct.pack(">I", zlib.crc32(tag + data) & 0xFFFFFFFF)

    Path(path).write_bytes(b"\x89PNG\r\n\x1a\n" + chunk(b"IHDR", struct.pack(">IIBBBBB", w, h, 8, 2, 0, 0, 0)) +
                           chunk(b"IDAT", zlib.compress(raw, 6)) + chunk(b"IEND", b""))


def load_policy(path):
    if path.suffix == ".npz":
        from tennisbot_rl_b200.ppo import load_sb3_policy_npz

        w = np.load(path)
        if "policy" in w:  # GpuPPO.save
            return torch.from_numpy(np.ascontiguousarray(w["policy"], np.float32))
        return load_sb3_policy_npz(path)
    return torch.from_numpy(np.load(path).astype(np.float32))


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("env_id", choices=["SwingRacket-v0", "Tennisbot-v0"])
    ap.add_argument("--envs", type=int, default=4, help="M envs, each a column of the contact sheet")
    ap.add_argument("--episodes", type=int, default=1, help="E episodes (Tennisbot-v0: --steps env steps per episode)")
    ap.add_argument("--steps", type=int, default=450, help="Tennisbot-v0: env steps per recorded episode")
    ap.add_argument("--tracker", action="store_true", help="Tennisbot-v0: the scripted ball tracker (TB_ACT_TRACK)")
    ap.add_argument("--policy", type=Path, help=".npy parameter vector or .npz SB3 MlpPolicy state dict")
    ap.add_argument("--vecnormalize", type=Path, help="with --policy: the VecNormalize record (npz) it was trained under")
    ap.add_argument("--stochastic", action="store_true", help="sample the policy's actions instead of taking the mean")
    ap.add_argument("--width", type=int, default=320)
    ap.add_argument("--height", type=int, default=240)
    ap.add_argument("--precision", default="f64")
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--racket-scale", type=float, default=1.0)
    ap.add_argument("--out", type=Path, default=Path("frames"))
    ap.add_argument("--sheet-every", type=int, default=0, help="contact sheet: every k-th frame (0: about 13 rows)")
    ap.add_argument("--flight-every", type=int, default=0,
                    help="SwingRacket-v0: also draw every k-th substep of the ball's flight in the 26th step (0: none)")
    a = ap.parse_args()
    if a.flight_every < 0:
        ap.error("--flight-every must be >= 0")
    if a.tracker and a.env_id != "Tennisbot-v0":
        ap.error("--tracker is Tennisbot-v0's scripted tracker")
    if a.tracker and a.policy:
        ap.error("--tracker and --policy are two action sources")
    if a.vecnormalize and not a.policy:
        ap.error("--vecnormalize normalises a --policy's observations")

    m = a.envs
    swing = a.env_id == "SwingRacket-v0"
    # a swing episode is exactly 26 env steps: without auto-reset its last frame shows its own end (the ball on the court)
    b = TennisBatch(a.env_id, m, seed=a.seed, precision=a.precision, auto_reset=not swing)
    b.set_param("racket_scale", a.racket_scale)
    cam = default_camera(a.env_id, a.width, a.height)
    per_episode = SWING_STEPS if swing else a.steps
    T = a.episodes * per_episode
    frames = []  # device frames [M, H, W, 3], copied to the host together at the end
    obs = torch.zeros((1, m, b.obs_dim), device=b.device)
    if a.policy:
        b.set_policy(load_policy(a.policy).to(b.device))
        if a.vecnormalize:  # frozen: the statistics the policy was trained with
            from tennisbot_rl_b200.ppo import load_vecnormalize_npz

            stats, cfg = load_vecnormalize_npz(a.vecnormalize, b.obs_dim)
            b.set_vecnorm(training=False, stats=stats.to(b.device), **cfg)
        rew, done = torch.zeros((1, m), device=b.device), torch.zeros((1, m), dtype=torch.uint8, device=b.device)
        last = torch.zeros((m, b.obs_dim), device=b.device)
        act = torch.zeros((1, m, b.act_dim), device=b.device)
    gen = torch.Generator(b.device).manual_seed(a.seed)
    flight_frames = 0
    for t in range(T):
        if t == 0 or (swing and t % per_episode == 0):  # a new episode: its first frame is the placement
            obs[0].copy_(b.reset())
            frames.append(b.render(cam)[0])
        flight = swing and a.flight_every > 0 and t % per_episode == per_episode - 1
        if flight:
            before = b.get_state()
        if a.policy:
            b.policy_rollout(obs, rew, done, last, actions=act, deterministic=not a.stochastic, noise_seed=a.seed)
            obs[0].copy_(last)  # raw, also with a normaliser (obs[0] now holds the normalised observation)
            taken = act[0].clamp(-1, 1)  # policy_rollout returns the unclipped action; the env step took it clipped
        elif a.tracker:
            b.rollout(1, _lib.ACT_TRACK)
        else:
            taken = torch.empty((m, b.act_dim), device=b.device).uniform_(-1, 1, generator=gen)
            b.step(taken)
        if flight:  # the flight inside this step: every k-th substep and the last (the landed ball, = the frame below)
            trace, _, substeps = b.trace_step(taken, before)[:3]
            last_k = int(substeps.max()) - 1
            ks = list(range(a.flight_every - 1, last_k, a.flight_every)) + [last_k]
            frames.extend(b.render(cam, trace[ks].reshape(-1, _lib.STATE_WORDS))[0].reshape(len(ks), m, a.height, a.width, 3))
            flight_frames += len(ks)
        frames.append(b.render(cam)[0])
    stats = b.read_stats()
    hits = int(stats[_lib.STAT_NAMES.index("racket_hits")])
    host = torch.stack(frames).cpu().numpy()  # the one copy to the host
    f = len(host)
    a.out.mkdir(parents=True, exist_ok=True)
    for t in range(f):
        for i in range(m):
            write_png(a.out / f"env{i:03d}_frame{t:04d}.png", host[t, i])
    every = a.sheet_every or max(1, (f + 12) // 13)
    rows = [np.concatenate(list(host[t]), axis=1) for t in range(0, f, every)]
    write_png(a.out / "contact_sheet.png", np.concatenate(rows, axis=0))
    src = "policy " + str(a.policy) if a.policy else ("tracker" if a.tracker else "uniform random")
    print(f"{a.env_id}: {m} envs x {T} env steps ({src}), {f} frames of {a.width}x{a.height} each -> {a.out}/; "
          f"rewarded racket-ball contact steps {hits}, episodes {int(stats[0])}, "
          f"mean return {stats[6] / 2 ** 20 / max(int(stats[0]), 1):.3f}; contact sheet: every {every} frames, one env per column"
          + (f"; {flight_frames} of the frames show flight substeps" if flight_frames else ""))
    b.close()


if __name__ == "__main__":
    main()
