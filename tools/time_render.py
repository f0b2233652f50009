"""Kernel time of tb_render (render_kernel) from CUDA events: frames/s and rays/s at three sizes, and the bytes written
against the HBM peak.

  python tools/time_render.py [--reps 100] [--precision f64] [--env SwingRacket-v0]

Sizes: 16 384 frames of 84x84 (pixel-observation scale), 1 024 of 320x240, 16 of 1280x720.  The records are the states of
a batch of that many envs after a few random steps, so racket, ball and goal sit where episodes put them.  One rendered
pixel writes 3 B of RGB, 4 B of depth and 1 B of body id (8 B with both optional outputs, 3 B without); the bound printed
is bytes / 7.7 TB/s (the HGX B200 data sheet's HBM3e bandwidth for one GPU) against the measured time."""
import argparse
import ctypes
import subprocess
import sys
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
from tennisbot_rl_b200.batch import TennisBatch  # noqa: E402
from tennisbot_rl_b200.render import default_camera  # noqa: E402

HBM_PEAK = 7.7e12
SIZES = [(16384, 84, 84), (1024, 320, 240), (16, 1280, 720)]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[torch.cuda.current_device()] if q else torch.cuda.get_device_name()


def time_calls(fn, reps):
    for _ in range(5):
        fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps * 1e-3


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=100)
    ap.add_argument("--precision", default="f64")
    ap.add_argument("--env", default="SwingRacket-v0")
    a = ap.parse_args()
    print("card (name, power limit, max SM clock):", card(), flush=True)
    for m, w, h in SIZES:
        b = TennisBatch(a.env, m, seed=1, precision=a.precision)
        b.reset()
        b.rollout(10)
        states = b.get_state()
        cam = default_camera(a.env, w, h)
        rgb = torch.empty((m, h, w, 3), dtype=torch.uint8, device=b.device)
        dep = torch.empty((m, h, w), dtype=torch.float32, device=b.device)
        bod = torch.empty((m, h, w), dtype=torch.uint8, device=b.device)
        c = cam.to_c()
        sp, stream = states.data_ptr(), b._stream()
        for label, d_ptr, b_ptr, bpp in (("rgb", None, None, 3), ("rgb+depth+body", dep.data_ptr(), bod.data_ptr(), 8)):
            def call():
                b.lib.tb_render(b.h, ctypes.byref(c), sp, m, rgb.data_ptr(), d_ptr, b_ptr, stream)
            s = time_calls(call, a.reps)
            rays = m * w * h
            byts = rays * bpp
            print(f"{a.env} {a.precision} {m:6d} x {w}x{h} {label:>15s}: {s * 1e3:8.3f} ms per launch, {m / s:.3e} frames/s, "
                  f"{rays / s:.3e} rays/s; {byts / 1e6:.1f} MB written = {byts / s / 1e12:.2f} TB/s, "
                  f"HBM bound {byts / HBM_PEAK * 1e3:.3f} ms = {byts / HBM_PEAK / s * 100:.0f} % of the time", flush=True)
        b.close()
        del rgb, dep, bod, states
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
