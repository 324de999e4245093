"""Command line front end with the reference's flags (eval/interpolator_cli.py:85-121) on the B200 engine.

    python -m frame_interpolation_b200.interpolator_cli --pattern "photos" --model_path synthetic \
        --times_to_interpolate 3 [--align 64 | --align 0 --any_size] [--block_height 2 --block_width 2] [--output_video --fps 30]

For every directory matching --pattern: the *.png/*.jpg/*.jpeg frames (natural order) are
interpolated recursively and written to <dir>/interpolated_frames/frame_%03d.png
(eval/interpolator_cli.py:127-177). No Beam runner: directories are processed in a loop, or, under
torchrun, sharded over ranks (one GPU each). --output_video pipes frames to ffmpeg if present.
"""
from __future__ import annotations

import argparse
import glob
import os
import subprocess
import sys
from typing import List

import numpy as np

from . import eval_util
from .interpolator import Interpolator

_INPUT_EXT = ["png", "jpg", "jpeg"]


def build_parser() -> argparse.ArgumentParser:
    p = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    p.add_argument("--pattern", required=True, help="The pattern to determine the directories with the input frames.")
    p.add_argument("--model_path", required=True,
                   help="FILMW1 weight file (tf_bundle.convert_saved_model output), or 'synthetic[:seed]' to opt in to "
                        "seeded random weights (plumbing tests only: the frames are meaningless).")
    p.add_argument("--times_to_interpolate", type=int, default=5,
                   help="Number of recursive midpoint interpolations; output has 2^times+1 frames per input pair.")
    p.add_argument("--fps", type=int, default=30)
    p.add_argument("--align", type=int, default=64)
    p.add_argument("--block_height", type=int, default=1)
    p.add_argument("--block_width", type=int, default=1)
    p.add_argument("--output_video", action="store_true")
    p.add_argument("--any_size", action="store_true",
                   help="Accept padded frame sizes that are not multiples of 64 (engine option any_size). Use with --align 0 to run frames at their own size, like the reference with align=None.")
    p.add_argument("--device", type=int, default=None, help="CUDA device ordinal (default: LOCAL_RANK or 0)")
    return p


class _VideoWriter:
    """Raw RGB frames piped to ffmpeg as they are produced; a failed encode raises with ffmpeg's own message."""

    def __init__(self, path: str, h: int, w: int, fps: int):
        ffmpeg = eval_util.get_ffmpeg_path()
        self.path = path
        # yuv420p needs even dimensions: pad by one replicated row/column instead of failing silently
        cmd = [ffmpeg, "-y", "-f", "rawvideo", "-pix_fmt", "rgb24", "-s", f"{w}x{h}", "-r", str(fps), "-i", "-",
               "-vf", "pad=ceil(iw/2)*2:ceil(ih/2)*2", "-pix_fmt", "yuv420p", path]
        self.proc = subprocess.Popen(cmd, stdin=subprocess.PIPE, stdout=subprocess.DEVNULL, stderr=subprocess.PIPE)

    def write(self, frame: np.ndarray) -> None:
        try:
            self.proc.stdin.write(eval_util.to_uint8(frame).tobytes())
        except BrokenPipeError:
            self.close()

    def close(self) -> None:
        if self.proc.stdin and not self.proc.stdin.closed:
            self.proc.stdin.close()
        err = self.proc.stderr.read().decode(errors="replace")
        rc = self.proc.wait()
        if rc != 0:
            raise RuntimeError(f"ffmpeg failed (exit {rc}) writing {self.path}: {err[-2000:]}")


def process_directory(directory: str, interpolator: Interpolator, times: int, fps: int, video: bool) -> int:
    """Frames are written (and piped to ffmpeg) as the generator yields them: nothing but the current input pair's
    sequence is ever held in memory (eval/interpolator_cli.py:164-177 materialises the whole list)."""
    names: List[str] = []
    for ext in _INPUT_EXT:
        names += eval_util.natural_sorted(glob.glob(os.path.join(directory, f"*.{ext}")))
    if len(names) < 2:
        print(f"[film_b200] {directory}: fewer than two input frames, skipped", file=sys.stderr)
        return 0
    frames_dir = os.path.join(directory, "interpolated_frames")
    if os.path.isdir(frames_dir):
        for old in glob.glob(os.path.join(frames_dir, "frame_*.png")):   # stale frames of a previous run
            os.remove(old)
    else:
        os.makedirs(frames_dir)
    writer = None
    n = 0
    for frame in eval_util.interpolate_recursively_from_files(names, times, interpolator):
        eval_util.write_image(os.path.join(frames_dir, f"frame_{n:03d}.png"), frame)
        if video:
            if writer is None:
                writer = _VideoWriter(os.path.join(directory, "interpolated.mp4"), frame.shape[0], frame.shape[1], fps)
            writer.write(frame)
        n += 1
    if writer is not None:
        writer.close()
    return n


def main(argv=None) -> int:
    args = build_parser().parse_args(argv)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    device = args.device if args.device is not None else int(os.environ.get("LOCAL_RANK", "0"))
    directories = sorted(d for d in glob.glob(args.pattern) if os.path.isdir(d))
    mine = directories[rank::world]            # directories are independent: shard them over ranks
    interpolator = Interpolator(args.model_path, args.align, [args.block_height, args.block_width], device=device)
    if args.any_size:
        interpolator.set_option("any_size", 1)
    for d in mine:
        n = process_directory(d, interpolator, args.times_to_interpolate, args.fps, args.output_video)
        print(f"[film_b200] {d}: wrote {n} frames to {d}/interpolated_frames", flush=True)
    return 0


if __name__ == "__main__":
    sys.exit(main())
