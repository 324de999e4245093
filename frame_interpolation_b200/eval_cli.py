"""Benchmark evaluator on the B200 engine -- TF-free counterpart of the reference's `eval/eval_cli.py:88-178`.

    python -m frame_interpolation_b200.eval_cli --triplets <dir> --model_path <weights.filmw> \
        --output_dir <out> [--max_examples N] [--metrics l1,l2,ssim,psnr] [--output_frames] [--align 0 --any_size]

The reference iterates a TFRecord of (x0, y, x1) triplets built by `datasets/create_*_tfrecord.py` from
folders of three frames (Vimeo-90K `im1/im2/im3.png`, Middlebury `frame10/frame10i11/frame11.png`, ...);
here the triplet FOLDERS are read directly (every sub-directory of --triplets holding exactly three images,
natural order: first, ground-truth middle, last), since TFRecords need TensorFlow. Per example, like
`run_evaluation`: predict the middle frame at t = 0.5, clip it to [0, 1] (eval_cli.py:162-165), evaluate the
metrics of losses/losses.py:72-74,98-113 (l1, l2, ssim, psnr; TF definitions restated in metrics.py), write
`results.csv` -- header `key, <metrics>`, one row per example, a final `mean` row -- and `readme.txt`;
--output_frames also saves inputs, ground truth and prediction as `<key>_<name>.png`.
"""
from __future__ import annotations

import argparse
import glob
import os
import sys
from typing import Callable, Dict, List, Optional, Sequence, Tuple

import numpy as np

from . import eval_util, metrics as M

_EXT = (".png", ".jpg", ".jpeg")
METRICS: Dict[str, Callable[[np.ndarray, np.ndarray], float]] = {
    "l1": M.l1, "l2": M.l2, "ssim": M.ssim, "psnr": M.psnr,
}


def find_triplets(root: str) -> List[Tuple[str, List[str]]]:
    """(key, [first, middle, last]) for every directory under `root` (recursively) with exactly three images."""
    out = []
    for d, _, files in sorted(os.walk(root)):
        imgs = eval_util.natural_sorted(f for f in files if f.lower().endswith(_EXT))
        if len(imgs) == 3:
            key = os.path.relpath(d, root).replace(os.sep, "_")
            out.append((key if key != "." else os.path.basename(os.path.abspath(d)), [os.path.join(d, f) for f in imgs]))
    return out


def run_evaluation(interpolator: Callable, triplets: Sequence[Tuple[str, List[str]]], output_dir: str,
                   max_examples: Optional[int] = None, metrics: Sequence[str] = ("l1", "l2", "ssim", "psnr"),
                   output_frames: bool = False, model_path: str = "", source: str = "") -> Dict[str, float]:
    for m in metrics:
        if m not in METRICS:
            raise ValueError(f"unknown metric {m!r} (available: {sorted(METRICS)}; vgg/style need the VGG-19 weights)")
    os.makedirs(output_dir, exist_ok=True)
    with open(os.path.join(output_dir, "readme.txt"), "w") as f:
        print("Results for:", file=f)
        print(f" model:   {model_path}", file=f)
        print(f" triplets: {source}", file=f)
    dt = np.full((1,), 0.5, np.float32)
    all_vals: Dict[str, List[float]] = {m: [] for m in metrics}
    with open(os.path.join(output_dir, "results.csv"), "w") as csv_file:
        print(", ".join(["key"] + list(metrics)), file=csv_file)
        for key, (p0, py, p1) in list(triplets)[:max_examples]:
            x0, y, x1 = (eval_util.read_image(p) for p in (p0, py, p1))
            pred = interpolator(x0[np.newaxis], x1[np.newaxis], dt)[0]
            if output_frames:
                for name, img in (("x0", x0), ("x1", x1), ("y", y), ("image", pred)):
                    eval_util.write_image(os.path.join(output_dir, f"{key}_{name}.png"), img)
            pred = np.clip(pred, 0.0, 1.0)                      # eval_cli.py:165: clipped in the eval loop only
            vals = [float(METRICS[m](pred[np.newaxis], y[np.newaxis])) for m in metrics]
            for m, v in zip(metrics, vals):
                all_vals[m].append(v)
            print(f"{key}, {', '.join(repr(v) for v in vals)}", file=csv_file)
        totals = {m: float(np.mean(v)) for m, v in all_vals.items() if v}
        if totals:
            print(f"mean, {', '.join(repr(totals[m]) for m in metrics)}", file=csv_file)
    return totals


def main(argv=None) -> int:
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--triplets", required=True, help="directory tree whose leaf folders hold three frames each")
    ap.add_argument("--model_path", required=True, help="FILMW1 weight file, or 'synthetic[:seed]'")
    ap.add_argument("--output_dir", required=True)
    ap.add_argument("--max_examples", type=int, default=None)
    ap.add_argument("--metrics", default="l1,l2,ssim,psnr")
    ap.add_argument("--output_frames", action="store_true")
    ap.add_argument("--align", type=int, default=64)
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--any_size", action="store_true",
                    help="Accept padded frame sizes that are not multiples of 64 (engine option any_size). Use with --align 0 to run frames at their own size, like the reference with align=None.")
    a = ap.parse_args(argv)
    from .interpolator import Interpolator
    interp = Interpolator(a.model_path, align=a.align, device=a.device)
    if a.any_size:
        interp.set_option("any_size", 1)
    trip = find_triplets(a.triplets)
    if not trip:
        print(f"[film_b200] no triplet folders under {a.triplets}", file=sys.stderr)
        return 1
    totals = run_evaluation(interp, trip, a.output_dir, a.max_examples, [m for m in a.metrics.split(",") if m],
                            a.output_frames, a.model_path, a.triplets)
    print("mean,", totals)
    return 0


if __name__ == "__main__":
    sys.exit(main())
