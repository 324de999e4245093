"""Cost of running frames at their own size (option "any_size", align=None) against padding them to a multiple of 64.

    python tools/any_size_bench.py [--rounds 5] [--calls 20] [--out results.json]

In one process, per configuration, the same frames alternate between an engine with align=64 and one with align=None +
any_size: 1080x1920 (padded: 1088x1920), 720x1280 (padded: 768x1280) and a 2160x3840 frame tiled 2x2 (1080x1920 tiles,
padded: 1088x1920 each).  Untiled configurations are timed on the device-pointer path with CUDA events around `--calls`
replays of the captured graph; the tiled one with a host clock around the synchronous tiled call (uploads and downloads
included, overlapped by the engine).  Per round both arms run back to back; the JSON reports the per-round numbers and
their medians.  For the untiled configurations eager calls with option time_ops give the per-op table (least of three), and
the rows that differ between the arms are reported (ops only one arm has, and shared ops whose time moved).

Needs a CUDA device (B200); there is no CPU fallback.  The card's name and power limit are read with a read-only
`nvidia-smi --query-gpu` and recorded beside the numbers.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from frame_interpolation_b200 import synthetic  # noqa: E402
from frame_interpolation_b200.interpolator import Interpolator  # noqa: E402

DT = np.full((1,), 0.5, np.float32)
CONFIGS = [
    ("1080p", 1080, 1920, None),
    ("720p", 720, 1280, None),
    ("4k_tiled_2x2", 2160, 3840, [2, 2]),
]


def gpu_info():
    q = "name,power.limit,clocks.max.sm,driver_version"
    try:
        r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True,
                           timeout=60)
        return {"query": q, "nvidia_smi": r.stdout.strip().splitlines()}
    except (OSError, subprocess.SubprocessError) as e:
        return {"query": q, "error": str(e)}


def frames(h, w, seed):
    if h > 1080:   # texture synthesis is O(pixels * waves): build 1080p once and tile it
        a, b = synthetic.frame_pair(1080, 1920, seed=seed, n_waves=6)
        return np.tile(a, (1, h // 1080, w // 1920, 1)), np.tile(b, (1, h // 1080, w // 1920, 1))
    return synthetic.frame_pair(h, w, seed=seed, n_waves=6)


def time_device(torch, stream, eng, d0, d1, dout, h, w, calls):
    # an explicit stream: a null stream handle would make the engine enqueue on its own stream, which the events
    # recorded on torch's default stream do not wait for
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    start.record(stream)
    for _ in range(calls):
        eng.interpolate_device(d0.data_ptr(), d1.data_ptr(), 1, h, w, dout.data_ptr(), stream=stream.cuda_stream)
    end.record(stream)
    end.synchronize()
    return start.elapsed_time(end) / calls


def time_host(eng, x0, x1, calls):
    t = time.perf_counter()
    for _ in range(calls):
        eng(x0, x1, DT)
    return (time.perf_counter() - t) * 1e3 / calls


def op_rows(eng, x0, x1, calls=3):
    """Per-op milliseconds of eager timed calls (option time_ops): per op name, the least over `calls` calls."""
    eng.set_option("time_ops", 1)
    best = {}
    for _ in range(calls):
        eng(x0, x1, DT)
        rows = {}
        for r in eng.op_table():
            rows[r["name"]] = rows.get(r["name"], 0.0) + r["ms"]
        best = {n: min(v, best.get(n, v)) for n, v in rows.items()}
    eng.set_option("time_ops", 0)
    return best


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--calls", type=int, default=20, help="timed calls per arm and round (tiled: a quarter of it)")
    ap.add_argument("--out", default=None, help="write the JSON here as well as to stdout")
    a = ap.parse_args(argv)
    import torch
    if not torch.cuda.is_available():
        sys.exit("any_size_bench: no CUDA device -- this measurement needs a B200")
    out = {"gpu": gpu_info(), "torch": torch.__version__, "rounds": a.rounds, "calls": a.calls, "configs": {}}
    for name, h, w, block in CONFIGS:
        x0, x1 = frames(h, w, seed=3)
        arms = {"padded_align64": Interpolator("synthetic", align=64, block_shape=block),
                "any_size_unpadded": Interpolator("synthetic", align=None, block_shape=block)}
        arms["any_size_unpadded"].set_option("any_size", 1)
        res = {"frame": [h, w], "block_shape": block, "ms_per_call": {k: [] for k in arms}}
        if block is None:
            d0, d1 = torch.from_numpy(x0).cuda(), torch.from_numpy(x1).cuda()
            dout = torch.empty_like(d0)
            stream = torch.cuda.Stream()
            run = lambda eng, n: time_device(torch, stream, eng, d0, d1, dout, h, w, n)   # noqa: E731
            calls = a.calls
        else:
            run = lambda eng, n: time_host(eng, x0, x1, n)   # noqa: E731
            calls = max(1, a.calls // 4)
        for k, eng in arms.items():   # warm-up: plan build, graph capture, first launches
            out_k = eng(x0, x1, DT)
            res.setdefault("finite", {})[k] = bool(np.isfinite(out_k).all())
            run(eng, 2)
            p = eng.profile()
            res.setdefault("network_size", {})[k] = [p["padded_h"], p["padded_w"]]
            res.setdefault("kernel_launches", {})[k] = p["kernel_launches"]
            res.setdefault("conv_flops", {})[k] = p["conv_flops"]
        for _ in range(a.rounds):
            for k, eng in arms.items():
                res["ms_per_call"][k].append(run(eng, calls))
        res["median_ms"] = {k: statistics.median(v) for k, v in res["ms_per_call"].items()}
        res["unpadded_over_padded"] = res["median_ms"]["any_size_unpadded"] / res["median_ms"]["padded_align64"]
        if block is None:
            ops = {k: op_rows(eng, x0, x1) for k, eng in arms.items()}
            pa, an = ops["padded_align64"], ops["any_size_unpadded"]
            res["ops_only_padded"] = {n: pa[n] for n in pa if n not in an}
            res["ops_only_unpadded"] = {n: an[n] for n in an if n not in pa}
            res["ops_shared_moved"] = {n: {"padded": pa[n], "unpadded": an[n]} for n in pa
                                       if n in an and abs(an[n] - pa[n]) > max(0.005, 0.1 * pa[n])}
            res["eager_op_sum_ms"] = {k: sum(v.values()) for k, v in ops.items()}
        for eng in arms.values():
            eng.close()
        out["configs"][name] = res
        print(name, json.dumps(res["median_ms"]), flush=True)
    text = json.dumps(out, indent=1)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")
    return 0


if __name__ == "__main__":
    sys.exit(main())
