"""Generates tests/golden/any_size/*.npz from the fp64 CPU oracle: frame sizes whose padded size is NOT a multiple of
64 (align=None, i.e. `align or None` with 0, or an align below 64), the case the engine computes with its option
"any_size".  Same format as tests/golden/make_golden.py; kept in their own directory because the vectors next to that
script are all 64-aligned.

    python tests/golden/any_size/make_any_size_golden.py
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
sys.path.insert(0, ROOT)
from frame_interpolation_b200 import synthetic, weights  # noqa: E402
from oracle.film_oracle import OracleInterpolator  # noqa: E402

# align 0 = no padding (the reference's `align or None`)
CASES = {
    "a72x80": dict(h=72, w=80, seed=41, align=0, block=None),            # odd only at the coarse levels, one axis
    "a97x131": dict(h=97, w=131, seed=42, align=0, block=None),          # odd at level 0 on both axes
    "a100x150_align32": dict(h=100, w=150, seed=43, align=32, block=None),
    "a64x97": dict(h=64, w=97, seed=44, align=0, block=None),            # the smallest height
    "a194x262_tiled2x2": dict(h=194, w=262, seed=45, align=0, block=[2, 2]),   # 97x131 tiles, unpadded
}


def main():
    torch.set_num_threads(4)
    w = weights.synthetic_weights(1234)
    here = os.path.dirname(os.path.abspath(__file__))
    for name, c in CASES.items():
        x0, x1 = synthetic.frame_pair(c["h"], c["w"], seed=c["seed"], n_waves=6)
        dt = np.full((1,), 0.5, np.float32)
        out32 = OracleInterpolator(w, align=c["align"], block_shape=c["block"])(x0, x1, dt)
        orc64 = OracleInterpolator(w, align=c["align"], block_shape=c["block"], dtype=torch.float64)
        out64 = orc64(x0, x1, dt)
        if c["block"] is None:
            aux = {}
            orc64.interpolate(x0, x1, dt, aux)
            fwd = aux["forward_flow_pyramid"][0][0].permute(1, 2, 0).numpy()
        else:
            fwd = np.zeros((0,), np.float32)
        np.savez_compressed(os.path.join(here, name + ".npz"), image=out64.astype(np.float32),
                            flow_fwd_l0=fwd.astype(np.float32),
                            weights_sha256=np.array(weights.digest(w)), x0_sum=np.float64(x0.sum()),
                            x1_sum=np.float64(x1.sum()), **{k: np.array(str(v)) for k, v in c.items()})
        print(name, out32.shape, float(np.abs(out32 - out64).max()))


if __name__ == "__main__":
    main()
