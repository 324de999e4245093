"""CPU side of frame sizes that are not multiples of 64 (engine option "any_size"): the oracle against the golden vectors
of tests/golden/any_size/, the independent numpy restatement against the oracle at an unaligned size, and the fp32 index
rule of the decoder's nearest-neighbour resize against the oracle's fp64 one."""
import ast
import glob
import importlib.util
import os

import numpy as np
import pytest
import torch

from frame_interpolation_b200 import synthetic, weights
from oracle.film_oracle import OracleInterpolator

HERE = os.path.dirname(os.path.abspath(__file__))
CASES = sorted(glob.glob(os.path.join(HERE, "golden", "any_size", "*.npz")))
DT = np.full((1,), 0.5, np.float32)


def load_case(path):
    z = np.load(path)
    c = dict(h=int(str(z["h"])), w=int(str(z["w"])), seed=int(str(z["seed"])), align=int(str(z["align"])),
             block=ast.literal_eval(str(z["block"])))
    return z, c


def test_any_size_golden_files_present_and_unaligned():
    assert len(CASES) == 5
    for p in CASES:
        _, c = load_case(p)
        h, w = c["h"], c["w"]
        if c["block"]:
            h, w = h // c["block"][0], w // c["block"][1]
        if c["align"]:
            h, w = -(-h // c["align"]) * c["align"], -(-w // c["align"]) * c["align"]
        assert h % 64 or w % 64, p                  # every vector exercises the unaligned case


@pytest.mark.parametrize("path", CASES, ids=[os.path.basename(p) for p in CASES])
def test_oracle_reproduces_any_size_golden(path):
    z, c = load_case(path)
    torch.set_num_threads(4)
    w = weights.synthetic_weights(1234)
    assert weights.digest(w) == str(z["weights_sha256"])
    x0, x1 = synthetic.frame_pair(c["h"], c["w"], seed=c["seed"], n_waves=6)
    assert abs(float(x0.sum()) - float(z["x0_sum"])) < 1e-2
    orc = OracleInterpolator(w, align=c["align"], block_shape=c["block"])
    out = orc(x0, x1, DT)
    assert out.shape == z["image"].shape == (1, c["h"], c["w"], 3)
    assert np.abs(out - z["image"]).max() < 1e-5
    if c["block"] is None:
        aux = {}
        orc.interpolate(x0, x1, DT, aux)
        fwd = aux["forward_flow_pyramid"][0][0].permute(1, 2, 0).numpy()
        assert np.abs(fwd - z["flow_fwd_l0"]).max() < 1e-4


def test_independent_numpy_restatement_agrees_with_the_oracle_unaligned():
    """72x80 without padding: levels 3..6 are 9x10, 4x5, 2x2, 1x1 -- odd sizes, floored pooling, a decoder level whose
    fine grid is not twice the coarse one (9 from 4) and a non-2x bilinear flow resize."""
    spec_ = importlib.util.spec_from_file_location("_film_numpy", os.path.join(HERE, "test_oracle_independent.py"))
    mod = importlib.util.module_from_spec(spec_)
    spec_.loader.exec_module(mod)
    w = weights.synthetic_weights()
    x0, x1 = synthetic.frame_pair(72, 80, seed=4, n_waves=6)
    ref = OracleInterpolator(w, align=None, dtype=torch.float64).interpolate(x0, x1, DT)[0]
    got = mod.film(w, x0[0].astype(np.float64), x1[0].astype(np.float64))
    assert got.shape == ref.shape == (72, 80, 3)
    assert np.abs(got - ref).max() < 1e-9, np.abs(got - ref).max()


def _nearest_fp32(n_in, n_out):
    d = np.arange(n_out, dtype=np.float32)
    s = np.float32(n_in) / np.float32(n_out)
    return np.minimum(np.floor((d + np.float32(0.5)) * s).astype(np.int64), n_in - 1)


def _nearest_fp64(n_in, n_out):
    return np.minimum(np.floor((np.arange(n_out) + 0.5) * (n_in / n_out)).astype(np.int64), n_in - 1)


def test_nearest_index_rule_fp32_equals_fp64_below_2585():
    """The engine's resize kernel computes TF2's nearest-neighbour index in fp32 (as TF does); the oracle in fp64. For the
    decoder's coarse -> fine maps (n -> 2n + 1, and n -> 2n) they agree for every coarse size below 2585, i.e. for every
    frame dimension below 5171; the first disagreement is at 2585 -> 5171."""
    for n in range(1, 2585):
        np.testing.assert_array_equal(_nearest_fp32(n, 2 * n + 1), _nearest_fp64(n, 2 * n + 1))
        np.testing.assert_array_equal(_nearest_fp32(n, 2 * n), _nearest_fp64(n, 2 * n))
    assert (_nearest_fp32(2585, 5171) != _nearest_fp64(2585, 5171)).any()
