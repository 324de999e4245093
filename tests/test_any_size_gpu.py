"""Frame sizes whose padded size is not a multiple of 64, computed behind the engine option "any_size" (default off):
parity with the fp64 oracle (golden vectors of tests/golden/any_size/, and the oracle itself at 1080p), stage-by-stage
intermediates at an odd size, the tiled / device / u8 / recursive paths, the CUDA-core validation path, and the option's
contract -- it never changes a 64-aligned result and turning it off restores the refusal even for a cached shape.
Bars as in test_engine_gpu.py: PLAN (4e-4) for the default precision plan, TIGHT (1e-4) with onepass_mask = 0."""
import ast
import glob
import os

import numpy as np
import pytest

from frame_interpolation_b200 import spec, synthetic

pytestmark = pytest.mark.gpu

PLAN = 4e-4
TIGHT = 1e-4
DT = np.full((1,), 0.5, np.float32)
GOLD = sorted(glob.glob(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "any_size", "*.npz")))


def _case(path):
    z = np.load(path)
    return z, dict(h=int(str(z["h"])), w=int(str(z["w"])), seed=int(str(z["seed"])), align=int(str(z["align"])),
                   block=ast.literal_eval(str(z["block"])))


def _engine(weights_path, align=None, block_shape=None, any_size=1, **options):
    from frame_interpolation_b200.interpolator import Interpolator
    eng = Interpolator(weights_path, align=align, block_shape=block_shape)
    if any_size:
        eng.set_option("any_size", 1)
    for k, v in options.items():
        eng.set_option(k, v)
    return eng


@pytest.fixture(scope="module")
def engine(synthetic_weights):
    eng = _engine(synthetic_weights[0])
    yield eng
    eng.close()


def _frames(c):
    return synthetic.frame_pair(c["h"], c["w"], seed=c["seed"], n_waves=6)


@pytest.mark.parametrize("path", GOLD, ids=[os.path.basename(p) for p in GOLD])
def test_any_size_matches_golden_vectors(path, synthetic_weights):
    """72x80 (odd only at the coarse levels), 97x131 (odd at level 0 on both axes), 100x150 with align=32, 64x97 (the
    smallest height) and 194x262 tiled 2x2 into unpadded 97x131 tiles -- the oracle's tiled path."""
    from frame_interpolation_b200 import weights
    z, c = _case(path)
    assert weights.digest(synthetic_weights[1]) == str(z["weights_sha256"])
    x0, x1 = _frames(c)
    eng = _engine(synthetic_weights[0], align=c["align"] or None, block_shape=c["block"])
    out = eng(x0, x1, DT)
    assert out.dtype == np.float32 and out.shape == z["image"].shape
    assert np.abs(out - z["image"]).max() < PLAN
    eng.set_option("onepass_mask", 0)
    assert np.abs(eng(x0, x1, DT) - z["image"]).max() < TIGHT
    eng.close()


def test_option_default_readback_and_minimum_size(synthetic_weights):
    eng = _engine(synthetic_weights[0], any_size=0)
    assert eng.get_option("any_size") == 0
    x0, x1 = synthetic.frame_pair(97, 131, seed=1, n_waves=4)
    with pytest.raises(RuntimeError, match="multiple of 64"):
        eng(x0, x1, DT)
    eng.set_option("any_size", 1)
    assert eng.get_option("any_size") == 1
    assert eng(x0, x1, DT).shape == (1, 97, 131, 3)
    # 63 rows: pyramid level 6 would be empty -- the reference graph fails there too (status 1, an argument error)
    y0, y1 = synthetic.frame_pair(63, 97, seed=1, n_waves=4)
    with pytest.raises(AssertionError, match="too small"):
        eng(y0, y1, DT)
    eng.close()


def test_turning_the_option_off_restores_the_refusal_for_a_cached_shape(engine):
    x0, x1 = synthetic.frame_pair(97, 131, seed=3, n_waves=6)
    a = engine(x0, x1, DT).copy()                   # the plan of this shape is now cached
    engine.set_option("any_size", 0)
    try:
        with pytest.raises(RuntimeError, match="multiple of 64"):
            engine(x0, x1, DT)
    finally:
        engine.set_option("any_size", 1)
    np.testing.assert_array_equal(engine(x0, x1, DT), a)


@pytest.mark.parametrize("h,w,align", [(128, 192, None), (100, 150, 64), (64, 64, None)])
def test_aligned_shapes_bit_identical_with_the_option_on(synthetic_weights, h, w, align):
    """The option only decides whether unaligned sizes are refused: a 64-aligned shape runs the same schedule."""
    x0, x1 = synthetic.frame_pair(h, w, seed=8, n_waves=6)
    on = _engine(synthetic_weights[0], align=align, any_size=1)
    off = _engine(synthetic_weights[0], align=align, any_size=0)
    np.testing.assert_array_equal(on(x0, x1, DT), off(x0, x1, DT))
    assert [r["name"] for r in on.op_table()] == [r["name"] for r in off.op_table()]
    assert not any("resize" in r["name"] or "up2x2" in r["name"] for r in on.op_table())
    on.close()
    off.close()


def test_op_table_and_flops_at_an_unaligned_size(engine):
    x0, x1 = synthetic.frame_pair(97, 131, seed=2, n_waves=4)
    engine(x0, x1, DT)
    p = engine.profile()
    assert (p["padded_h"], p["padded_w"]) == (97, 131)
    assert abs(p["conv_flops"] - 2 * spec.conv_macs(97, 131)["total"]) / p["conv_flops"] < 1e-9
    rows = {r["name"]: r for r in engine.op_table()}
    sizes = spec.level_sizes(97, 131)
    # levels 0 (97x131 from 48x65) and 1 (48x65 from 24x32) take the general path, levels 2 and 3 the parity classes
    for i in (0, 1):
        hh, ww = sizes[i]
        r = rows[f"fusion_up2x2@L{i}"]
        assert r["category"] == 0
        assert r["ref_flops"] == 2 * 4 * spec.fusion_filters(i + 1) * spec.fusion_filters(i) * hh * ww
        assert f"fusion_resize0@L{i}" in rows and f"fusion_up@L{i}" not in rows
    for i in (2, 3):
        assert f"fusion_up@L{i}" in rows and f"fusion_up2x2@L{i}" not in rows


def test_intermediate_tensors_match_oracle_at_97x131(synthetic_weights):
    """Three-pass engine with keep_debug: the feature pyramid at every level (odd levels show the floored fused pool of
    the conv epilogues), residual flows, flows and warped pyramids (<= 5e-4), and the decoder's resized tensors against
    the oracle's resize_nearest of the engine's own coarse tensor (a pure copy: exact)."""
    import torch
    from oracle import film_oracle as O
    h, w = 97, 131
    x0, x1 = synthetic.frame_pair(h, w, seed=9, n_waves=8)
    eng = _engine(synthetic_weights[0], onepass_mask=0, keep_debug=1)
    eng.interpolate(x0, x1, DT)
    aux = {}
    O.OracleInterpolator(synthetic_weights[1], align=None).interpolate(x0, x1, DT, aux)
    sizes = spec.level_sizes(h, w)

    def nhwc(t):
        return t[0].permute(1, 2, 0).contiguous().numpy().reshape(-1)
    for l in range(spec.PYRAMID_LEVELS):
        for k in range(2):
            got, want = eng.debug_read(f"feat{k}/{l}"), nhwc(aux["feature_pyramids"][k][l])
            assert got.size == want.size == sizes[l][0] * sizes[l][1] * spec.feature_channels(l)
            assert np.abs(got - want).max() < 1e-3 * max(1.0, np.abs(want).max()), (l, k)
        assert np.abs(eng.debug_read(f"res_fwd/{l}") - nhwc(aux["forward_residual_flow_pyramid"][l])).max() < 5e-4
        assert np.abs(eng.debug_read(f"res_bwd/{l}") - nhwc(aux["backward_residual_flow_pyramid"][l])).max() < 5e-4
    for l in range(spec.FUSION_PYRAMID_LEVELS):
        assert np.abs(eng.debug_read(f"flow_fwd/{l}") - nhwc(aux["forward_flow_pyramid"][l])).max() < 5e-4
        assert np.abs(eng.debug_read(f"flow_bwd/{l}") - nhwc(aux["backward_flow_pyramid"][l])).max() < 5e-4
        C = spec.feature_channels(l)
        al = aux["aligned_pyramid"][l]
        scale = max(1.0, float(al.abs().max()))
        assert np.abs(eng.debug_read(f"warped0/{l}") - nhwc(al[:, 3:3 + C])).max() < 5e-4 * scale
        assert np.abs(eng.debug_read(f"warped1/{l}") - nhwc(al[:, 6 + C:6 + 2 * C])).max() < 5e-4 * scale
    for i in (0, 1):
        nf = spec.fusion_filters(i + 1)
        (hc, wc), (hf, wf) = sizes[i + 1], sizes[i]
        coarse = torch.from_numpy(eng.debug_read(f"fusion_net/{i + 1}").reshape(1, hc, wc, nf)).permute(0, 3, 1, 2)
        want = nhwc(O.resize_nearest(coarse, (hf, wf)))
        np.testing.assert_array_equal(eng.debug_read(f"fusion_resized0/{i}"), want)
    eng.close()


def test_resized_coarsest_aligned_level_at_72x80(synthetic_weights):
    """72x80: decoder level 3 (9x10 from 4x5) takes the general path; its sources are the two warped feature batches of
    level 4 and the side tensor (warped images + flows), each resized on its own."""
    import torch
    from oracle import film_oracle as O
    x0, x1 = synthetic.frame_pair(72, 80, seed=10, n_waves=8)
    eng = _engine(synthetic_weights[0], onepass_mask=0, keep_debug=1)
    eng.interpolate(x0, x1, DT)
    (hc, wc), (hf, wf) = spec.level_sizes(72, 80)[4], spec.level_sizes(72, 80)[3]
    C = spec.feature_channels(4)

    def rs(flat, c):
        t = torch.from_numpy(flat.reshape(1, hc, wc, c)).permute(0, 3, 1, 2)
        return O.resize_nearest(t, (hf, wf))[0].permute(1, 2, 0).contiguous().numpy()
    for k in range(2):
        np.testing.assert_array_equal(eng.debug_read(f"fusion_resized{k}/3").reshape(hf, wf, C), rs(eng.debug_read(f"warped{k}/4"), C))
    side = eng.debug_read("fusion_resized2/3").reshape(hf, wf, -1)
    np.testing.assert_array_equal(side[..., :10], rs(eng.debug_read("aligned_side/4"), 10))
    assert not side[..., 10:].any()                 # padding channels of the side tensor stay zero
    eng.close()


def test_device_u8_and_recursive_paths_at_97x131(engine):
    import torch
    from frame_interpolation_b200 import eval_util
    h, w = 97, 131
    x0, x1 = synthetic.frame_pair(h, w, seed=7, n_waves=8)
    host = engine(x0, x1, DT).copy()
    d0, d1 = torch.from_numpy(x0).cuda(), torch.from_numpy(x1).cuda()
    out = torch.empty_like(d0)
    torch.cuda.synchronize()
    engine.interpolate_device(d0.data_ptr(), d1.data_ptr(), 1, h, w, out.data_ptr())
    engine.synchronize()
    np.testing.assert_array_equal(out.cpu().numpy(), host)
    # u8 front / back end
    u0, u1 = eval_util.to_uint8(x0), eval_util.to_uint8(x1)
    f0 = u0.astype(np.float32) / np.float32(255.0)
    f1 = u1.astype(np.float32) / np.float32(255.0)
    np.testing.assert_array_equal(engine.interpolate_u8(u0, u1), eval_util.to_uint8(engine(f0, f1, DT)))
    # device-resident recursion == recursion through __call__
    seq = engine.interpolate_recursively(x0[0], x1[0], 2)
    assert seq.shape == (5, h, w, 3)

    def rec(a, b, n):
        if n == 0:
            return [a]
        m = engine(a[None], b[None], DT)[0].copy()
        return rec(a, m, n - 1) + rec(m, b, n - 1)
    for got, want in zip(seq, rec(x0[0], x1[0], 2) + [x1[0]]):
        np.testing.assert_array_equal(got, want)
    np.testing.assert_array_equal(engine.interpolate_recursively_u8(u0[0], u1[0], 2),
                                  eval_util.to_uint8(engine.interpolate_recursively(f0[0], f1[0], 2)))


def test_validation_path_and_tensor_core_first_layer_at_97x131(synthetic_weights):
    x0, x1 = synthetic.frame_pair(97, 131, seed=11, n_waves=8)
    a = _engine(synthetic_weights[0], onepass_mask=0)
    b = _engine(synthetic_weights[0], conv_impl=1)
    assert np.abs(a(x0, x1, DT) - b(x0, x1, DT)).max() < 1e-4
    default = _engine(synthetic_weights[0])
    fe0 = _engine(synthetic_weights[0], fe_conv0_tc=1)
    assert np.abs(fe0(x0, x1, DT) - default(x0, x1, DT)).max() < 2.5e-4
    for e in (fe0, default):
        e.set_option("onepass_mask", 0)
    assert np.abs(fe0(x0, x1, DT) - default(x0, x1, DT)).max() < 5e-5
    for e in (a, b, default, fe0):
        e.close()


def test_cli_any_size_flag(tmp_path, synthetic_weights):
    """`interpolator_cli` and `eval_cli` with --align 0: refused without --any_size, the engine's frame with it."""
    from frame_interpolation_b200 import eval_cli, eval_util, interpolator_cli
    x0, x1 = synthetic.frame_pair(97, 131, seed=5, n_waves=6)
    scene = tmp_path / "scene"
    scene.mkdir()
    eval_util.write_image(str(scene / "a1.png"), x0[0])
    eval_util.write_image(str(scene / "a2.png"), x0[0] * 0.5 + x1[0] * 0.5)
    eval_util.write_image(str(scene / "a3.png"), x1[0])
    eng = _engine(synthetic_weights[0])
    r0, r1 = eval_util.read_image(str(scene / "a1.png")), eval_util.read_image(str(scene / "a3.png"))
    want = eval_util.to_uint8(eng(r0[None], r1[None], DT)[0])
    eng.close()
    # interpolator_cli on the first and last frame only
    pair = tmp_path / "pair"
    pair.mkdir()
    for n in ("a1.png", "a3.png"):
        (pair / n).write_bytes((scene / n).read_bytes())
    args = ["--pattern", str(pair), "--model_path", synthetic_weights[0], "--times_to_interpolate", "1", "--align", "0"]
    with pytest.raises(RuntimeError, match="multiple of 64"):
        interpolator_cli.main(args)
    assert interpolator_cli.main(args + ["--any_size"]) == 0
    mid = eval_util.read_image(str(pair / "interpolated_frames" / "frame_001.png"))
    np.testing.assert_array_equal(eval_util.to_uint8(mid), want)
    # eval_cli on the triplet (first, middle, last)
    out = tmp_path / "eval"
    args = ["--triplets", str(scene), "--model_path", synthetic_weights[0], "--output_dir", str(out), "--align", "0",
            "--output_frames"]
    with pytest.raises(RuntimeError, match="multiple of 64"):
        eval_cli.main(args)
    assert eval_cli.main(args + ["--any_size"]) == 0
    pred = eval_util.read_image(str(out / "scene_image.png"))
    np.testing.assert_array_equal(eval_util.to_uint8(pred), want)


@pytest.mark.timeout(900)
def test_full_size_1080p_unpadded(synthetic_weights):
    """1080x1920 without padding: the decoder's level 3 (135x240 from 67x120) takes the general path."""
    import torch
    from oracle.film_oracle import OracleInterpolator
    x0, x1 = synthetic.frame_pair(1080, 1920, seed=0, n_waves=6)
    eng = _engine(synthetic_weights[0])
    out = eng(x0, x1, DT)
    assert out.shape == (1, 1080, 1920, 3) and np.isfinite(out).all()
    assert engine_padded(eng) == (1080, 1920)
    assert "fusion_up2x2@L3" in [r["name"] for r in eng.op_table()]
    torch.set_num_threads(min(32, os.cpu_count() or 1))
    ref = OracleInterpolator(synthetic_weights[1], align=None)(x0, x1, DT)
    err = np.abs(out.astype(np.float64) - ref).max()
    assert err < PLAN, err
    eng.set_option("onepass_mask", 0)
    err3 = np.abs(eng(x0, x1, DT).astype(np.float64) - ref).max()
    assert err3 < TIGHT, err3
    eng.close()


def engine_padded(eng):
    p = eng.profile()
    return p["padded_h"], p["padded_w"]
