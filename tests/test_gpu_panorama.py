"""The equirectangular camera on the GPU (bt_scene_set_camera_projection / Scene.set_camera_projection): camera-ray and image
parity with the oracle on identical sample sets, the pooled and lane kernels bit for bit, switching back to the perspective
camera, the round trip through an environment map, and the plumbing (host buffers, multi-device engines, work counters,
the CLI)."""
import json
import os
import subprocess

import numpy as np
import pytest

import oracle_camera as OC
from common import LENS_SCENE, LENS_VOLUME, mae_per_channel, oracle_render, synthetic_scene
from test_gpu_environment import _read_png, render, smooth_map, write_pfm
from test_panorama import camera_doc, filtered_map, round_trip_error, rotation

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EQ = OC.EQUIRECTANGULAR


def engine_scene(name, w, h, lens=None, precision=None, projection=EQ):
    import bendy_tracer_b200 as bt
    import oracle_ffi as O
    sc = bt.Scene.load(O.scene_path(name))
    cam = sc.find_by_tag("camera")
    sc.set_camera_aspect(cam, float(np.float32(w) / np.float32(h)))
    if lens is not None:
        sc.set_lenses(lens)
    if precision:
        sc.set_precision(precision)
    if projection is not None:
        sc.set_camera_projection(cam, projection)
    return sc, cam


def bvh_pair():
    """synthetic_scene (its camera among the primitives: the panorama sees them in every direction), both sides panoramic"""
    import bendy_tracer_b200 as bt
    doc = synthetic_scene(200, 100, 20, seed=5)
    osc, esc = OC.CameraOracleScene(doc), bt.Scene.from_json(json.dumps(doc))
    cam = esc.find_by_tag("camera")
    osc.set_projection(cam, EQ)
    esc.set_camera_projection(cam, EQ)
    assert esc.info()["n_bvh_nodes"] > 0
    return osc, esc, cam


# ---- camera rays --------------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("subsample", [0, 2])
@pytest.mark.parametrize("precision", ["exact", "fast"])
def test_camera_rays(precision, subsample):
    """scene.json.gz's camera (it has a focus: a panorama ignores it) at 128 x 64: the exact flavour is the oracle bit for bit,
    the fast one within test_gpu_parity's bar (its jitter's FMA contraction moves u, v by an ulp)"""
    import bendy_tracer_b200 as bt
    import oracle_ffi as O
    w, h = 128, 64
    osc, esc, cam = OC.load_pair("scene", w, h)
    esc.set_precision(precision)
    rng = np.random.default_rng(2)
    n = 8192
    xs, ys, pi = rng.integers(0, w, n), rng.integers(0, h, n), rng.integers(0, 64, n)
    xs[:w], ys[:w] = np.arange(w), 0                                  # the pole rows
    xs[w:2 * w], ys[w:2 * w] = np.arange(w), h - 1
    ref = osc.camera_rays(cam, O.make_config(samples=16, subsample=subsample), w, h, xs, ys, pi, seed=7, sample_base=3)
    got = bt.Tracer(bt.Config(), seed=7).camera_rays(esc, cam, bt.RenderConfig.with_samples_subsample(16, bt.Subsample(subsample)),
                                                    w, h, xs, ys, pi, sample_base=3)
    assert np.array_equal(got[:, :3], ref[:, :3])                     # the camera's position: a pinhole
    if precision == "exact":
        assert np.array_equal(got, ref), f"{(got != ref).any(1).sum()} of {n} rays differ, by up to {np.abs(got - ref).max()}"
    assert np.abs(got - ref).max() <= 2e-6


# ---- image parity -----------------------------------------------------------------------------------------------------------------

PARITY = [("cornell2", None, False), ("scene", None, False), ("cloud", None, False), ("scene", LENS_SCENE, True),
          ("cloud", LENS_VOLUME, True), ("bvh", None, False)]


@pytest.mark.parametrize("name,lens,env", PARITY, ids=["cornell2", "scene", "cloud", "scene+lens+map", "cloud+lens+map", "bvh"])
@pytest.mark.parametrize("precision", ["exact", "fast"])
def test_parity_with_oracle(name, lens, env, precision):
    """identical sample sets at subsample 2; test_gpu_environment's bars: exact MAE <= 1e-5, fast <= 1e-3.
    Fast cloud + lens is skipped there and here: its volume march flips scatter decisions above the bar in any camera.
    Fast scene + lens runs with BT_LENS_EXACT_RSQRT: with the default MUFU.RSQ stepper a panorama of this scene measured a
    blue-channel MAE of 1.06e-3 / 1.10e-3 at 64 / 256 spp (128 x 64, the same with or without the map, >= 44 % of it in the
    worst 1 % of pixels: rare paths whose outcome differs between the two steppers, which more samples do not average out),
    against 7.1e-4 for the perspective frame of the same size; with BT_LENS_EXACT_RSQRT this sample set measures 9.2e-4, so the
    margin is small and the remaining difference lies in the fast flavour's other arithmetic.  The exact flavour is within
    1e-8 of the oracle on every case."""
    import bendy_tracer_b200 as bt
    if precision == "fast" and name == "cloud" and lens is not None:
        pytest.skip("the fast stepper through a volume is above the bar with or without a panorama; AUTO renders it exact")
    w, h, passes = 128, 64, 2
    osc, esc, cam = bvh_pair() if name == "bvh" else OC.load_pair(name, w, h, lenses=lens)
    esc.set_precision(precision)
    if precision == "fast" and lens is not None:
        esc.set_lenses(lens, bt.LensConfig(exact_rsqrt=True))
    if env:
        m = smooth_map(64, 128, 1)
        osc.set_environment(m)
        esc.set_environment(m)
    ref, n, _ = oracle_render(osc, cam, w, h, passes, 2, seed=2)
    got = render(esc, cam, w, h, passes, 2, seed=2)
    mae = mae_per_channel(got, ref, n)
    print(f"{name}{'+lens' if lens is not None else ''} {precision}: MAE vs oracle {mae}")
    assert (mae <= (1e-5 if precision == "exact" else 1e-3)).all(), mae


@pytest.mark.parametrize("output", [0, 1, 2, 3])
def test_parity_subsample_none_and_aov_outputs(output):
    """the lensed scene with a map, exact flavour, subsample None, colour and the three AOV outputs"""
    w, h = 128, 64
    osc, esc, cam = OC.load_pair("scene", w, h, lenses=LENS_SCENE)
    esc.set_precision("exact")
    m = smooth_map(32, 64, 4)
    osc.set_environment(m)
    esc.set_environment(m)
    ref, n, _ = oracle_render(osc, cam, w, h, 4, 0, output=output, seed=6)
    got = render(esc, cam, w, h, 4, 0, output=output, seed=6)
    assert (mae_per_channel(got, ref, n) <= 1e-5).all(), output


# ---- the schedulers agree ---------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("precision", ["fast", "exact"])
def test_pool_equals_lane_kernel(precision):
    """a lensed panorama with a map: the pooled kernel (default pool_w) and the lane kernel (pool_w = 0), bit for bit"""
    w, h = 160, 80
    sc, cam = engine_scene("scene", w, h, LENS_SCENE, precision)
    sc.set_environment(smooth_map(32, 64, 2))
    assert np.array_equal(render(sc, cam, w, h, 2, 2), render(sc, cam, w, h, 2, 2, pool_w=0))


def test_pool_bvh_equals_lane_kernel():
    w, h = 128, 64
    _, sc, cam = bvh_pair()
    sc.set_precision("exact")
    ref = render(sc, cam, w, h, 2, 2, pool_w=0)
    assert np.array_equal(render(sc, cam, w, h, 2, 2, pool_w=3), ref)


# ---- the projection's state ---------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("name,lens", [("cornell", None), ("scene", LENS_SCENE), ("cloud", None)])
@pytest.mark.parametrize("precision", ["fast", "exact"])
def test_back_to_perspective_is_bit_identical(name, lens, precision):
    w, h = 96, 54
    plain, cam = engine_scene(name, w, h, lens, precision, projection=None)
    ref = render(plain, cam, w, h, 1, 2)
    sc, _ = engine_scene(name, w, h, lens, precision)
    pano = render(sc, cam, w, h, 1, 2)
    sc.set_camera_projection(cam, OC.PERSPECTIVE)
    assert np.array_equal(render(sc, cam, w, h, 1, 2), ref)
    assert not np.array_equal(pano, ref)


def test_projection_survives_scene_edits_and_rejected_calls():
    """the projection set before apply_transform, commit and set_camera_aspect renders what a projection set after them
    renders; rejected calls leave it as it was"""
    import bendy_tracer_b200 as bt
    from bendy_tracer_b200 import _ffi
    w, h = 128, 64
    affine = np.concatenate([rotation(9).T.ravel(), [0.3, -0.2, 0.5]]).astype(np.float32)
    scenes = []
    for early in (True, False):
        sc, cam = engine_scene("scene", w, h, LENS_SCENE, projection=EQ if early else None)
        render(sc, cam, w, h, 1, 2)                                   # flattened and uploaded before the edits
        sc.apply_transform(cam, affine)
        sc.commit()
        sc.set_camera_aspect(cam, 1.25)
        if not early:
            sc.set_camera_projection(cam, EQ)
        scenes.append((sc, cam))
    ref = render(*scenes[1], w, h, 1, 2)
    sc, cam = scenes[0]
    assert np.array_equal(render(sc, cam, w, h, 1, 2), ref)
    assert _ffi.lib.bt_scene_set_camera_projection(sc.handle, cam, 2) == _ffi.ERR_INVALID_ARG
    with pytest.raises(bt.ScenePanic):
        sc.set_camera_projection(1, bt.Projection.PERSPECTIVE)
    assert np.array_equal(render(sc, cam, w, h, 1, 2), ref)
    sc.set_camera_projection(cam, bt.Projection.PERSPECTIVE)
    assert not np.array_equal(render(sc, cam, w, h, 1, 2), ref)


# ---- the round trip ---------------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("precision", ["fast", "exact"])
def test_round_trip_reproduces_the_map(precision):
    """test_panorama.py's round trip at 256 x 128 and 2 x 256 spp: a panorama of an empty scene is the filtered map within
    the Monte-Carlo noise"""
    import bendy_tracer_b200 as bt
    h, w, spp = 128, 256, 256
    env = smooth_map(h, w, 22)
    sc = bt.Scene.from_json(json.dumps(camera_doc()))
    sc.set_precision(precision)
    sc.set_environment(env)
    sc.set_camera_projection(0, EQ)
    a, b = render(sc, 0, w, h, spp, 0, seed=1), render(sc, 0, w, h, spp, 0, seed=2)
    err, noise = round_trip_error(a, b, spp, env)
    print(f"round trip {precision}: MAE {err:.2e}, noise {noise:.2e}")
    assert err <= 1.5 * noise, (err, noise)
    assert np.abs(filtered_map(env) - filtered_map(np.roll(env, 1, axis=1))).mean() / 2 > 10 * noise


# ---- plumbing -----------------------------------------------------------------------------------------------------------------------

def test_host_buffer_equals_device_buffer():
    w, h = 256, 128
    sc, cam = engine_scene("scene", w, h, LENS_SCENE)
    sc.set_environment(smooth_map(64, 128, 4))
    ref = render(sc, cam, w, h, 1, 2)
    for bands in (1, 3):
        assert np.array_equal(render(sc, cam, w, h, 1, 2, device=None, host_bands=bands), ref), bands


def test_multi_device_engine():
    import bendy_tracer_b200 as bt
    w, h = 128, 64
    sc, cam = engine_scene("scene", w, h, LENS_SCENE)
    ref = render(sc, cam, w, h, 4, 2)
    sc2, cam2 = engine_scene("scene", w, h, LENS_SCENE)
    got = render(sc2, cam2, w, h, 4, 2, engine=bt.Engine(devices=[0, 0]))
    assert np.allclose(got[..., :3], ref[..., :3], rtol=2e-6, atol=2e-5)    # f32 summation order only


@pytest.mark.parametrize("lens", [None, LENS_SCENE])
def test_render_stats_count_every_path(lens):
    import bendy_tracer_b200 as bt
    w, h = 96, 48
    sc, cam = engine_scene("scene", w, h, lens)
    stats = bt.Tracer(bt.Config(), seed=5).render_stats(sc, cam, bt.RenderConfig.with_samples_subsample(2, bt.Subsample(2)), w, h)
    assert stats["paths"] == w * h * 8


def test_cli_renders_a_panorama(tmp_path):
    """bendy_b200_cli --projection equirectangular --lens --environment renders what the API renders with the same seed"""
    import bendy_tracer_b200 as bt
    import oracle_ffi as O
    w, h, samples = 128, 64, 8
    env = smooth_map(32, 64, 10)
    env[:8] *= 3.0
    write_pfm(tmp_path / "sky.pfm", env)
    cli = os.path.join(ROOT, "bendy_tracer_b200", "csrc", "bendy_b200_cli")
    r = subprocess.run([cli, "--output", "full", "--width", str(w), "--height", str(h), "--samples", str(samples), "--scene",
                        O.scene_path("scene"), "--lens", ",".join(str(float(x)) for x in LENS_SCENE[0]), "--environment",
                        str(tmp_path / "sky.pfm"), "--projection", "equirectangular", "--screenshot", str(tmp_path / "out.png")],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    sc, cam = engine_scene("scene", w, h, LENS_SCENE)
    sc.set_environment(env)
    buf = bt.Buffer(w, h)
    tracer = bt.Tracer(bt.Config(chunks_x=8, chunks_y=4), seed=0)
    while buf.samples() < samples:
        tracer.render(sc, cam, bt.RenderConfig.with_samples_subsample(1, bt.Subsample(2)), buf)
    want = buf.preview(bt.Engine.default(0))
    got = _read_png(tmp_path / "out.png")
    assert got.shape == want.shape and np.array_equal(got, want)
