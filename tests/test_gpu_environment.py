"""The environment map on the GPU (bt_scene_set_environment / Scene.set_environment): parity with the oracle on identical
sample sets, bit-identity of an all-ones map with no map in every kernel, pooled = lane kernel with a map, what the map
must not touch (AOV outputs, work counters) and the plumbing (host buffers, multi-device engines, clear, replacement
between asynchronous renders, the CLI's PFM reader)."""
import json
import os
import subprocess

import numpy as np
import pytest

from common import LENS_SCENE, LENS_VOLUME, SCENES, mae_per_channel, oracle_render, synthetic_scene
from oracle_env import load_pair

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def smooth_map(h, w, seed):
    """a random smooth, strictly positive map: a few low-frequency waves per channel"""
    rng = np.random.default_rng(seed)
    r, c = np.meshgrid((np.arange(h) + 0.5) / h, (np.arange(w) + 0.5) / w, indexing="ij")
    out = np.zeros((h, w, 3))
    for ch in range(3):
        out[..., ch] = 1.0
        for _ in range(4):
            kx, ky = rng.integers(1, 5), rng.integers(1, 4)
            out[..., ch] += 0.2 * np.sin(2 * np.pi * kx * c + rng.uniform(0, 6.3)) * np.cos(np.pi * ky * r + rng.uniform(0, 6.3))
    return np.maximum(out, 0.05).astype(np.float32)


def lens_for(name):
    """one mass 4 units in front of the scene's camera"""
    import oracle_ffi as O
    m = np.array(O.read_scene_json(O.scene_path(name))["objects"]["collection"]["0"]["transform"]["transform_world"], np.float64)
    return np.array([[*(m[9:12] - 4.0 * m[6:9] / np.linalg.norm(m[6:9])), 0.05]], np.float32)


def render(sc, cam, w, h, passes, sub, output=0, seed=3, device="cuda:0", engine=None, **tuning):
    import bendy_tracer_b200 as bt
    eng = engine or bt.Engine.default(0)
    eng.set_tuning(**tuning)
    try:
        buf = bt.Buffer(w, h, device=device)
        bt.Tracer(bt.Config(output=bt.Output(output)), engine=eng, seed=seed).render(
            sc, cam, bt.RenderConfig.with_samples_subsample(passes, bt.Subsample(sub)), buf)
        return buf.data.cpu().numpy() if device else np.array(buf.data)
    finally:
        eng.set_tuning(**{k: None for k in tuning})


def engine_scene(name, w, h, lens=None, precision=None):
    import bendy_tracer_b200 as bt
    import oracle_ffi as O
    sc = bt.Scene.load(O.scene_path(name))
    cam = sc.find_by_tag("camera")
    sc.set_camera_aspect(cam, float(np.float32(w) / np.float32(h)))
    if lens is not None:
        sc.set_lenses(lens)
    if precision:
        sc.set_precision(precision)
    return sc, cam


def bvh_pair(w, h):
    import bendy_tracer_b200 as bt
    from oracle_env import EnvOracleScene
    doc = synthetic_scene(200, 100, 20, seed=5)
    osc, esc = EnvOracleScene(doc), bt.Scene.from_json(json.dumps(doc))
    cam = esc.find_by_tag("camera")
    aspect = float(np.float32(w) / np.float32(h))
    osc.set_camera_aspect(cam, aspect)
    esc.set_camera_aspect(cam, aspect)
    assert esc.info()["n_bvh_nodes"] > 0
    return osc, esc, cam


# ---- parity with the oracle ---------------------------------------------------------------------------------------------

PARITY = [("scene", None), ("cloud", None), ("scene", LENS_SCENE), ("cloud", LENS_VOLUME), ("bvh", None)]


@pytest.mark.parametrize("name,lens", PARITY, ids=["scene", "cloud", "scene+lens", "cloud+lens", "bvh"])
@pytest.mark.parametrize("precision", ["exact", "fast"])
def test_parity_with_oracle(name, lens, precision):
    """identical sample sets; exact flavour MAE <= 1e-5, fast <= 1e-3 (the north-star bar).  The lensed fast case needs
    64 spp like smoke(): the MUFU.RSQ stepper flips a Fresnel decision on ~1e-4 .. 1e-3 of the paths.  Fast cloud + lens
    is not asserted: its volume march flips scatter decisions above the bar without a map too (AUTO renders it exact)."""
    if precision == "fast" and name == "cloud" and lens is not None:
        pytest.skip("the fast stepper through a volume is above the bar with or without a map; AUTO renders it exact")
    w, h = (96, 54) if precision == "fast" and lens is not None else (128, 72)
    passes = 16 if precision == "fast" and lens is not None else 2
    osc, esc, cam = bvh_pair(w, h) if name == "bvh" else load_pair(name, w, h, lenses=lens)
    esc.set_precision(precision)
    plain, _, _ = oracle_render(osc, cam, w, h, passes, 2, seed=2)
    env = smooth_map(64, 128, 1)
    osc.set_environment(env)
    esc.set_environment(env)
    ref, n, _ = oracle_render(osc, cam, w, h, passes, 2, seed=2)
    got = render(esc, cam, w, h, passes, 2, seed=2)
    mae = mae_per_channel(got, ref, n)
    print(f"{name}{'+lens' if lens is not None else ''} {precision}: MAE vs oracle {mae}")
    assert (mae <= (1e-5 if precision == "exact" else 1e-3)).all(), mae
    assert mae_per_channel(ref, plain, n).min() > 2e-3                 # the map really changes the image


# ---- an all-ones map is no map ------------------------------------------------------------------------------------------

@pytest.mark.parametrize("name", SCENES)
@pytest.mark.parametrize("lensed", [False, True])
@pytest.mark.parametrize("precision", ["fast", "exact"])
def test_all_ones_map_is_bit_identical(name, lensed, precision):
    w, h = 64, 36
    sc, cam = engine_scene(name, w, h, lens_for(name) if lensed else None, precision)
    for pool_w in (4, 0):
        ref = render(sc, cam, w, h, 1, 2, pool_w=pool_w)
        for shape in ((1, 1), (3, 5), (64, 128)):
            sc.set_environment(np.ones(shape + (3,), np.float32))
            got = render(sc, cam, w, h, 1, 2, pool_w=pool_w)
            assert np.array_equal(got, ref), (pool_w, shape, f"{(got != ref).any(-1).sum()} pixels differ")
        sc.set_environment(None)


@pytest.mark.parametrize("precision", ["fast", "exact"])
def test_all_ones_map_is_bit_identical_bvh(precision):
    w, h = 96, 54
    _, sc, cam = bvh_pair(w, h)
    sc.set_precision(precision)
    for pool_w in (3, 0):
        ref = render(sc, cam, w, h, 1, 2, pool_w=pool_w)
        sc.set_environment(np.ones((1, 1, 3), np.float32))
        assert np.array_equal(render(sc, cam, w, h, 1, 2, pool_w=pool_w), ref), pool_w
        sc.set_environment(None)


# ---- the two schedulers agree with a map ----------------------------------------------------------------------------------

POOL_CASES = [(n, None) for n in SCENES] + [("scene", LENS_SCENE), ("cloud", LENS_VOLUME), ("cornell2", np.array([[0.0, 2.5, 4.0, 0.1]], np.float32))]


@pytest.mark.parametrize("name,lens", POOL_CASES, ids=[f"{n}{'+lens' if l is not None else ''}" for n, l in POOL_CASES])
def test_pool_equals_lane_kernel_with_map(name, lens):
    w, h = 136, 76
    sc, cam = engine_scene(name, w, h, lens)
    sc.set_environment(smooth_map(32, 64, 2))
    ref = render(sc, cam, w, h, 2, 2, pool_w=0)
    got = render(sc, cam, w, h, 2, 2, pool_w=4)
    assert np.array_equal(got, ref), f"{(got != ref).any(-1).sum()} pixels differ"


# ---- what the map must not touch ------------------------------------------------------------------------------------------

@pytest.mark.parametrize("name,lens", [("scene", None), ("scene", LENS_SCENE), ("cloud", None), ("cloud", LENS_VOLUME)])
def test_aov_outputs_and_work_counters_ignore_the_map(name, lens):
    import bendy_tracer_b200 as bt
    w, h = 96, 54
    sc, cam = engine_scene(name, w, h, lens)
    env = smooth_map(32, 64, 3)
    rc = bt.RenderConfig.with_samples_subsample(2, bt.Subsample(2))
    tracer = bt.Tracer(bt.Config(), seed=5)
    for output in (1, 2, 3):
        sc.set_environment(None)
        ref = render(sc, cam, w, h, 1, 2, output=output)
        sc.set_environment(env)
        assert np.array_equal(render(sc, cam, w, h, 1, 2, output=output), ref), output
    sc.set_environment(None)
    stats = tracer.render_stats(sc, cam, rc, w, h)
    sc.set_environment(env)
    assert tracer.render_stats(sc, cam, rc, w, h) == stats
    assert stats["paths"] == w * h * 8


# ---- plumbing -------------------------------------------------------------------------------------------------------------

def test_host_buffer_equals_device_buffer():
    w, h = 200, 120
    sc, cam = engine_scene("scene", w, h, LENS_SCENE)
    sc.set_environment(smooth_map(64, 128, 4))
    ref = render(sc, cam, w, h, 1, 2)
    for bands in (1, 3):
        assert np.array_equal(render(sc, cam, w, h, 1, 2, device=None, host_bands=bands), ref), bands


def test_multi_device_engine_uploads_the_map_everywhere():
    import bendy_tracer_b200 as bt
    w, h = 128, 72
    sc, cam = engine_scene("scene", w, h, LENS_SCENE)
    sc.set_environment(smooth_map(64, 128, 5))
    ref = render(sc, cam, w, h, 4, 2)
    sc2, cam2 = engine_scene("scene", w, h, LENS_SCENE)
    sc2.set_environment(smooth_map(64, 128, 5))
    multi = bt.Engine(devices=[0, 0])
    got = render(sc2, cam2, w, h, 4, 2, engine=multi)
    assert np.allclose(got[..., :3], ref[..., :3], rtol=2e-6, atol=2e-5)    # f32 summation order only
    sc2.set_environment(None)                                               # ... and a clear reaches every copy
    plain = render(engine_scene("scene", w, h, LENS_SCENE)[0], cam, w, h, 4, 2)
    assert np.allclose(render(sc2, cam2, w, h, 4, 2, engine=multi)[..., :3], plain[..., :3], rtol=2e-6, atol=2e-5)


def test_clear_and_invalid_calls():
    """clearing restores the no-map image bit for bit; rejected calls leave the map that was set"""
    import bendy_tracer_b200 as bt
    from bendy_tracer_b200 import _ffi
    w, h = 96, 54
    sc, cam = engine_scene("scene", w, h, LENS_SCENE)
    plain = render(sc, cam, w, h, 1, 2)
    env = smooth_map(32, 64, 6)
    sc.set_environment(env)
    mapped = render(sc, cam, w, h, 1, 2)
    assert np.abs(mapped - plain).mean() > 1e-3
    bad = env.copy()
    bad[3, 3, 0] = np.nan
    for call in (lambda: sc.set_environment(bad), lambda: sc.set_environment(-env), lambda: sc.set_environment(env[..., :2])):
        with pytest.raises((bt.BendyError, ValueError)):
            call()
    assert _ffi.lib.bt_scene_set_environment(sc.handle, None, 4, 4) == _ffi.ERR_INVALID_ARG
    assert np.array_equal(render(sc, cam, w, h, 1, 2), mapped)
    sc.set_environment(None)
    assert np.array_equal(render(sc, cam, w, h, 1, 2), plain)


def test_replacing_the_map_between_async_renders():
    """two sync=False renders on one stream with the map replaced in between: each gets the map set when it was
    enqueued (the re-upload waits for the first render; same size -- in place -- and a different size -- reallocated)"""
    import torch

    import bendy_tracer_b200 as bt
    w, h = 384, 216
    env1, env2, env3 = smooth_map(64, 128, 7), smooth_map(64, 128, 8), smooth_map(16, 32, 9)
    refs = []
    for env in (env1, env2, env3):
        sc, cam = engine_scene("scene", w, h, LENS_SCENE)
        sc.set_environment(env)
        refs.append(render(sc, cam, w, h, 2, 2))
    sc, cam = engine_scene("scene", w, h, LENS_SCENE)
    tracer = bt.Tracer(bt.Config(), seed=3)
    rc = bt.RenderConfig.with_samples_subsample(2, bt.Subsample(2))
    bufs = [bt.Buffer(w, h, device="cuda:0") for _ in range(3)]
    for env, buf in zip((env1, env2, env3), bufs):
        sc.set_environment(env)
        tracer.render(sc, cam, rc, buf, sync=False)
    torch.cuda.current_stream(0).synchronize()
    for buf, ref in zip(bufs, refs):
        assert np.array_equal(buf.data.cpu().numpy(), ref)


def write_pfm(path, rgb):
    h, w, _ = rgb.shape
    with open(path, "wb") as f:
        f.write(f"PF\n{w} {h}\n-1.0\n".encode() + np.ascontiguousarray(rgb[::-1], "<f4").tobytes())


def test_cli_renders_with_a_pfm_map(tmp_path):
    """bendy_b200_cli --environment sky.pfm renders what the API renders with the same map (the PFM's bottom-first rows
    flipped): the CLI runs one pass per iteration into a host buffer; so does the loop here"""
    import bendy_tracer_b200 as bt
    import oracle_ffi as O
    w, h, samples = 96, 54, 8
    env = smooth_map(32, 64, 10)
    env[:8] *= 3.0                                                     # an up / down asymmetry a wrong flip would show
    write_pfm(tmp_path / "sky.pfm", env)
    cli = os.path.join(ROOT, "bendy_tracer_b200", "csrc", "bendy_b200_cli")
    r = subprocess.run([cli, "--output", "full", "--width", str(w), "--height", str(h), "--samples", str(samples), "--scene",
                        O.scene_path("scene"), "--lens", ",".join(str(float(x)) for x in LENS_SCENE[0]), "--environment",
                        str(tmp_path / "sky.pfm"), "--screenshot", str(tmp_path / "out.png")], capture_output=True, text=True)
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


def _read_png(path):
    import zlib
    data = open(path, "rb").read()
    i, w, h, idat = 8, 0, 0, b""
    while i < len(data):
        n = int.from_bytes(data[i:i + 4], "big")
        kind, body = data[i + 4:i + 8], data[i + 8:i + 8 + n]
        if kind == b"IHDR":
            w, h = int.from_bytes(body[:4], "big"), int.from_bytes(body[4:8], "big")
        elif kind == b"IDAT":
            idat += body
        i += 12 + n
    raw = np.frombuffer(zlib.decompress(idat), np.uint8).reshape(h, w * 4 + 1)
    assert (raw[:, 0] == 0).all()                                      # filter type None: what the CLI writes
    return raw[:, 1:].reshape(h, w, 4)
