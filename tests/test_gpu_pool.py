"""The pooled render kernel (csrc/render_pool.cuh) against the one-path-per-lane kernel (render_body).

Both run the same per-path arithmetic and form every pixel sum in path order (the pooled kernel retires
finished paths in order), so their images must be BIT-IDENTICAL for every scene, output, frame shape,
pool size, CTA size and arithmetic flavour -- whatever the scheduling.  Parity with the CPU oracle is
asserted on the default path in test_gpu_parity.py; this file pins the two schedulers to each other.
"""
import numpy as np
import pytest

from common import LENS_SCENE, LENS_VOLUME, SCENES, cornell_with_cuboid_light

pytestmark = pytest.mark.gpu


def _render(scene, cam, w, h, passes, sub, output=0, seed=3, sample_base=0, device="cuda:0", **tuning):
    import bendy_tracer_b200 as bt
    eng = bt.Engine.default(0)
    eng.set_tuning(**tuning)
    try:
        buf = bt.Buffer(w, h, device=device)
        tr = bt.Tracer(bt.Config(output=bt.Output(output)), engine=eng, seed=seed)
        tr.render(scene, cam, bt.RenderConfig.with_samples_subsample(passes, bt.Subsample(sub)), buf, sample_base=sample_base)
        return buf.data.cpu().numpy() if device else buf.data.copy()
    finally:
        eng.set_tuning(**{k: None for k in tuning})


def _scene(name, w, h, lens=None, precision=None):
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


CASES = [(n, None) for n in SCENES] + [("scene", LENS_SCENE), ("cloud", LENS_VOLUME), ("cornell2", np.array([[0.0, 2.5, 4.0, 0.1]], np.float32))]


@pytest.mark.parametrize("name,lens", CASES, ids=[f"{n}{'+lens' if l is not None else ''}" for n, l in CASES])
@pytest.mark.parametrize("pool_w", [1, 3, 4])
def test_pool_equals_lane_kernel(name, lens, pool_w):
    w, h = 136, 76                                   # 17 x 19 tiles of 8 x 4
    sc, cam = _scene(name, w, h, lens)
    ref = _render(sc, cam, w, h, 3, 2, pool_w=0)
    got = _render(sc, cam, w, h, 3, 2, pool_w=pool_w)
    assert np.array_equal(got, ref), f"{(got != ref).any(-1).sum()} pixels differ"
    assert np.isfinite(got).all() and got[..., :3].sum() > 0


@pytest.mark.parametrize("name,lens", [("cornell", None), ("scene", LENS_SCENE), ("volume", None)])
@pytest.mark.parametrize("output", [1, 2, 3])
def test_pool_aov_outputs(name, lens, output):
    w, h = 96, 64
    sc, cam = _scene(name, w, h, lens)
    ref = _render(sc, cam, w, h, 2, 2, output=output, pool_w=0)
    got = _render(sc, cam, w, h, 2, 2, output=output, pool_w=3)
    assert np.array_equal(got, ref)


@pytest.mark.parametrize("w,h", [(1, 1), (7, 3), (9, 5), (64, 33), (250, 17)])
def test_pool_ragged_frames(w, h):
    """frames that are not whole 8 x 4 tiles, down to one pixel"""
    for name, lens in (("cornell2", None), ("scene", LENS_SCENE)):
        sc, cam = _scene(name, w, h, lens)
        ref = _render(sc, cam, w, h, 5, 0, pool_w=0)
        got = _render(sc, cam, w, h, 5, 0, pool_w=2)
        assert np.array_equal(got, ref)


@pytest.mark.parametrize("passes,sub", [(1, 0), (1, 3), (40, 0), (7, 2)])
def test_pool_path_counts(passes, sub):
    """1 .. 40 paths per pixel: fewer than, equal to and more than the in-order retirement window (16)"""
    w, h = 64, 32
    for name, lens in (("cornell", None), ("scene", LENS_SCENE), ("cloud", None)):
        sc, cam = _scene(name, w, h, lens)
        ref = _render(sc, cam, w, h, passes, sub, sample_base=5, pool_w=0)
        got = _render(sc, cam, w, h, passes, sub, sample_base=5, pool_w=3)
        assert np.array_equal(got, ref)


@pytest.mark.parametrize("knobs", [dict(pool_threads=32), dict(pool_threads=64), dict(pool_threads=128), dict(pool_threads=1024),
                                   dict(pool_refill=1), dict(pool_refill=32), dict(pool_step_min=0), dict(pool_step_min=32)])
def test_pool_scheduling_knobs_change_nothing(knobs):
    w, h = 120, 68
    for name, lens in (("scene", LENS_SCENE), ("cloud", LENS_VOLUME), ("cornell2", None)):
        sc, cam = _scene(name, w, h, lens)
        ref = _render(sc, cam, w, h, 2, 2, pool_w=0)
        got = _render(sc, cam, w, h, 2, 2, pool_w=3, **knobs)
        assert np.array_equal(got, ref), (name, knobs)


@pytest.mark.parametrize("precision", ["fast", "exact"])
def test_pool_flavours_and_generic_kernels(precision):
    """Both arithmetic flavours; lens tables of 2 masses (shared-memory walk), the exact-rsqrt stepper and a
    LIGHT Cuboid run the generic (not content-specialised) pooled kernels.  The EXACT flavour (every operation
    written out, no contraction) is bit-identical across the two kernels everywhere.  In the FAST flavour the
    compiler contracts a * b + c per kernel: the content-specialised pairs still agree bit for bit, two
    separately compiled generic kernels agree to rounding (DESIGN.md, "Two arithmetic flavours")."""
    import json

    import bendy_tracer_b200 as bt
    w, h = 96, 64
    two = np.array([[1.362, 1.577, 6.114, 0.15], [0.5, 1.0, 3.0, 0.05]], np.float32)
    for name, lens, cfg, generic in (("scene", LENS_SCENE, None, False), ("scene", two, None, True),
                                     ("scene", LENS_SCENE, bt.LensConfig(exact_rsqrt=True), True), ("cloud", None, None, False),
                                     ("cloud", LENS_VOLUME, None, False), ("cornell2", None, None, False)):
        sc, cam = _scene(name, w, h, None, precision)
        if lens is not None:
            sc.set_lenses(lens, cfg)
        ref = _render(sc, cam, w, h, 2, 2, pool_w=0)
        got = _render(sc, cam, w, h, 2, 2, pool_w=3)
        if precision == "exact" or not generic:
            assert np.array_equal(got, ref), (name, precision)
        else:
            assert (np.abs(got - ref).mean(axis=(0, 1)) / 8 <= 1e-6).all(), (name, precision)
    sc = bt.Scene.from_json(json.dumps(cornell_with_cuboid_light()))
    sc.set_precision(precision)
    cam = sc.find_by_tag("camera")
    sc.set_camera_aspect(cam, 1.5)
    got, ref = _render(sc, cam, w, h, 2, 2, pool_w=3), _render(sc, cam, w, h, 2, 2, pool_w=0)
    assert np.array_equal(got, ref) if precision == "exact" else (np.abs(got - ref).mean(axis=(0, 1)) / 8 <= 1e-6).all()


def test_pool_falls_back_beyond_its_counters():
    """max_bounces above 254 does not fit the pooled kernel's packed counters: the lane kernel renders the call"""
    import bendy_tracer_b200 as bt
    w, h = 64, 32
    sc, cam = _scene("cornell2", w, h)
    eng = bt.Engine.default(0)
    imgs = []
    for pool_w in (0, 3):
        eng.set_tuning(pool_w=pool_w)
        try:
            buf = bt.Buffer(w, h, device="cuda:0")
            bt.Tracer(bt.Config(max_bounces=300), engine=eng, seed=1).render(sc, cam, bt.RenderConfig.with_samples(3), buf)
            imgs.append(buf.data.cpu().numpy())
        finally:
            eng.set_tuning(pool_w=None)
    assert np.array_equal(imgs[0], imgs[1])


def test_pool_host_buffer_bands():
    """bt_render with a host frame pipelines row bands through the pooled kernel: same bits as one piece"""
    w, h = 256, 200
    sc, cam = _scene("scene", w, h, LENS_SCENE)
    ref = _render(sc, cam, w, h, 1, 2, pool_w=0)
    for bands in (1, 3):
        got = _render(sc, cam, w, h, 1, 2, device=None, pool_w=3, host_bands=bands)
        assert np.array_equal(got, ref)


def test_pool_full_size_c3_slice():
    """the C3 frame (3840 x 2160) at 4 spp: persistent grid, > 100 tiles per warp"""
    w, h = 3840, 2160
    sc, cam = _scene("scene", w, h, LENS_SCENE)
    ref = _render(sc, cam, w, h, 1, 2, pool_w=0)
    got = _render(sc, cam, w, h, 1, 2, pool_w=3)
    assert np.array_equal(got, ref)


@pytest.mark.parametrize("precision", ["exact", "fast"])
def test_pool_bvh_traversal_equals_lane_kernel(precision):
    """BVH scenes under a flat field: the pooled kernel runs the traversal as NODE / LEAF phases over its slots
    (stack: 8 levels in shared memory, the rest in the arena).  Same rays, same tests, same tie rule as the lane
    kernel's traversal: bit-identical in the exact flavour, to contraction rounding in the fast one (generic kernels)."""
    import json

    import bendy_tracer_b200 as bt
    from common import synthetic_scene
    w, h = 136, 76
    docs = [json.dumps(synthetic_scene(300, 100, 20, seed=4)), json.dumps(synthetic_scene(3000, 500, 100, seed=5, extent=6.0))]
    scenes = [bt.Scene.from_json(d) for d in docs]
    sc2, _ = _scene("cornell2", w, h)
    sc2.set_accel("bvh")
    for sc in scenes + [sc2]:
        sc.set_precision(precision)
        cam = sc.find_by_tag("camera")
        sc.set_camera_aspect(cam, float(np.float32(w) / np.float32(h)))
        assert sc.info()["n_bvh_nodes"] > 0
        ref = _render(sc, cam, w, h, 2, 2, pool_w=0)
        for pool_w, turn in ((1, 1), (2, 2), (3, 4)):
            got = _render(sc, cam, w, h, 2, 2, pool_w=pool_w, steps_per_turn=turn)
            if precision == "exact":
                assert np.array_equal(got, ref), (pool_w, f"{(got != ref).any(-1).sum()} pixels differ")
            else:
                assert (np.abs(got - ref).mean(axis=(0, 1)) / 8 <= 1e-6).all(), pool_w
        for output in (1, 2, 3):
            ref = _render(sc, cam, w, h, 1, 2, output=output, pool_w=0)
            got = _render(sc, cam, w, h, 1, 2, output=output, pool_w=2)
            assert np.array_equal(got, ref) if precision == "exact" else np.abs(got - ref).mean() <= 1e-5, output
        # the traversal stack's slow tail (local memory in the lane kernel, the arena in the pooled one) holds everything
        # beyond ONE shared-memory level here: same images
        ref = _render(sc, cam, w, h, 2, 2, pool_w=0)
        for pool_w in (0, 3):
            got = _render(sc, cam, w, h, 2, 2, pool_w=pool_w, bvh_stack_k=1)
            if precision == "exact" or pool_w == 0:
                assert np.array_equal(got, ref), (pool_w, "bvh_stack_k=1")
            else:
                assert (np.abs(got - ref).mean(axis=(0, 1)) / 8 <= 1e-6).all(), pool_w


def test_pool_stats_only_from_the_pooled_kernel():
    """bt_render_pool_stats reports the pooled kernel's scheduling counters, or BT_ERR_UNSUPPORTED when the call would not run
    a content-specialised pooled kernel: a BVH scene, or max_bounces beyond the pooled kernel's packed counters"""
    import json

    import bendy_tracer_b200 as bt
    from common import synthetic_scene
    w, h, passes = 64, 32, 2
    rc = bt.RenderConfig.with_samples_subsample(passes, bt.Subsample(2))
    sc, cam = _scene("scene", w, h, LENS_SCENE)
    stats = bt.Tracer(bt.Config(), seed=1).render_pool_stats(sc, cam, rc, w, h)
    assert stats["paths_issued"] == stats["paths_retired"] == w * h * passes * 4
    with pytest.raises(bt.BendyError) as e:
        bt.Tracer(bt.Config(max_bounces=300), seed=1).render_pool_stats(sc, cam, rc, w, h)
    assert e.value.code == bt._ffi.ERR_UNSUPPORTED
    bvh = bt.Scene.from_json(json.dumps(synthetic_scene()))
    assert bvh.info()["n_bvh_nodes"] > 0
    cam = bvh.find_by_tag("camera")
    bvh.set_camera_aspect(cam, float(np.float32(w) / np.float32(h)))
    with pytest.raises(bt.BendyError) as e:
        bt.Tracer(bt.Config(), seed=1).render_pool_stats(bvh, cam, rc, w, h)
    assert e.value.code == bt._ffi.ERR_UNSUPPORTED
