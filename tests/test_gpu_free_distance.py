"""The free-distance grid refresh of the lensed stepper (kernels.cu: grid_bound_fetch): one straight sequence for lanes inside
and outside the grid's box, the scene-spanning ("far") spheres evaluated from the call's constants.  A chord the bound skips
could never hit anything, so every frame must equal, bit for bit, the frame that intersects every chord (BT_LENS_NO_SKIP) --
in cases chosen to send the refresh down each of its paths: rays that leave the box in every direction, a camera outside
the box, 0, 1 and 2 far spheres, rects and boxes.  The pooled kernel's counters tell which paths ran."""
import json

import numpy as np
import pytest

from common import LENS_SCENE, synthetic_scene

pytestmark = pytest.mark.gpu

LENS_CORNELL2 = np.array([[0.3, 2.2, 2.0, 0.1]], np.float32)


def _render(sc, cam, w, h, passes=2, seed=3):
    import bendy_tracer_b200 as bt
    buf = bt.Buffer(w, h, device="cuda:0")
    bt.Tracer(bt.Config(), seed=seed).render(sc, cam, bt.RenderConfig.with_samples_subsample(passes, bt.Subsample(2)), buf)
    return buf.data.cpu().numpy()


def _pool_stats(sc, cam, w, h, passes=2, seed=3):
    import bendy_tracer_b200 as bt
    rc = bt.RenderConfig.with_samples_subsample(passes, bt.Subsample(2))
    return bt.Tracer(bt.Config(), seed=seed).render_pool_stats(sc, cam, rc, w, h)


def _skip_equals_no_skip(sc, cam, lens, w, h, stats=True):
    """the frame with chord skipping equals the one without; returns the pooled kernel's counters of the skipping render
    (stats: the scene is one a content-specialised pooled kernel with counters renders)"""
    import bendy_tracer_b200 as bt
    sc.set_lenses(lens)
    got = _render(sc, cam, w, h)
    stats = _pool_stats(sc, cam, w, h) if stats else None
    sc.set_lenses(lens, bt.LensConfig(no_skip=True))
    ref = _render(sc, cam, w, h)
    sc.set_lenses(lens)
    assert np.isfinite(got).all()
    assert np.array_equal(got, ref)
    return stats


def _check_counters(st):
    """the refresh counters are consistent with one another and with the STEP iterations"""
    lanes = st["refresh_lanes_grid"] + st["refresh_lanes_outside"]
    assert st["refresh_mixed_iterations"] <= st["refresh_iterations"] <= st["step_iterations"]
    assert st["refresh_iterations"] <= lanes <= 32 * st["refresh_iterations"]
    assert lanes <= st["step_lanes"]
    if st["refresh_lanes_grid"] == 0 or st["refresh_lanes_outside"] == 0:
        assert st["refresh_mixed_iterations"] == 0


def _load(name, w, h):
    import bendy_tracer_b200 as bt
    import oracle_ffi as O
    sc = bt.Scene.load(O.scene_path(name))
    cam = sc.find_by_tag("camera")
    sc.set_camera_aspect(cam, float(np.float32(w) / np.float32(h)))
    return sc, cam


def test_panorama_inside_the_scene_leaves_the_box_everywhere():
    """an equirectangular panorama from the camera of scene.json.gz: bent rays leave the grid's box in every direction"""
    import bendy_tracer_b200 as bt
    w, h = 128, 64
    sc, cam = _load("scene", w, h)
    sc.set_camera_projection(cam, bt.Projection.EQUIRECTANGULAR)
    st = _skip_equals_no_skip(sc, cam, LENS_SCENE, w, h)
    _check_counters(st)
    assert st["refresh_lanes_grid"] > 0 and st["refresh_lanes_outside"] > 0 and st["refresh_mixed_iterations"] > 0


def test_camera_outside_the_box():
    """the camera pulled back 40 units (far outside the grid's box, inside the ground sphere's reach): every path starts
    with out-of-box refreshes"""
    w, h = 128, 72
    sc, cam = _load("scene", w, h)
    sc.apply_transform(cam, [1, 0, 0, 0, 1, 0, 0, 0, 1, 0.0, 3.0, 40.0])
    sc.commit()
    st = _skip_equals_no_skip(sc, cam, LENS_SCENE, w, h)
    _check_counters(st)
    assert st["refresh_lanes_outside"] > 0


def _sphere_scene(n_far):
    """synthetic spheres (a linear-scan scene) with 0, 1 or 2 scene-spanning spheres"""
    doc = synthetic_scene(24, 0, 0, seed=4, extent=3.0)
    objs = doc["objects"]["collection"]
    if n_far == 0:
        del objs["1"]                                  # the r = 100 ground
    if n_far == 2:
        key = doc["objects"]["next_key"]
        sky = json.loads(json.dumps(objs["1"]))
        sky["object_ref"] = key
        sky["inner"]["Sphere"]["radius"] = 80.0
        for t in ("transform_world", "transform_local"):
            sky["transform"][t][9:12] = [0.0, 0.0, -95.0]
        objs[str(key)] = sky
        doc["objects"]["next_key"] = key + 1
    return doc


@pytest.mark.parametrize("n_far", [0, 1, 2])
def test_far_spheres_from_the_constants(n_far):
    import bendy_tracer_b200 as bt
    w, h = 128, 72
    sc = bt.Scene.from_json(json.dumps(_sphere_scene(n_far)))
    assert sc.info()["n_bvh_nodes"] == 0
    cam = sc.find_by_tag("camera")
    sc.set_camera_aspect(cam, float(np.float32(w) / np.float32(h)))
    for projection in (bt.Projection.PERSPECTIVE, bt.Projection.EQUIRECTANGULAR):
        sc.set_camera_projection(cam, projection)
        st = _skip_equals_no_skip(sc, cam, LENS_SCENE, w, h)
        _check_counters(st)
        assert st["refresh_lanes_grid"] > 0                # the grid serves this scene


def test_cornell2_rects_and_boxes():
    w, h = 128, 72
    sc, cam = _load("cornell2", w, h)
    _skip_equals_no_skip(sc, cam, LENS_CORNELL2, w, h, stats=False)    # (a generic kernel renders it: no counters)


def test_commit_moves_the_far_sphere_constants():
    """a transform edit of the ground sphere (a far sphere: evaluated from the call's constants outside the box), committed,
    renders what the same state flattened from scratch renders -- and not what the old position rendered"""
    import bendy_tracer_b200 as bt
    w, h = 128, 64
    sc, cam = _load("scene", w, h)
    sc.set_camera_projection(cam, bt.Projection.EQUIRECTANGULAR)
    sc.set_lenses(LENS_SCENE)
    before = _render(sc, cam, w, h)
    sc.apply_transform(1, [1, 0, 0, 0, 1, 0, 0, 0, 1, 0.0, -100.6, 0.0])
    sc.commit()
    after = _render(sc, cam, w, h)
    fresh = bt.Scene.from_json(sc.to_json())
    fresh.set_camera_aspect(cam, float(np.float32(w) / np.float32(h)))
    fresh.set_camera_projection(cam, bt.Projection.EQUIRECTANGULAR)
    fresh.set_lenses(LENS_SCENE)
    assert np.array_equal(after, _render(fresh, cam, w, h))
    assert not np.array_equal(after, before)
    sc.set_lenses(LENS_SCENE, bt.LensConfig(no_skip=True))
    assert np.array_equal(after, _render(sc, cam, w, h))
