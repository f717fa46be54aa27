"""The equirectangular camera (bt_scene_set_camera_projection / Scene.set_camera_projection) on the host: the direction's
known answers in the oracle, the convention shared with the environment map (every ray lands in its pixel's texel, and a
panorama of an empty scene reproduces the map, filtered), an Einstein ring in a panorama, the API's argument checks and the
CLI's --projection.

The oracle side is tests/oracle_camera.cpp: the unchanged CPU oracle with the environment map (oracle_env.cpp) and the
projection routed into its camera_ray.  Semantics (DESIGN.md §3.6): pixel (x, y) with zero jitter looks at the centre of
texel (x, y) of a map of the image's size; the centre column looks along camera -z, columns grow towards camera +x, row 0
is the +y pole; a pinhole."""
import json
import os
import subprocess

import numpy as np
import pytest

import bendy_tracer_b200 as bt
import oracle_camera as OC
import oracle_env as OE
import oracle_ffi as O
from bendy_tracer_b200 import _ffi
from common import LENS_SCENE, oracle_render
from test_environment import DISC, D_L, R_S, disc_map, einstein_angle_f64, ring_scene
from test_gpu_environment import smooth_map

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CLI = os.path.join(ROOT, "bendy_tracer_b200", "csrc", "bendy_b200_cli")
F = np.float32


def pixel_dir(x, y, w, h):
    """the oracle's zero-jitter camera-space direction of pixel (x, y), u and v formed in f32 as camera_ray forms them"""
    pw, ph = F(2) * (F(1) / F(w)), F(2) * (F(1) / F(h))
    return OC.equirect_dir(F(x) * pw - F(1), F(y) * ph - F(1), pw, ph)


def texel_dir(r, c, h, w):
    """f64: the direction through the centre of texel (r, c) of an h x w map (env_lookup's convention)"""
    phi = ((c + 0.5) / w - 0.5) * 2 * np.pi
    theta = (0.5 - (r + 0.5) / h) * np.pi
    return np.array([np.cos(theta) * np.sin(phi), np.sin(theta), -np.cos(theta) * np.cos(phi)])


def texel_coords(d):
    """f64: env_lookup's texel coordinates (x, y) of directions d (n, 3), in units of texels of a 1 x 1 map"""
    phi = np.arctan2(d[:, 0], -d[:, 2])
    theta = np.arctan2(d[:, 1], np.hypot(d[:, 0], d[:, 2]))
    return 0.5 + phi / (2 * np.pi), 0.5 - theta / np.pi


# ---- the direction ------------------------------------------------------------------------------------------------------

def test_centre_pixel_looks_forward():
    """odd sizes: the centre pixel's zero-jitter direction is camera -z; the exact NDC origin too, bit for bit"""
    for w, h in ((9, 5), (255, 127)):
        assert np.allclose(pixel_dir(w // 2, h // 2, w, h), [0, 0, -1], atol=1e-6)
    assert np.array_equal(OC.equirect_dir(F(-0.0625), F(-0.125), F(0.125), F(0.25)), F([0, -0.0, -1]))


def test_left_edge_looks_backwards():
    """u' = -1: phi = -pi, the direction +z (sin of the rounded pi is 8.7e-8, the azimuth -pi or +pi)"""
    d = OC.equirect_dir(F(-1.125), F(-0.25), F(0.25), F(0.5))        # u' = -1, v' = 0
    assert np.allclose(d, [0, 0, 1], atol=1e-7)
    assert abs(abs(np.arctan2(d[0], -d[2])) - np.pi) < 1e-6


@pytest.mark.parametrize("w,h", [(16, 8), (33, 17), (64, 32)])
def test_every_pixel_looks_at_its_texel_centre(w, h):
    """rows: row 0 next to the +y pole, the last row next to -y; columns: the quarter columns along -x and +x; all pixels at
    their f64 texel centre to f32 rounding"""
    got = np.array([[pixel_dir(x, y, w, h) for x in range(w)] for y in range(h)], np.float64)
    want = np.array([[texel_dir(y, x, h, w) for x in range(w)] for y in range(h)])
    assert np.abs(got - want).max() < 2e-6
    assert (got[0, :, 1] > np.cos(np.pi / h)).all() and (got[-1, :, 1] < -np.cos(np.pi / h)).all()
    if w % 4 == 0:                                                  # u' = -1/2 and +1/2 lie on column boundaries
        pw, ph = F(2) / F(w), F(2) / F(h)
        for u, x in ((-0.5, -1.0), (0.5, 1.0)):
            d = OC.equirect_dir(F(u) - pw / F(2), F(-ph / F(2)), pw, ph)
            assert np.allclose(d, [x, 0, 0], atol=1e-7), (u, d)


def camera_doc(rotation=None, translation=(0.0, 0.0, 0.0), focus=None):
    """a scene of one camera (scene.json.gz's lens parameters) and one tiny black sphere 10 units along world +x, root
    Emissive{white, 1}"""
    base = O.read_scene_json(O.scene_path("scene"))
    cam = json.loads(json.dumps(base["objects"]["collection"]["0"]))
    cam["inner"]["Camera"]["focus"] = focus
    m = [float(F(v)) for v in (np.eye(3) if rotation is None else np.asarray(rotation)).T.ravel()] + [float(F(v)) for v in translation]
    cam["transform"] = {"transform_world": m, "transform_local": m, "transform_parent": None}
    at = [float(F(v)) for v in np.add(translation, [10.0, 0.0, 0.0])]
    sphere = {"object_ref": 1, "tag": None, "flags": {"bits": 0},
              "transform": {"transform_world": [1, 0, 0, 0, 1, 0, 0, 0, 1] + at,
                            "transform_local": [1, 0, 0, 0, 1, 0, 0, 0, 1] + at, "transform_parent": None},
              "inner": {"Sphere": {"material": 1, "volume": None, "radius": 1e-3}}, "children": None}
    doc = {"roots": [], "root_material": 0, "objects": {"collection": {"0": cam, "1": sphere}, "next_key": 2},
           "data": {"collection": {"0": {"inner": {"Material": {"Emissive": {"albedo": {"r": 1.0, "g": 1.0, "b": 1.0}, "intensity": 1.0}}}},
                                   "1": {"inner": {"Material": {"Flat": {"albedo": {"r": 0.0, "g": 0.0, "b": 0.0}}}}}},
                    "next_key": 2}}
    return json.loads(json.dumps(doc))


def rotation(seed):
    q = np.random.default_rng(seed).normal(size=4)
    w, x, y, z = q / np.linalg.norm(q)
    return np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w)],
                     [2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w)],
                     [2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)]])


def panorama_rays(osc, w, h, spp, seed=1):
    """the oracle's camera rays of every pixel, spp each, subsample None: (h * w * spp, 6) origins and directions"""
    xs, ys = np.meshgrid(np.arange(w), np.arange(h))
    xs, ys = np.repeat(xs.ravel(), spp), np.repeat(ys.ravel(), spp)
    return osc.camera_rays(0, O.make_config(samples=spp), w, h, xs, ys, np.tile(np.arange(spp), w * h), seed=seed)


def test_rotated_camera_rotates_every_direction():
    """the same draws through a rotated, translated camera: every direction is R times the unrotated one, every origin the
    camera's position"""
    w, h, spp = 24, 12, 3
    rays = {}
    for key, r, t in (("plain", None, (0, 0, 0)), ("rotated", rotation(3), (1.5, -2.0, 0.25))):
        osc = OC.CameraOracleScene(camera_doc(r, t))
        osc.set_projection(0, OC.EQUIRECTANGULAR)
        rays[key] = panorama_rays(osc, w, h, spp)
    R = rotation(3).astype(np.float32).astype(np.float64)
    assert np.abs(rays["rotated"][:, 3:] - rays["plain"][:, 3:] @ R.T).max() < 1e-6
    assert np.array_equal(rays["rotated"][:, :3], np.tile(F([1.5, -2.0, 0.25]), (len(rays["rotated"]), 1)))
    assert np.array_equal(rays["plain"][:, :3], np.zeros_like(rays["plain"][:, :3]))


# ---- the convention: every ray in its pixel's texel ------------------------------------------------------------------------

@pytest.mark.parametrize("focus", [None, 12.5])
def test_every_ray_lands_in_its_pixels_texel(focus):
    """subsample None: a ray of pixel (x, y) converted with env_lookup's formula lands in [x - 0.5, x + 0.5] x [y - 0.5, y + 0.5]
    (texel units), up to atan2 rounding.  On the first and last rows the azimuth of a ray at the pole is undefined (cos of the
    rounded pi/2 is -4.4e-8): there it may come out half a turn off.  Focus or not, every origin is the camera position."""
    w, h, spp = 40, 20, 8
    R, t = rotation(5), (0.5, 1.0, -3.0)
    osc = OC.CameraOracleScene(camera_doc(R, t, focus))
    osc.set_projection(0, OC.EQUIRECTANGULAR)
    rays = panorama_rays(osc, w, h, spp, seed=7)
    assert np.array_equal(rays[:, :3], np.tile(F(t), (len(rays), 1)))
    d = rays[:, 3:].astype(np.float64) @ R.astype(np.float32).astype(np.float64)   # back to camera space
    u, v = texel_coords(d)
    tx, ty = u * w - 0.5, v * h - 0.5
    xs, ys = np.repeat(np.tile(np.arange(w), h), spp), np.repeat(np.repeat(np.arange(h), w), spp)
    eps = 1e-3

    def col_ok(tx):
        off = (tx - xs + w / 2) % w - w / 2                           # columns wrap
        return np.abs(off) <= 0.5 + eps

    ok = col_ok(tx) & (np.abs(ty - ys) <= 0.5 + eps)
    pole = (ys == 0) | (ys == h - 1)
    assert ok[~pole].all(), np.flatnonzero(~ok & ~pole)[:10]
    assert (ok | (pole & col_ok(tx + w / 2) & (np.abs(ty - ys) <= 0.5 + eps)))[pole].all()


# ---- the round trip: a panorama of an empty scene is the map, filtered --------------------------------------------------------

def filtered_map(env):
    """what a panorama of env at env's size converges to: bilinear lookups under box jitter, the separable kernel
    [1/8, 3/4, 1/8]; columns wrap; rows clamp, so the first and last rows keep 7/8 of their own texel and take 1/8 of the
    next one inwards"""
    e = env.astype(np.float64)
    cols = 0.75 * e + 0.125 * (np.roll(e, 1, axis=1) + np.roll(e, -1, axis=1))
    out = 0.75 * cols
    out[1:] += 0.125 * cols[:-1]
    out[:-1] += 0.125 * cols[1:]
    out[0] += 0.125 * cols[0]
    out[-1] += 0.125 * cols[-1]
    return out


def sphere_mask(w, h):
    """the pixels around world +x, where camera_doc's tiny sphere is"""
    mask = np.zeros((h, w), bool)
    cx, cy = int(0.75 * w), h // 2
    mask[cy - 2:cy + 2, cx - 2:cx + 2] = True
    return mask


def round_trip_error(img_a, img_b, n, env):
    """(MAE of the mean of two independent renders against the filtered map, MAE of their half-difference: the noise
    of that mean) over the pixels away from the sphere"""
    h, w, _ = env.shape
    keep = ~sphere_mask(w, h)
    mean = (img_a[..., :3].astype(np.float64) + img_b[..., :3]) / (2 * n)
    noise = np.abs(img_a[..., :3].astype(np.float64) - img_b[..., :3]) / (2 * n)
    return np.abs(mean - filtered_map(env))[keep].mean(), noise[keep].mean()


def test_round_trip_reproduces_the_map():
    """camera_doc at the identity, a smooth map, the panorama at the map's size and 2 x 128 spp: the mean image equals the
    filtered map within the Monte-Carlo noise (the mean of two independent renders against the mean absolute half-difference
    of the two); a half-texel shift of the convention would be ~20 x that"""
    h, w, spp = 24, 48, 128
    env = smooth_map(h, w, 21)
    osc = OC.CameraOracleScene(camera_doc())
    osc.set_environment(env)
    osc.set_projection(0, OC.EQUIRECTANGULAR)
    a, n, _ = oracle_render(osc, 0, w, h, spp, seed=1)
    b, _, _ = oracle_render(osc, 0, w, h, spp, seed=2)
    err, noise = round_trip_error(a, b, n, env)
    shifted = np.abs(filtered_map(env) - filtered_map(np.roll(env, 1, axis=1))).mean() / 2
    print(f"round trip: MAE {err:.2e}, noise {noise:.2e}, half-texel shift {shifted:.2e}")
    assert err <= 1.5 * noise, (err, noise)
    assert shifted > 10 * noise
    assert (filtered_map(np.ones((4, 6, 3))) == 1).all()            # the kernel's weights sum to one, rows included


# ---- an Einstein ring in a panorama -------------------------------------------------------------------------------------------

def test_einstein_ring_in_a_panorama():
    """test_environment.py's ring on a 512 x 256 panorama at 4 spp: the ring's intensity-weighted angle to the axis is the f64
    Einstein angle within half a pixel plus the disc's radius; without the lens the light is a spot at the panorama's centre"""
    doc, pos, fwd, right = ring_scene()
    theta_e = einstein_angle_f64(pos, fwd, right)
    w, h, spp = 512, 256, 4
    osc = OC.CameraOracleScene(doc)
    osc.set_projection(0, OC.EQUIRECTANGULAR)
    osc.set_environment(disc_map(fwd))
    dirs = panorama_rays(osc, w, h, spp)[:, 3:].astype(np.float64)
    ang = np.arccos(np.clip((dirs @ fwd) / np.linalg.norm(dirs, axis=1), -1, 1)).reshape(h, w, spp).mean(-1)
    pixel = np.pi / h
    for lensed in (True, False):
        osc.set_lenses(np.array([[*(pos + D_L * fwd), R_S]], np.float32) if lensed else np.zeros((0, 4), np.float32))
        img, n, _ = osc.render(0, O.make_config(samples=spp), w, h, seed=1)
        lum = img[..., :3].mean(-1) / n
        assert lum.sum() > 0
        mean_angle = float((lum * ang).sum() / lum.sum())
        yy, xx = np.mgrid[:h, :w]
        cy, cx = (lum * yy).sum() / lum.sum(), (lum * xx).sum() / lum.sum()
        assert abs(cy - (h - 1) / 2) < 1.5 and abs(cx - (w - 1) / 2) < 1.5, (cx, cy)    # centred on the axis either way
        if lensed:
            assert abs(mean_angle - theta_e) <= pixel / 2 + DISC, (mean_angle, theta_e)
        else:
            assert mean_angle <= DISC + pixel / 2, mean_angle
            assert (ang[lum > 0] <= DISC + 2 * np.pi / 2048 + pixel).all()


# ---- the oracle without a projection is oracle_env --------------------------------------------------------------------------

def test_camera_oracle_without_a_projection_is_the_env_oracle():
    for name, lens, env in (("scene", LENS_SCENE, smooth_map(16, 32, 3)), ("cloud", None, None), ("cornell", None, None)):
        w, h = 48, 27
        env_osc = OE.load_pair(name, w, h, lenses=lens)[0]
        osc, _, cam = OC.load_pair(name, w, h, lenses=lens, projection=OC.PERSPECTIVE)
        if env is not None:
            env_osc.set_environment(env)
            osc.set_environment(env)
        ref = oracle_render(env_osc, cam, w, h, 1, 2, seed=4)[0]
        assert np.array_equal(oracle_render(osc, cam, w, h, 1, 2, seed=4)[0], ref), name
        osc.set_projection(cam, OC.EQUIRECTANGULAR)
        assert not np.array_equal(oracle_render(osc, cam, w, h, 1, 2, seed=4)[0], ref), name
        osc.set_projection(cam, OC.PERSPECTIVE)
        assert np.array_equal(oracle_render(osc, cam, w, h, 1, 2, seed=4)[0], ref), name


# ---- host API -----------------------------------------------------------------------------------------------------------------

def test_invalid_calls_are_rejected():
    sc = bt.Scene.load(O.scene_path("scene"))
    cam = sc.find_by_tag("camera")
    before = sc.to_json()
    with pytest.raises(bt.ScenePanic) as aspect:
        sc.set_camera_aspect(1, 1.5)                                  # object 1 is not a camera
    with pytest.raises(bt.ScenePanic) as proj:
        sc.set_camera_projection(1, bt.Projection.EQUIRECTANGULAR)
    assert proj.value.message == aspect.value.message
    with pytest.raises(bt.ScenePanic):
        sc.set_camera_projection(10 ** 6, bt.Projection.EQUIRECTANGULAR)
    for bad in (-1, 2, 7, 1 << 30):
        assert _ffi.lib.bt_scene_set_camera_projection(sc.handle, cam, bad) == _ffi.ERR_INVALID_ARG, bad
    with pytest.raises(bt.BendyError) as e:
        sc.set_camera_projection(cam, 5)
    assert e.value.code == _ffi.ERR_INVALID_ARG
    assert _ffi.lib.bt_scene_set_camera_projection(None, cam, 1) == _ffi.ERR_INVALID_ARG
    assert sc.to_json() == before
    # that the rejected calls left the projection as it was is checked on the GPU (test_gpu_panorama.py)


def test_projection_is_not_part_of_the_wire_format():
    for name in ("scene", "cloud", "cornell"):
        sc = bt.Scene.load(O.scene_path(name))
        cam = sc.find_by_tag("camera")
        plain = sc.to_json()
        sc.set_camera_projection(cam, bt.Projection.EQUIRECTANGULAR)
        assert sc.to_json() == plain
        sc.set_camera_aspect(cam, 2.0)
        aspect = sc.to_json()
        sc.set_camera_projection(cam, bt.Projection.PERSPECTIVE)
        assert sc.to_json() == aspect
        assert bt.Scene.from_json(aspect).to_json() == aspect


# ---- CLI: --projection ----------------------------------------------------------------------------------------------------------

def run_cli(*args):
    return subprocess.run([CLI, "--output", "full", "--width", "64", "--height", "32", "--samples", "0",
                           "--scene", O.scene_path("scene"), *args], capture_output=True, text=True)


def test_cli_projection_dry_run(tmp_path):
    r = run_cli("--projection", "equirectangular")
    assert r.returncode == 0 and "projection equirectangular: 64 x 32" in r.stderr, r.stderr
    r = run_cli("--projection", "perspective")
    assert r.returncode == 0 and "projection" not in r.stderr, r.stderr
    sky = tmp_path / "sky.pfm"
    sky.write_bytes(b"PF\n4 2\n-1.0\n" + np.ones(24, "<f4").tobytes())
    r = run_cli("--projection", "equirectangular", "--lens", ",".join(str(float(x)) for x in LENS_SCENE[0]), "--environment", str(sky))
    assert r.returncode == 0 and "projection equirectangular" in r.stderr and "environment map" in r.stderr, r.stderr


@pytest.mark.parametrize("value", ["fisheye", "Equirectangular", ""])
def test_cli_projection_bad_value(value):
    r = run_cli("--projection", value)
    assert r.returncode != 0 and "\nerror: " in "\n" + r.stderr and "--projection" in r.stderr, (r.returncode, r.stderr)
    r = run_cli("--projection")
    assert r.returncode != 0 and "missing value for --projection" in r.stderr, r.stderr
