"""The environment map (bt_scene_set_environment / Scene.set_environment) on the host: the lookup's known answers in the
oracle, the Einstein ring it makes visible under a lens, the API's argument checks and the CLI's PFM reader.

The oracle side is oracle/bendy_oracle.cpp with a map set (OracleScene.set_environment): its sample_root multiplies the
colour by the map's lookup.  Semantics (DESIGN.md §3.5): an escaping path's colour is sample_root's colour times the bilinear lookup of
an equirectangular map in its escape direction; row 0 is the +y pole, the centre column looks along -z."""
import ctypes as C
import json
import os
import subprocess

import numpy as np
import pytest

import bendy_tracer_b200 as bt
import oracle_ffi as O
from bendy_tracer_b200 import _ffi
from common import LENS_SCENE, LENS_VOLUME, load_pair, oracle_render

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CLI = os.path.join(ROOT, "bendy_tracer_b200", "csrc", "bendy_b200_cli")


def random_map(h, w, seed):
    return np.random.default_rng(seed).uniform(0.0, 1.0, (h, w, 3)).astype(np.float32)


def texel_dir(r, c, h, w):
    """the direction through the centre of texel (r, c)"""
    phi = ((c + 0.5) / w - 0.5) * 2 * np.pi
    theta = (0.5 - (r + 0.5) / h) * np.pi
    return np.array([np.cos(theta) * np.sin(phi), np.sin(theta), -np.cos(theta) * np.cos(phi)])


def lerp(a, b, t):
    return a + (b - a) * np.float32(t)


# ---- the lookup ---------------------------------------------------------------------------------------------------

def test_texel_centre_returns_the_texel():
    h, w = 16, 32
    env = random_map(h, w, 1)
    for r in range(h):
        for c in range(0, w, 3):
            got = O.env_lookup(env, texel_dir(r, c, h, w))
            assert np.allclose(got, env[r, c], atol=2e-5), (r, c)


def test_forward_direction_is_the_map_centre():
    """d = (0, 0, -1): u = v = 0.5, i.e. the corner shared by the four central texels of an even-sized map"""
    h, w = 8, 12
    env = random_map(h, w, 2)
    got = O.env_lookup(env, [0.0, 0.0, -1.0])
    r, c = h // 2 - 1, w // 2 - 1
    want = lerp(lerp(env[r, c], env[r, c + 1], 0.5), lerp(env[r + 1, c], env[r + 1, c + 1], 0.5), 0.5)
    assert np.array_equal(got, want)
    # odd-sized: the centre texel exactly
    env = random_map(7, 9, 3)
    assert np.array_equal(O.env_lookup(env, [0.0, 0.0, -1.0]), env[3, 4])
    # +x is a quarter turn right of the centre column (x = 0.75 W - 0.5), -x a quarter turn left, +z the seam
    assert np.allclose(O.env_lookup(env, [1.0, 0.0, 0.0]), lerp(env[3, 6], env[3, 7], 0.25), atol=1e-5)
    assert np.allclose(O.env_lookup(env, [-1.0, 0.0, 0.0]), lerp(env[3, 1], env[3, 2], 0.75), atol=1e-5)
    assert np.allclose(O.env_lookup(env, [0.0, 0.0, 1.0]), lerp(env[3, 8], env[3, 0], 0.5), atol=1e-5)


def test_poles_reach_the_first_and_last_rows():
    h, w = 10, 20
    env = random_map(h, w, 4)
    env[0] = [0.25, 0.5, 0.75]
    env[-1] = [1.0, 2.0, 3.0]
    for d in ([0, 1, 0], [0.0, 1.0, 1e-4], [0.01, 1.0, -0.01], [-0.03, 1.0, 0.02]):
        assert np.array_equal(O.env_lookup(env, d), env[0, 0]), d
    for d in ([0, -1, 0], [0.0, -1.0, 1e-4], [0.02, -1.0, 0.01]):
        assert np.array_equal(O.env_lookup(env, d), env[-1, 0]), d


def test_seam_is_continuous():
    """phi = pi - eps and -pi + eps lie on either side of the +z seam: the lookups agree to O(eps)"""
    h, w = 16, 32
    env = random_map(h, w, 5)
    for eps in (1e-2, 1e-3, 1e-4):
        for theta in (-0.7, 0.0, 0.3, 1.2):
            a = O.env_lookup(env, [np.cos(theta) * np.sin(np.pi - eps), np.sin(theta), -np.cos(theta) * np.cos(np.pi - eps)])
            b = O.env_lookup(env, [np.cos(theta) * np.sin(-np.pi + eps), np.sin(theta), -np.cos(theta) * np.cos(-np.pi + eps)])
            assert np.abs(a - b).max() <= 2 * eps / (2 * np.pi) * w + 1e-5, (eps, theta, a, b)
    # exactly on the seam: the midpoint of the last and the first column
    r = 5
    d = texel_dir(r, 0, h, w)
    d = np.array([0.0, d[1], np.cos(np.arcsin(d[1]))])
    assert np.allclose(O.env_lookup(env, d), lerp(env[r, -1], env[r, 0], 0.5), atol=1e-5)


def test_bilinear_midpoint_is_the_average():
    h, w = 12, 24
    env = random_map(h, w, 6)
    for r, c in ((0, 0), (3, 7), (10, 22)):
        phi = ((c + 1) / w - 0.5) * 2 * np.pi
        theta = (0.5 - (r + 1) / h) * np.pi
        d = [np.cos(theta) * np.sin(phi), np.sin(theta), -np.cos(theta) * np.cos(phi)]
        want = (env[r, c] + env[r, c + 1] + env[r + 1, c] + env[r + 1, c + 1]) / 4
        assert np.allclose(O.env_lookup(env, d), want, atol=2e-5), (r, c)


@pytest.mark.parametrize("h,w", [(1, 1), (1, 3), (2, 1), (5, 7), (64, 128)])
def test_any_direction_returns_a_value_of_the_map(h, w):
    """non-unit, zero, huge, tiny, NaN and infinite components: the result is finite and inside the map's range,
    a scaled direction looks up the same texels, and a fully invalid one returns a texel exactly"""
    env = random_map(h, w, 7) + 0.5
    lo, hi = env.reshape(-1, 3).min(0), env.reshape(-1, 3).max(0)
    rng = np.random.default_rng(8)
    unit = rng.normal(size=(200, 3))
    unit /= np.linalg.norm(unit, axis=1, keepdims=True)
    base = O.env_lookup(env, unit)
    for k in (1e-3, 0.37, 1.01, 7.5, 1e3):                        # (not 1e-30 / 1e30: d.x^2 + d.z^2 under- / overflows)
        assert np.allclose(O.env_lookup(env, unit * k), base, atol=1e-4), k
    nan, inf = float("nan"), float("inf")
    odd = [[0, 0, 0], [-0.0, 0.0, -0.0], [nan, nan, nan], [nan, 0, -1], [0, nan, -1], [1, 0, nan], [inf, 0, 0],
           [-inf, inf, 0], [inf, inf, inf], [0, -inf, 0], [nan, inf, -inf], [1e38, 1e38, 1e38], [1e-45, 0, -1e-45],
           [np.nextafter(np.float32(0), np.float32(1)), 0, 0], [0, 0, 1], [-1e-7, 0, 1], [1e-7, 0, 1]]
    got = O.env_lookup(env, odd)
    assert np.isfinite(got).all()
    assert ((got >= lo - 1e-6) & (got <= hi + 1e-6)).all()
    texels = {tuple(t) for t in env.reshape(-1, 3)}
    assert tuple(got[2]) in texels                                   # all-NaN: one texel, no blend


def test_all_ones_map_is_bit_identical_to_no_map():
    """the lookup of a constant map returns the constant exactly, so an all-ones map changes no bit"""
    for name, lens in (("scene", None), ("scene", LENS_SCENE), ("cloud", LENS_VOLUME), ("cornell", None)):
        w, h = 48, 27
        osc, _, cam = load_pair(name, w, h, lenses=lens)
        ref, n, _ = oracle_render(osc, cam, w, h, 1, 2, seed=3)
        for shape in ((1, 1), (5, 9)):
            osc.set_environment(np.ones(shape + (3,), np.float32))
            got, n2, _ = oracle_render(osc, cam, w, h, 1, 2, seed=3)
            assert n == n2 and np.array_equal(got, ref), (name, shape)
        osc.set_environment(random_map(8, 16, 9))
        mapped, _, _ = oracle_render(osc, cam, w, h, 1, 2, seed=3)
        if name != "cornell":                                        # Flat{black} root: nothing to multiply
            assert np.abs(mapped - ref).mean() > 1e-3, name
        osc.set_environment(None)
        assert np.array_equal(oracle_render(osc, cam, w, h, 1, 2, seed=3)[0], ref)


# ---- the Einstein ring ----------------------------------------------------------------------------------------------

D_L, R_S, DISC = 6.0, 0.0075, np.radians(0.3)


def ring_scene():
    """the camera of scene.json.gz (without its focus: a pinhole, so that every ray starts on the axis), root
    Emissive{white, 1} and one small black sphere behind the camera, out of view"""
    base = O.read_scene_json(O.scene_path("scene"))
    cam = json.loads(json.dumps(base["objects"]["collection"]["0"]))
    cam["inner"]["Camera"]["focus"] = None
    m = np.array(cam["transform"]["transform_world"], np.float64)
    pos, fwd = m[9:12], -m[6:9] / np.linalg.norm(m[6:9])
    behind = [float(np.float32(x)) for x in pos - 3.0 * fwd]
    sphere = {"object_ref": 1, "tag": None, "flags": {"bits": 0},
              "transform": {"transform_world": [1, 0, 0, 0, 1, 0, 0, 0, 1] + behind,
                            "transform_local": [1, 0, 0, 0, 1, 0, 0, 0, 1] + behind, "transform_parent": None},
              "inner": {"Sphere": {"material": 1, "volume": None, "radius": 0.1}}, "children": None}
    doc = {"roots": [], "root_material": 0, "objects": {"collection": {"0": cam, "1": sphere}, "next_key": 2},
           "data": {"collection": {"0": {"inner": {"Material": {"Emissive": {"albedo": {"r": 1.0, "g": 1.0, "b": 1.0}, "intensity": 1.0}}}},
                                   "1": {"inner": {"Material": {"Flat": {"albedo": {"r": 0.0, "g": 0.0, "b": 0.0}}}}}},
                    "next_key": 2}}
    return json.loads(json.dumps(doc)), pos, fwd, m[0:3] / np.linalg.norm(m[0:3])


def disc_map(fwd, h=1024, w=2048):
    """black, except a bright disc of angular radius DISC around `fwd`"""
    r, c = np.meshgrid(np.arange(h), np.arange(w), indexing="ij")
    theta = (0.5 - (r + 0.5) / h) * np.pi
    phi = ((c + 0.5) / w - 0.5) * 2 * np.pi
    d = np.stack([np.cos(theta) * np.sin(phi), np.sin(theta), -np.cos(theta) * np.cos(phi)], -1)
    lit = np.arccos(np.clip(d @ fwd, -1, 1)) < DISC
    env = np.zeros((h, w, 3), np.float32)
    env[lit] = 1.0
    return env


def einstein_angle_f64(pos, fwd, right):
    """the launch angle from the camera at which the f64 stepper's ray leaves the lens exactly along the axis"""
    lens = np.array([[*(pos + D_L * fwd), R_S]], np.float32)

    def final_tilt(theta):
        d = np.cos(theta) * fwd + np.sin(theta) * right
        out = O.integrate(lens, np.array([[*pos, *d]], np.float32), 3000, use_f64=True)[0]
        assert np.linalg.norm(out[:3] - pos) > 1e3                   # far beyond the lens: the deflection is complete
        return float(out[3:] @ right) / float(np.linalg.norm(out[3:]))

    lo, hi = 0.01, 0.2
    assert final_tilt(lo) < 0 < final_tilt(hi)
    for _ in range(40):
        mid = 0.5 * (lo + hi)
        lo, hi = (mid, hi) if final_tilt(mid) < 0 else (lo, mid)
    return 0.5 * (lo + hi)


def test_einstein_ring():
    """A point mass on the camera axis D_L in front of it and a small bright disc on the axis far behind it: the disc
    is imaged as a ring at the Einstein angle.  The ring's intensity-weighted angle to the axis must be the angle at
    which the f64 stepper sends a ray from the camera exactly along the axis -- which checks the bent rays' escape
    directions and the map's orientation together -- and that angle is the weak-field sqrt(2 r_s / D_L) to 5 %."""
    doc, pos, fwd, right = ring_scene()
    theta_e = einstein_angle_f64(pos, fwd, right)
    assert abs(theta_e - np.sqrt(2 * R_S / D_L)) <= 0.05 * np.sqrt(2 * R_S / D_L), theta_e

    size, spp = 192, 4
    osc = O.OracleScene(doc)
    osc.set_camera_aspect(0, 1.0)
    osc.set_environment(disc_map(fwd))
    cfg = O.make_config(samples=spp)
    xs, ys = np.meshgrid(np.arange(size), np.arange(size))
    xs, ys = np.repeat(xs.ravel(), spp), np.repeat(ys.ravel(), spp)
    rays = osc.camera_rays(0, cfg, size, size, xs, ys, np.tile(np.arange(spp), size * size))
    dirs = rays[:, 3:].astype(np.float64)
    ang = np.arccos(np.clip((dirs @ fwd) / np.linalg.norm(dirs, axis=1), -1, 1)).reshape(size, size, spp).mean(-1)
    pixel = ang.max() / (size / 2 * np.sqrt(2))                      # angle of one pixel (corners are sqrt(2) half-widths out)
    assert 2.5 * theta_e < ang[size // 2].max() < 4 * theta_e        # the ring sits about a third of the way out

    for lensed in (True, False):
        osc.set_lenses(np.array([[*(pos + D_L * fwd), R_S]], np.float32) if lensed else np.zeros((0, 4), np.float32))
        img, n, _ = osc.render(0, cfg, size, size, seed=1)
        lum = img[..., :3].mean(-1) / n
        assert lum.sum() > 0
        mean_angle = float((lum * ang).sum() / lum.sum())
        if lensed:
            assert abs(mean_angle - theta_e) <= pixel / 2 + DISC, (mean_angle, theta_e)
            lit = lum > 0.5
            assert (ang[lit] > theta_e - 2 * DISC - pixel).all() and (ang[lit] < theta_e + 2 * DISC + pixel).all()
            # a ring, not an arc: every quadrant of the image holds a quarter of its light
            yy, xx = np.mgrid[:size, :size] - (size - 1) / 2
            for q in ((xx > 0) & (yy > 0), (xx < 0) & (yy > 0), (xx < 0) & (yy < 0), (xx > 0) & (yy < 0)):
                assert abs(lum[q].sum() / lum.sum() - 0.25) < 0.05
        else:                                                        # a spot of the disc's radius at the image centre
            texel = 2 * np.pi / 2048                                   # bilinear filtering blurs the disc's edge by one texel
            assert mean_angle <= DISC + pixel / 2, mean_angle
            assert (ang[lum > 0] <= DISC + texel + pixel).all()
            yy, xx = np.mgrid[:size, :size]
            cy, cx = (lum * yy).sum() / lum.sum(), (lum * xx).sum() / lum.sum()
            assert abs(cy - (size - 1) / 2) < 1.5 and abs(cx - (size - 1) / 2) < 1.5, (cx, cy)


# ---- host API -------------------------------------------------------------------------------------------------------

def test_invalid_maps_are_rejected():
    sc = bt.Scene.load(O.scene_path("scene"))
    good = random_map(4, 8, 10)
    sc.set_environment(good)
    buf = np.ones(12, np.float32)
    for rgb, w, h in ((buf.ctypes.data, 0, 4), (buf.ctypes.data, 4, 0), (buf.ctypes.data, 0, 0), (None, 2, 2), (None, 0, 1),
                      (buf.ctypes.data, 1 << 16, 1 << 15), (buf.ctypes.data, 0xffffffff, 0xffffffff)):
        assert lib_call(sc, rgb, w, h) == _ffi.ERR_INVALID_ARG, (w, h)
    for bad in (float("nan"), float("inf"), -float("inf"), -1e-6, -1.0):
        rgb = good.copy()
        rgb[2, 5, 1] = bad
        with pytest.raises(bt.BendyError) as e:
            sc.set_environment(rgb)
        assert e.value.code == _ffi.ERR_INVALID_ARG and "texel 21" in e.value.message
    for shape in ((4, 8), (4, 8, 4), (4, 8, 1), (0, 8, 3), (4, 0, 3), (2, 4, 8, 3)):
        with pytest.raises(ValueError):
            sc.set_environment(np.ones(shape, np.float32))
    assert lib_call(None, buf.ctypes.data, 2, 2) == _ffi.ERR_INVALID_ARG
    # that the scene still renders with `good` after these calls is checked on the GPU (test_gpu_environment.py)
    sc.set_environment(np.zeros((1, 1, 3), np.float32))              # zero is a valid (black) map
    sc.set_environment(None)
    sc.set_environment(None)


def lib_call(sc, rgb, w, h):
    return _ffi.lib.bt_scene_set_environment(sc.handle if sc is not None else None, rgb, w, h)


def test_map_is_not_part_of_the_wire_format():
    for name in ("scene", "cloud", "cornell"):
        sc = bt.Scene.load(O.scene_path(name))
        plain = sc.to_json()
        sc.set_lenses(LENS_SCENE)
        lensed = sc.to_json()
        sc.set_environment(random_map(16, 32, 11))
        assert sc.to_json() == lensed
        sc.set_environment(None)
        assert sc.to_json() == lensed
        sc.set_lenses(np.zeros((0, 4), np.float32))
        sc.set_environment(random_map(2, 2, 12))
        assert sc.to_json() == plain


# ---- CLI: --environment sky.pfm ---------------------------------------------------------------------------------------

def write_pfm(path, rgb, little=True, header=None, cut=0):
    """PFM: "PF\\nW H\\nscale\\n", scale < 0 = little-endian, rows bottom first"""
    h, w, _ = rgb.shape
    data = np.ascontiguousarray(rgb[::-1], "<f4" if little else ">f4").tobytes()
    head = header if header is not None else f"PF\n{w} {h}\n{-1.0 if little else 1.0}\n".encode()
    with open(path, "wb") as f:
        f.write(head + data[:len(data) - cut])
    return path


def run_cli(*args):
    return subprocess.run([CLI, "--output", "full", "--width", "64", "--height", "36", "--samples", "0",
                           "--scene", O.scene_path("scene"), *args], capture_output=True, text=True)


def test_cli_environment_dry_run(tmp_path):
    rgb = random_map(6, 10, 12)
    for little in (True, False):
        p = write_pfm(tmp_path / f"sky_{little}.pfm", rgb, little)
        r = run_cli("--environment", str(p))
        assert r.returncode == 0 and "environment map" in r.stderr and "10 x 6" in r.stderr, r.stderr
    grey = tmp_path / "grey.pfm"
    with open(grey, "wb") as f:
        f.write(b"Pf\n3 2\n-1.0\n" + np.ones(6, "<f4").tobytes())
    assert run_cli("--environment", str(grey)).returncode == 0


@pytest.mark.parametrize("case", ["truncated", "empty", "magic", "width", "height", "scale", "no_newline", "negative", "nan", "missing"])
def test_cli_environment_malformed(tmp_path, case):
    rgb = random_map(6, 10, 13)
    p = tmp_path / "bad.pfm"
    if case == "truncated":
        write_pfm(p, rgb, cut=5)
    elif case == "empty":
        p.write_bytes(b"")
    elif case == "magic":
        write_pfm(p, rgb, header=b"P6\n10 6\n-1.0\n")
    elif case == "width":
        write_pfm(p, rgb, header=b"PF\n-10 6\n-1.0\n")
    elif case == "height":
        write_pfm(p, rgb, header=b"PF\n10 x\n-1.0\n")
    elif case == "scale":
        write_pfm(p, rgb, header=b"PF\n10 6\n0\n")
    elif case == "no_newline":
        p.write_bytes(b"PF\n10 6\n-1.0")
    elif case == "negative":
        rgb[1, 2, 0] = -1.0
        write_pfm(p, rgb)
    elif case == "nan":
        rgb[0, 0, 2] = np.nan
        write_pfm(p, rgb)
    r = run_cli("--environment", str(p))
    assert r.returncode != 0 and "\nerror: " in "\n" + r.stderr, (case, r.returncode, r.stderr)
    assert "bad.pfm" in r.stderr, r.stderr


def test_pfm_header_is_parsed_like_the_writers_write_it(tmp_path):
    """whitespace variants of the header (one token per line, or all on one line) and a trailing byte count check"""
    rgb = random_map(3, 4, 14)
    data = np.ascontiguousarray(rgb[::-1], "<f4").tobytes()
    for head in (b"PF\n4 3\n-1\n", b"PF 4 3 -1.000000\n", b"PF\n4\n3\n-1.0\n", b"PF\r\n4 3\r\n-1.0\n"):
        p = tmp_path / "h.pfm"
        p.write_bytes(head + data)
        r = run_cli("--environment", str(p))
        assert r.returncode == 0, (head, r.stderr)
