"""Shared helpers of the parity tests: load the same scene into the oracle and the engine."""
import numpy as np

import oracle_ffi as O

SCENES = ["cornell", "cornell2", "scene", "volume", "cloud"]

# C3/C4 synthetic lens (SURVEY 8d): a mass 6 units in front of the camera of scene.json.gz
LENS_SCENE = np.array([[1.362, 1.577, 6.114, 0.2]], np.float32)
LENS_VOLUME = np.array([[2.4 - 6 * 0.1705, 2.7 - 6 * 0.1908, 12.0 - 6 * 0.9667, 0.2]], np.float32)


def load_pair(name, width, height, lenses=None, projection=None):
    """(oracle scene, engine scene, camera ref) with camera.aspect_ratio = width / height (main.rs:218-223), and the
    lenses and the camera projection, when given, set on both"""
    import bendy_tracer_b200 as bt
    path = O.scene_path(name)
    osc = O.OracleScene.load(path)
    esc = bt.Scene.load(path)
    cam = esc.find_by_tag("camera")
    assert cam == osc.find_by_tag("camera")
    aspect = float(np.float32(width) / np.float32(height))
    osc.set_camera_aspect(cam, aspect)
    esc.set_camera_aspect(cam, aspect)
    if lenses is not None:
        osc.set_lenses(lenses)
        esc.set_lenses(lenses)
    if projection is not None:
        osc.set_projection(cam, projection)
        esc.set_camera_projection(cam, projection)
    return osc, esc, cam


def oracle_render(osc, cam, width, height, samples, subsample=0, output=0, seed=0, sample_base=0, **cfg):
    c = O.make_config(samples=samples, subsample=subsample, output=output, **cfg)
    buf, n, status = osc.render(cam, c, width, height, seed=seed, sample_base=sample_base)
    return buf, n, status


def engine_render(esc, cam, width, height, samples, subsample=0, output=0, seed=0, sample_base=0, device=None,
                  buffer=None, **cfg):
    import bendy_tracer_b200 as bt
    tracer = bt.Tracer(bt.Config(chunks_x=8, chunks_y=4, output=bt.Output(output), **cfg), seed=seed)
    if buffer is None:
        buffer = bt.Buffer(width, height, device=device)
    rc = bt.RenderConfig.with_samples_subsample(samples, bt.Subsample(subsample))
    status = tracer.render(esc, cam, rc, buffer, sample_base=sample_base)
    data = buffer.data if isinstance(buffer.data, np.ndarray) else buffer.data.cpu().numpy()
    return data, buffer.samples(), status


def mae_per_channel(a, b, n):
    """per-channel mean absolute error of the resolved (sum / samples) images"""
    return np.abs(a[..., :3].astype(np.float64) - b[..., :3].astype(np.float64)).mean(axis=(0, 1)) / n


def synthetic_scene(n_spheres=200, n_rects=100, n_cuboids=20, seed=0, extent=6.0):
    """A many-primitive scene in the reference's wire format: random diffuse / metallic / glass spheres,
    rects and cuboids inside a box of half-size `extent`, a ground sphere, one emissive sphere light
    (ObjectFlags::LIGHT) and the camera of scene.json.gz.  Exercises the BVH path."""
    import json
    rng = np.random.default_rng(seed)
    base = O.read_scene_json(O.scene_path("scene"))
    objs = {"0": base["objects"]["collection"]["0"]}          # camera
    data = {
        "0": {"inner": {"Material": {"Flat": {"albedo": {"r": 0.0, "g": 0.0, "b": 0.0}}}}},
        "1": {"inner": {"Material": {"Emissive": {"albedo": {"r": 1.0, "g": 1.0, "b": 1.0}, "intensity": 0.3}}}},
        "2": {"inner": {"Material": {"Emissive": {"albedo": {"r": 1.0, "g": 0.9, "b": 0.8}, "intensity": 12.0}}}},
        "3": {"inner": {"Material": {"Diffuse": {"albedo": {"r": 0.3, "g": 0.4, "b": 0.6}, "roughness": 0.8}}}},
    }
    n_mats = 12
    for m in range(n_mats):
        a = [float(np.float32(x)) for x in rng.uniform(0.2, 0.9, 3)]
        alb = {"r": a[0], "g": a[1], "b": a[2]}
        kind = ["Diffuse", "Diffuse", "Metallic", "Glass"][m % 4]
        body = {"albedo": alb, "roughness": float(np.float32(rng.uniform(0.0, 0.3)))}
        if kind == "Glass":
            body["ior"] = 1.4
        data[str(4 + m)] = {"inner": {"Material": {kind: body}}}

    def f(x):
        return float(np.float32(x))

    def obj(key, inner, t, flags=0, m=None):
        m = m if m is not None else [1, 0, 0, 0, 1, 0, 0, 0, 1]
        tf = [f(x) for x in m] + [f(x) for x in t]
        objs[str(key)] = {"object_ref": key, "tag": None, "flags": {"bits": flags},
                          "transform": {"transform_world": tf, "transform_local": tf, "transform_parent": None},
                          "inner": inner, "children": None}

    def rot():
        q = rng.normal(size=4)
        q /= np.linalg.norm(q)
        w, x, y, z = q
        return [1 - 2 * (y * y + z * z), 2 * (x * y + z * w), 2 * (x * z - y * w),
                2 * (x * y - z * w), 1 - 2 * (x * x + z * z), 2 * (y * z + x * w),
                2 * (x * z + y * w), 2 * (y * z - x * w), 1 - 2 * (x * x + y * y)]

    def rect(mat, hw, hh, x=(1, 0, 0), y=(0, 1, 0)):
        z = np.cross(x, y)
        return {"material": mat, "half_width": f(hw), "half_height": f(hh), "x": [f(v) for v in x],
                "y": [f(v) for v in y], "z": [f(v) for v in z]}

    key = 1
    obj(key, {"Sphere": {"material": 3, "volume": None, "radius": 100.0}}, (0, -101, 0)); key += 1
    obj(key, {"Sphere": {"material": 2, "volume": None, "radius": 2.0}}, (6, 10, 0), flags=1); key += 1
    for _ in range(n_spheres):
        p = rng.uniform(-extent, extent, 3)
        p[1] = rng.uniform(-0.5, extent)
        obj(key, {"Sphere": {"material": int(rng.integers(4, 4 + n_mats)), "volume": None,
                             "radius": f(rng.uniform(0.05, 0.35))}}, p); key += 1
    for _ in range(n_rects):
        p = rng.uniform(-extent, extent, 3)
        p[1] = rng.uniform(-0.5, extent)
        obj(key, {"Rect": rect(int(rng.integers(4, 4 + n_mats)), rng.uniform(0.1, 0.5), rng.uniform(0.1, 0.5))}, p, m=rot()); key += 1
    for _ in range(n_cuboids):
        p = rng.uniform(-extent, extent, 3)
        p[1] = rng.uniform(-0.5, extent)
        hx, hy, hz = rng.uniform(0.1, 0.4, 3)
        mat = int(rng.integers(4, 4 + n_mats))
        ex, ey, ez = np.eye(3)
        faces = [[[0, 0, f(-hz)], rect(mat, hx, hy, ex, ey)], [[0, 0, f(hz)], rect(mat, hx, hy, -ex, ey)],
                 [[f(-hx), 0, 0], rect(mat, hz, hy, ez, ey)], [[f(hx), 0, 0], rect(mat, hz, hy, -ez, ey)],
                 [[0, f(-hy), 0], rect(mat, hx, hz, ex, ez)], [[0, f(hy), 0], rect(mat, hx, hz, ex, -ez)]]
        obj(key, {"Cuboid": {"faces": faces}}, p, m=rot()); key += 1
    scene = {"roots": [], "root_material": 1, "objects": {"collection": objs, "next_key": key},
             "data": {"collection": data, "next_key": 4 + n_mats}}
    return json.loads(json.dumps(scene))


def cornell_with_cuboid_light(extra_rect_light=True):
    """cornell.json.gz with the short box (object 8) turned into an emissive LIGHT Cuboid
    (Cuboid::random_point / Cuboid::pdf, cuboid.rs:48-81); the ceiling rect light stays (two LIGHT
    objects: Uniform::new(0, 2) picks between them) unless extra_rect_light is False."""
    import copy
    doc = copy.deepcopy(O.read_scene_json(O.scene_path("cornell")))
    objs = doc["objects"]["collection"]
    data = doc["data"]["collection"]
    key = doc["data"]["next_key"]
    data[str(key)] = {"inner": {"Material": {"Emissive": {"albedo": {"r": 0.9, "g": 0.6, "b": 0.3}, "intensity": 4.0}}}}
    doc["data"]["next_key"] = key + 1
    box = objs["8"]
    assert "Cuboid" in box["inner"]
    box["flags"]["bits"] = 1
    for _, rect in box["inner"]["Cuboid"]["faces"]:
        rect["material"] = key
    if not extra_rect_light:
        objs["6"]["flags"]["bits"] = 0
    return doc


def skewed_scene(n_coincident=200, n_chain=200, chain_radius=0.0):
    """synthetic_scene's fixtures plus n_coincident spheres on one spot and a geometric chain x = 8 * 2^-i that makes
    every SAH split lopsided (the BVH builder's depth budget / median fallback; deep, narrow trees for the traversal).
    chain_radius > 0: the chain spheres get radius chain_radius * x (disjoint, visible), else 0.01."""
    import json
    doc = synthetic_scene(0, 0, 0, seed=3)
    objs = doc["objects"]["collection"]
    key = doc["objects"]["next_key"]
    proto = objs["2"]
    for i in range(n_coincident + n_chain):
        o = json.loads(json.dumps(proto))
        o["object_ref"] = key
        o["flags"] = {"bits": 0}
        x = 0.0 if i < n_coincident else float(np.float32(2.0 ** -(i - n_coincident) * 8.0))
        o["inner"]["Sphere"]["radius"] = float(np.float32(chain_radius * x)) if chain_radius > 0 and i >= n_coincident else 0.01
        t = o["transform"]["transform_world"]
        t[9:12] = [x, 0.5, 0.0]
        o["transform"]["transform_local"] = list(t)
        objs[str(key)] = o
        key += 1
    doc["objects"]["next_key"] = key
    return doc
