"""ctypes binding of the CPU oracle (oracle/libbendy_oracle.so) -- TEST INFRASTRUCTURE ONLY.

The scene JSON is parsed here with Python's `json`, independently of the engine's C++ loader, and
handed to the oracle as the flat `orc_object` / `orc_data` arrays of oracle/bendy_oracle.h.
"""
import ctypes as C
import gzip
import json
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(ROOT, "oracle")
SCENE_DIR = os.path.join(ROOT, "tests", "golden", "scenes")

EMPTY, CAMERA, SPHERE, RECT, CUBOID = range(5)
FLAT, DIFFUSE, METALLIC, GLASS, EMISSIVE = range(5)
OUT_FULL, OUT_ALBEDO, OUT_NORMAL, OUT_DEPTH = range(4)
CS_NONE, CS_NORMAL, CS_LINEAR, CS_SRGB = range(4)
FACE_MISS, FACE_CAPTURED = -1, -2
PERSPECTIVE, EQUIRECTANGULAR = 0, 1


class OrcRect(C.Structure):
    _fields_ = [("material", C.c_uint64), ("half_width", C.c_float), ("half_height", C.c_float),
                ("x", C.c_float * 3), ("y", C.c_float * 3), ("z", C.c_float * 3)]


class OrcObject(C.Structure):
    _fields_ = [("object_ref", C.c_uint64), ("kind", C.c_uint32), ("flags", C.c_uint32),
                ("transform", C.c_float * 12), ("material", C.c_uint64), ("volume", C.c_int64),
                ("radius", C.c_float), ("sensor_size", C.c_float), ("focal_length", C.c_float),
                ("aspect_ratio", C.c_float), ("fstop", C.c_float), ("focus", C.c_float),
                ("has_focus", C.c_int32), ("rect", OrcRect), ("face_offset", (C.c_float * 3) * 6),
                ("faces", OrcRect * 6)]


class OrcData(C.Structure):
    _fields_ = [("data_ref", C.c_uint64), ("kind", C.c_uint32), ("mat_kind", C.c_uint32),
                ("albedo", C.c_float * 3), ("roughness", C.c_float), ("ior", C.c_float),
                ("intensity", C.c_float), ("width", C.c_uint32), ("height", C.c_uint32),
                ("depth", C.c_uint32), ("size", C.c_float * 3), ("buffer", C.POINTER(C.c_float))]


class OrcConfig(C.Structure):
    _fields_ = [("max_bounces", C.c_uint64), ("max_volume_bounces", C.c_uint64),
                ("clip_min", C.c_float), ("clip_max", C.c_float), ("volume_step", C.c_float),
                ("chunks_x", C.c_uint32), ("chunks_y", C.c_uint32), ("output", C.c_int32),
                ("samples", C.c_uint64), ("subsample", C.c_uint32),
                ("has_output", C.c_int32), ("r_output", C.c_int32),
                ("has_max_bounces", C.c_int32), ("r_max_bounces", C.c_uint64),
                ("has_max_volume_bounces", C.c_int32), ("r_max_volume_bounces", C.c_uint64),
                ("has_volume_step", C.c_int32), ("r_volume_step", C.c_float)]


class OrcLensConfig(C.Structure):
    _fields_ = [("kappa", C.c_float), ("h_min", C.c_float), ("h_max", C.c_float),
                ("r_far", C.c_float), ("max_steps", C.c_uint32)]


class OrcProbeResult(C.Structure):
    _fields_ = [("face", C.c_int32), ("steps", C.c_uint32), ("object_ref", C.c_uint64),
                ("t", C.c_double), ("position", C.c_double * 3), ("normal", C.c_double * 3),
                ("direction", C.c_double * 3)]


_lib = None


def build():
    subprocess.run(["make", "-C", ORACLE_DIR, "-s"], check=True)


def lib():
    global _lib
    if _lib is not None:
        return _lib
    build()                                      # make: rebuilds a library older than its sources, else a no-op
    L = C.CDLL(os.path.join(ORACLE_DIR, "libbendy_oracle.so"))
    L.orc_scene_create.restype = C.c_void_p
    L.orc_scene_create.argtypes = [C.POINTER(OrcObject), C.c_int, C.POINTER(OrcData), C.c_int, C.c_uint64]
    L.orc_scene_set_lenses.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.POINTER(OrcLensConfig)]
    L.orc_scene_set_camera_aspect.argtypes = [C.c_void_p, C.c_uint64, C.c_float]
    L.orc_scene_set_environment.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32]
    L.orc_scene_set_camera_projection.argtypes = [C.c_void_p, C.c_uint64, C.c_int]
    L.orc_scene_destroy.argtypes = [C.c_void_p]
    L.orc_render.argtypes = [C.c_void_p, C.c_uint64, C.POINTER(OrcConfig), C.c_uint64, C.c_uint64,
                             C.c_void_p, C.c_uint32, C.c_uint32, C.c_int, C.POINTER(C.c_uint64)]
    L.orc_resolve_u8.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint64, C.c_int, C.c_void_p]
    L.orc_probe.argtypes = [C.c_void_p, C.POINTER(OrcConfig), C.c_int, C.c_void_p, C.c_void_p, C.c_int,
                            C.POINTER(OrcProbeResult)]
    L.orc_camera_rays.argtypes = [C.c_void_p, C.c_uint64, C.POINTER(OrcConfig), C.c_uint64, C.c_uint64,
                                  C.c_uint32, C.c_uint32, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                  C.c_void_p]
    L.orc_integrate.argtypes = [C.c_void_p, C.c_int, C.POINTER(OrcLensConfig), C.c_int, C.c_void_p,
                                C.c_uint32, C.c_int, C.c_void_p, C.c_void_p]
    L.orc_last_error.restype = C.c_char_p
    L.orc_xoshiro_from_seed.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
    L.orc_xoshiro_seed_from_u64.argtypes = [C.c_uint64, C.c_void_p]
    L.orc_path_seed.restype = C.c_uint64
    L.orc_path_seed.argtypes = [C.c_uint64, C.c_uint64, C.c_uint64]
    L.orc_uniform_f32.argtypes = [C.c_uint64, C.c_float, C.c_float, C.c_int, C.c_void_p, C.c_int, C.POINTER(C.c_float)]
    L.orc_standard_f32.argtypes = [C.c_uint64, C.c_void_p, C.c_int]
    L.orc_gen_bool.argtypes = [C.c_uint64, C.c_double, C.c_void_p, C.c_int]
    L.orc_uniform_usize.argtypes = [C.c_uint64, C.c_uint64, C.c_void_p, C.c_int]
    L.orc_with_frustum.argtypes = [C.c_float, C.c_float, C.c_float, C.c_float, C.c_void_p]
    L.orc_environment_lookup.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p]
    L.orc_equirect_dir.argtypes = [C.c_float, C.c_float, C.c_float, C.c_float, C.c_void_p]
    L.orc_any_orthonormal_pair.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    L.orc_distr.argtypes = [C.c_int, C.c_uint64, C.c_void_p, C.c_void_p, C.c_int]
    L.orc_sphere_hit.argtypes = [C.c_void_p, C.c_float, C.c_void_p, C.c_void_p, C.c_float, C.c_float,
                                 C.POINTER(C.c_float), C.c_void_p, C.POINTER(C.c_int)]
    L.orc_rect_hit.argtypes = [C.POINTER(OrcRect), C.c_void_p, C.c_void_p, C.c_void_p, C.c_float, C.c_float,
                               C.POINTER(C.c_float), C.c_void_p, C.POINTER(C.c_int)]
    L.orc_density_sample.restype = C.c_float
    L.orc_density_sample.argtypes = [C.POINTER(OrcData), C.c_void_p]
    L.orc_reflect.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    L.orc_refract.argtypes = [C.c_void_p, C.c_void_p, C.c_float, C.c_void_p]
    L.orc_fresnel.restype = C.c_float
    L.orc_fresnel.argtypes = [C.c_void_p, C.c_void_p, C.c_float]
    L.orc_linear_to_srgb.restype = C.c_float
    L.orc_linear_to_srgb.argtypes = [C.c_float]
    L.orc_rk4_step_f32.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_float]
    L.orc_rk4_step_f64.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_double]
    _lib = L
    return L


class OraclePanic(RuntimeError):
    pass


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def f3(v):
    return np.ascontiguousarray(v, dtype=np.float32)


def _fill_rect(dst, src):
    dst.material = src["material"]
    dst.half_width = src["half_width"]
    dst.half_height = src["half_height"]
    for k in ("x", "y", "z"):
        getattr(dst, k)[:] = src[k]


def read_scene_json(path):
    opener = gzip.open if str(path).endswith(".gz") else open
    with opener(path, "rt") as f:
        return json.load(f)


def scene_path(name):
    return os.path.join(SCENE_DIR, name + ".json.gz")


DEFAULT_LENS_CONFIG = dict(kappa=0.05, h_min=0.02, h_max=5.0, r_far=500.0, max_steps=4096)


def make_config(samples=1, subsample=0, output=OUT_FULL, chunks=(8, 4), max_bounces=8,
                max_volume_bounces=32, clip_min=0.01, clip_max=1000.0, volume_step=0.1,
                r_output=None, r_max_bounces=None, r_max_volume_bounces=None, r_volume_step=None):
    c = OrcConfig()
    c.max_bounces, c.max_volume_bounces = max_bounces, max_volume_bounces
    c.clip_min, c.clip_max, c.volume_step = clip_min, clip_max, volume_step
    c.chunks_x, c.chunks_y = chunks
    c.output = output
    c.samples, c.subsample = samples, subsample
    for name, val in (("output", r_output), ("max_bounces", r_max_bounces),
                      ("max_volume_bounces", r_max_volume_bounces), ("volume_step", r_volume_step)):
        setattr(c, "has_" + name, 0 if val is None else 1)
        setattr(c, "r_" + name, 0 if val is None else val)
    return c


class OracleScene:
    """Scene model of the reference (src/scene/mod.rs:84-90) held by the oracle."""

    def __init__(self, scene_json):
        L = lib()
        self.json = scene_json
        objs = scene_json["objects"]["collection"]
        datas = scene_json["data"]["collection"]
        oa = (OrcObject * max(len(objs), 1))()
        self.tags = {}
        for i, (key, o) in enumerate(objs.items()):
            dst = oa[i]
            dst.object_ref = int(key)
            dst.flags = o["flags"]["bits"]
            dst.transform[:] = o["transform"]["transform_world"]
            dst.volume = -1
            if o.get("tag") is not None:
                self.tags.setdefault(o["tag"], int(key))
            inner = o["inner"]
            if inner == "Empty":
                dst.kind = EMPTY
            elif "Camera" in inner:
                cam = inner["Camera"]
                dst.kind = CAMERA
                dst.sensor_size, dst.focal_length = cam["sensor_size"], cam["focal_length"]
                dst.aspect_ratio, dst.fstop = cam["aspect_ratio"], cam["fstop"]
                dst.has_focus = 0 if cam["focus"] is None else 1
                dst.focus = 0.0 if cam["focus"] is None else cam["focus"]
            elif "Sphere" in inner:
                s = inner["Sphere"]
                dst.kind = SPHERE
                dst.material = s["material"]
                dst.volume = -1 if s["volume"] is None else s["volume"]
                dst.radius = s["radius"]
            elif "Rect" in inner:
                dst.kind = RECT
                _fill_rect(dst.rect, inner["Rect"])
            elif "Cuboid" in inner:
                dst.kind = CUBOID
                for f, (offset, rect) in enumerate(inner["Cuboid"]["faces"]):
                    dst.face_offset[f][:] = offset
                    _fill_rect(dst.faces[f], rect)
            else:
                raise ValueError(f"unknown object kind {inner!r}")
        da = (OrcData * max(len(datas), 1))()
        self._buffers = []
        for i, (key, d) in enumerate(datas.items()):
            dst = da[i]
            dst.data_ref = int(key)
            inner = d["inner"]
            if "Material" in inner:
                (kind, m), = inner["Material"].items()
                dst.kind = 0
                dst.mat_kind = ["Flat", "Diffuse", "Metallic", "Glass", "Emissive"].index(kind)
                dst.albedo[:] = [m["albedo"]["r"], m["albedo"]["g"], m["albedo"]["b"]]
                dst.roughness = m.get("roughness", 0.0)
                dst.ior = m.get("ior", 0.0)
                dst.intensity = m.get("intensity", 0.0)
            else:
                dm = inner["Volume"]["DensityMap"]
                dst.kind = 1
                dst.width, dst.height, dst.depth = dm["width"], dm["height"], dm["depth"]
                dst.size[:] = dm["size"]
                buf = np.asarray(dm["buffer"], dtype=np.float32)
                self._buffers.append(buf)
                dst.buffer = buf.ctypes.data_as(C.POINTER(C.c_float))
        self.handle = L.orc_scene_create(oa, len(objs), da, len(datas), scene_json["root_material"])
        self.lenses = np.zeros((0, 4), np.float32)

    @classmethod
    def load(cls, path):
        return cls(read_scene_json(path))

    def __del__(self):
        if getattr(self, "handle", None):
            lib().orc_scene_destroy(self.handle)
            self.handle = None

    def find_by_tag(self, tag):
        return self.tags.get(tag)

    def set_camera_aspect(self, camera_ref, aspect):
        if lib().orc_scene_set_camera_aspect(self.handle, camera_ref, aspect) != 0:
            raise OraclePanic(lib().orc_last_error().decode())

    def set_lenses(self, xyzr, **cfg):
        xyzr = np.ascontiguousarray(xyzr, dtype=np.float32).reshape(-1, 4)
        c = OrcLensConfig(**{**DEFAULT_LENS_CONFIG, **cfg})
        self.lenses = xyzr
        lib().orc_scene_set_lenses(self.handle, _p(xyzr), len(xyzr), C.byref(c))

    def set_environment(self, rgb):
        """(H, W, 3) RGB, row 0 = +y pole, centre column along -z; None clears it"""
        if rgb is None:
            lib().orc_scene_set_environment(self.handle, None, 0, 0)
            return
        rgb = np.ascontiguousarray(rgb, np.float32)
        h, w, _ = rgb.shape
        lib().orc_scene_set_environment(self.handle, _p(rgb), w, h)

    def set_projection(self, camera_ref, projection):
        """PERSPECTIVE or EQUIRECTANGULAR"""
        if lib().orc_scene_set_camera_projection(self.handle, camera_ref, int(projection)) != 0:
            raise OraclePanic(lib().orc_last_error().decode())

    def render(self, camera_ref, cfg, width, height, seed=0, sample_base=0, buffer=None, n_threads=None):
        """Tracer::render into an RGBA32F buffer (alpha 1, as Buffer::new). Returns (buffer, samples, status)."""
        if buffer is None:
            buffer = np.zeros((height, width, 4), np.float32)
            buffer[..., 3] = 1.0
        samples = C.c_uint64(0)
        if n_threads is None:
            n_threads = os.cpu_count() or 1
        st = lib().orc_render(self.handle, camera_ref, C.byref(cfg), seed, sample_base, _p(buffer), width, height,
                              n_threads, C.byref(samples))
        if st < 0:
            raise OraclePanic(lib().orc_last_error().decode())
        return buffer, samples.value, st

    def probe(self, cfg, origins, dirs, use_f64=False):
        origins, dirs = f3(origins).reshape(-1, 3), f3(dirs).reshape(-1, 3)
        n = len(origins)
        out = (OrcProbeResult * n)()
        if lib().orc_probe(self.handle, C.byref(cfg), n, _p(origins), _p(dirs), int(use_f64), out) != 0:
            raise OraclePanic(lib().orc_last_error().decode())
        return dict(
            face=np.array([r.face for r in out], np.int32),
            steps=np.array([r.steps for r in out], np.uint32),
            object_ref=np.array([r.object_ref for r in out], np.uint64),
            t=np.array([r.t for r in out]),
            position=np.array([list(r.position) for r in out]).reshape(n, 3),
            normal=np.array([list(r.normal) for r in out]).reshape(n, 3),
            direction=np.array([list(r.direction) for r in out]).reshape(n, 3),
        )

    def camera_rays(self, camera_ref, cfg, width, height, xs, ys, path_index, seed=0, sample_base=0):
        xs = np.ascontiguousarray(xs, np.uint32)
        ys = np.ascontiguousarray(ys, np.uint32)
        pi = np.ascontiguousarray(path_index, np.uint64)
        out = np.zeros((len(xs), 6), np.float32)
        if lib().orc_camera_rays(self.handle, camera_ref, C.byref(cfg), seed, sample_base, width, height, len(xs),
                                 _p(xs), _p(ys), _p(pi), _p(out)) != 0:
            raise OraclePanic(lib().orc_last_error().decode())
        return out


def resolve_u8(buffer, samples, color_space):
    h, w, _ = buffer.shape
    out = np.zeros((h, w, 4), np.uint8)
    lib().orc_resolve_u8(_p(np.ascontiguousarray(buffer, np.float32)), w, h, samples, color_space, _p(out))
    return out


def env_lookup(rgb, d):
    """the map's factor for direction(s) d ((3,) or (n, 3)) in the (H, W, 3) map rgb"""
    rgb = np.ascontiguousarray(rgb, np.float32)
    h, w, _ = rgb.shape
    d = np.ascontiguousarray(d, np.float32)
    flat = d.reshape(-1, 3)
    out = np.zeros_like(flat)
    for i in range(len(flat)):
        lib().orc_environment_lookup(_p(rgb), w, h, _p(flat[i]), _p(out[i]))
    return out.reshape(d.shape)


def equirect_dir(u, v, pixel_width, pixel_height):
    """camera-space direction of an equirectangular camera for the NDC (u, v) before the half-pixel offset"""
    out = np.zeros(3, np.float32)
    lib().orc_equirect_dir(u, v, pixel_width, pixel_height, _p(out))
    return out


def integrate(xyzr, xv, n_steps, use_f64=False, **cfg):
    xyzr = np.ascontiguousarray(xyzr, np.float32).reshape(-1, 4)
    xv = np.ascontiguousarray(xv, np.float32).reshape(-1, 6)
    c = OrcLensConfig(**{**DEFAULT_LENS_CONFIG, **cfg})
    o32 = np.zeros_like(xv)
    o64 = np.zeros(xv.shape, np.float64)
    lib().orc_integrate(_p(xyzr), len(xyzr), C.byref(c), len(xv), _p(xv), n_steps, int(use_f64), _p(o32), _p(o64))
    return o64 if use_f64 else o32
