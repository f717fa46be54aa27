"""The CPU oracle with the environment map and the equirectangular camera (tests/oracle_camera.cpp) -- TEST INFRASTRUCTURE ONLY.

oracle_camera.cpp includes oracle_env.cpp (the unchanged oracle with the map in sample_root) and routes the oracle's two
camera_ray calls through the projection set per camera.  The library is built on first use into a cache directory keyed by
the sources' contents, like oracle_env's.  `CameraOracleScene` is an `oracle_env.EnvOracleScene` on this library with
`set_projection`; `equirect_dir` is the camera-space direction for single (u, v).
"""
import contextlib
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

import oracle_env as OE
import oracle_ffi as O

HERE = os.path.dirname(os.path.abspath(__file__))
SOURCES = [os.path.join(HERE, "oracle_camera.cpp"), *OE.SOURCES]
PERSPECTIVE, EQUIRECTANGULAR = 0, 1

_lib = None


def lib():
    global _lib
    if _lib is not None:
        return _lib
    key = hashlib.sha256(b"".join(open(p, "rb").read() for p in SOURCES) + " ".join(OE.CXXFLAGS).encode()).hexdigest()[:16]
    out_dir = os.path.join(tempfile.gettempdir(), f"bendy_oracle_camera_{os.getuid()}")
    path = os.path.join(out_dir, f"liboracle_camera_{key}.so")
    if not os.path.exists(path):
        os.makedirs(out_dir, exist_ok=True)
        tmp = f"{path}.{os.getpid()}.tmp"
        subprocess.run([os.environ.get("CXX", "g++"), *OE.CXXFLAGS, "-o", tmp, SOURCES[0]], check=True)
        os.replace(tmp, path)
    L = C.CDLL(path)
    for name, fn in vars(O.lib()).items():       # the oracle's signatures, as oracle_ffi declares them
        if name.startswith("orc_"):
            f = getattr(L, name)
            f.argtypes, f.restype = fn.argtypes, fn.restype
    L.orc_env_set.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32]
    L.orc_env_scene_destroy.argtypes = [C.c_void_p]
    L.orc_env_lookup.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p]
    L.orc_cam_set_projection.argtypes = [C.c_void_p, C.c_uint64, C.c_int]
    L.orc_cam_scene_destroy.argtypes = [C.c_void_p]
    L.orc_cam_equirect_dir.argtypes = [C.c_float, C.c_float, C.c_float, C.c_float, C.c_void_p]
    _lib = L
    return L


@contextlib.contextmanager
def _this_library():
    """EnvOracleScene's methods run on oracle_env.lib(): point it at this library for the duration of one call"""
    saved = OE._lib
    OE._lib = lib()
    try:
        yield
    finally:
        OE._lib = saved


def _on_this_library(method):
    def wrapped(self, *args, **kw):
        with _this_library():
            return method(self, *args, **kw)
    wrapped.__doc__ = method.__doc__
    return wrapped


class CameraOracleScene(OE.EnvOracleScene):
    """oracle_env.EnvOracleScene on the oracle with the camera projection"""
    __init__ = _on_this_library(OE.EnvOracleScene.__init__)
    set_camera_aspect = _on_this_library(OE.EnvOracleScene.set_camera_aspect)
    set_lenses = _on_this_library(OE.EnvOracleScene.set_lenses)
    set_environment = _on_this_library(OE.EnvOracleScene.set_environment)
    render = _on_this_library(OE.EnvOracleScene.render)
    probe = _on_this_library(OE.EnvOracleScene.probe)
    camera_rays = _on_this_library(OE.EnvOracleScene.camera_rays)

    @classmethod
    def load(cls, path):
        return cls(O.read_scene_json(path))

    def set_projection(self, camera_ref, projection):
        """PERSPECTIVE (0) or EQUIRECTANGULAR (1); raises RuntimeError for a non-camera reference or another value"""
        if lib().orc_cam_set_projection(self.handle, camera_ref, int(projection)) != 0:
            raise RuntimeError(lib().orc_last_error().decode())

    def __del__(self):
        if getattr(self, "handle", None):
            lib().orc_cam_scene_destroy(self.handle)
            self.handle = None


def equirect_dir(u, v, pixel_width, pixel_height):
    """camera-space direction of an equirectangular camera for the NDC (u, v) before the half-pixel offset"""
    out = np.zeros(3, np.float32)
    lib().orc_cam_equirect_dir(u, v, pixel_width, pixel_height, out.ctypes.data)
    return out


def load_pair(name, width, height, lenses=None, projection=EQUIRECTANGULAR):
    """oracle_env.load_pair on this library, both cameras set to `projection`: (oracle scene, engine scene, camera ref)"""
    import bendy_tracer_b200 as bt
    path = O.scene_path(name)
    osc = CameraOracleScene.load(path)
    esc = bt.Scene.load(path)
    cam = esc.find_by_tag("camera")
    assert cam == osc.find_by_tag("camera")
    aspect = float(np.float32(width) / np.float32(height))
    osc.set_camera_aspect(cam, aspect)
    esc.set_camera_aspect(cam, aspect)
    if lenses is not None:
        osc.set_lenses(lenses)
        esc.set_lenses(lenses)
    osc.set_projection(cam, projection)
    esc.set_camera_projection(cam, projection)
    return osc, esc, cam
