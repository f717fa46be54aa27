"""The CPU oracle with the environment-map extension (tests/oracle_env.cpp) -- TEST INFRASTRUCTURE ONLY.

oracle_env.cpp compiles oracle/bendy_oracle.cpp unchanged, with sample_root's colour multiplied by the map's lookup in the
escape direction when a scene has a map.  The library is built on first use into a cache directory keyed by the sources'
contents (the tree may be read-only), with the oracle's own compiler flags.  `EnvOracleScene` is an `oracle_ffi.OracleScene`
that runs on this library and has `set_environment`; `env_lookup` is the lookup for single directions.
"""
import contextlib
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

import oracle_ffi as O

HERE = os.path.dirname(os.path.abspath(__file__))
SOURCES = [os.path.join(HERE, "oracle_env.cpp"), os.path.join(O.ORACLE_DIR, "bendy_oracle.cpp"),
           os.path.join(O.ORACLE_DIR, "bendy_oracle.h")]
CXXFLAGS = ["-O3", "-std=c++17", "-ffp-contract=off", "-march=x86-64-v3", "-fPIC", "-pthread", "-shared"]   # oracle/Makefile's

_lib = None


def lib():
    global _lib
    if _lib is not None:
        return _lib
    key = hashlib.sha256(b"".join(open(p, "rb").read() for p in SOURCES) + " ".join(CXXFLAGS).encode()).hexdigest()[:16]
    out_dir = os.path.join(tempfile.gettempdir(), f"bendy_oracle_env_{os.getuid()}")
    path = os.path.join(out_dir, f"liboracle_env_{key}.so")
    if not os.path.exists(path):
        os.makedirs(out_dir, exist_ok=True)
        tmp = f"{path}.{os.getpid()}.tmp"
        subprocess.run([os.environ.get("CXX", "g++"), *CXXFLAGS, "-o", tmp, SOURCES[0]], check=True)
        os.replace(tmp, path)
    L = C.CDLL(path)
    for name, fn in vars(O.lib()).items():       # the oracle's signatures, as oracle_ffi declares them
        if name.startswith("orc_"):
            f = getattr(L, name)
            f.argtypes, f.restype = fn.argtypes, fn.restype
    L.orc_env_set.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32]
    L.orc_env_scene_destroy.argtypes = [C.c_void_p]
    L.orc_env_lookup.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p]
    _lib = L
    return L


@contextlib.contextmanager
def _this_library():
    """oracle_ffi's methods call oracle_ffi.lib(): point it at this library for the duration of one call"""
    saved = O._lib
    O._lib = lib()
    try:
        yield
    finally:
        O._lib = saved


def _on_this_library(method):
    def wrapped(self, *args, **kw):
        with _this_library():
            return method(self, *args, **kw)
    wrapped.__doc__ = method.__doc__
    return wrapped


class EnvOracleScene(O.OracleScene):
    """oracle_ffi.OracleScene on the environment-map oracle"""
    __init__ = _on_this_library(O.OracleScene.__init__)
    set_camera_aspect = _on_this_library(O.OracleScene.set_camera_aspect)
    set_lenses = _on_this_library(O.OracleScene.set_lenses)
    render = _on_this_library(O.OracleScene.render)
    probe = _on_this_library(O.OracleScene.probe)
    camera_rays = _on_this_library(O.OracleScene.camera_rays)

    @classmethod
    def load(cls, path):
        return cls(O.read_scene_json(path))

    def set_environment(self, rgb):
        """(H, W, 3) RGB, row 0 = +y pole, centre column along -z; None clears it"""
        if rgb is None:
            self._env = None
            lib().orc_env_set(self.handle, None, 0, 0)
            return
        self._env = np.ascontiguousarray(rgb, np.float32)
        h, w, _ = self._env.shape
        lib().orc_env_set(self.handle, self._env.ctypes.data, w, h)

    def __del__(self):
        if getattr(self, "handle", None):
            lib().orc_env_scene_destroy(self.handle)
            self.handle = None


def env_lookup(rgb, d):
    """the map's factor for direction(s) d ((3,) or (n, 3)) in the (H, W, 3) map rgb"""
    rgb = np.ascontiguousarray(rgb, np.float32)
    h, w, _ = rgb.shape
    d = np.ascontiguousarray(d, np.float32)
    flat = d.reshape(-1, 3)
    out = np.zeros_like(flat)
    for i in range(len(flat)):
        lib().orc_env_lookup(rgb.ctypes.data, w, h, flat[i].ctypes.data, out[i].ctypes.data)
    return out.reshape(d.shape)


def load_pair(name, width, height, lenses=None):
    """common.load_pair with the oracle side on this library: (oracle scene, engine scene, camera ref)"""
    import bendy_tracer_b200 as bt
    path = O.scene_path(name)
    osc = EnvOracleScene.load(path)
    esc = bt.Scene.load(path)
    cam = esc.find_by_tag("camera")
    assert cam == osc.find_by_tag("camera")
    aspect = float(np.float32(width) / np.float32(height))
    osc.set_camera_aspect(cam, aspect)
    esc.set_camera_aspect(cam, aspect)
    if lenses is not None:
        osc.set_lenses(lenses)
        esc.set_lenses(lenses)
    return osc, esc, cam
