"""ctypes binding of include/bendy_b200.h (csrc/libbendy_b200.so).

The library is loaded eagerly and loudly: if it is missing the package raises instead of falling
back to anything -- there is no CPU path in this package.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("BENDY_B200_LIB") or os.path.join(_HERE, "csrc", "libbendy_b200.so")

OK, ERR_INVALID_ARG, ERR_PARSE, ERR_SCENE, ERR_CUDA, ERR_UNSUPPORTED = 0, -1, -2, -3, -4, -5
MEM_HOST, MEM_DEVICE = 0, 1


class BtConfig(C.Structure):
    _fields_ = [("max_bounces", C.c_uint64), ("max_volume_bounces", C.c_uint64),
                ("clip_min", C.c_float), ("clip_max", C.c_float), ("volume_step", C.c_float),
                ("chunks_x", C.c_uint32), ("chunks_y", C.c_uint32), ("output", C.c_int32)]


class BtRenderConfig(C.Structure):
    _fields_ = [("subsample", C.c_uint32), ("samples", C.c_uint64),
                ("has_output", C.c_int32), ("output", C.c_int32),
                ("has_max_bounces", C.c_int32), ("max_bounces", C.c_uint64),
                ("has_max_volume_bounces", C.c_int32), ("max_volume_bounces", C.c_uint64),
                ("has_volume_step", C.c_int32), ("volume_step", C.c_float)]


class BtLensConfig(C.Structure):
    _fields_ = [("kappa", C.c_float), ("h_min", C.c_float), ("h_max", C.c_float),
                ("r_far", C.c_float), ("max_steps", C.c_uint32), ("flags", C.c_uint32)]


class BtSegment(C.Structure):
    _fields_ = [("face", C.c_int32), ("steps", C.c_uint32), ("object_ref", C.c_uint64),
                ("t", C.c_float), ("position", C.c_float * 3), ("normal", C.c_float * 3),
                ("direction", C.c_float * 3)]


class BtSceneInfo(C.Structure):
    _fields_ = [("n_objects", C.c_uint32), ("n_data", C.c_uint32), ("n_primitives", C.c_uint32),
                ("n_lights", C.c_uint32), ("n_volumes", C.c_uint32), ("n_lenses", C.c_uint32),
                ("n_bvh_nodes", C.c_uint32), ("n_boxes", C.c_uint32), ("root_material", C.c_uint64)]


# every symbol include/bendy_b200.h declares: (restype, argtypes)
_P = C.c_void_p
SIGNATURES = {
    "bt_engine_create": (C.c_int, [C.c_int, C.POINTER(_P)]),
    "bt_engine_create_multi": (C.c_int, [C.POINTER(C.c_int), C.c_int, C.POINTER(_P)]),
    "bt_engine_device_count": (C.c_int, [_P]),
    "bt_engine_destroy": (None, [_P]),
    "bt_engine_launch_count": (C.c_uint64, [_P]),
    "bt_engine_set_tuning": (C.c_int, [_P, C.c_char_p, C.c_int64]),
    "bt_scene_create_json": (C.c_int, [_P, _P, C.c_size_t, C.POINTER(_P)]),
    "bt_scene_to_json": (C.c_int, [_P, C.POINTER(_P), C.POINTER(C.c_size_t)]),
    "bt_free": (None, [_P]),
    "bt_scene_destroy": (None, [_P]),
    "bt_scene_find_by_tag": (C.c_int, [_P, C.c_char_p, C.POINTER(C.c_uint64)]),
    "bt_scene_set_camera_aspect": (C.c_int, [_P, C.c_uint64, C.c_float]),
    "bt_scene_apply_transform": (C.c_int, [_P, C.c_uint64, C.POINTER(C.c_float)]),
    "bt_scene_commit": (C.c_int, [_P]),
    "bt_scene_set_lenses": (C.c_int, [_P, _P, C.c_uint32, C.POINTER(BtLensConfig)]),
    "bt_lens_config_default": (None, [C.POINTER(BtLensConfig)]),
    "bt_scene_set_environment": (C.c_int, [_P, _P, C.c_uint32, C.c_uint32]),
    "bt_scene_set_accel": (C.c_int, [_P, C.c_int]),
    "bt_scene_set_precision": (C.c_int, [_P, C.c_int]),
    "bt_scene_get_info": (C.c_int, [_P, C.POINTER(BtSceneInfo)]),
    "bt_scene_copy_bvh": (C.c_int, [_P, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_uint64]),
    "bt_config_default": (None, [C.POINTER(BtConfig)]),
    "bt_render_config_default": (None, [C.POINTER(BtRenderConfig)]),
    "bt_render": (C.c_int, [_P, _P, C.c_uint64, C.POINTER(BtConfig), C.POINTER(BtRenderConfig), C.c_uint64,
                            C.c_uint64, _P, C.c_int, C.c_uint32, C.c_uint32, C.POINTER(C.c_uint64),
                            C.POINTER(C.c_int32)]),
    "bt_render_async": (C.c_int, [_P, _P, C.c_uint64, C.POINTER(BtConfig), C.POINTER(BtRenderConfig), C.c_uint64,
                                  C.c_uint64, _P, C.c_uint32, C.c_uint32, C.POINTER(C.c_uint64),
                                  C.POINTER(C.c_int32), _P]),
    "bt_render_stats": (C.c_int, [_P, _P, C.c_uint64, C.POINTER(BtConfig), C.POINTER(BtRenderConfig), C.c_uint64,
                                  C.c_uint64, C.c_uint32, C.c_uint32, C.POINTER(C.c_uint64)]),
    "bt_render_pool_stats": (C.c_int, [_P, _P, C.c_uint64, C.POINTER(BtConfig), C.POINTER(BtRenderConfig), C.c_uint64,
                                       C.c_uint64, C.c_uint32, C.c_uint32, C.POINTER(C.c_uint64)]),
    "bt_resolve_u8": (C.c_int, [_P, _P, C.c_int, C.c_uint32, C.c_uint32, C.c_uint64, C.c_int, _P]),
    "bt_trace_segments": (C.c_int, [_P, _P, C.POINTER(BtConfig), C.c_uint32, _P, _P, C.POINTER(BtSegment)]),
    "bt_camera_rays": (C.c_int, [_P, _P, C.c_uint64, C.POINTER(BtConfig), C.POINTER(BtRenderConfig), C.c_uint64,
                                 C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint32, _P, _P, _P, _P]),
    "bt_geodesic_integrate": (C.c_int, [_P, _P, C.c_uint32, C.POINTER(BtLensConfig), C.c_uint32, _P, C.c_int,
                                        C.c_uint32, _P]),
    "bt_fp32_peak": (C.c_int, [_P, C.c_uint32, C.POINTER(C.c_double)]),
    "bt_last_error": (C.c_char_p, []),
}


class BendyError(RuntimeError):
    """A BT_ERR_* return code from the engine (code, message from bt_last_error)."""

    def __init__(self, code, message):
        super().__init__(f"bendy_b200 error {code}: {message}")
        self.code = code
        self.message = message


class ScenePanic(BendyError):
    """BT_ERR_SCENE: a condition on which the reference panics."""


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `make -C bendy_tracer_b200/csrc` "
            "(or __graft_entry__.build()); bendy_tracer_b200 has no CPU fallback")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError here = the .so does not export the header's symbol
        fn.restype = res
        fn.argtypes = args
    return lib


lib = _load()


def check(code):
    if code == OK:
        return
    msg = (lib.bt_last_error() or b"").decode(errors="replace")
    if code == ERR_SCENE:
        raise ScenePanic(code, msg)
    raise BendyError(code, msg)
