"""Host-side mirror of the reference's public render API over the C ABI.

Same names, argument meaning and error behaviour as the Rust crate `bendy_tracer`
(reference src/lib.rs:1-4): `Tracer`, `Config`, `RenderConfig`, `Subsample`, `Output`, `Status`
(src/tracer/mod.rs:16-203), `Buffer`, `ColorSpace` (src/tracer/buffer.rs:11-193) and `Scene`
(src/scene/mod.rs:84-151).  Panics of the reference surface as `ScenePanic`.

torch is used only for device memory and streams (plumbing); every computation happens in
csrc/libbendy_b200.so.
"""
import ctypes as C
import enum
import gzip
import threading
from dataclasses import dataclass, field
from typing import Optional

import numpy as np

from . import _ffi
from ._ffi import BendyError, ScenePanic, check, lib  # noqa: F401


class Output(enum.IntEnum):
    """reference src/tracer/mod.rs:108-115"""
    Full = 0
    Albedo = 1
    Normal = 2
    Depth = 3


class Status(enum.IntEnum):
    """reference src/tracer/mod.rs:159-163"""
    Done = 0
    InProgress = 1


class ColorSpace(enum.IntEnum):
    """reference src/tracer/buffer.rs:11-17"""
    NONE = 0
    Normal = 1
    Linear = 2
    SRgb = 3


@dataclass(frozen=True)
class Subsample:
    """reference src/tracer/mod.rs:47-106. `Subsample.none()` / `Subsample.subpixel(n)`."""
    count: int = 0  # 0 = Subsample::None

    @staticmethod
    def none():
        return Subsample(0)

    @staticmethod
    def subpixel(count):
        return Subsample(int(count))

    def subpixel_size(self):
        return 1.0 if self.count == 0 else float(np.float32(1.0) / np.float32(self.count))

    def subpixel_count(self):
        return 1 if self.count == 0 else self.count * self.count

    def __iter__(self):
        if self.count == 0:
            yield (0.0, 0.0)
            return
        width = np.float32(1.0) / np.float32(self.count)
        for k in range(self.count * self.count):
            yield (float(np.float32(k % self.count) * width), float(np.float32(k // self.count) * width))


@dataclass
class Config:
    """reference src/tracer/mod.rs:16-45 (Config::DEFAULT :29-38)"""
    max_bounces: int = 8
    max_volume_bounces: int = 32
    clip_min: float = 0.01
    clip_max: float = 1000.0
    volume_step: float = 0.1
    chunks_x: int = 4
    chunks_y: int = 2
    output: Output = Output.Full

    def _c(self):
        return _ffi.BtConfig(self.max_bounces, self.max_volume_bounces, self.clip_min, self.clip_max,
                             self.volume_step, self.chunks_x, self.chunks_y, int(self.output))


@dataclass
class RenderConfig:
    """reference src/tracer/mod.rs:117-157"""
    subsample: Subsample = field(default_factory=Subsample.none)
    samples: int = 64
    output: Optional[Output] = None
    max_bounces: Optional[int] = None
    max_volume_bounces: Optional[int] = None
    volume_step: Optional[float] = None

    @staticmethod
    def with_samples(samples):
        return RenderConfig(samples=samples)

    @staticmethod
    def with_samples_subsample(samples, subsample):
        return RenderConfig(samples=samples, subsample=subsample)

    def _c(self):
        c = _ffi.BtRenderConfig()
        c.subsample = self.subsample.count
        c.samples = self.samples
        for name in ("output", "max_bounces", "max_volume_bounces", "volume_step"):
            v = getattr(self, name)
            setattr(c, "has_" + name, 0 if v is None else 1)
            if v is not None:
                setattr(c, name, int(v) if name != "volume_step" else float(v))
        return c


@dataclass
class LensConfig:
    """stepping parameters of the lens-field extension (DESIGN.md "Geodesic model")"""
    kappa: float = 0.05
    h_min: float = 0.02
    h_max: float = 5.0
    r_far: float = 500.0
    max_steps: int = 4096
    exact_rsqrt: bool = False   # BT_LENS_EXACT_RSQRT: bit-identical to the CPU oracle, slower
    no_skip: bool = False       # BT_LENS_NO_SKIP: intersect every chord (the oracle's literal loop)

    def _c(self):
        return _ffi.BtLensConfig(self.kappa, self.h_min, self.h_max, self.r_far, self.max_steps,
                                 (1 if self.exact_rsqrt else 0) | (2 if self.no_skip else 0))


class Engine:
    """One CUDA device (replaces the reference's implicit rayon global pool, mod.rs:194)."""

    _default = {}
    _lock = threading.Lock()

    def __init__(self, device=0, devices=None):
        """`devices=[0, 1, ...]`: one engine over several GPUs of the box (bt_engine_create_multi): every render call
        splits its passes across them and sums the slices on devices[0], where device buffers must live"""
        h = C.c_void_p()
        if devices is not None:
            devices = [int(d) for d in devices]
            arr = (C.c_int * len(devices))(*devices)
            check(lib.bt_engine_create_multi(arr, len(devices), C.byref(h)))
            device = devices[0]
        else:
            check(lib.bt_engine_create(int(device), C.byref(h)))
        self.handle = h
        self.device = int(device)
        self.devices = devices or [self.device]

    @classmethod
    def default(cls, device=0):
        with cls._lock:
            if device not in cls._default:
                cls._default[device] = cls(device)
            return cls._default[device]

    @property
    def launch_count(self):
        return int(lib.bt_engine_launch_count(self.handle))

    def set_tuning(self, **knobs):
        """scheduling knobs of the kernels (bt_engine_set_tuning): never change an image; None restores the default"""
        for name, value in knobs.items():
            check(lib.bt_engine_set_tuning(self.handle, name.encode(), -1 if value is None else int(value)))

    def fp32_peak_tflops(self, iters=4096):
        t = C.c_double()
        check(lib.bt_fp32_peak(self.handle, iters, C.byref(t)))
        return t.value

    def geodesic_integrate(self, lenses, xv, n_steps, lens_config=None, stream=None):
        """n_steps RK4 steps of the rays `xv` ((n, 6) x,v) through point masses `lenses` ((m, 4) x,y,z,r_s).

        numpy in -> numpy out (blocking, host copies inside); CUDA torch tensor in -> updated in
        place on `stream` (torch's current stream by default) without synchronising."""
        lenses = np.ascontiguousarray(lenses, np.float32).reshape(-1, 4)
        cfg = (lens_config or LensConfig())._c()
        if isinstance(xv, np.ndarray):
            out = np.ascontiguousarray(xv, np.float32).reshape(-1, 6).copy()
            check(lib.bt_geodesic_integrate(self.handle, lenses.ctypes.data, len(lenses), C.byref(cfg), len(out),
                                            out.ctypes.data, _ffi.MEM_HOST, n_steps, None))
            return out
        import torch
        assert xv.is_cuda and xv.dtype == torch.float32 and xv.is_contiguous()
        s = stream if stream is not None else torch.cuda.current_stream(xv.device).cuda_stream
        check(lib.bt_geodesic_integrate(self.handle, lenses.ctypes.data, len(lenses), C.byref(cfg), xv.numel() // 6,
                                        xv.data_ptr(), _ffi.MEM_DEVICE, n_steps, C.c_void_p(s)))
        return xv

    def __del__(self):
        h, self.handle = getattr(self, "handle", None), None
        if h:
            lib.bt_engine_destroy(h)


class Scene:
    """reference src/scene/mod.rs:84-151 (read side) + the scene wire format (src/main.rs:93-102)."""

    def __init__(self, data: bytes):
        h = C.c_void_p()
        buf = bytes(data)
        check(lib.bt_scene_create_json(None, buf, len(buf), C.byref(h)))
        self.handle = h

    @classmethod
    def load(cls, path):
        """serde_json::from_reader over a GzDecoder or a plain file (src/main.rs:93-102)"""
        with open(path, "rb") as f:
            return cls(f.read())

    @classmethod
    def from_json(cls, text):
        return cls(text.encode() if isinstance(text, str) else text)

    def to_json(self) -> str:
        """serde_json::to_writer (src/main.rs:299-313)"""
        out, n = C.c_void_p(), C.c_size_t()
        check(lib.bt_scene_to_json(self.handle, C.byref(out), C.byref(n)))
        try:
            return C.string_at(out, n.value).decode()
        finally:
            lib.bt_free(out)

    def save(self, path):
        text = self.to_json().encode()
        if str(path).endswith(".gz"):
            with gzip.open(path, "wb") as f:
                f.write(text)
        else:
            with open(path, "wb") as f:
                f.write(text)

    def find_by_tag(self, tag) -> Optional[int]:
        """Scene::find_by_tag (src/scene/mod.rs:124-129): None when no object carries the tag"""
        ref = C.c_uint64()
        code = lib.bt_scene_find_by_tag(self.handle, tag.encode(), C.byref(ref))
        if code == _ffi.ERR_SCENE:
            return None
        check(code)
        return ref.value

    def set_camera_aspect(self, camera_ref, aspect_ratio):
        """the update main pushes through its UpdateQueue (src/main.rs:218-223)"""
        check(lib.bt_scene_set_camera_aspect(self.handle, camera_ref, aspect_ratio))

    def apply_transform(self, object_ref, affine):
        """Object::apply_transform + UpdateQueue::commit (src/scene/object/mod.rs:212-223)"""
        a = (C.c_float * 12)(*[float(x) for x in np.asarray(affine, np.float32).reshape(12)])
        check(lib.bt_scene_apply_transform(self.handle, object_ref, a))

    def commit(self):
        """UpdateQueue::commit (src/scene/mod.rs:204-213): apply the queued edits to the flattened scene now (transform edits in
        place: records rewritten, BVH refit); otherwise the next render does it"""
        check(lib.bt_scene_commit(self.handle))

    def set_lenses(self, xyzr, lens_config=None):
        xyzr = np.ascontiguousarray(xyzr, np.float32).reshape(-1, 4)
        cfg = (lens_config or LensConfig())._c()
        check(lib.bt_scene_set_lenses(self.handle, xyzr.ctypes.data, len(xyzr), C.byref(cfg)))

    def set_environment(self, rgb):
        """environment map (bt_scene_set_environment): an equirectangular (H, W, 3) RGB image that multiplies the colour of
        every escaping path, looked up in its escape direction; row 0 is the +y pole, the centre column looks along -z.
        None clears it.  Negative or non-finite values raise BendyError (BT_ERR_INVALID_ARG), a wrong shape ValueError."""
        if rgb is None:
            check(lib.bt_scene_set_environment(self.handle, None, 0, 0))
            return
        rgb = np.ascontiguousarray(rgb, np.float32)
        if rgb.ndim != 3 or rgb.shape[2] != 3 or rgb.shape[0] == 0 or rgb.shape[1] == 0:
            raise ValueError(f"environment map must be a non-empty (H, W, 3) array, got shape {rgb.shape}")
        if rgb.shape[0] * rgb.shape[1] >= 1 << 31:
            raise ValueError(f"environment map of {rgb.shape[0]} x {rgb.shape[1]} texels: width * height must be below 2^31")
        check(lib.bt_scene_set_environment(self.handle, rgb.ctypes.data, rgb.shape[1], rgb.shape[0]))

    def set_accel(self, accel):
        """closest-hit structure: "auto" (linear scan up to 64 primitives, BVH beyond), "linear", "bvh",
        "linear_faces" (the scan with every cuboid as six rect tests, no box slab test)"""
        check(lib.bt_scene_set_accel(self.handle, {"auto": 0, "linear": 1, "bvh": 2, "linear_faces": 3}[accel]))

    def set_precision(self, precision):
        """arithmetic flavour of the kernels: "auto" (exact for volumetric scenes, fast otherwise),
        "fast" (MUFU reciprocals / square roots, ~1 ulp) or "exact" (IEEE, bit-identical to the oracle)"""
        check(lib.bt_scene_set_precision(self.handle, {"auto": 0, "fast": 1, "exact": 2}[precision]))

    def info(self):
        i = _ffi.BtSceneInfo()
        check(lib.bt_scene_get_info(self.handle, C.byref(i)))
        return {k: getattr(i, k) for k, _ in i._fields_}

    def bvh(self):
        """the acceleration structure as of the last flatten / commit (bt_scene_copy_bvh): `nodes` float32 [n, 8, 4]
        (min.x max.x min.y max.y min.z max.z of the four children, then the child references -- see `refs`),
        `refs` uint32 [n, 4], `order` uint32 [n_primitives] (tree position -> canonical index), `bounds` float32
        [n_primitives, 6] (canonical order)"""
        i = self.info()
        nodes = np.zeros((i["n_bvh_nodes"], 8, 4), np.float32)
        order = np.zeros(i["n_primitives"], np.uint32)
        bounds = np.zeros((i["n_primitives"], 6), np.float32)
        check(lib.bt_scene_copy_bvh(self.handle, nodes.ctypes.data, nodes.shape[0], order.ctypes.data, bounds.ctypes.data, order.shape[0]))
        return {"nodes": nodes, "refs": nodes[:, 6, :].copy().view(np.uint32), "order": order, "bounds": bounds}

    def __del__(self):
        h, self.handle = getattr(self, "handle", None), None
        if h:
            lib.bt_scene_destroy(h)


class Buffer:
    """reference src/tracer/buffer.rs:32-193: RGBA32F running sums + sample counter + u8 preview.

    `device=None` keeps the sums in host memory (numpy; every render copies them to the GPU and
    back, like a host caller of the C ABI); `device="cuda:0"` keeps them in HBM as a torch tensor.
    """

    def __init__(self, width, height, color_space=ColorSpace.SRgb, device=None):
        self.color_space = ColorSpace(color_space)
        self.device = device
        self._samples = 0
        self._preview = None
        self._alloc(width, height)

    def _alloc(self, width, height):
        if self.device is None:
            self.data = np.zeros((height, width, 4), np.float32)
            self.data[..., 3] = 1.0  # BLACK_ALPHA_ONE, buffer.rs:9,43
        else:
            import torch
            self.data = torch.zeros((height, width, 4), dtype=torch.float32, device=self.device)
            self.data[..., 3] = 1.0

    def width(self):
        return self.data.shape[1]

    def height(self):
        return self.data.shape[0]

    def dimensions(self):
        return (self.width(), self.height())

    def samples(self):
        return self._samples

    def pixel_width(self):
        return float(np.float32(2.0) * (np.float32(1.0) / np.float32(self.width())))

    def pixel_height(self):
        return float(np.float32(2.0) * (np.float32(1.0) / np.float32(self.height())))

    def into_buffer(self):
        return self.data

    def clear(self):
        self.data[..., :3] = 0.0
        self.data[..., 3] = 1.0
        self._samples = 0

    def resize(self, width, height):
        self._alloc(width, height)
        self._preview = None
        self._samples = 0

    def chunks(self, chunks_x, chunks_y):
        """Buffer::chunks + Chunks::next (buffer.rs:102-115, 293-326): ceil-div tile size, row-major
        enumeration, last row / column clipped.  Yields (min_x, min_y, max_x, max_y).  The engine does not
        schedule by these tiles (Config.chunks_* only ever affected scheduling); the iterator is kept
        for callers that walk the reference's tiles."""
        w, h = self.width(), self.height()
        if chunks_x <= 0 or chunks_y <= 0:
            raise ZeroDivisionError("attempt to calculate the remainder with a divisor of zero")   # the reference panics
        cw = w // chunks_x if w % chunks_x == 0 else w // chunks_x + 1
        ch = h // chunks_y if h % chunks_y == 0 else h // chunks_y + 1
        ox = oy = 0
        done = False
        while not done:
            tw, th = min(cw, w - ox), min(ch, h - oy)
            yield (ox, oy, ox + tw, oy + th)
            ox += tw
            if ox == w:
                ox = 0
                oy += th
            if oy == h:
                done = True

    def _ptr_mem(self):
        if isinstance(self.data, np.ndarray):
            return self.data.ctypes.data, _ffi.MEM_HOST
        return self.data.data_ptr(), _ffi.MEM_DEVICE

    def preview(self, engine=None):
        """Buffer::preview (buffer.rs:117-138): RGBA8 numpy array (H, W, 4)"""
        engine = engine or Engine.default(_device_index(self.device))
        ptr, mem = self._ptr_mem()
        h, w = self.height(), self.width()
        if mem == _ffi.MEM_HOST:
            out = np.zeros((h, w, 4), np.uint8)
            check(lib.bt_resolve_u8(engine.handle, ptr, mem, w, h, self._samples, int(self.color_space), out.ctypes.data))
        else:
            import torch
            torch.cuda.current_stream(self.data.device).synchronize()
            dev = torch.zeros((h, w, 4), dtype=torch.uint8, device=self.data.device)
            check(lib.bt_resolve_u8(engine.handle, ptr, mem, w, h, self._samples, int(self.color_space), dev.data_ptr()))
            out = dev.cpu().numpy()
        self._preview = out
        return out

    def preview_or_update(self, engine=None):
        return self._preview if self._preview is not None else self.preview(engine)

    def maybe_preview(self):
        return self._preview

    def take_preview(self):
        p, self._preview = self._preview, None
        return p


def _device_index(device):
    if device is None:
        return 0
    import torch
    d = torch.device(device)
    return d.index or 0


class Tracer:
    """reference src/tracer/mod.rs:165-203"""

    def __init__(self, config: Optional[Config] = None, engine: Optional[Engine] = None, seed: int = 0):
        self.config = config or Config()
        self.engine = engine
        self.seed = seed

    @staticmethod
    def with_config(config, **kw):
        return Tracer(config, **kw)

    def render(self, scene: Scene, camera: int, config: RenderConfig, buffer: Buffer, *, sample_base=None,
               stream=None, sync=True) -> Status:
        """Tracer::render (mod.rs:179-202): add `samples * subpixel_count` samples per pixel to `buffer`.

        The RNG stream is keyed by (self.seed, pixel, global pass index); the global pass index of
        this call starts at `sample_base` (default: the passes already in `buffer`).  With a
        device buffer and sync=False the call only enqueues work on `stream` / torch's current
        stream."""
        engine = self.engine or Engine.default(_device_index(buffer.device))
        cfg, rc = self.config._c(), config._c()
        if sample_base is None:
            sample_base = buffer.samples() // config.subsample.subpixel_count()
        ptr, mem = buffer._ptr_mem()
        samples = C.c_uint64(buffer._samples)
        status = C.c_int32(0)
        if mem == _ffi.MEM_HOST:
            check(lib.bt_render(engine.handle, scene.handle, camera, C.byref(cfg), C.byref(rc), self.seed, sample_base,
                                ptr, mem, buffer.width(), buffer.height(), C.byref(samples), C.byref(status)))
        else:
            import torch
            s = stream if stream is not None else torch.cuda.current_stream(buffer.data.device).cuda_stream
            check(lib.bt_render_async(engine.handle, scene.handle, camera, C.byref(cfg), C.byref(rc), self.seed,
                                      sample_base, ptr, buffer.width(), buffer.height(), C.byref(samples),
                                      C.byref(status), C.c_void_p(s)))
            if sync:   # the stream the work was enqueued on, which need not be torch's current one
                (torch.cuda.ExternalStream(s, device=buffer.data.device) if stream is not None
                 else torch.cuda.current_stream(buffer.data.device)).synchronize()
        buffer._samples = samples.value
        return Status(status.value)

    def render_stats(self, scene: Scene, camera: int, config: RenderConfig, width, height, sample_base=0):
        """work counters of the render call with these arguments (bt_render_stats): dict"""
        engine = self.engine or Engine.default(0)
        cfg, rc = self.config._c(), config._c()
        out = (C.c_uint64 * 4)()
        check(lib.bt_render_stats(engine.handle, scene.handle, camera, C.byref(cfg), C.byref(rc), self.seed, sample_base,
                                  width, height, out))
        return dict(paths=out[0], scans=out[1], rk4_steps=out[2], events=out[3])

    def render_pool_stats(self, scene: Scene, camera: int, config: RenderConfig, width, height, sample_base=0):
        """scheduling counters of the pooled kernel for the render call with these arguments (bt_render_pool_stats)"""
        engine = self.engine or Engine.default(0)
        cfg, rc = self.config._c(), config._c()
        out = (C.c_uint64 * 17)()
        check(lib.bt_render_pool_stats(engine.handle, scene.handle, camera, C.byref(cfg), C.byref(rc), self.seed, sample_base,
                                       width, height, out))
        keys = ("step_iterations", "step_lanes", "refill_rounds", "step_entries", "scan_passes", "scan_slots", "shade_passes",
                "shade_slots", "regen_passes", "paths_issued", "paths_retired", "turns", "clk_step", "clk_scan", "clk_shade", "clk_regen",
                "clk_total")
        d = dict(zip(keys, [int(v) for v in out]))
        d["lanes_per_step"] = d["step_lanes"] / max(d["step_iterations"], 1)
        d["lanes_per_scan"] = d["scan_slots"] / max(d["scan_passes"], 1)
        d["lanes_per_shade"] = d["shade_slots"] / max(d["shade_passes"], 1)
        d["lanes_per_regen"] = d["paths_issued"] / max(d["regen_passes"], 1)
        for k in ("step", "scan", "shade", "regen"):
            d["time_share_" + k] = d["clk_" + k] / max(d["clk_total"], 1)
        return d

    def trace_segments(self, scene: Scene, origins, dirs):
        """ChunkState::try_hit (mod.rs:389-402) / the geodesic segment for each ray; dict of numpy arrays"""
        engine = self.engine or Engine.default(0)
        o = np.ascontiguousarray(origins, np.float32).reshape(-1, 3)
        d = np.ascontiguousarray(dirs, np.float32).reshape(-1, 3)
        out = (_ffi.BtSegment * max(len(o), 1))()
        cfg = self.config._c()
        check(lib.bt_trace_segments(engine.handle, scene.handle, C.byref(cfg), len(o), o.ctypes.data, d.ctypes.data, out))
        a = np.frombuffer(out, dtype=np.dtype(_ffi.BtSegment))[:len(o)]
        return {k: a[k].copy() for k in ("face", "steps", "object_ref", "t", "position", "normal", "direction")}

    def camera_rays(self, scene: Scene, camera: int, config: RenderConfig, width, height, xs, ys, path_index, sample_base=0):
        """the rays render_samples generates (mod.rs:272-302) for (x, y, path index) triples; (n, 6)"""
        engine = self.engine or Engine.default(0)
        xs = np.ascontiguousarray(xs, np.uint32)
        ys = np.ascontiguousarray(ys, np.uint32)
        pi = np.ascontiguousarray(path_index, np.uint64)
        out = np.zeros((len(xs), 6), np.float32)
        cfg, rc = self.config._c(), config._c()
        check(lib.bt_camera_rays(engine.handle, scene.handle, camera, C.byref(cfg), C.byref(rc), self.seed, sample_base,
                                 width, height, len(xs), xs.ctypes.data, ys.ctypes.data, pi.ctypes.data, out.ctypes.data))
        return out
