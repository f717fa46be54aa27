"""bendy_tracer_b200 -- B200-native engine for bendy-tracer's per-sample render loop.

Python mirror of the reference crate's public render API (see api.py) over the C ABI declared in
include/bendy_b200.h.  Importing this package loads csrc/libbendy_b200.so and fails loudly when
it is missing; there is no CPU fallback.
"""
from .api import (BendyError, Buffer, ColorSpace, Config, Engine, LensConfig, Output, Projection, RenderConfig,
                  Scene, ScenePanic, Status, Subsample, Tracer)
from .distributed import render_sharded, shard_passes

__all__ = ["BendyError", "Buffer", "ColorSpace", "Config", "Engine", "LensConfig", "Output", "Projection", "RenderConfig",
           "Scene", "ScenePanic", "Status", "Subsample", "Tracer", "render_sharded", "shard_passes"]
