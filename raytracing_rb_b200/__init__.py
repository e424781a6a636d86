"""raytracing_rb_b200 — B200-native tracing core for raytracing_rb's per-pixel hot path
(Camera#render_at -> RayTracer#trace_sync), behind the reference's World/Camera API.

Host side mirrors the reference classes (World, Camera, Sphere, Plane, SpotLight, Texture,
ConfigurableObject, Vec3); the hot path is hand-written CUDA for sm_100a in csrc/, reached through
the C ABI of include/rtrb_b200.h.  No CPU fallback exists."""
from . import _abi
from ._abi import PREC_DEFAULT, PREC_FAST64, PREC_STRICT, RNG_CTR, RNG_MT
from .camera import Camera, write_png, write_png_scanlines
from .configurable_object import ConfigurableObject
from .lights import Light, SpotLight
from .objects import Box, Plane, Sphere, WorldObject
from .ray_tracer import Ray, RayTracer
from .renderer import (RAY_HIT_DTYPE, Frame, Progressive, Renderer, deal_frames, device_count, ipc_close, ipc_open,
                       make_opts, make_ray_opts, measure_fma_peak, png_max_bytes, progressive_schedule, render_multi,
                       tile_partition)
from .texture import Texture
from .vec3 import Vec3
from .world import World

__all__ = [
    "Camera", "World", "Sphere", "Plane", "Box", "WorldObject", "Light", "SpotLight", "Texture", "Vec3",
    "ConfigurableObject", "Renderer", "Frame", "make_opts", "render_multi", "measure_fma_peak",
    "device_count", "deal_frames", "ipc_open", "ipc_close", "write_png", "write_png_scanlines", "tile_partition",
    "png_max_bytes", "Progressive", "progressive_schedule", "Ray", "RayTracer", "RAY_HIT_DTYPE", "make_ray_opts",
    "PREC_STRICT", "PREC_FAST64", "PREC_DEFAULT", "RNG_CTR", "RNG_MT",
]
