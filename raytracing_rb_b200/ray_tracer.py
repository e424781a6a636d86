"""Mirror of the reference's ray-level entry points below the camera: Alex::Ray (src/libs/algebra.rb:3-17) and
Alex::RayTracer#trace_sync (src/ray_tracer.rb:16-46).  Tracing runs on the GPU through rtrb_trace_rays; World#intersect
is World.intersect (world.py) through rtrb_intersect_rays."""
import numpy as np

from . import _abi
from .vec3 import Vec3


class Ray:
    """Ray(front, position), algebra.rb: `front` is not normalised."""

    def __init__(self, front, position):
        self.front, self.position = front, position

    def to_a(self):
        """(position, front) as six floats, the rtrb_ray layout."""
        return list(self.position.to_a()) + list(self.front.to_a())

    def distance(self, pos):  # algebra.rb:10-12
        return (self.position - pos).r


def rays_array(rays):
    """Ray objects, or rows of (position, front), -> [n, 6] float64."""
    rays = list(rays) if not isinstance(rays, np.ndarray) else rays
    if len(rays) and isinstance(rays[0], Ray):
        return np.array([r.to_a() for r in rays], np.float64).reshape(-1, 6)
    return np.ascontiguousarray(rays, np.float64).reshape(-1, 6)


class RayTracer:
    """RayTracer.new(world, trace_depth, width, height, mc): trace_sync(x, y, ray) traces one ray for pixel (x, y) of a
    width x height frame; its Monte-Carlo rays are keyed as that pixel's sample 0 (pixel y * width + x), as the frame's
    first sample of the pixel is."""

    def __init__(self, world, trace_depth, width, height, monte_carlo_diffusion_times=0, seed=1,
                 precision=_abi.PREC_DEFAULT, device=0):
        self.world, self.trace_depth, self.width, self.height = world, trace_depth, width, height
        self.monte_carlo_diffusion_times = monte_carlo_diffusion_times
        self.seed, self.precision, self.device = seed, precision, device
        self.last_stats = None

    def trace_batch(self, xs, ys, rays):
        """trace_sync for many (x, y, ray) at once -> (rgb [n, 3] float64, status code); raises nothing, see last_stats."""
        xs, ys = np.asarray(xs, np.int64).reshape(-1), np.asarray(ys, np.int64).reshape(-1)
        arr = rays_array(rays)
        keys = np.stack([ys * self.width + xs, np.zeros_like(xs)], axis=1).astype(np.uint32)
        rgb, _, stats, code = self.world.renderer(self.device).trace_rays(
            arr, self.trace_depth, self.monte_carlo_diffusion_times, self.seed, keys, self.precision)
        self.last_stats = stats
        return rgb, code

    def trace_sync(self, x, y, ray):
        """ray_tracer.rb:16-46: the colour (unclamped) for one ray.  Raises RuntimeError where the reference raises."""
        rgb, code = self.trace_batch([x], [y], [ray])
        if code == _abi.RTRB_ERR_RAISED:
            raise RuntimeError("the reference would have raised: status 0x%x" % self.last_stats["status"])
        return Vec3(*[float(v) for v in rgb[0]])
