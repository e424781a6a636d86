"""Mirror of Alex::Camera (reference src/camera.rb:15-158).  Ruby (here: Python, because this image
has no Ruby) stays the host: it parses camera.yml, owns the canvas and saves the PNG.  The pixel
loops render_sync (:101-110) / render_fork (:41-68) are replaced by ONE frame-level call into the
CUDA core, `render_cuda`, which returns the finished RGBA8 rows.

There is deliberately no CPU `render_sync` here: the product has no CPU path.  `render_at(x, y)`
is kept for API parity and runs the same kernels on a one-pixel window."""
import os
import struct
import zlib

import numpy as np

from . import _abi
from .configurable_object import ConfigurableObject
from .renderer import make_opts, progressive_schedule, render_multi
from .world import synced_renderer


def write_png(path, rgba):
    """Minimal RGBA8 PNG writer (the reference uses the `png` gem, camera.rb:36-39)."""
    h, w = rgba.shape[:2]
    raw = np.concatenate([np.zeros((h, 1), np.uint8), rgba.reshape(h, w * 4)], axis=1).tobytes()

    def chunk(tag, data):
        c = struct.pack(">I", len(data)) + tag + data
        return c + struct.pack(">I", zlib.crc32(tag + data) & 0xFFFFFFFF)

    with open(path, "wb") as f:
        f.write(b"\x89PNG\r\n\x1a\n")
        f.write(chunk(b"IHDR", struct.pack(">IIBBBBB", w, h, 8, 6, 0, 0, 0)))
        f.write(chunk(b"IDAT", zlib.compress(raw, 6)))
        f.write(chunk(b"IEND", b""))


def write_png_scanlines(path, scanlines, width, height):
    """PNG (8-bit RGB) from RTRB_FMT_PNG_RGB8 scanlines: the device already laid the rows out the way IDAT wants them
    (filter byte + pixels), so the host only deflates and frames the chunks."""
    def chunk(tag, data):
        c = struct.pack(">I", len(data)) + tag + data
        return c + struct.pack(">I", zlib.crc32(tag + data) & 0xFFFFFFFF)

    with open(path, "wb") as f:
        f.write(b"\x89PNG\r\n\x1a\n")
        f.write(chunk(b"IHDR", struct.pack(">IIBBBBB", width, height, 8, 2, 0, 0, 0)))
        f.write(chunk(b"IDAT", zlib.compress(np.ascontiguousarray(scanlines).tobytes(), 6)))
        f.write(chunk(b"IEND", b""))


class Camera(ConfigurableObject):
    # camera.rb:17-24 accessors
    position = up = front = None
    width = height = 0
    image_distance = focal_distance = aperture_radius = None
    retina_width = retina_height = None
    trace_depth = None
    max_sample_times = pre_sample_times = variant_threshold = None
    monte_carlo_diffusion_times = None

    def __init__(self, world, config_file, device=0):
        self.width = 0
        self.height = 0
        super().__init__(config_file)
        self.world = world
        self.device = device
        self._renderers = {}
        self.canvas = np.zeros((self.height, self.width, 4), np.uint8)  # PNG::Canvas.new(w, h, Black), :33
        self.canvas[..., 3] = 255
        self.last_frame = None

    # -- flattening -------------------------------------------------------------------------------
    def camera_desc(self):
        c = _abi.CameraDesc()
        c.position = (_abi.D3)(*self.position.to_a())
        c.up = (_abi.D3)(*self.up.to_a())
        c.front = (_abi.D3)(*self.front.to_a())
        c.retina_width, c.retina_height = float(self.retina_width), float(self.retina_height)
        c.aperture_radius = float(self.aperture_radius)
        c.image_distance, c.focal_distance = float(self.image_distance), float(self.focal_distance)
        c.variant_threshold = float(self.variant_threshold)
        c.width, c.height = int(self.width), int(self.height)
        c.pre_sample_times, c.max_sample_times = int(self.pre_sample_times), int(self.max_sample_times)
        c.trace_depth = int(self.trace_depth)
        c.monte_carlo_diffusion_times = int(self.monte_carlo_diffusion_times)
        return c

    def renderer(self, device=None):
        """This camera's renderer on `device` (one per device, made on first use), brought up to date with the world:
        edits of its objects and lights since the last call reach the next frame."""
        return synced_renderer(self._renderers, self.device if device is None else device, self.world)

    # -- the hot path -----------------------------------------------------------------------------
    def render_frame(self, gpus=1, seed=1, precision=_abi.PREC_DEFAULT, window=None, count_detail=False,
                     want_rgb=True, want_hit=True, rng_mode=_abi.RNG_CTR):
        """One frame on `gpus` GPUs -> Frame (see renderer.Frame)."""
        opts = make_opts(seed=seed, precision=precision, window=window, count_detail=count_detail, rng_mode=rng_mode)
        cam = self.camera_desc()
        if gpus <= 1:
            frame = self.renderer().render(cam, opts, want_rgb=want_rgb, want_hit=want_hit)
        else:
            frame = render_multi([self.renderer(d) for d in range(gpus)], cam, opts, want_rgb=want_rgb,
                                 want_hit=want_hit)
        self.last_frame = frame
        return frame

    @staticmethod
    def _raise_for(stats):
        names = [n for b, n in ((_abi.ST_COLOR_GT_1, "color greater than 1"),
                                (_abi.ST_ZERO_VECTOR, "zero vector detected"),
                                (_abi.ST_MATH_DOMAIN, "Math::DomainError"),
                                (_abi.ST_STACK_OVERFLOW, "device bounce stack overflow"),
                                (_abi.ST_NAN_TO_INT, "FloatDomainError")) if stats["status"] & b]
        raise RuntimeError("%s at pixel (%d, %d)" % (", ".join(names), stats["first_bad_x"], stats["first_bad_y"]))

    def render_cuda(self, file_path=None, gpus=1, seed=1, **kw):
        """Drop-in for render_sync(file_path) / render_fork(file_path, n) (camera.rb:41-68,101-110).
        Raises RuntimeError where the reference would have raised mid-frame (ray_tracer.rb:294-296,
        fast_4d_matrix.c:124,291), after the whole frame has been produced."""
        frame = self.render_frame(gpus=gpus, seed=seed, **kw)
        self.canvas[...] = frame.rgba
        if file_path:
            self.save_image(file_path)
        if frame.raised:
            self._raise_for(frame.stats)
        return frame

    def render_png(self, file_path, seed=1, **kw):
        """render_cuda(file_path) with the PNG encoded on the GPU: one GPU renders the frame in RGB8 and deflates it in
        device memory, and only the file crosses PCIe (8-bit RGB, where save_image writes RGBA with alpha 255; the
        pixels are the same).  `canvas` is left as it was.  Raises RuntimeError as render_cuda does, after the file
        has been written.  Returns the frame's stats dict."""
        opts = make_opts(seed=seed, skip_outputs=_abi.SKIP_RGB | _abi.SKIP_HIT, pixel_format=_abi.FMT_RGB8, **kw)
        r = self.renderer()
        stats, code = r.render_device(self.camera_desc(), opts)
        png = r.encode_png(self.width, self.height, _abi.FMT_RGB8)
        d = os.path.dirname(os.path.abspath(file_path))
        os.makedirs(d, exist_ok=True)
        with open(file_path, "wb") as f:
            f.write(png)
        if code == _abi.RTRB_ERR_RAISED:
            self._raise_for(stats)
        return stats

    def render_progressive(self, file_path=None, schedule=None, seed=1, **kw):
        """render_cuda in passes, for previews and time-budgeted renders: a generator that yields (samples_done, Frame)
        after every pass of `schedule` (increasing sample counts, the last one pre_sample_times; default
        progressive_schedule(pre_sample_times)).  A preview after e samples is the frame of pre = max = e samples; the
        final pass gives render_frame's frame.  With file_path the PNG is rewritten after every pass by the GPU encoder,
        as render_png writes it.  Raises RuntimeError as render_cuda does when the final frame raised.  kw: make_opts
        options (precision, window, count_detail, pixel_format, ...)."""
        cam = self.camera_desc()
        r = self.renderer()
        prog = r.progressive(cam, make_opts(seed=seed, **kw))
        try:
            frame = None
            for e in schedule or progressive_schedule(cam.pre_sample_times):
                prog.pass_to(e)
                frame = prog.download()
                if file_path:
                    png = r.encode_png(self.width, self.height, prog.opts.pixel_format, src=prog.frame_ptr())
                    os.makedirs(os.path.dirname(os.path.abspath(file_path)), exist_ok=True)
                    with open(file_path, "wb") as f:
                        f.write(png)
                yield e, frame
            self.last_frame = frame
            if frame is not None and prog.done == cam.pre_sample_times and frame.raised:
                self._raise_for(frame.stats)
        finally:
            prog.close()

    def render_fork(self, file_path, threads, out_dir="out", seed=1, **kw):
        """Drop-in for render_fork(file_path, threads) (camera.rb:41-68) for tooling that consumes its
        intermediate files: ONE GPU frame, then the same `out/file_<i>.json` per column strip the forked
        children write (camera.rb:53-65: strip i = x in [int(i/threads*W), int((i+1)/threads*W)), items in
        x-outer / y-inner order, each {position: [x, H-1-y], color: [r, g, b]} as render_at returns them),
        then the image as the parent does (:42-52)."""
        import json
        frame = self.render_frame(seed=seed, want_rgb=True, want_hit=False, **kw)
        os.makedirs(out_dir, exist_ok=True)
        W, H = self.width, self.height
        for i in range(threads):
            start_x, end_x = int(float(i) / threads * W), int(float(i + 1) / threads * W)
            data = [{"position": [x, H - 1 - y], "color": [float(c) for c in frame.rgb[y, x]]}
                    for x in range(start_x, end_x) for y in range(H)]
            with open(os.path.join(out_dir, "file_%d.json" % i), "w") as f:
                json.dump(data, f)
        self.canvas[...] = frame.rgba
        if file_path:
            self.save_image(file_path)
        return frame

    def render_at(self, x, y, seed=1, precision=_abi.PREC_DEFAULT):
        """camera.rb:70-99 — {position: [x, H-1-y], color: [r, g, b]} for one pixel (GPU, 1x1 window)."""
        f = self.render_frame(seed=seed, precision=precision, window=(x, y, x + 1, y + 1))
        return {"position": [x, self.height - 1 - y], "color": [float(c) for c in f.rgb[y, x]]}

    def array_to_color(self, arr):  # camera.rb:153-156
        return tuple(int(min(c * 256.0, 255)) for c in arr) + (255,)

    def save_image(self, file_path):  # camera.rb:36-39
        d = os.path.dirname(os.path.abspath(file_path))
        os.makedirs(d, exist_ok=True)
        write_png(file_path, self.canvas)
