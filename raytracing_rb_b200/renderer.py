"""Thin object wrapper over the C ABI (include/rtrb_b200.h): one Renderer = one baked scene on one
GPU.  Frames come back as numpy arrays in the layout Camera#render_at defines (row = y, col = x)."""
import ctypes as C

import numpy as np

from . import _abi
from ._lib import check, lib


class Frame:
    """One rendered frame: rgba uint8 [H,W,4]; rgb float64 [H,W,3] (render_at's unclamped colour) or
    None; hit int32 [H,W] primary hit ids or None; stats dict; status word."""

    def __init__(self, rgba, rgb, hit, stats, code):
        self.rgba, self.rgb, self.hit, self.stats, self.code = rgba, rgb, hit, stats, code

    @property
    def status(self):
        return self.stats["status"]

    @property
    def raised(self):
        return self.code == _abi.RTRB_ERR_RAISED


def make_opts(rng_mode=_abi.RNG_CTR, precision=_abi.PREC_DEFAULT, seed=1, window=None, tile_rank=0, tile_world=1,
              count_detail=False, stream=None, rgba_device_out=None, skip_outputs=0, pixel_format=_abi.FMT_RGBA8):
    o = _abi.RenderOpts()
    o.rng_mode, o.precision, o.seed = rng_mode, precision, seed
    if window:
        o.x0, o.y0, o.x1, o.y1 = window
    o.tile_rank, o.tile_world = tile_rank, tile_world
    o.count_detail = 1 if count_detail else 0
    o.skip_outputs = skip_outputs
    o.stream = stream
    o.rgba_device_out = rgba_device_out
    o.pixel_format = pixel_format
    return o


# numpy view of rtrb_ray_hit (World#intersect's answer for one ray)
RAY_HIT_DTYPE = np.dtype([("object", "<i4"), ("direction", "<i4"), ("face", "<i4"), ("reserved0", "<i4"),
                          ("distance", "<f8"), ("intersection", "<f8", (3,)), ("delta", "<f8", (3,))])
assert RAY_HIT_DTYPE.itemsize == C.sizeof(_abi.RayHit)


def make_ray_opts(precision=_abi.PREC_DEFAULT, seed=1, trace_depth=1, mc=0, count_detail=False, window=None,
                  device_buffers=False, stream=None):
    o = _abi.RayOpts()
    o.precision, o.seed = precision, seed
    o.trace_depth, o.monte_carlo_diffusion_times = trace_depth, mc
    o.count_detail = 1 if count_detail else 0
    if window:
        o.x0, o.y0, o.x1, o.y1 = window
    o.device_buffers = 1 if device_buffers else 0
    o.stream = stream
    return o


def _frame_shape(width, height, pixel_format):
    """numpy shape of an 8-bit frame in `pixel_format`."""
    if pixel_format == _abi.FMT_PNG_RGB8:   # H scanlines of (filter byte 0, W x RGB8): IDAT's payload before deflate
        return (height, width * 3 + 1)
    return (height, width, 3 if pixel_format == _abi.FMT_RGB8 else 4)


def progressive_schedule(pre, first=1):
    """The doubling pass schedule of a progressive frame of `pre` samples per pixel: first, 2*first, 4*first, ... while
    below pre, then pre itself (always the last entry).  Pure host logic."""
    if pre < 1 or first < 1:
        raise ValueError("pre and first must be >= 1")
    out, e = [], first
    while e < pre:
        out.append(e)
        e *= 2
    out.append(pre)
    return out


def _is_tensor(x):
    return type(x).__module__.startswith("torch")


def _torch_stream(device):
    """torch.cuda.current_stream(device) as a cudaStream_t for the C ABI.  torch reports its default stream as 0, which
    the ABI reads as "the renderer's own stream"; the legacy default stream's handle is cudaStreamLegacy (0x1)."""
    import torch
    return torch.cuda.current_stream(device).cuda_stream or 1


class Renderer:
    def __init__(self, scene, device=0):
        self._scene = scene  # SceneDescHolder of the last create / update; kept for introspection
        self._h = C.c_void_p()
        self.device = device
        self._png_pending = {}  # submit_png ticket -> (host buffer, byte count that rtrb_wait fills in)
        self.synced_to = None   # (world, edit count) it was last brought up to date with (world.synced_renderer)
        check(lib().rtrb_renderer_create(C.byref(scene.desc), device, C.byref(self._h)))

    def close(self):
        if self._h:
            lib().rtrb_renderer_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def handle(self):
        return self._h

    def update(self, scene, stream=None):
        """Replaces the baked scene with `scene` (a SceneDescHolder) in stream order (rtrb_scene_update): work queued
        before the call sees the old scene, work issued after it the new one; an unchanged scene queues nothing.
        stream: a cudaStream_t handle, a torch.cuda.Stream, or None for the renderer's own stream."""
        if stream is not None and not isinstance(stream, int):
            stream = stream.cuda_stream or 1  # torch's default stream reports 0: cudaStreamLegacy, as _torch_stream
        check(lib().rtrb_scene_update(self._h, C.byref(scene.desc), C.c_void_p(stream) if stream else None))
        self._scene = scene

    def render_device(self, cam, opts=None, want_stats=True):
        """Frame stays in device memory.  Returns (stats dict or None, status code)."""
        opts = opts or make_opts()
        st = _abi.Stats()
        code = lib().rtrb_render_device(self._h, C.byref(cam), C.byref(opts), C.byref(st) if want_stats else None)
        check(code, allow_raised=True)
        return (st.as_dict() if want_stats else None), code

    def download(self, width, height, want_rgb=True, want_hit=True, channels=4):
        rgba = np.empty((height, width, channels), np.uint8)
        rgb = np.empty((height, width, 3), np.float64) if want_rgb else None
        hit = np.empty((height, width), np.int32) if want_hit else None
        check(lib().rtrb_download(self._h, rgba.ctypes.data, rgb.ctypes.data if want_rgb else None,
                                  hit.ctypes.data if want_hit else None))
        return rgba, rgb, hit

    def render(self, cam, opts=None, want_rgb=True, want_hit=True, out_rgba=None):
        """The frame-level call the Ruby shim binds (host buffers in, host buffers out)."""
        opts = opts or make_opts()
        H, W = cam.height, cam.width
        rgba = out_rgba if out_rgba is not None else np.empty(_frame_shape(W, H, opts.pixel_format), np.uint8)
        rgb = np.empty((H, W, 3), np.float64) if want_rgb else None
        hit = np.empty((H, W), np.int32) if want_hit else None
        st = _abi.Stats()
        code = lib().rtrb_render(self._h, C.byref(cam), C.byref(opts), rgba.ctypes.data,
                                 rgb.ctypes.data if want_rgb else None, hit.ctypes.data if want_hit else None,
                                 C.byref(st))
        check(code, allow_raised=True)
        return Frame(rgba, rgb, hit, st.as_dict(), code)

    def submit(self, cam, out_rgba, opts=None):
        """Pipelined frame: returns a ticket at once; the RGBA8 frame lands in `out_rgba` (a numpy view
        of pinned host memory for full speed) by the time `wait(ticket)` returns.  Up to four in flight."""
        opts = opts or make_opts()
        t = C.c_int()
        check(lib().rtrb_submit(self._h, C.byref(cam), C.byref(opts), out_rgba.ctypes.data, C.byref(t)))
        return t.value

    def wait(self, ticket):
        st = _abi.Stats()
        code = lib().rtrb_wait(self._h, ticket, C.byref(st))
        check(code, allow_raised=True)
        return st.as_dict(), code

    def encode_png(self, width, height, pixel_format=_abi.FMT_RGB8, src=None, stream=None):
        """PNG file (bytes) of a width x height image in device memory, encoded on the device: `src` (a device pointer)
        or, if None, the renderer's framebuffer; ordered after the work on `stream` (None = the renderer's own)."""
        cap = png_max_bytes(width, height)
        out = np.empty(cap, np.uint8)
        n = C.c_size_t()
        check(lib().rtrb_encode_png(self._h, C.c_void_p(src) if src else None, width, height, pixel_format,
                                    C.c_void_p(stream) if stream else None, out.ctypes.data, cap, C.byref(n)))
        return out[:n.value].tobytes()

    def submit_png(self, cam, out_pinned, opts=None):
        """Pipelined frame encoded as a PNG file on the device: returns a ticket at once; the file lands in `out_pinned`
        (a uint8 numpy view of page-locked, device-mapped host memory of at least png_max_bytes(W, H) bytes) by the time
        `wait_png(ticket)` returns.  Shares the four slots and the ticket order of `submit`."""
        opts = opts or make_opts()
        t = C.c_int()
        n = C.c_size_t()
        check(lib().rtrb_submit_png(self._h, C.byref(cam), C.byref(opts), out_pinned.ctypes.data, out_pinned.nbytes,
                                    C.byref(n), C.byref(t)))
        self._png_pending[t.value] = (out_pinned, n)
        return t.value

    def wait_png(self, ticket):
        """-> (PNG bytes, stats dict, status code) of a submit_png frame."""
        out, n = self._png_pending.get(ticket, (None, None))
        stats, code = self.wait(ticket)
        del self._png_pending[ticket]
        return out[:n.value].tobytes(), stats, code

    # -- ray-level queries (rtrb_trace_rays / rtrb_intersect_rays / rtrb_camera_rays) ----------------------------------
    # Rays are [n, 6] float64 rows (position, front).  numpy arrays take the blocking host-buffer path; CUDA torch
    # tensors on this renderer's device take the device-buffer path on torch.cuda.current_stream() and give torch outputs.
    def _device_rays(self, rays):
        import torch
        if not rays.is_cuda or rays.device.index != self.device:
            raise ValueError("ray tensors must live on cuda:%d" % self.device)
        return rays.to(torch.float64).reshape(-1, 6).contiguous(), _torch_stream(self.device)

    def trace_rays(self, rays, trace_depth=1, mc=0, seed=1, keys=None, precision=_abi.PREC_DEFAULT, count_detail=False,
                   want_stats=True):
        """RayTracer#trace_sync on every ray -> (rgb [n, 3] float64, hit [n] int32, stats dict or None, status code).
        keys: [n, 2] (pixel, sample) Philox keys of the Monte-Carlo rays; None keys ray i as (i, 0).  On the device
        path the call synchronises only when want_stats (stats is None otherwise)."""
        st = _abi.Stats()
        if _is_tensor(rays):
            import torch
            rays, stream = self._device_rays(rays)
            n = rays.shape[0]
            if keys is not None:
                keys = keys.reshape(-1, 2).to(device=rays.device, dtype=torch.int32).contiguous()
                assert keys.shape[0] == n
            rgb = torch.empty((n, 3), dtype=torch.float64, device=rays.device)
            hit = torch.empty((n,), dtype=torch.int32, device=rays.device)
            opts = make_ray_opts(precision, seed, trace_depth, mc, count_detail, device_buffers=True, stream=stream)
            code = lib().rtrb_trace_rays(self._h, C.byref(opts), n, rays.data_ptr(), keys.data_ptr() if keys is not None else None,
                                         rgb.data_ptr(), hit.data_ptr(), C.byref(st) if want_stats else None)
        else:
            rays = np.ascontiguousarray(rays, np.float64).reshape(-1, 6)
            n = rays.shape[0]
            if keys is not None:
                keys = np.ascontiguousarray(keys, np.uint32).reshape(-1, 2)
                assert keys.shape[0] == n
            rgb = np.empty((n, 3), np.float64)
            hit = np.empty((n,), np.int32)
            opts = make_ray_opts(precision, seed, trace_depth, mc, count_detail)
            code = lib().rtrb_trace_rays(self._h, C.byref(opts), n, rays.ctypes.data, keys.ctypes.data if keys is not None else None,
                                         rgb.ctypes.data, hit.ctypes.data, C.byref(st))
            want_stats = True
        check(code, allow_raised=True)
        return rgb, hit, (st.as_dict() if want_stats else None), code

    def intersect_rays(self, rays, precision=_abi.PREC_DEFAULT):
        """World#intersect on every ray.  numpy input -> structured array of RAY_HIT_DTYPE; torch input -> dict of
        tensors (object, direction, face int32; distance float64; intersection, delta [n, 3] float64) that view one
        [n, 9] float64 buffer of rtrb_ray_hit records."""
        if _is_tensor(rays):
            import torch
            rays, stream = self._device_rays(rays)
            n = rays.shape[0]
            raw = torch.empty((n, 9), dtype=torch.float64, device=rays.device)
            opts = make_ray_opts(precision, device_buffers=True, stream=stream)
            check(lib().rtrb_intersect_rays(self._h, C.byref(opts), n, rays.data_ptr(), raw.data_ptr()))
            ints = raw[:, :2].view(torch.int32)
            return {"object": ints[:, 0], "direction": ints[:, 1], "face": ints[:, 2], "distance": raw[:, 2],
                    "intersection": raw[:, 3:6], "delta": raw[:, 6:9], "raw": raw}
        rays = np.ascontiguousarray(rays, np.float64).reshape(-1, 6)
        out = np.empty(rays.shape[0], RAY_HIT_DTYPE)
        opts = make_ray_opts(precision)
        check(lib().rtrb_intersect_rays(self._h, C.byref(opts), rays.shape[0], rays.ctypes.data, out.ctypes.data))
        return out

    def camera_rays(self, cam, seed=1, window=None, samples=None, device_buffers=False):
        """Camera#lens_func for every pixel of `window` (x0, y0, x1, y1; None = the whole frame) and every sample j in
        `samples` = (begin, end) (None = the pre samples, (0, pre_sample_times)) -> (rays [n, 6], keys [n, 2]); ray
        (x, y, j) is row ((y - y0) * (x1 - x0) + (x - x0)) * (end - begin) + (j - begin) and its key is (y * W + x, j).
        numpy arrays (keys uint32), or with device_buffers torch tensors on this renderer's device (keys int32)."""
        b, e = samples if samples is not None else (0, cam.pre_sample_times)
        x0, y0, x1, y1 = window if window else (0, 0, cam.width, cam.height)
        n = max(0, x1 - x0) * max(0, y1 - y0) * max(0, e - b)
        if device_buffers:
            import torch
            dev = torch.device("cuda", self.device)
            rays = torch.empty((n, 6), dtype=torch.float64, device=dev)
            keys = torch.empty((n, 2), dtype=torch.int32, device=dev)
            opts = make_ray_opts(seed=seed, window=window, device_buffers=True,
                                 stream=_torch_stream(self.device))
            check(lib().rtrb_camera_rays(self._h, C.byref(cam), C.byref(opts), b, e, rays.data_ptr(), keys.data_ptr()))
            return rays, keys
        rays = np.empty((n, 6), np.float64)
        keys = np.empty((n, 2), np.uint32)
        opts = make_ray_opts(seed=seed, window=window)
        check(lib().rtrb_camera_rays(self._h, C.byref(cam), C.byref(opts), b, e, rays.ctypes.data, keys.ctypes.data))
        return rays, keys

    def progressive(self, cam, opts=None):
        """A progressive frame of `cam` on this renderer (rtrb_progressive_create) -> Progressive."""
        return Progressive(self, cam, opts)

    def apng(self, width, height, delay=(1, 25)):
        """An animated PNG of width x height frames on this renderer, each shown delay[0] / delay[1] seconds
        (rtrb_apng_create) -> Apng."""
        return Apng(self, width, height, delay)

    def peer_push(self, src_ptr, dst_peer_ptr, nbytes, after_stream=None):
        """Copy-engine gather: queue a D2D copy to a peer mapping behind `after_stream` (see rtrb_peer_push)."""
        check(lib().rtrb_peer_push(self._h, C.c_void_p(src_ptr), C.c_void_p(dst_peer_ptr), nbytes,
                                   C.c_void_p(after_stream) if after_stream else None))

    def peer_push_join(self, stream=None):
        check(lib().rtrb_peer_push_join(self._h, C.c_void_p(stream) if stream else None))

    def last_mt_passes(self):
        """Passes the last RNG_MT frame needed to reach the fixed point of its stream offsets."""
        return int(lib().rtrb_last_mt_passes(self._h))

    def framebuffer_ptr(self, width, height):
        p = C.c_void_p()
        check(lib().rtrb_framebuffer_device_ptr(self._h, width, height, C.byref(p)))
        return p.value

    def framebuffer_download(self, width, height, out):
        check(lib().rtrb_framebuffer_download(self._h, width, height, out.ctypes.data))
        return out

    def framebuffer_copy_async(self, nbytes, out, stream=None):
        """Queues framebuffer[:nbytes] -> `out` (pinned host memory) on `stream`; the caller synchronises."""
        check(lib().rtrb_framebuffer_copy_async(self._h, nbytes, out.ctypes.data, C.c_void_p(stream) if stream else None))

    def framebuffer_ipc_export(self, width, height):
        buf = (C.c_uint8 * 64)()
        check(lib().rtrb_framebuffer_ipc_export(self._h, width, height, buf))
        return bytes(buf)


class Progressive:
    """A frame whose pre_sample_times samples are traced in passes (rtrb_progressive_*, include/rtrb_b200.h).  After a
    pass to e < pre samples its outputs and stats are those of the frame with pre = max = e; the pass that reaches pre
    gives the frame of the camera as given.  Holds a reference to its Renderer, which must outlive it."""

    def __init__(self, renderer, cam, opts=None):
        self.renderer = renderer
        self.cam = cam
        self.opts = opts or make_opts()
        self.done = 0
        self.stats, self.code = None, _abi.RTRB_OK
        self._h = C.c_void_p()
        check(lib().rtrb_progressive_create(renderer.handle, C.byref(cam), C.byref(self.opts), C.byref(self._h)))

    def pass_to(self, sample_end, want_stats=True):
        """Traces samples [done, sample_end) -> (stats dict or None, status code).  Synchronises only when want_stats."""
        st = _abi.Stats()
        code = lib().rtrb_progressive_pass(self._h, sample_end, C.byref(st) if want_stats else None)
        check(code, allow_raised=True)
        self.done = sample_end
        self.stats, self.code = (st.as_dict() if want_stats else None), code
        return self.stats, code

    def download(self, want_rgb=True, want_hit=True):
        """The outputs of the passes so far -> Frame (rgba is None when the 8-bit frame goes to rgba_device_out; stats
        and code are those of the last pass)."""
        H, W = self.cam.height, self.cam.width
        rgba = None if self.opts.rgba_device_out else np.empty(_frame_shape(W, H, self.opts.pixel_format), np.uint8)
        rgb = np.empty((H, W, 3), np.float64) if want_rgb else None
        hit = np.empty((H, W), np.int32) if want_hit else None
        check(lib().rtrb_progressive_download(self._h, rgba.ctypes.data if rgba is not None else None,
                                              rgb.ctypes.data if want_rgb else None, hit.ctypes.data if want_hit else None))
        return Frame(rgba, rgb, hit, self.stats, self.code)

    def frame_ptr(self):
        """Device pointer of the 8-bit frame (e.g. for Renderer.encode_png(src=...))."""
        p = C.c_void_p()
        check(lib().rtrb_progressive_frame_ptr(self._h, C.byref(p)))
        return p.value

    def close(self):
        if self._h:
            lib().rtrb_progressive_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Apng:
    """An animated PNG built frame by frame on the device (rtrb_apng_*, include/rtrb_b200.h): frame 0 is the whole
    canvas, every later frame only the rectangle of pixels that changed since the frame before.  The file is
    header(), then the chunk bytes of every frame in the order they were added, then TRAILER.  Holds a reference to its
    Renderer, which must outlive it."""

    TRAILER = b"\x00\x00\x00\x00IEND\xaeB`\x82"

    def __init__(self, renderer, width, height, delay=(1, 25)):
        self.renderer = renderer
        self.width, self.height = width, height
        self.delay = tuple(delay)
        self.frames = 0
        self._pending = {}  # submit ticket -> (host buffer, byte count that rtrb_wait fills in)
        self._h = C.c_void_p()
        check(lib().rtrb_apng_create(renderer.handle, width, height, self.delay[0], self.delay[1], C.byref(self._h)))

    def add(self, src=None, pixel_format=_abi.FMT_RGB8, stream=None):
        """Appends the frame at device pointer `src` (None = the renderer's framebuffer) in pixel_format, ordered after
        the work on `stream` (None = the renderer's own) -> the frame's chunk bytes."""
        cap = apng_frame_max_bytes(self.width, self.height)
        out = np.empty(cap, np.uint8)
        n = C.c_size_t()
        check(lib().rtrb_apng_add(self._h, C.c_void_p(src) if src else None, pixel_format,
                                  C.c_void_p(stream) if stream else None, out.ctypes.data, cap, C.byref(n)))
        self.frames += 1
        return out[:n.value].tobytes()

    def submit(self, cam, out_pinned, opts=None):
        """Pipelined frame rendered and appended on the device (rtrb_submit_apng): returns a ticket at once; the chunk
        bytes land in `out_pinned` (a uint8 numpy view of page-locked, device-mapped host memory of at least
        apng_frame_max_bytes(W, H) bytes) by the time `wait(ticket)` returns.  Shares the renderer's four slots."""
        opts = opts or make_opts(pixel_format=_abi.FMT_RGB8)
        t = C.c_int()
        n = C.c_size_t()
        check(lib().rtrb_submit_apng(self.renderer.handle, self._h, C.byref(cam), C.byref(opts),
                                     out_pinned.ctypes.data, out_pinned.nbytes, C.byref(n), C.byref(t)))
        self.frames += 1
        self._pending[t.value] = (out_pinned, n)
        return t.value

    def wait(self, ticket):
        """-> (chunk bytes, stats dict, status code) of a submitted frame."""
        out, n = self._pending.pop(ticket)
        stats, code = self.renderer.wait(ticket)
        return out[:n.value].tobytes(), stats, code

    def header(self, num_plays=0):
        """Signature, IHDR and acTL for the frames added so far; num_plays 0 loops forever."""
        return apng_header(self.width, self.height, self.frames, num_plays)

    def close(self):
        if self._h:
            lib().rtrb_apng_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def ipc_open(device, handle_bytes):
    buf = (C.c_uint8 * 64).from_buffer_copy(handle_bytes)
    p = C.c_void_p()
    check(lib().rtrb_ipc_open(device, buf, C.byref(p)))
    return p.value


def ipc_close(device, ptr):
    check(lib().rtrb_ipc_close(device, C.c_void_p(ptr)))


def render_multi(renderers, cam, opts=None, want_rgb=True, want_hit=True):
    """In-process multi-GPU frame: image tiles interleaved over len(renderers) GPUs, written through
    peer mappings into renderers[0]'s framebuffer (no collective)."""
    opts = opts or make_opts()
    n = len(renderers)
    arr = (C.c_void_p * n)(*[r.handle for r in renderers])
    H, W = cam.height, cam.width
    rgba = np.empty((H, W, 4), np.uint8)
    rgb = np.empty((H, W, 3), np.float64) if want_rgb else None
    hit = np.empty((H, W), np.int32) if want_hit else None
    st = _abi.Stats()
    code = lib().rtrb_render_multi(arr, n, C.byref(cam), C.byref(opts), rgba.ctypes.data,
                                   rgb.ctypes.data if want_rgb else None, hit.ctypes.data if want_hit else None,
                                   C.byref(st))
    check(code, allow_raised=True)
    return Frame(rgba, rgb, hit, st.as_dict(), code)


def tile_partition(width, height, tile_rank=0, tile_world=1, window=None):
    """The super-tile ids (ty * ceil(width/32) + tx) `tile_rank` of `tile_world` renders.  Pure host logic."""
    win = (C.c_int32 * 4)(*(window or (0, 0, 0, 0)))
    n = C.c_int()
    check(lib().rtrb_tile_partition(width, height, win, tile_rank, tile_world, None, 0, C.byref(n)))
    out = (C.c_int32 * max(1, n.value))()
    check(lib().rtrb_tile_partition(width, height, win, tile_rank, tile_world, out, n.value, C.byref(n)))
    return list(out[:n.value])


def deal_frames(rank, world, frames_per_gpu):
    """Whole-frame dealing of a batch of small frames (DESIGN.md 8): rank r renders frames
    [r*B, (r+1)*B) of the step and frame f lands in slot f of rank 0's framebuffer.  Returns the list of
    (frame index, slot) pairs of `rank`.  Pure host logic."""
    if world < 1 or not 0 <= rank < world or frames_per_gpu < 0:
        raise ValueError("bad rank/world/frames_per_gpu")
    first = rank * frames_per_gpu
    return [(first + f, first + f) for f in range(frames_per_gpu)]


def png_max_bytes(width, height):
    """Bytes that always suffice for a device-encoded PNG of width x height.  Pure host logic."""
    n = C.c_size_t()
    check(lib().rtrb_png_max_bytes(width, height, C.byref(n)))
    return n.value


def apng_frame_max_bytes(width, height):
    """Bytes that always suffice for one APNG frame's chunks of a width x height animation.  Pure host logic."""
    n = C.c_size_t()
    check(lib().rtrb_apng_frame_max_bytes(width, height, C.byref(n)))
    return n.value


def apng_header(width, height, num_frames, num_plays=0):
    """Signature, IHDR and acTL chunks of a width x height animation of num_frames frames.  Pure host logic."""
    out = (C.c_uint8 * 53)()
    check(lib().rtrb_apng_header(width, height, num_frames, num_plays, out))
    return bytes(out)


def measure_fma_peak(device=0, fp64=True):
    v = C.c_double()
    check(lib().rtrb_measure_fma_peak(device, 1 if fp64 else 0, C.byref(v)))
    return v.value


def device_count():
    n = C.c_int()
    check(lib().rtrb_device_count(C.byref(n)))
    return n.value
