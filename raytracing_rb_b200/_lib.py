"""Loader for the C-ABI CUDA library (include/rtrb_b200.h).  There is no CPU fallback: if the
library is missing the import of anything that renders fails loudly."""
import ctypes as C
import os

from . import _abi

_HERE = os.path.dirname(os.path.abspath(__file__))
# RTRB_B200_LIB selects another build of the same library (A/B runs of kernel variants); never a fallback
LIB_PATH = os.environ.get("RTRB_B200_LIB") or os.path.join(_HERE, "csrc", "librtrb_b200.so")

EXPORTS = (
    "rtrb_abi_version", "rtrb_last_error", "rtrb_device_count",
    "rtrb_renderer_create", "rtrb_renderer_destroy", "rtrb_scene_update",
    "rtrb_render_device", "rtrb_download", "rtrb_render", "rtrb_submit", "rtrb_wait",
    "rtrb_framebuffer_device_ptr", "rtrb_framebuffer_download", "rtrb_framebuffer_copy_async", "rtrb_framebuffer_ipc_export", "rtrb_ipc_open", "rtrb_ipc_close",
    "rtrb_peer_push", "rtrb_peer_push_join",
    "rtrb_render_multi", "rtrb_tile_partition", "rtrb_measure_fma_peak", "rtrb_launch_count", "rtrb_last_mt_passes",
    "rtrb_png_max_bytes", "rtrb_encode_png", "rtrb_submit_png",
    "rtrb_trace_rays", "rtrb_intersect_rays", "rtrb_camera_rays",
    "rtrb_progressive_create", "rtrb_progressive_pass", "rtrb_progressive_download", "rtrb_progressive_frame_ptr",
    "rtrb_progressive_destroy",
    "rtrb_apng_header", "rtrb_apng_frame_max_bytes", "rtrb_apng_create", "rtrb_apng_add", "rtrb_submit_apng",
    "rtrb_apng_destroy",
)

_lib = None


class RtrbError(RuntimeError):
    def __init__(self, code, message):
        super().__init__("rtrb error %d: %s" % (code, message))
        self.code = code


def lib():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise ImportError(
            "CUDA extension %s is not built (run `python -c 'import __graft_entry__ as g; g.build()'` or "
            "`make -C raytracing_rb_b200/csrc`); there is no CPU fallback" % LIB_PATH)
    L = C.CDLL(LIB_PATH)
    P = C.POINTER
    L.rtrb_abi_version.restype = C.c_int
    L.rtrb_last_error.restype = C.c_char_p
    L.rtrb_device_count.argtypes = [P(C.c_int)]
    L.rtrb_renderer_create.argtypes = [P(_abi.SceneDesc), C.c_int, P(C.c_void_p)]
    L.rtrb_renderer_destroy.argtypes = [C.c_void_p]
    L.rtrb_scene_update.argtypes = [C.c_void_p, P(_abi.SceneDesc), C.c_void_p]
    L.rtrb_render_device.argtypes = [C.c_void_p, P(_abi.CameraDesc), P(_abi.RenderOpts), P(_abi.Stats)]
    L.rtrb_download.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.rtrb_render.argtypes = [C.c_void_p, P(_abi.CameraDesc), P(_abi.RenderOpts), C.c_void_p, C.c_void_p,
                              C.c_void_p, P(_abi.Stats)]
    L.rtrb_submit.argtypes = [C.c_void_p, P(_abi.CameraDesc), P(_abi.RenderOpts), C.c_void_p, P(C.c_int)]
    L.rtrb_wait.argtypes = [C.c_void_p, C.c_int, P(_abi.Stats)]
    L.rtrb_framebuffer_device_ptr.argtypes = [C.c_void_p, C.c_int, C.c_int, P(C.c_void_p)]
    L.rtrb_framebuffer_download.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p]
    L.rtrb_framebuffer_copy_async.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p]
    L.rtrb_framebuffer_ipc_export.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p]
    L.rtrb_ipc_open.argtypes = [C.c_int, C.c_void_p, P(C.c_void_p)]
    L.rtrb_ipc_close.argtypes = [C.c_int, C.c_void_p]
    L.rtrb_peer_push.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]
    L.rtrb_peer_push_join.argtypes = [C.c_void_p, C.c_void_p]
    L.rtrb_render_multi.argtypes = [P(C.c_void_p), C.c_int, P(_abi.CameraDesc), P(_abi.RenderOpts), C.c_void_p,
                                    C.c_void_p, C.c_void_p, P(_abi.Stats)]
    L.rtrb_tile_partition.argtypes = [C.c_int, C.c_int, P(C.c_int32), C.c_int, C.c_int, P(C.c_int32), C.c_int, P(C.c_int)]
    L.rtrb_measure_fma_peak.argtypes = [C.c_int, C.c_int, P(C.c_double)]
    L.rtrb_launch_count.restype = C.c_uint64
    L.rtrb_last_mt_passes.argtypes = [C.c_void_p]
    L.rtrb_png_max_bytes.argtypes = [C.c_int, C.c_int, P(C.c_size_t)]
    L.rtrb_encode_png.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_size_t,
                                  P(C.c_size_t)]
    L.rtrb_submit_png.argtypes = [C.c_void_p, P(_abi.CameraDesc), P(_abi.RenderOpts), C.c_void_p, C.c_size_t,
                                  P(C.c_size_t), P(C.c_int)]
    L.rtrb_trace_rays.argtypes = [C.c_void_p, P(_abi.RayOpts), C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                  P(_abi.Stats)]
    L.rtrb_intersect_rays.argtypes = [C.c_void_p, P(_abi.RayOpts), C.c_int, C.c_void_p, C.c_void_p]
    L.rtrb_camera_rays.argtypes = [C.c_void_p, P(_abi.CameraDesc), P(_abi.RayOpts), C.c_int, C.c_int, C.c_void_p,
                                   C.c_void_p]
    L.rtrb_progressive_create.argtypes = [C.c_void_p, P(_abi.CameraDesc), P(_abi.RenderOpts), P(C.c_void_p)]
    L.rtrb_progressive_pass.argtypes = [C.c_void_p, C.c_int, P(_abi.Stats)]
    L.rtrb_progressive_download.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.rtrb_progressive_frame_ptr.argtypes = [C.c_void_p, P(C.c_void_p)]
    L.rtrb_progressive_destroy.argtypes = [C.c_void_p]
    L.rtrb_apng_header.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]
    L.rtrb_apng_frame_max_bytes.argtypes = [C.c_int, C.c_int, P(C.c_size_t)]
    L.rtrb_apng_create.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, P(C.c_void_p)]
    L.rtrb_apng_add.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_size_t, P(C.c_size_t)]
    L.rtrb_submit_apng.argtypes = [C.c_void_p, C.c_void_p, P(_abi.CameraDesc), P(_abi.RenderOpts), C.c_void_p,
                                   C.c_size_t, P(C.c_size_t), P(C.c_int)]
    L.rtrb_apng_destroy.argtypes = [C.c_void_p]
    for name in EXPORTS:
        getattr(L, name)
    if L.rtrb_abi_version() != _abi.ABI_VERSION:
        raise ImportError("librtrb_b200.so ABI %d != expected %d" % (L.rtrb_abi_version(), _abi.ABI_VERSION))
    _lib = L
    return L


def check(code, allow_raised=False):
    if code == _abi.RTRB_OK:
        return code
    if allow_raised and code == _abi.RTRB_ERR_RAISED:
        return code
    msg = lib().rtrb_last_error()
    raise RtrbError(code, msg.decode("utf-8", "replace") if msg else "?")
