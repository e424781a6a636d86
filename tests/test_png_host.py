"""Host-side checks of the device PNG encoder's C ABI: the size bound, the exports, and no CPU fallback."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def L():
    subprocess.check_call(["make", "-C", os.path.join(ROOT, "raytracing_rb_b200", "csrc"), "-j4", "-s", "all"])
    from raytracing_rb_b200 import _lib
    return _lib.lib()


@pytest.mark.parametrize("w,h", [(1, 1), (1, 1080), (1920, 1), (85, 128), (85, 129), (341, 64), (1920, 1080),
                                 (3840, 2160), (7, 9999)])
def test_max_bytes_bounds(L, w, h):
    """At least the stored-block worst case (every 32 KiB segment a stored block + sync flush in its own IDAT chunk,
    plus signature, IHDR, zlib header, Adler-32 and IEND chunks); at most the raw stream + 1 % + 1 KiB."""
    from raytracing_rb_b200 import _abi, png_max_bytes
    raw = h * (3 * w + 1)
    segs = -(-raw // _abi.PNG_SEGMENT_BYTES)
    stored = 8 + 25 + (12 + 2) + segs * (12 + 10) + raw + (12 + 4) + 12
    got = png_max_bytes(w, h)
    assert stored <= got <= raw + raw // 100 + 1024


def test_max_bytes_rejects_bad_sizes(L):
    from raytracing_rb_b200 import _abi
    n = C.c_size_t()
    for w, h in ((0, 5), (5, 0), (-1, 3)):
        assert L.rtrb_png_max_bytes(w, h, C.byref(n)) == _abi.RTRB_ERR_INVALID
    assert L.rtrb_png_max_bytes(4, 4, None) == _abi.RTRB_ERR_INVALID


def test_png_symbols_are_exported(L):
    from raytracing_rb_b200 import _abi, _lib
    for name in ("rtrb_png_max_bytes", "rtrb_encode_png", "rtrb_submit_png"):
        assert name in _lib.EXPORTS and hasattr(L, name)
    assert L.rtrb_abi_version() == _abi.ABI_VERSION == 4


def test_encode_png_without_a_device_fails_with_cuda_error(L):
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from raytracing_rb_b200 import Renderer, _abi, png_max_bytes
    from raytracing_rb_b200._lib import RtrbError
    r = Renderer.__new__(Renderer)  # no renderer can be created without a device; the entry point must still refuse
    r._h = C.c_void_p()
    with pytest.raises(RtrbError) as e:
        r.encode_png(64, 36)
    assert e.value.code == _abi.RTRB_ERR_CUDA
    out = np.zeros(png_max_bytes(64, 36), np.uint8)
    n = C.c_size_t()
    assert L.rtrb_encode_png(None, C.c_void_p(1 << 20), 64, 36, _abi.FMT_RGBA8, None, out.ctypes.data, out.nbytes,
                             C.byref(n)) == _abi.RTRB_ERR_CUDA
