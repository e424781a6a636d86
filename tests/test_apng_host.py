"""Host-side checks of the animated PNG C ABI: the header bytes, the per-frame size bound, the exports, and no CPU
fallback."""
import ctypes as C
import os
import struct
import subprocess
import zlib

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def L():
    subprocess.check_call(["make", "-C", os.path.join(ROOT, "raytracing_rb_b200", "csrc"), "-j4", "-s", "all"])
    from raytracing_rb_b200 import _lib
    return _lib.lib()


def chunks(data):
    pos, out = 0, []
    while pos < len(data):
        n, = struct.unpack(">I", data[pos:pos + 4])
        tag, body = data[pos + 4:pos + 8], data[pos + 8:pos + 8 + n]
        crc, = struct.unpack(">I", data[pos + 8 + n:pos + 12 + n])
        out.append((tag, body, crc))
        pos += 12 + n
    assert pos == len(data)
    return out


@pytest.mark.parametrize("w,h,frames,plays", [(1, 1, 1, 0), (1920, 1080, 12, 0), (160, 90, 3, 7), (7, 9999, 65536, 1)])
def test_header_bytes(L, w, h, frames, plays):
    from raytracing_rb_b200 import apng_header
    hdr = apng_header(w, h, frames, plays)
    assert len(hdr) == 53
    assert hdr[:8] == b"\x89PNG\r\n\x1a\n"
    cs = chunks(hdr[8:])
    assert [t for t, _, _ in cs] == [b"IHDR", b"acTL"]
    for tag, body, crc in cs:
        assert crc == zlib.crc32(tag + body) & 0xFFFFFFFF
    assert struct.unpack(">IIBBBBB", cs[0][1]) == (w, h, 8, 2, 0, 0, 0)
    assert struct.unpack(">II", cs[1][1]) == (frames, plays)


def test_header_rejects_bad_arguments(L):
    from raytracing_rb_b200 import _abi
    out = (C.c_uint8 * 53)()
    for w, h, f, p in ((0, 5, 1, 0), (5, 0, 1, 0), (-1, 3, 1, 0), (4, 4, 0, 0), (4, 4, -2, 0), (4, 4, 1, -1)):
        assert L.rtrb_apng_header(w, h, f, p, out) == _abi.RTRB_ERR_INVALID, (w, h, f, p)
    assert L.rtrb_apng_header(4, 4, 1, 0, None) == _abi.RTRB_ERR_INVALID


@pytest.mark.parametrize("w,h", [(1, 1), (1, 1080), (1920, 1), (85, 128), (85, 129), (341, 64), (1920, 1080),
                                 (3840, 2160), (7, 9999)])
def test_frame_max_bytes_bounds(L, w, h):
    """At least the stored-block worst case of the whole canvas: fcTL, then every 32 KiB segment a stored block + sync
    flush in its own fdAT chunk (sequence number included), plus the zlib-header and Adler-32 fdAT chunks."""
    from raytracing_rb_b200 import _abi, apng_frame_max_bytes
    raw = h * (3 * w + 1)
    segs = -(-raw // _abi.PNG_SEGMENT_BYTES)
    stored = (12 + 26) + (12 + 4 + 2) + segs * (12 + 4 + 10) + raw + (12 + 4 + 4)
    got = apng_frame_max_bytes(w, h)
    assert stored <= got <= raw + raw // 100 + 1024


def test_frame_max_bytes_rejects_bad_sizes(L):
    from raytracing_rb_b200 import _abi
    n = C.c_size_t()
    for w, h in ((0, 5), (5, 0), (-1, 3)):
        assert L.rtrb_apng_frame_max_bytes(w, h, C.byref(n)) == _abi.RTRB_ERR_INVALID
    assert L.rtrb_apng_frame_max_bytes(4, 4, None) == _abi.RTRB_ERR_INVALID


def test_apng_symbols_are_exported(L):
    from raytracing_rb_b200 import _abi, _lib
    for name in ("rtrb_apng_header", "rtrb_apng_frame_max_bytes", "rtrb_apng_create", "rtrb_apng_add",
                 "rtrb_submit_apng", "rtrb_apng_destroy"):
        assert name in _lib.EXPORTS and hasattr(L, name)
    assert L.rtrb_abi_version() == _abi.ABI_VERSION == 4
    assert L.rtrb_apng_destroy(None) == _abi.RTRB_OK


def test_create_checks_arguments_before_the_device(L):
    from raytracing_rb_b200 import _abi
    h = C.c_void_p()
    for w, ht, dn, dd in ((0, 4, 1, 25), (4, -1, 1, 25), (4, 4, 65536, 25), (4, 4, 1, 70000), (4, 4, -1, 25)):
        assert L.rtrb_apng_create(None, w, ht, dn, dd, C.byref(h)) == _abi.RTRB_ERR_INVALID, (w, ht, dn, dd)
    assert L.rtrb_apng_create(None, 4, 4, 1, 25, None) == _abi.RTRB_ERR_INVALID


def test_create_without_a_device_fails_with_cuda_error(L):
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from raytracing_rb_b200 import _abi
    h = C.c_void_p()
    assert L.rtrb_apng_create(C.c_void_p(1 << 20), 64, 36, 1, 25, C.byref(h)) == _abi.RTRB_ERR_CUDA
    assert not h.value
    out = np.zeros(16, np.uint8)
    n = C.c_size_t()
    assert L.rtrb_apng_add(None, None, _abi.FMT_RGB8, None, out.ctypes.data, out.nbytes, C.byref(n)) == _abi.RTRB_ERR_INVALID
