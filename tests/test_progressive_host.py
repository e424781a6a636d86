"""Host-side checks of progressive frames: the doubling schedule, the exports of rtrb_progressive_*, and the argument
and device checks that come before any device work."""
import ctypes as C

import pytest

from raytracing_rb_b200 import _abi, make_opts, progressive_schedule


@pytest.fixture(scope="module")
def L():
    from raytracing_rb_b200 import _lib
    return _lib.lib()


@pytest.mark.parametrize("pre, first, want", [
    (1, 1, [1]), (2, 1, [1, 2]), (3, 1, [1, 2, 3]), (4, 1, [1, 2, 4]), (10, 1, [1, 2, 4, 8, 10]),
    (64, 1, [1, 2, 4, 8, 16, 32, 64]), (64, 3, [3, 6, 12, 24, 48, 64]), (5, 8, [5]), (16, 16, [16]),
])
def test_progressive_schedule_doubles_and_ends_at_pre(pre, first, want):
    assert progressive_schedule(pre, first) == want


@pytest.mark.parametrize("pre, first", [(0, 1), (4, 0), (-1, 1)])
def test_progressive_schedule_rejects_bad_counts(pre, first):
    with pytest.raises(ValueError):
        progressive_schedule(pre, first)


def test_progressive_symbols_are_exported_abi_unchanged(L):
    from raytracing_rb_b200 import _lib
    for n in ("rtrb_progressive_create", "rtrb_progressive_pass", "rtrb_progressive_download",
              "rtrb_progressive_frame_ptr", "rtrb_progressive_destroy"):
        assert hasattr(L, n), n
        assert n in _lib.EXPORTS, n
    assert L.rtrb_abi_version() == 4


def camera():
    from raytracing_rb_b200 import Camera, World, scenes
    w, c = scenes.build(1)
    return Camera(World(w), c).camera_desc()


def test_null_arguments_are_invalid(L):
    cam = camera()
    opts = make_opts()
    out = C.c_void_p()
    fake = C.create_string_buffer(64)  # never dereferenced: the argument checks come first
    assert L.rtrb_progressive_create(None, C.byref(cam), C.byref(opts), C.byref(out)) == _abi.RTRB_ERR_INVALID
    assert L.rtrb_progressive_create(fake, None, C.byref(opts), C.byref(out)) == _abi.RTRB_ERR_INVALID
    assert L.rtrb_progressive_create(fake, C.byref(cam), C.byref(opts), None) == _abi.RTRB_ERR_INVALID
    assert out.value is None
    assert L.rtrb_progressive_pass(None, 1, None) == _abi.RTRB_ERR_INVALID
    assert L.rtrb_progressive_download(None, None, None, None) == _abi.RTRB_ERR_INVALID
    assert L.rtrb_progressive_frame_ptr(None, C.byref(C.c_void_p())) == _abi.RTRB_ERR_INVALID
    assert L.rtrb_progressive_destroy(None) == _abi.RTRB_OK


def test_bad_camera_and_options_are_rejected_before_the_device(L):
    cam = camera()
    fake = C.create_string_buffer(64)
    out = C.c_void_p()
    bad_cam = _abi.CameraDesc.from_buffer_copy(cam)
    bad_cam.pre_sample_times = 0
    assert L.rtrb_progressive_create(fake, C.byref(bad_cam), None, C.byref(out)) == _abi.RTRB_ERR_INVALID
    assert L.rtrb_progressive_create(fake, C.byref(cam), C.byref(make_opts(rng_mode=_abi.RNG_MT)),
                                     C.byref(out)) == _abi.RTRB_ERR_UNSUPPORTED
    assert L.rtrb_progressive_create(fake, C.byref(cam), C.byref(make_opts(pixel_format=7)), C.byref(out)) == _abi.RTRB_ERR_INVALID
    assert L.rtrb_progressive_create(fake, C.byref(cam), C.byref(make_opts(window=(0, 0, 10**6, 5))),
                                     C.byref(out)) == _abi.RTRB_ERR_INVALID


def test_create_without_a_device_fails_with_cuda_error(L):
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    cam = camera()
    fake = C.create_string_buffer(64)  # never dereferenced: the device check comes before any use of the renderer
    out = C.c_void_p()
    assert L.rtrb_progressive_create(fake, C.byref(cam), C.byref(make_opts()), C.byref(out)) == _abi.RTRB_ERR_CUDA
    assert out.value is None
