"""Frame overlap: consecutive depth-1 FAST64 frames on one stream run with programmatic dependent launch (the next
frame's kernel traces under the tail of the previous one and waits for it only to write) and take their control
blocks from a ring that each kernel zeroes one slot ahead.  Frames and per-frame stats must be exactly what the same
frames give one at a time with RTRB_FRAME_OVERLAP=0: into distinct buffers and into one shared buffer (the last
frame wins), with more frames than control blocks in the ring, with frames that set status bits between clean
ones, and interleaved with every other call that enqueues work on the renderer's stream."""
import numpy as np
import pytest

from raytracing_rb_b200 import Camera, Renderer, World, _abi, make_opts, png_max_bytes, scenes

pytestmark = pytest.mark.gpu

RING = 4  # control blocks of the synchronous frame path (RTRB_CTL_RING)
STAT_KEYS = ("rays", "shadow_queries", "samples", "status", "first_bad_x", "first_bad_y", "max_stack")
SKIP = _abi.SKIP_RGB | _abi.SKIP_HIT


def renderer(world, monkeypatch, overlap):
    if overlap:
        monkeypatch.delenv("RTRB_FRAME_OVERLAP", raising=False)  # on by default
    else:
        monkeypatch.setenv("RTRB_FRAME_OVERLAP", "0")
    r = Renderer(world.to_scene_desc(), 0)
    monkeypatch.delenv("RTRB_FRAME_OVERLAP", raising=False)
    return r


def dolly(world, cdoc, n):
    cams = []
    for f in range(n):
        c = Camera(world, cdoc).camera_desc()
        c.position[1] = c.position[1] + 0.02 * (f % 64)
        cams.append(c)
    return cams


def stats_of(st):
    return {k: st[k] for k in STAT_KEYS}


def solo_frames(world, cams, monkeypatch, opts=None):
    """The frames and stats one at a time, frame overlap off."""
    r = renderer(world, monkeypatch, overlap=False)
    frames, stats = [], []
    for cam in cams:
        fr = r.render(cam, opts or make_opts(seed=1, pixel_format=_abi.FMT_RGB8), want_rgb=False, want_hit=False)
        frames.append(fr.rgba)
        stats.append(stats_of(fr.stats))
    r.close()
    return frames, stats


def generic_two_lights(width, height):
    """Config 2 with a second light: no longer a lean scene, so its depth-1 frames run the generic build."""
    wdoc, cdoc = scenes.build(2, width=width, height=height)
    second = scenes.light([2, 5, 6], 0.0)
    wdoc = dict(wdoc, lights=list(wdoc["lights"]) + [second])
    for l in wdoc["lights"]:
        l["properties"]["color"] = [0.5, 0.5, 0.5]
    return wdoc, cdoc


@pytest.mark.parametrize("scene", ["config2_lean_1080p", "generic_two_lights_480x270"])
def test_back_to_back_frames_equal_solo_frames(monkeypatch, scene):
    import torch
    if scene == "config2_lean_1080p":
        wdoc, cdoc = scenes.build(2)
        n = 32
    else:
        wdoc, cdoc = generic_two_lights(480, 270)
        n = 12
    world = World(wdoc)
    cams = dolly(world, cdoc, n)
    W, H = cams[0].width, cams[0].height
    frame_bytes, slot_bytes = W * H * 3, W * H * 4
    want, want_stats = solo_frames(world, cams, monkeypatch)
    assert len({f.tobytes() for f in want}) > 1  # the dolly moves the picture

    r = renderer(world, monkeypatch, overlap=True)
    s = torch.cuda.Stream()
    base = r.framebuffer_ptr(W, H * n)
    shared = torch.zeros(frame_bytes, dtype=torch.uint8, device="cuda")

    def opts(out):
        return make_opts(seed=1, stream=s.cuda_stream, rgba_device_out=out, skip_outputs=SKIP,
                         pixel_format=_abi.FMT_RGB8)

    for f in range(n):  # distinct slots
        r.render_device(cams[f], opts(base + f * slot_bytes), want_stats=False)
    for f in range(n):  # one shared buffer: every frame overwrites the previous one
        r.render_device(cams[f], opts(shared.data_ptr()), want_stats=False)
    torch.cuda.synchronize()
    got = np.zeros((H * n, W, 4), np.uint8)
    r.framebuffer_download(W, H * n, got)
    got = got.reshape(n, slot_bytes)[:, :frame_bytes]
    for f in range(n):
        assert np.array_equal(got[f], want[f].reshape(-1)), "frame %d differs" % f
    assert np.array_equal(shared.cpu().numpy(), want[-1].reshape(-1))

    # per-frame stats of frames between unread ones: every third frame reports none, so the ring wraps with
    # blocks that unread frames counted into
    for f in range(n):
        if f % 3 == 1:
            r.render_device(cams[f], opts(base + f * slot_bytes), want_stats=False)
        else:
            st, _ = r.render_device(cams[f], opts(base + f * slot_bytes))
            assert stats_of(st) == want_stats[f], "frame %d" % f
    r.close()


def bright_ground_world():
    """test_status_word_color_greater_than_one's scene: the ground's ambient alone makes a lit pixel exceed 1, so a
    window on the ground raises and a window on the sky does not."""
    g = scenes.ground()
    g["properties"]["ambient"] = [0.9, 0.9, 0.9]
    return World({"max_distance": 10000, "soft_shadow_exponent": 2, "lights": [scenes.light([5, -4, 4], 0.0)],
                  "world_objects": [g, scenes.matte("m", [6, 0, 0], 0.6, (1, 1, 1))]})


def test_status_frames_between_clean_frames(monkeypatch):
    world = bright_ground_world()
    _, cdoc = scenes.build(2, width=96, height=54)
    n = 5 * RING
    cams = dolly(world, cdoc, n)
    W, H = cams[0].width, cams[0].height
    windows = [(0, 0, W, 8) if f % 2 == 0 else (0, H - 20, W, H) for f in range(n)]  # sky strip / ground strip

    def opts(f, stream=None, out=None):
        return make_opts(seed=1, window=windows[f], skip_outputs=SKIP, pixel_format=_abi.FMT_RGB8, stream=stream,
                         rgba_device_out=out)

    solo = renderer(world, monkeypatch, overlap=False)
    want = [stats_of(solo.render_device(cams[f], opts(f))[0]) for f in range(n)]
    solo.close()
    assert all(want[f]["status"] == 0 for f in range(0, n, 2))
    assert all(want[f]["status"] & _abi.ST_COLOR_GT_1 and want[f]["first_bad_x"] >= 0 for f in range(1, n, 2))

    r = renderer(world, monkeypatch, overlap=True)
    for f in range(n):
        if f % 3 == 1:  # raised or clean frames nobody reads, ahead of frames that are read
            _, code = r.render_device(cams[f], opts(f), want_stats=False)
            assert code == _abi.RTRB_OK
        else:
            st, code = r.render_device(cams[f], opts(f))
            assert stats_of(st) == want[f], "frame %d" % f
            assert code == (_abi.RTRB_ERR_RAISED if want[f]["status"] else _abi.RTRB_OK)
    r.close()


def interleaved_calls(r, cams, bufs):
    """Overlapping frames on the renderer's own stream with every other call that enqueues work there between them.
    Returns everything the calls delivered."""
    import torch
    W, H = cams[0].width, cams[0].height
    out = []
    quiet = make_opts(seed=1, skip_outputs=SKIP, pixel_format=_abi.FMT_RGB8)
    for k in range(2):
        c = cams[4 * k:4 * k + 4]
        r.render_device(c[0], quiet, want_stats=False)
        st, _ = r.render_device(c[1], quiet)
        out.append(stats_of(st))
        r.render_device(c[2], quiet, want_stats=False)
        rgb, hit, st, _ = r.trace_rays(r.camera_rays(c[2], window=(0, 0, 32, 16))[0])
        out += [rgb, hit, stats_of(st)]
        r.render_device(c[3], quiet, want_stats=False)
        out.append(r.encode_png(W, H, _abi.FMT_RGB8))
        t = r.submit(c[0], bufs["rgb"], make_opts(seed=1, pixel_format=_abi.FMT_RGB8))
        r.render_device(c[1], quiet, want_stats=False)
        st, _ = r.wait(t)
        out += [bufs["rgb"].copy(), stats_of(st)]
        png, st, _ = r.wait_png(r.submit_png(c[2], bufs["png"], make_opts(seed=1, pixel_format=_abi.FMT_RGB8)))
        out += [png, stats_of(st)]
        r.render_device(c[3], quiet, want_stats=False)
        torch.cuda.synchronize()
        fb = np.zeros((H, W, 4), np.uint8)
        r.framebuffer_download(W, H, fb)
        out.append(fb.reshape(-1)[:W * H * 3].copy())
    return out


def test_interleaved_with_stats_submit_rays_and_png(monkeypatch):
    import torch
    world = World(scenes.build(2, width=480, height=270)[0])
    _, cdoc = scenes.build(2, width=480, height=270)
    cams = dolly(world, cdoc, 8)
    W, H = cams[0].width, cams[0].height
    bufs = {"rgb": torch.zeros((H, W, 3), dtype=torch.uint8).pin_memory().numpy(),
            "png": torch.zeros(png_max_bytes(W, H), dtype=torch.uint8).pin_memory().numpy()}
    results = []
    for overlap in (False, True):
        r = renderer(world, monkeypatch, overlap)
        results.append(interleaved_calls(r, cams, bufs))
        r.close()
    off, on = results
    assert len(off) == len(on)
    for i, (a, b) in enumerate(zip(off, on)):
        if isinstance(a, np.ndarray):
            assert np.array_equal(a, b), "result %d" % i
        else:
            assert a == b, "result %d" % i
