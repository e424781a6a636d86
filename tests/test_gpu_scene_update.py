"""rtrb_scene_update: a renderer whose scene is replaced in place renders exactly what a renderer created from the new
scene renders (RGBA8 bytes, float RGB, hit ids and every counter except the FAST64 refine count and the timings), across
scene-class and filter changes, buffer growth, frames and ray calls in flight on several streams, and through the
Python mirror's Camera / World."""
import copy

import numpy as np
import pytest

from raytracing_rb_b200 import (Camera, Renderer, World, _abi, device_count, make_opts, render_multi, scenes,
                                PREC_FAST64, PREC_STRICT)
from raytracing_rb_b200._lib import RtrbError
from raytracing_rb_b200.vec3 import Vec3

pytestmark = pytest.mark.gpu

VOLATILE = ("exact_tests", "device_ms", "trace_ms")
SKIP = _abi.SKIP_RGB | _abi.SKIP_HIT


# ---- scenes ------------------------------------------------------------------------------------------------------
def moved(wdoc, dx=0.25, dy=-0.15):
    """Every sphere of the world moved by (dx, dy, 0)."""
    w = copy.deepcopy(wdoc)
    for o in w["world_objects"]:
        if o["type"] == "Sphere":
            c = o["properties"]["center"]
            o["properties"]["center"] = [c[0] + dx, c[1] + dy, c[2]]
    return w


def with_lights(wdoc, lights):
    return dict(copy.deepcopy(wdoc), lights=lights)


def grid_world(n):
    """Ground + n matte spheres: 31 keeps the linear filter with its apex tables, 40 takes the BVH."""
    objs = [scenes.ground()]
    for k in range(n):
        objs.append(scenes.matte("s%d" % k, (4 + 1.1 * (k // 8), -4 + 1.1 * (k % 8), -0.6), 0.4,
                                 (0.4 + 0.07 * (k % 8), 0.5, 0.9 - 0.05 * (k % 8))))
    return scenes._world(objs, [scenes.light([5, -4, 4], 0.0)])


def textured_sphere():
    return [o for o in scenes._config3_objects() if o["properties"]["name"] == "rails sphere"][0]


def c2(w=192, h=108):
    return scenes.build(2, width=w, height=h)


EMPTY = {"max_distance": 10000, "soft_shadow_exponent": 2, "lights": [], "world_objects": []}


def pair(name):
    """(world A, world B, camera doc) of each scene pair."""
    w2, cam2 = c2()
    if name == "c2_moved":
        return w2, moved(w2), cam2
    if name == "c2_lean_to_one_light":
        return w2, with_lights(w2, [scenes.light([5, -4, 4], 0.8)]), cam2
    if name == "c2_one_light_to_generic":
        three = [scenes.light([5, -4, 4], 0.8), scenes.light([2, 5, 6], 0.0), scenes.light([8, 0, 5], 0.3)]
        for l in three:
            l["properties"]["color"] = [0.3, 0.3, 0.3]
        return with_lights(w2, [scenes.light([5, -4, 4], 0.8)]), with_lights(w2, three), cam2
    if name in ("31_to_40", "40_to_31"):
        a, b = grid_world(31), grid_world(40)
        return (a, b, cam2) if name == "31_to_40" else (b, a, cam2)
    if name in ("c2_to_c7", "c7_to_c2"):
        w7, cam7 = scenes.build(7, width=96, height=54)
        return (w2, w7, cam7) if name == "c2_to_c7" else (w7, w2, cam7)
    if name == "add_textured_sphere":
        w = copy.deepcopy(w2)
        w["world_objects"].append(textured_sphere())
        return w2, w, scenes.build(3, width=96, height=54)[1]
    if name in ("empty_to_c1", "c1_to_empty"):
        w1, cam1 = scenes.build(1)
        return (EMPTY, w1, cam1) if name == "empty_to_c1" else (w1, EMPTY, cam1)
    if name == "c5_all_moved":
        w5, cam5 = scenes.build(5, width=96, height=54, spp=2)
        return w5, moved(w5, 0.05, 0.03), cam5
    raise KeyError(name)


PAIRS = ["c2_moved", "c2_lean_to_one_light", "c2_one_light_to_generic", "31_to_40", "40_to_31", "c2_to_c7", "c7_to_c2",
         "add_textured_sphere", "empty_to_c1", "c1_to_empty", "c5_all_moved"]


# ---- frames ------------------------------------------------------------------------------------------------------
def desc(wdoc):
    return World(copy.deepcopy(wdoc)).to_scene_desc()


def cam_desc(wdoc, cdoc):
    return Camera(World(copy.deepcopy(wdoc)), copy.deepcopy(cdoc)).camera_desc()


def frame(r, cam, precision):
    return r.render(cam, make_opts(seed=1, precision=precision, count_detail=True))


def assert_same(got, want, what=""):
    assert np.array_equal(got.rgba, want.rgba), what + ": RGBA8"
    assert np.array_equal(got.rgb, want.rgb), what + ": float RGB"
    assert np.array_equal(got.hit, want.hit), what + ": hit ids"
    assert got.code == want.code, what
    a = {k: v for k, v in got.stats.items() if k not in VOLATILE}
    b = {k: v for k, v in want.stats.items() if k not in VOLATILE}
    assert a == b, what


def fresh(wdoc, cam, precision):
    r = Renderer(desc(wdoc), 0)
    f = frame(r, cam, precision)
    r.close()
    return f


@pytest.mark.parametrize("precision", [PREC_STRICT, PREC_FAST64])
@pytest.mark.parametrize("name", PAIRS)
def test_update_equals_fresh_renderer(name, precision):
    wa, wb, cdoc = pair(name)
    cam = cam_desc(wa, cdoc)
    r = Renderer(desc(wa), 0)
    first = frame(r, cam, precision)
    assert_same(first, fresh(wa, cam, precision), "A before the update")
    r.update(desc(wb))
    assert_same(frame(r, cam, precision), fresh(wb, cam, precision), "after the update to B")
    r.close()


@pytest.mark.parametrize("precision", [PREC_STRICT, PREC_FAST64])
def test_a_b_a_reproduces_a(precision):
    wa, wb, cdoc = pair("c2_to_c7")
    cam = cam_desc(wa, cdoc)
    r = Renderer(desc(wa), 0)
    first = frame(r, cam, precision)
    r.update(desc(wb))
    frame(r, cam, precision)
    r.update(desc(wa))
    assert_same(frame(r, cam, precision), first, "A -> B -> A")
    r.close()


def test_unchanged_scene_is_a_no_op():
    wdoc, cdoc = c2()
    cam = cam_desc(wdoc, cdoc)
    r = Renderer(desc(wdoc), 0)
    first = frame(r, cam, PREC_FAST64)
    for _ in range(3):
        r.update(desc(wdoc))
    assert_same(frame(r, cam, PREC_FAST64), first, "unchanged scene")
    r.close()


# ---- rejected updates --------------------------------------------------------------------------------------------
def broken(wdoc, how):
    h = desc(wdoc)
    o = h.desc.objects[3]
    if how == "sphere_without_refractive_rate":
        o.has_refraction = 0
    elif how == "unknown_type":
        o.type = 7
    else:
        o.texture = 5
    return h


@pytest.mark.parametrize("how", ["sphere_without_refractive_rate", "unknown_type", "bad_texture_index"])
def test_rejected_update_keeps_the_old_scene(how):
    wdoc, cdoc = c2()
    cam = cam_desc(wdoc, cdoc)
    r = Renderer(desc(wdoc), 0)
    before = frame(r, cam, PREC_FAST64)
    with pytest.raises(RtrbError) as e:
        r.update(broken(moved(wdoc), how))
    assert e.value.code in (_abi.RTRB_ERR_INVALID, _abi.RTRB_ERR_UNSUPPORTED)
    assert_same(frame(r, cam, PREC_FAST64), before, "after a rejected update")
    r.close()


# ---- stream order ------------------------------------------------------------------------------------------------
def rgb8_fresh(wdoc, cam):
    r = Renderer(desc(wdoc), 0)
    f = r.render(cam, make_opts(seed=1, pixel_format=_abi.FMT_RGB8), want_rgb=False, want_hit=False).rgba
    r.close()
    return f


def three_scenes(kind):
    if kind == "depth1":
        w, cdoc = c2(480, 270)
    else:
        w, cdoc = scenes.build(3, width=160, height=90)
    return [w, moved(w), moved(w, 0.6, 0.4)], cdoc


@pytest.mark.parametrize("kind", ["depth1", "ray_tree"])
def test_pipelined_submit_update_submit(kind):
    import torch
    worlds, cdoc = three_scenes(kind)
    cam = cam_desc(worlds[0], cdoc)
    want = [rgb8_fresh(w, cam) for w in worlds]
    assert len({f.tobytes() for f in want}) == 3
    r = Renderer(desc(worlds[0]), 0)
    outs = [torch.zeros((cam.height, cam.width, 3), dtype=torch.uint8).pin_memory().numpy() for _ in range(3)]
    opts = make_opts(seed=1, pixel_format=_abi.FMT_RGB8)
    tickets = [r.submit(cam, outs[0], opts)]
    r.update(desc(worlds[1]))
    tickets.append(r.submit(cam, outs[1], opts))
    r.update(desc(worlds[2]))
    tickets.append(r.submit(cam, outs[2], opts))
    for t in tickets:
        r.wait(t)
    for i in range(3):
        assert np.array_equal(outs[i], want[i]), "frame %d" % i
    r.close()


@pytest.mark.parametrize("on_torch_stream", [False, True])
@pytest.mark.parametrize("kind", ["depth1", "ray_tree"])
def test_render_device_update_render_device(kind, on_torch_stream):
    import torch
    worlds, cdoc = three_scenes(kind)
    cam = cam_desc(worlds[0], cdoc)
    want = [rgb8_fresh(w, cam) for w in worlds]
    W, H = cam.width, cam.height
    r = Renderer(desc(worlds[0]), 0)
    base = r.framebuffer_ptr(W, H * 6)
    s = torch.cuda.Stream() if on_torch_stream else None
    handle = s.cuda_stream if s is not None else None

    def launch(slot):
        r.render_device(cam, make_opts(seed=1, stream=handle, rgba_device_out=base + slot * W * H * 4, skip_outputs=SKIP,
                                       pixel_format=_abi.FMT_RGB8), want_stats=False)

    # two frames of each scene back to back: the second one overlaps the first again
    launch(0); launch(1)
    r.update(desc(worlds[1]), stream=handle)
    launch(2); launch(3)
    r.update(desc(worlds[2]), stream=s)
    launch(4); launch(5)
    torch.cuda.synchronize()
    got = np.zeros((H * 6, W, 4), np.uint8)
    r.framebuffer_download(W, H * 6, got)
    got = got.reshape(6, W * H * 4)[:, :W * H * 3]
    for slot in range(6):
        assert np.array_equal(got[slot], want[slot // 2].reshape(-1)), "slot %d" % slot
    r.close()


def test_cross_stream_update_waits_for_the_frame_in_flight():
    import torch
    wa, cdoc = scenes.build(5, width=960, height=540, spp=32)
    wb = moved(wa, 0.05, 0.03)
    cam = cam_desc(wa, cdoc)
    want = [rgb8_fresh(w, cam) for w in (wa, wb)]
    W, H = cam.width, cam.height
    r = Renderer(desc(wa), 0)
    base = r.framebuffer_ptr(W, H * 2)
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    hb = desc(wb)  # flattened before the frame, so the update is issued while the frame runs

    def launch(slot):
        r.render_device(cam, make_opts(seed=1, stream=s1.cuda_stream, rgba_device_out=base + slot * W * H * 4,
                                       skip_outputs=SKIP, pixel_format=_abi.FMT_RGB8), want_stats=False)

    launch(0)
    r.update(hb, stream=s2.cuda_stream)
    launch(1)
    torch.cuda.synchronize()
    got = np.zeros((H * 2, W, 4), np.uint8)
    r.framebuffer_download(W, H * 2, got)
    got = got.reshape(2, W * H * 4)[:, :W * H * 3]
    assert np.array_equal(got[0], want[0].reshape(-1)), "the frame queued before the update"
    assert np.array_equal(got[1], want[1].reshape(-1)), "the frame issued after the update"
    r.close()


def test_growth_while_frames_are_in_flight():
    import torch
    small = scenes._world([scenes.ground(), scenes.matte("a", (5, 0, -0.5), 0.5, (1, 0.5, 0.5)),
                           scenes.matte("b", (7, 2, -0.4), 0.6, (0.5, 1, 0.5))], [scenes.light([5, -4, 4], 0.0)])
    big = scenes.config5(width=480, height=270, spp=1, grid=45)[0]  # 2 027 objects
    big["world_objects"] = big["world_objects"][:2000]
    _, cdoc = c2(480, 270)
    cam = cam_desc(small, cdoc)
    want_small, want_big = rgb8_fresh(small, cam), rgb8_fresh(big, cam)
    r = Renderer(desc(small), 0)
    outs = [torch.zeros((cam.height, cam.width, 3), dtype=torch.uint8).pin_memory().numpy() for _ in range(5)]
    opts = make_opts(seed=1, pixel_format=_abi.FMT_RGB8)
    tickets = [r.submit(cam, outs[i], opts) for i in range(4)]
    r.update(desc(big))
    for t in tickets:
        r.wait(t)
    r.wait(r.submit(cam, outs[4], opts))
    for i in range(4):
        assert np.array_equal(outs[i], want_small), "small-scene frame %d" % i
    assert np.array_equal(outs[4], want_big)
    r.close()


def test_ray_queries_after_an_update():
    wa, cdoc = c2(64, 36)
    wb = moved(wa)
    cam = cam_desc(wa, cdoc)
    r = Renderer(desc(wa), 0)
    rays, keys = r.camera_rays(cam)
    r.trace_rays(rays, keys=keys)
    r.update(desc(wb))
    fr = Renderer(desc(wb), 0)
    got, want = r.trace_rays(rays, keys=keys, count_detail=True), fr.trace_rays(rays, keys=keys, count_detail=True)
    assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1])
    assert {k: v for k, v in got[2].items() if k not in VOLATILE} == {k: v for k, v in want[2].items() if k not in VOLATILE}
    assert np.array_equal(r.intersect_rays(rays), fr.intersect_rays(rays))
    r.close()
    fr.close()


def test_multi_gpu_update_keeps_the_framebuffer():
    n = device_count()
    if n < 2:
        pytest.skip("needs two devices")
    wa, cdoc = c2(480, 270)
    wb = moved(wa)
    cam = cam_desc(wa, cdoc)
    rs = [Renderer(desc(wa), d) for d in range(2)]
    ptr = rs[0].framebuffer_ptr(cam.width, cam.height)
    render_multi(rs, cam, make_opts(seed=1))
    for r in rs:
        r.update(desc(wb))
    assert rs[0].framebuffer_ptr(cam.width, cam.height) == ptr
    many = render_multi(rs, cam, make_opts(seed=1))
    solo = Renderer(desc(wb), 0)
    one = solo.render(cam, make_opts(seed=1))
    assert np.array_equal(many.rgba, one.rgba) and np.array_equal(many.rgb, one.rgb)
    assert np.array_equal(many.hit, one.hit)
    for r in rs + [solo]:
        r.close()


# ---- the Python mirror -------------------------------------------------------------------------------------------
def test_world_edits_reach_render_cuda_and_intersect(tmp_path):
    wdoc, cdoc = c2(160, 90)
    wp, cp = scenes.write_yaml(2, str(tmp_path / "before"), width=160, height=90)
    world = World(wp)
    cam = Camera(world, cp)
    cam.render_cuda(None)
    r = cam.renderer()
    wr = world.renderer()
    ray = [[0, 0, 0, 1, -0.05, -0.12]]
    world.intersect_batch(ray)

    k = 5
    x, y, z = world.world_objects[k].center.to_a()
    world.world_objects[k].center = Vec3(x + 0.4, y - 0.3, z)
    world.lights[0].color = Vec3(0.8, 0.7, 0.6)
    got = cam.render_cuda(None)

    edited = copy.deepcopy(wdoc)
    props = edited["world_objects"][k]["properties"]
    props["center"] = [props["center"][0] + 0.4, props["center"][1] - 0.3, props["center"][2]]
    edited["lights"][0]["properties"]["color"] = [0.8, 0.7, 0.6]
    import yaml
    (tmp_path / "edited.yml").write_text(yaml.safe_dump(edited))
    fresh_world = World(str(tmp_path / "edited.yml"))
    want = Camera(fresh_world, cp).render_cuda(None)
    assert np.array_equal(got.rgba, want.rgba) and np.array_equal(got.rgb, want.rgb)
    assert np.array_equal(got.hit, want.hit)
    assert not np.array_equal(got.rgba, Camera(World(wp), cp).render_cuda(None).rgba)
    assert cam.renderer() is r and world.renderer() is wr
    rays = np.array([[0, 0, 0, 1, -0.05 + 0.01 * i, -0.12] for i in range(-20, 20)], np.float64)
    assert np.array_equal(world.intersect_batch(rays), fresh_world.intersect_batch(rays))
