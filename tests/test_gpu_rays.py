"""Ray-level queries on the GPU (rtrb_trace_rays, rtrb_intersect_rays, rtrb_camera_rays) driven with adversarial rays:
origins inside spheres or just off surfaces, grazing tangents, rays parallel to planes, origins thousands of units out,
unnormalised directions from 1e-6 to 1e6 long, and zero / NaN / infinite directions.  STRICT must match the oracle's
RayTracer#trace_sync and World#intersect, FAST64 must equal STRICT bit for bit, and camera rays traced with their keys
must rebuild the frames render_frame produces."""
import ctypes as C

import numpy as np
import pytest

from raytracing_rb_b200 import PREC_FAST64, PREC_STRICT, Camera, World, _abi, make_opts, scenes
from raytracing_rb_b200._lib import lib
from raytracing_rb_b200.renderer import make_ray_opts
from test_gpu_fuzz import random_scene, structural_scene

pytestmark = pytest.mark.gpu

TRACE_COUNTERS = ("samples", "rays", "shadow_queries", "hits", "refractions", "mc_rays", "sphere_tests", "plane_tests",
                  "box_tests")
FAST_COUNTERS = ("samples", "rays", "shadow_queries", "hits", "highlight_hits", "local_shaded", "lit_lights", "mc_rays",
                 "texel_fetches", "status")


def small_config(cid):
    kw = {1: {}, 2: dict(width=96, height=54), 3: dict(width=96, height=54), 4: dict(width=96, height=54),
          5: dict(width=64, height=36, spp=2)}[cid]
    return scenes.build(cid, **kw)


# (name, scene builder, trace_depth, mc): every scene gets a different (depth, mc), together covering 0..8 and 0..2
SCENES = ([("config%d" % c, (lambda c=c: small_config(c)), d, m) for c, d, m in
           ((1, 4, 1), (2, 1, 0), (3, 8, 0), (4, 3, 2), (5, 2, 1))] +
          [("random%d" % s, (lambda s=s: random_scene(s)), [0, 1, 2, 5, 6, 7][s % 6], s % 3) for s in range(0, 36, 5)] +
          [("structural%d" % s, (lambda s=s: structural_scene(s)), [1, 2, 3, 4][s % 4], [0, 1, 2][s % 3])
           for s in range(0, 24, 3)])


def _unit(rs, n):
    v = rs.normal(size=(n, 3))
    return v / np.linalg.norm(v, axis=1, keepdims=True)


def scene_geometry(world):
    sd = world.to_scene_desc().desc
    sph, pl = [], []
    for i in range(sd.n_objects):
        o = sd.objects[i]
        if o.type == _abi.OBJ_SPHERE:
            sph.append((np.array(o.point[:]), o.radius))
        elif o.type == _abi.OBJ_PLANE:
            pl.append((np.array(o.point[:]), np.array(o.front[:])))
        else:  # a box: its bounding sphere stands in for the geometry of the ray sets
            sph.append((np.array(o.point[:]), 0.5 * float(np.linalg.norm([o.width_front, o.width_up, o.width_left]))))
    return sph, pl


def adversarial_rays(world, cam, renderer, seed, n_each=160):
    """[n, 6] rays of every kind the module docstring lists."""
    rs = np.random.RandomState(seed)
    sph, pl = scene_geometry(world)
    cpos = np.array(cam.position.to_a())
    pts = [c for c, _ in sph] + [cpos]
    lo, hi = np.min(pts, axis=0) - 2.0, np.max(pts, axis=0) + 2.0
    sets = []
    # the camera's own rays
    desc = cam.camera_desc()
    cr, _ = renderer.camera_rays(desc, seed=seed, samples=(0, 1))
    sets.append(cr[rs.choice(len(cr), min(n_each, len(cr)), replace=False)])
    # random origins in the scene's bounds, directions of length 1e-6 .. 1e6
    o = rs.uniform(lo, hi, size=(n_each, 3))
    d = _unit(rs, n_each) * (10.0 ** rs.uniform(-6, 6, size=(n_each, 1)))
    sets.append(np.hstack([o, d]))
    # origins at intersection +- delta of real hits
    probe = np.hstack([rs.uniform(lo, hi, size=(4 * n_each, 3)), _unit(rs, 4 * n_each)])
    h = renderer.intersect_rays(probe, PREC_STRICT)
    h = h[h["object"] >= 0][:n_each // 2]
    for sgn in (1.0, -1.0):
        sets.append(np.hstack([h["intersection"] + sgn * h["delta"], _unit(rs, len(h))]))
    if sph:
        k = rs.randint(len(sph), size=n_each)
        c = np.array([sph[i][0] for i in k]); r = np.array([sph[i][1] for i in k])[:, None]
        v = _unit(rs, n_each)
        u = np.cross(v, _unit(rs, n_each)); u /= np.linalg.norm(u, axis=1, keepdims=True)
        f = np.where(rs.rand(n_each, 1) < 0.5, 1.0 + 1e-12, 1.0 - 1e-12)
        sets.append(np.hstack([c + u * r * f - v * rs.uniform(0.5, 20, (n_each, 1)), v]))       # tangents at R(1 +- 1e-12)
        sets.append(np.hstack([c + _unit(rs, n_each) * r * rs.uniform(0, 0.9, (n_each, 1)), _unit(rs, n_each)]))  # inside
    if pl:
        k = rs.randint(len(pl), size=n_each)
        p = np.array([pl[i][0] for i in k]); nrm = np.array([pl[i][1] for i in k])
        par = np.cross(nrm, _unit(rs, n_each))                                                     # parallel to the plane
        on = rs.rand(n_each, 1) < 0.5
        o = np.where(on, p + np.cross(nrm, _unit(rs, n_each)), rs.uniform(lo, hi, size=(n_each, 3)))
        sets.append(np.hstack([o, par]))
    far = np.array([3000.0, -2000.0, 500.0])
    sets.append(np.hstack([rs.uniform(lo, hi, size=(n_each, 3)) + far, _unit(rs, n_each)]))
    sets.append(np.hstack([far + cpos + rs.normal(size=(n_each, 3)), np.tile(np.mean(pts, axis=0) - far - cpos, (n_each, 1))
                           + rs.normal(size=(n_each, 3))]))
    odd = np.array([[0, 0, 0], [np.nan, 0, 1], [np.inf, 0, 0], [0, -np.inf, 1], [np.nan] * 3, [1e-300, 0, 0], [1e300, 1e300, 0]])
    o = rs.uniform(lo, hi, size=(len(odd), 3))
    sets.append(np.hstack([o, odd]))
    sets.append(np.hstack([cpos + np.zeros((len(odd), 3)), odd]))
    return np.ascontiguousarray(np.vstack(sets), np.float64)


def _build(maker):
    wdoc, cdoc = maker()
    world = World(wdoc)
    cam = Camera(world, cdoc)
    return world, cam


def _assert_same_nan(a, b, **kw):
    assert np.array_equal(np.isnan(a), np.isnan(b))
    m = ~np.isnan(a)
    if kw:
        np.testing.assert_allclose(a[m], b[m], rtol=0, **kw)
    else:
        assert np.array_equal(a[m], b[m])


@pytest.mark.parametrize("name,maker,depth,mc", SCENES, ids=[s[0] for s in SCENES])
def test_trace_rays_strict_oracle_fast(name, maker, depth, mc):
    import rays_oracle
    world, cam = _build(maker)
    r = cam.renderer()
    rays = adversarial_rays(world, cam, r, seed=len(name) * 7 + depth)
    if depth >= 5:
        rays = rays[::2]
    keys = np.stack([np.arange(len(rays)) * 3 + 1, np.arange(len(rays)) % 5], axis=1).astype(np.uint32)
    a_rgb, a_hit, a_st, a_code = r.trace_rays(rays, depth, mc, seed=5, keys=keys, precision=PREC_STRICT, count_detail=True)
    b_rgb, b_hit, b_st, b_code = r.trace_rays(rays, depth, mc, seed=5, keys=keys, precision=PREC_FAST64, count_detail=True)
    # FAST64 == STRICT, bit for bit
    assert np.array_equal(a_rgb, b_rgb, equal_nan=True), "FAST64 must equal STRICT bit for bit"
    assert np.array_equal(a_hit, b_hit) and a_code == b_code
    for k in FAST_COUNTERS + ("first_bad_x", "first_bad_y"):
        assert a_st[k] == b_st[k], k
    # STRICT == oracle (up to libm in the colours)
    o_rgb, o_hit, o_st, o_code = rays_oracle.RayOracle(world.to_scene_desc()).trace_rays(rays, depth, mc, 5, keys)
    assert np.array_equal(a_hit, o_hit)
    assert a_code == o_code
    for k in TRACE_COUNTERS + ("status", "first_bad_x", "first_bad_y"):
        assert a_st[k] == o_st[k], k
    _assert_same_nan(a_rgb, o_rgb, atol=1e-12)
    print("%s depth %d mc %d: %d rays, %d traced items, status 0x%x, first bad %d, hits %d" % (
        name, depth, mc, len(rays), a_st["rays"], a_st["status"], a_st["first_bad_x"], int((a_hit >= 0).sum())))


@pytest.mark.parametrize("name,maker,depth,mc", SCENES, ids=[s[0] for s in SCENES])
def test_intersect_rays_equal_oracle(name, maker, depth, mc):
    import rays_oracle
    world, cam = _build(maker)
    r = cam.renderer()
    rays = adversarial_rays(world, cam, r, seed=len(name) * 11 + 3)
    want = rays_oracle.RayOracle(world.to_scene_desc()).intersect_rays(rays)
    for prec in (PREC_STRICT, PREC_FAST64):
        got = r.intersect_rays(rays, prec)
        for f in ("object", "direction", "face"):
            assert np.array_equal(got[f], want[f]), (prec, f)
        for f in ("distance", "intersection", "delta"):
            assert np.array_equal(got[f], want[f], equal_nan=True), (prec, f)
    miss = want["object"] < 0
    assert np.all(want["face"][miss] == -1) and np.all(got["distance"][miss] == 0)
    assert miss.any() and (~miss).any()


def _restate_render_at(rgb_pre, rgb_extra, pre, mx, threshold):
    """render_at (camera.rb:70-99) from the sample colours, in the reference's order.  rgb_pre: [npx, pre, 3]."""
    npx = rgb_pre.shape[0]
    avg = np.zeros((npx, 3))
    for j in range(pre):
        avg = avg + rgb_pre[:, j]
    avg = avg / float(pre)
    var = np.zeros(npx)
    for j in range(pre):
        d = rgb_pre[:, j] - avg
        m = np.fmax(d[:, 0], np.fmax(d[:, 1], d[:, 2]))
        var = var + m * m
    var = var / float(pre)
    adaptive = var >= threshold
    if mx > pre:
        cv = np.zeros((npx, 3))
        for j in range(mx - pre):
            cv = cv + rgb_extra[:, j]
    else:
        cv = np.zeros((npx, 3))
    avg[adaptive] = (avg[adaptive] * float(pre) + cv[adaptive]) / float(mx)
    return avg


COMPOSITION = [(1, {}, None), (2, dict(width=96, height=54), None), (3, {}, (832, 476, 1088, 604))]


@pytest.mark.parametrize("prec", [PREC_STRICT, PREC_FAST64])
@pytest.mark.parametrize("cid,kw,window", COMPOSITION)
def test_camera_rays_traced_with_keys_rebuild_the_frame(cid, kw, window, prec):
    world, cam = _build(lambda: scenes.build(cid, **kw))
    r = cam.renderer()
    d = cam.camera_desc()
    x0, y0, x1, y1 = window or (0, 0, d.width, d.height)
    pre, mx = d.pre_sample_times, d.max_sample_times
    rays, keys = r.camera_rays(d, seed=3, window=window, samples=(0, pre))
    rgb, hit, st, _ = r.trace_rays(rays, d.trace_depth, d.monte_carlo_diffusion_times, seed=3, keys=keys, precision=prec)
    npx = (x1 - x0) * (y1 - y0)
    rgb_extra = None
    if mx > pre:
        er, ek = r.camera_rays(d, seed=3, window=window, samples=(pre, mx))
        rgb_extra = r.trace_rays(er, d.trace_depth, d.monte_carlo_diffusion_times, seed=3, keys=ek, precision=prec)[0]
        rgb_extra = rgb_extra.reshape(npx, mx - pre, 3)
    got = _restate_render_at(rgb.reshape(npx, pre, 3), rgb_extra, pre, mx, d.variant_threshold)
    frame = cam.render_frame(seed=3, precision=prec, window=window)
    want = frame.rgb[y0:y1, x0:x1].reshape(npx, 3)
    assert np.array_equal(got, want), "max abs diff %g" % np.nanmax(np.abs(got - want))
    assert np.array_equal(hit.reshape(npx, pre)[:, 0], frame.hit[y0:y1, x0:x1].reshape(npx))
    assert st["status"] == frame.stats["status"]


@pytest.mark.parametrize("aperture", [0.0, 0.001])
def test_camera_rays_equal_oracle_lens_func(oracle_mod, aperture):
    world, cam = _build(lambda: scenes.build(1))
    cam.aperture_radius = aperture
    d = cam.camera_desc()
    rays, keys = cam.renderer().camera_rays(d, seed=9, window=(5, 7, 45, 27), samples=(2, 5))
    assert rays.shape == (40 * 20 * 3, 6)
    rs = np.random.RandomState(1)
    for i in rs.choice(len(rays), 300, replace=False):
        j = 2 + i % 3
        x = 5 + (i // 3) % 40
        y = 7 + (i // 3) // 40
        assert tuple(keys[i]) == (y * d.width + x, j)
        a, b = oracle_mod.philox(9, 0, [int(keys[i][0]), j, 0, 0])[:2]
        theta = ((a >> 5) * 67108864.0 + (b >> 6)) * (1.0 / 9007199254740992.0)
        front, pos = oracle_mod.lens_ray(d, x, y, theta)
        want = np.array(pos + front)
        if aperture == 0.0:
            assert np.array_equal(rays[i], want), i
        else:
            np.testing.assert_allclose(rays[i], want, rtol=1e-15, atol=0)


def test_device_buffers_and_batching():
    import torch
    world, cam = _build(lambda: random_scene(5))
    r = cam.renderer()
    rays = adversarial_rays(world, cam, r, seed=2)
    keys = np.stack([np.arange(len(rays)), np.zeros(len(rays))], axis=1).astype(np.uint32)
    h_rgb, h_hit, h_st, h_code = r.trace_rays(rays, 4, 1, seed=2, keys=keys, count_detail=True)
    dev = torch.device("cuda", r.device)
    d_rgb, d_hit, d_st, d_code = r.trace_rays(torch.from_numpy(rays).to(dev), 4, 1, seed=2,
                                              keys=torch.from_numpy(keys.astype(np.int32)).to(dev), count_detail=True)
    assert d_rgb.cpu().numpy().tobytes() == h_rgb.tobytes() and np.array_equal(d_hit.cpu().numpy(), h_hit)
    assert d_code == h_code and all(d_st[k] == h_st[k] for k in FAST_COUNTERS + ("first_bad_x",))
    # without stats the device path does not synchronise; torch's stream orders the outputs
    n_rgb, _, n_st, _ = r.trace_rays(torch.from_numpy(rays).to(dev), 4, 1, seed=2, keys=torch.from_numpy(keys.astype(np.int32)).to(dev),
                                     want_stats=False)
    assert n_st is None and n_rgb.cpu().numpy().tobytes() == h_rgb.tobytes()
    hh = r.intersect_rays(rays)
    hd = r.intersect_rays(torch.from_numpy(rays).to(dev))
    assert hd["raw"].cpu().numpy().tobytes() == hh.tobytes()
    cr, ck = r.camera_rays(cam.camera_desc(), seed=4, samples=(0, 2))
    dr, dk = r.camera_rays(cam.camera_desc(), seed=4, samples=(0, 2), device_buffers=True)
    assert dr.cpu().numpy().tobytes() == cr.tobytes() and dk.cpu().numpy().view(np.uint32).tobytes() == ck.tobytes()
    # one call of 10 000 rays == seven calls with the same keys
    big = np.vstack([rays] * (10000 // len(rays) + 1))[:10000]
    bkeys = np.stack([np.arange(10000) // 3, np.arange(10000) % 3], axis=1).astype(np.uint32)
    one, one_hit, _, _ = r.trace_rays(big, 3, 2, seed=8, keys=bkeys)
    parts = np.array_split(np.arange(10000), 7)
    seven = np.vstack([r.trace_rays(big[p], 3, 2, seed=8, keys=bkeys[p])[0] for p in parts])
    seven_hit = np.concatenate([r.trace_rays(big[p], 3, 2, seed=8, keys=bkeys[p])[1] for p in parts])
    assert seven.tobytes() == one.tobytes() and np.array_equal(seven_hit, one_hit)
    # without keys ray i is keyed (i, 0)
    nk = r.trace_rays(big[:500], 3, 2, seed=8)[0]
    wk = r.trace_rays(big[:500], 3, 2, seed=8, keys=np.stack([np.arange(500), np.zeros(500)], 1).astype(np.uint32))[0]
    assert nk.tobytes() == wk.tobytes()
    # n = 0
    e_rgb, e_hit, e_st, e_code = r.trace_rays(np.zeros((0, 6)), 2, 0)
    assert e_rgb.shape == (0, 3) and e_code == _abi.RTRB_OK and e_st["rays"] == 0
    assert r.intersect_rays(np.zeros((0, 6))).shape == (0,)


def test_ray_calls_leave_frames_alone():
    import torch
    world, cam = _build(lambda: scenes.build(2, width=96, height=54))
    r = cam.renderer()
    d = cam.camera_desc()
    solo = r.render(d, make_opts(seed=4))
    rays = adversarial_rays(world, cam, r, seed=1)
    r.render_device(d, make_opts(seed=4))
    r.trace_rays(rays, 5, 1, seed=3)
    r.intersect_rays(rays)
    r.camera_rays(Camera(world, scenes.build(3, width=40, height=30)[1]).camera_desc(), samples=(0, 2))
    rgba, rgb, hit = r.download(d.width, d.height)
    assert np.array_equal(rgba, solo.rgba) and np.array_equal(rgb, solo.rgb) and np.array_equal(hit, solo.hit)
    r.render_device(d, make_opts(seed=4, pixel_format=_abi.FMT_RGB8))
    png0 = r.encode_png(d.width, d.height, _abi.FMT_RGB8)
    r.render_device(d, make_opts(seed=4, pixel_format=_abi.FMT_RGB8))
    r.trace_rays(rays, 5, 1, seed=3)
    assert r.encode_png(d.width, d.height, _abi.FMT_RGB8) == png0
    # frames in flight on the pipeline slots
    bufs = [torch.zeros((54, 96, 4), dtype=torch.uint8).pin_memory().numpy() for _ in range(2)]
    other = r.render(d, make_opts(seed=6))
    t0 = r.submit(d, bufs[0], make_opts(seed=4))
    t1 = r.submit(d, bufs[1], make_opts(seed=6))
    r.trace_rays(rays, 8, 0, seed=3)
    r.intersect_rays(torch.from_numpy(rays).cuda(r.device))
    r.wait(t0)
    r.wait(t1)
    assert np.array_equal(bufs[0], solo.rgba) and np.array_equal(bufs[1], other.rgba)


def test_ray_call_errors():
    world, cam = _build(lambda: scenes.build(2, width=96, height=54))
    r = cam.renderer()
    L = lib()
    h = r.handle
    rays = np.array([[0, 0, 0, 1, 0, 0]] * 4, np.float64)
    rgb, hit = np.zeros((4, 3)), np.zeros(4, np.int32)
    hits = np.zeros(4 * 72, np.uint8)
    st = _abi.Stats()
    o = make_ray_opts()
    inv, uns = _abi.RTRB_ERR_INVALID, _abi.RTRB_ERR_UNSUPPORTED
    assert L.rtrb_trace_rays(h, C.byref(o), -1, rays.ctypes.data, None, rgb.ctypes.data, None, None) == inv
    assert L.rtrb_trace_rays(h, C.byref(o), 4, None, None, rgb.ctypes.data, None, None) == inv
    assert L.rtrb_trace_rays(h, C.byref(o), 4, rays.ctypes.data, None, None, None, None) == inv
    assert L.rtrb_trace_rays(h, None, 4, rays.ctypes.data, None, rgb.ctypes.data, None, None) == inv
    assert L.rtrb_intersect_rays(h, C.byref(o), -2, rays.ctypes.data, hits.ctypes.data) == inv
    assert L.rtrb_intersect_rays(h, C.byref(o), 4, rays.ctypes.data, None) == inv
    bad = make_ray_opts(precision=7)
    assert L.rtrb_trace_rays(h, C.byref(bad), 4, rays.ctypes.data, None, rgb.ctypes.data, None, None) == inv
    assert L.rtrb_intersect_rays(h, C.byref(bad), 4, rays.ctypes.data, hits.ctypes.data) == inv
    for depth, mc in ((43, 2), (1 << 30, 1)):  # 43 * 3 + 1 = 130 > 128; 2^30 * 2 + 1 does not fit in 32 bits
        deep = make_ray_opts(trace_depth=depth, mc=mc)
        assert L.rtrb_trace_rays(h, C.byref(deep), 4, rays.ctypes.data, None, rgb.ctypes.data, None, None) == uns
    assert L.rtrb_trace_rays(h, C.byref(make_ray_opts(trace_depth=-1)), 4, rays.ctypes.data, None, rgb.ctypes.data, None, None) == inv
    # device_buffers = 1 with host memory
    dv = make_ray_opts(device_buffers=True)
    assert L.rtrb_trace_rays(h, C.byref(dv), 4, rays.ctypes.data, None, rgb.ctypes.data, None, None) == inv
    assert L.rtrb_intersect_rays(h, C.byref(dv), 4, rays.ctypes.data, hits.ctypes.data) == inv
    d = cam.camera_desc()
    out, keys = np.zeros((96 * 54 * 2, 6)), np.zeros((96 * 54 * 2, 2), np.uint32)
    assert L.rtrb_camera_rays(h, C.byref(d), C.byref(dv), 0, 1, out.ctypes.data, keys.ctypes.data) == inv
    for win in ((0, 0, 97, 54), (-1, 0, 10, 10), (5, 5, 5, 9), (0, 50, 10, 55)):
        assert L.rtrb_camera_rays(h, C.byref(d), C.byref(make_ray_opts(window=win)), 0, 1, out.ctypes.data, None) == inv
    for b, e in ((0, 0), (3, 2), (-1, 1)):
        assert L.rtrb_camera_rays(h, C.byref(d), C.byref(o), b, e, out.ctypes.data, None) == inv
    assert L.rtrb_camera_rays(h, C.byref(d), C.byref(o), 0, 1, None, None) == inv
    assert L.rtrb_trace_rays(h, C.byref(o), 0, None, None, None, None, C.byref(st)) == _abi.RTRB_OK
    assert L.rtrb_intersect_rays(h, C.byref(o), 0, None, None) == _abi.RTRB_OK
    # rays that raise: zero and NaN directions (Vec3#normalize / #cos on a zero vector), outputs still written
    raising = np.array([[0, 0, 0, 2.0, -0.001, 0.0], [0, 0, 0, 0, 0, 0], [0, 0.001, 0, 2.0, -0.001, 0.0], [0, 0, 0, 0, 0, 0]])
    for prec in (PREC_STRICT, PREC_FAST64):
        rgb2, hit2, st2, code = r.trace_rays(raising, 2, 0, precision=prec)
        assert code == _abi.RTRB_ERR_RAISED and st2["status"] & _abi.ST_ZERO_VECTOR
        assert (st2["first_bad_x"], st2["first_bad_y"]) == (1, 0)
        clean_rgb, clean_hit, _, clean_code = r.trace_rays(raising[[0, 2]], 2, 0, precision=prec,
                                                           keys=np.array([[0, 0], [2, 0]], np.uint32))
        assert clean_code == _abi.RTRB_OK
        assert rgb2[[0, 2]].tobytes() == clean_rgb.tobytes() and np.array_equal(hit2[[0, 2]], clean_hit)
