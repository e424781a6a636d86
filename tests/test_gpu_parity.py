"""GPU parity tests proper: the CUDA path (through the C ABI, raytracing_rb_b200/csrc) against the
CPU oracle on the same seeded inputs.  Tiers (BASELINE.json north_star):
  * deterministic configs: 8-bit output within +-1 LSB on >= 99.9% of pixels, max abs diff stated;
  * primary hit ids bit-exact;
  * ray / shadow-query counters exactly equal.
STRICT mode is additionally held to a much tighter bar (float RGB within 1e-12)."""
import numpy as np
import pytest

from helpers_rtrb import compare_u8, load_scene
from raytracing_rb_b200 import PREC_FAST64, PREC_STRICT, make_opts

pytestmark = pytest.mark.gpu

COUNTERS = ("samples", "rays", "shadow_queries", "highlight_hits", "hits", "local_shaded", "lit_lights", "mc_rays",
            "refractions", "texel_fetches", "sphere_tests", "sphere_accepts", "plane_tests", "plane_accepts",
            "cover_sphere", "cover_sphere_full", "cover_sphere_penumbra", "cover_plane", "cover_plane_accepts",
            "adaptive_pixels")


def run_both(oracle_mod, config_id, precision, seed=1, **kw):
    world, cam = load_scene(config_id, **kw)
    ref = oracle_mod.OracleScene(world.to_scene_desc()).render(cam.camera_desc(), make_opts(seed=seed))
    got = cam.render_frame(seed=seed, precision=precision, count_detail=True)
    return ref, got


def check(ref, got, strict):
    frac, maxdiff, ndiff = compare_u8(got.rgba, ref.rgba)
    print("within+-1LSB=%.6f max_abs_diff=%d differing_px=%d" % (frac, maxdiff, ndiff))
    assert frac >= 0.999
    assert np.array_equal(got.hit, ref.hit), "primary hit ids must be bit-exact"
    for k in COUNTERS:
        if strict or k in ("samples", "rays", "shadow_queries", "hits", "highlight_hits", "local_shaded",
                           "lit_lights", "mc_rays", "texel_fetches", "adaptive_pixels"):
            assert got.stats[k] == ref.stats[k], k
    assert got.stats["status"] == ref.stats["status"]
    if strict:
        assert np.abs(got.rgb - ref.rgb).max() <= 1e-12
        assert maxdiff <= 1
    assert (got.rgba[..., 3] == 255).all()


@pytest.mark.parametrize("precision", [PREC_STRICT, PREC_FAST64])
def test_config1_default_scene(oracle_mod, precision):
    ref, got = run_both(oracle_mod, 1, precision)
    check(ref, got, precision == PREC_STRICT)
    assert got.stats["max_stack"] == ref.stats["max_stack"] or precision != PREC_STRICT


@pytest.mark.parametrize("precision", [PREC_STRICT, PREC_FAST64])
def test_config2_full_size_deterministic(oracle_mod, precision):
    ref, got = run_both(oracle_mod, 2, precision)  # 1920x1080
    check(ref, got, precision == PREC_STRICT)


@pytest.mark.parametrize("precision", [PREC_STRICT, PREC_FAST64])
def test_config3_recursion_texture(oracle_mod, precision):
    ref, got = run_both(oracle_mod, 3, precision, width=480, height=270)
    check(ref, got, precision == PREC_STRICT)


@pytest.mark.parametrize("precision", [PREC_STRICT, PREC_FAST64])
def test_config4_soft_shadow_mc(oracle_mod, precision):
    ref, got = run_both(oracle_mod, 4, precision, width=240, height=135)
    check(ref, got, precision == PREC_STRICT)


@pytest.mark.parametrize("precision", [PREC_STRICT, PREC_FAST64])
def test_config5_many_spheres(oracle_mod, precision):
    ref, got = run_both(oracle_mod, 5, precision, width=96, height=54, spp=2)
    check(ref, got, precision == PREC_STRICT)


@pytest.mark.parametrize("config_id,kw", [
    (2, {}),                                    # full 1920x1080
    (3, {}),                                    # full 1920x1080, depth 8, 4 spp, glass + textures
    (4, dict(width=960, height=540)),           # soft shadows + MC rays
    (5, dict(width=480, height=270, spp=4)),    # 1024 spheres
    (6, dict(width=960, height=540)),           # default scene + boxes (linear filter, box bounding spheres)
    (7, dict(width=960, height=540)),           # boxes among 64 spheres (BVH filter), one box without a bound
])
def test_fast64_is_bit_identical_to_strict(config_id, kw):
    """Size-independent property used at BASELINE sizes, where the CPU oracle is too slow: the FP32
    filter + exact refine path must reproduce STRICT bit for bit (float RGB, hit ids, counters)."""
    world, cam = load_scene(config_id, **kw)
    a = cam.render_frame(seed=3, precision=PREC_STRICT, count_detail=True)
    b = cam.render_frame(seed=3, precision=PREC_FAST64, count_detail=True)
    assert np.array_equal(a.rgb, b.rgb)
    assert np.array_equal(a.rgba, b.rgba)
    assert np.array_equal(a.hit, b.hit)
    for k in ("samples", "rays", "shadow_queries", "hits", "highlight_hits", "local_shaded", "lit_lights", "mc_rays",
              "texel_fetches", "adaptive_pixels", "status"):
        assert a.stats[k] == b.stats[k], k
    print("config %d: exact tests per (ray + shadow query) in FAST64 = %.3f; strict %.3f ms, fast %.3f ms" % (
        config_id, b.stats["exact_tests"] / max(1, b.stats["rays"] + b.stats["shadow_queries"]),
        a.stats["trace_ms"], b.stats["trace_ms"]))


def test_window_and_tiles_compose(oracle_mod):
    """A column strip (render_fork's child_work, camera.rb:53-65) and an interleaved tile subset
    reproduce exactly the same pixels as the full frame (counter RNG keyed by pixel)."""
    world, cam = load_scene(3, width=200, height=120)
    full = cam.render_frame(seed=7)
    strip = cam.render_frame(seed=7, window=(50, 0, 100, 120))
    assert np.array_equal(strip.rgba[:, 50:100], full.rgba[:, 50:100])
    assert (strip.hit[:, :50] == -3).all() and (strip.hit[:, 100:] == -3).all()
    r = cam.renderer()
    c = cam.camera_desc()
    acc = np.zeros_like(full.rgba)
    rays = 0
    for rank in range(3):
        f = r.render(c, make_opts(seed=7, tile_rank=rank, tile_world=3))
        mask = f.hit != -3
        acc[mask] = f.rgba[mask]
        rays += f.stats["rays"]
    assert np.array_equal(acc, full.rgba)
    assert rays == full.stats["rays"]


def test_render_at_matches_frame(oracle_mod):
    world, cam = load_scene(1)
    full = cam.render_frame(seed=1)
    for (x, y) in ((0, 0), (96, 54), (191, 107), (130, 60)):
        item = cam.render_at(x, y, seed=1)
        assert item["position"] == [x, cam.height - 1 - y]
        assert item["color"] == [float(v) for v in full.rgb[y, x]]


def test_status_word_color_greater_than_one(oracle_mod):
    from raytracing_rb_b200 import Camera, World, scenes, _abi
    g = scenes.ground()
    g["properties"]["ambient"] = [0.9, 0.9, 0.9]
    w = World({"max_distance": 10000, "soft_shadow_exponent": 2, "lights": [scenes.light([5, -4, 4], 0.0)],
               "world_objects": [g]})
    _, cdoc = scenes.build(2, width=64, height=36)
    cam = Camera(w, cdoc)
    ref = oracle_mod.OracleScene(w.to_scene_desc()).render(cam.camera_desc())
    got = cam.render_frame()
    assert got.raised and got.stats["status"] & _abi.ST_COLOR_GT_1
    assert (got.stats["first_bad_x"], got.stats["first_bad_y"]) == (ref.stats["first_bad_x"], ref.stats["first_bad_y"])
    assert np.array_equal(got.rgba, ref.rgba)
    with pytest.raises(RuntimeError, match="color greater than 1"):
        cam.render_cuda(None)


def test_device_rejects_what_it_cannot_do(oracle_mod):
    from raytracing_rb_b200 import _abi
    from raytracing_rb_b200._lib import RtrbError
    world, cam = load_scene(1)
    with pytest.raises(RtrbError):  # MT stream mode is serial by construction: no tile partition, 32-bit seeds
        cam.renderer().render(cam.camera_desc(), make_opts(rng_mode=_abi.RNG_MT, tile_rank=0, tile_world=2))
    with pytest.raises(RtrbError):
        cam.renderer().render(cam.camera_desc(), make_opts(rng_mode=_abi.RNG_MT, seed=1 << 40))
    c = cam.camera_desc()
    c.trace_depth = 100
    c.monte_carlo_diffusion_times = 4
    with pytest.raises(RtrbError):
        cam.renderer().render(c, make_opts())


def test_multi_gpu_tiles_compose_in_process():
    """rtrb_render_multi: tiles dealt round-robin to every visible GPU, written through peer mappings
    into GPU 0's framebuffer; the composed frame must equal the single-GPU frame bit for bit."""
    from raytracing_rb_b200 import device_count
    n = device_count()
    if n < 2:
        pytest.skip("needs >= 2 GPUs")
    world, cam = load_scene(3, width=640, height=360)
    one = cam.render_frame(gpus=1, seed=5, count_detail=True)
    many = cam.render_frame(gpus=min(n, 8), seed=5, count_detail=True)
    assert np.array_equal(one.rgba, many.rgba)
    assert np.array_equal(one.rgb, many.rgb)
    assert np.array_equal(one.hit, many.hit)
    for k in ("samples", "rays", "shadow_queries", "hits", "texel_fetches"):
        assert one.stats[k] == many.stats[k], k


def test_pipelined_submit_wait_matches_blocking_render():
    """rtrb_submit / rtrb_wait (two frames in flight) must deliver the same bytes and counters as the
    blocking rtrb_render, frame after frame, including when the camera changes between frames."""
    import torch
    world, cam = load_scene(3, width=320, height=180)
    r = cam.renderer()
    cams = []
    for k in range(5):
        c = cam.camera_desc()
        c.position[1] = 0.05 * k
        cams.append(c)
    want = [r.render(c, make_opts(seed=2), want_rgb=False, want_hit=False) for c in cams]
    bufs = [torch.empty((180, 320, 4), dtype=torch.uint8).pin_memory().numpy() for _ in range(2)]
    got, stats, tickets = [], [], []
    for k, c in enumerate(cams):
        tickets.append(r.submit(c, bufs[k & 1], make_opts(seed=2)))
        if k >= 1:
            st, _ = r.wait(tickets[k - 1])
            stats.append(st)
            got.append(bufs[(k - 1) & 1].copy())
    st, _ = r.wait(tickets[-1])
    stats.append(st)
    got.append(bufs[(len(cams) - 1) & 1].copy())
    for k in range(len(cams)):
        assert np.array_equal(got[k], want[k].rgba), k
        assert stats[k]["rays"] == want[k].stats["rays"] and stats[k]["shadow_queries"] == want[k].stats["shadow_queries"]
    assert not np.array_equal(got[0], got[-1])


@pytest.mark.parametrize("precision", [PREC_STRICT, PREC_FAST64])
def test_depth1_with_mc_rays(oracle_mod, precision):
    """trace_depth 1 with Monte-Carlo rays configured: every child is born dead, but the counters
    (mc_rays spawned) and the image must still match the oracle (exercises the depth-1 kernel)."""
    from raytracing_rb_b200 import Camera, World, scenes
    wdoc, cdoc = scenes.build(4, width=160, height=90)
    cdoc["trace_depth"] = 1
    cdoc["pre_sample_times"] = cdoc["max_sample_times"] = 2
    world = World(wdoc)
    cam = Camera(world, cdoc)
    ref = oracle_mod.OracleScene(world.to_scene_desc()).render(cam.camera_desc(), make_opts(seed=9))
    got = cam.render_frame(seed=9, precision=precision, count_detail=True)
    check(ref, got, precision == PREC_STRICT)
    assert got.stats["mc_rays"] == ref.stats["mc_rays"] > 0


BOX_COUNTERS = ("box_tests", "box_accepts", "cover_box", "cover_box_accepts")


@pytest.mark.parametrize("precision", [PREC_STRICT, PREC_FAST64])
@pytest.mark.parametrize("config_id,kw", [(6, {}), (7, dict(width=160, height=90))])
def test_box_scenes(oracle_mod, config_id, kw, precision):
    """SURVEY 8f rank 2: the Box primitive (box.rb) against the oracle - image, primary hit ids (boxes are
    hit), ray counters; STRICT additionally reproduces the per-object test counters."""
    ref, got = run_both(oracle_mod, config_id, precision, **kw)
    check(ref, got, precision == PREC_STRICT)
    world, _ = load_scene(config_id, **kw)
    from raytracing_rb_b200 import Box
    box_ids = [i for i, o in enumerate(world.world_objects) if isinstance(o, Box)]
    assert box_ids and np.isin(got.hit, box_ids).sum() > 0
    if precision == PREC_STRICT:
        for k in BOX_COUNTERS:
            assert got.stats[k] == ref.stats[k] > 0, k


def test_rgb8_frame_is_rgba8_without_alpha():
    """RTRB_FMT_RGB8: the same bytes minus the constant alpha, through the blocking call and through
    rtrb_submit / rtrb_wait."""
    import torch
    from raytracing_rb_b200 import _abi
    world, cam = load_scene(3, width=200, height=120)
    r, c = cam.renderer(), cam.camera_desc()
    a = r.render(c, make_opts(seed=4), want_rgb=False, want_hit=False)
    b = r.render(c, make_opts(seed=4, pixel_format=_abi.FMT_RGB8), want_rgb=False, want_hit=False)
    assert b.rgba.shape == (120, 200, 3)
    assert np.array_equal(a.rgba[..., :3], b.rgba)
    buf = torch.zeros((120, 200, 3), dtype=torch.uint8).pin_memory().numpy()
    st, _ = r.wait(r.submit(c, buf, make_opts(seed=4, pixel_format=_abi.FMT_RGB8)))
    assert np.array_equal(buf, b.rgba) and st["rays"] == a.stats["rays"]
    assert st["device_ms"] == 0.0  # pipelined frames are not timed


def test_peer_push_carries_a_frame_between_renderers():
    """rtrb_peer_push / rtrb_peer_push_join (copy-engine gather): a frame rendered by one renderer lands in
    a frame slot of another renderer's framebuffer (same GPU here; a peer mapping on a multi-GPU box)."""
    world, cam = load_scene(2, width=320, height=180)
    from raytracing_rb_b200 import Renderer
    src, dst = cam.renderer(), Renderer(world.to_scene_desc(), 0)
    c = cam.camera_desc()
    W, H = 320, 180
    want = src.render(c, make_opts(seed=1), want_rgb=False, want_hit=False).rgba
    sp = src.framebuffer_ptr(W, H)
    dp = dst.framebuffer_ptr(W, H * 3)
    src.render_device(c, make_opts(seed=1), want_stats=False)
    src.peer_push(sp, dp + 2 * W * H * 4, W * H * 4)
    src.peer_push_join()
    src.render_device(c, make_opts(seed=1))  # stats => synchronises the stream the join was queued on
    out = np.zeros((H * 3, W, 4), np.uint8)
    dst.framebuffer_download(W, H * 3, out)
    assert np.array_equal(out[2 * H:], want)
    assert not out[:2 * H].any()


def test_render_fork_json_files(tmp_path):
    """Camera#render_fork's intermediate files (camera.rb:53-65) from one GPU frame: strip bounds, item
    order (x outer, y inner), position = [x, H-1-y], colour = render_at's floats."""
    import json
    world, cam = load_scene(2, width=50, height=20)
    frame = cam.render_fork(str(tmp_path / "img.png"), 3, out_dir=str(tmp_path / "out"))
    items = []
    bounds = [int(float(i) / 3 * 50) for i in range(4)]
    for i in range(3):
        data = json.load(open(tmp_path / "out" / ("file_%d.json" % i)))
        assert len(data) == (bounds[i + 1] - bounds[i]) * 20
        assert data[0]["position"] == [bounds[i], 19] and data[1]["position"] == [bounds[i], 18]
        items += data
    assert len(items) == 50 * 20
    for it in items[::37]:
        x, y = it["position"][0], 19 - it["position"][1]
        assert it["color"] == [float(c) for c in frame.rgb[y, x]]
    assert (tmp_path / "img.png").stat().st_size > 100


@pytest.mark.parametrize("config_id,kw,window", [
    (1, {}, None),                                   # default scene: adaptive 3..10 samples + Monte-Carlo rays
    (4, dict(width=96, height=54), None),            # 16 spp, MC rays in every shadow
    (3, dict(width=160, height=90), (40, 0, 80, 90)),  # a render_fork column strip: the stream restarts at its first pixel
])
def test_mt19937_stream_mode_matches_oracle(oracle_mod, config_id, kw, window):
    """SURVEY 8f rank 4: RTRB_RNG_MT on the device - the reference's own random stream (Random.srand(1),
    main.rb:10) consumed in its own order.  Same stream, same order => the frame must equal the oracle's MT
    frame, including which pixels take the adaptive branch and every ray counter."""
    from raytracing_rb_b200 import RNG_MT
    world, cam = load_scene(config_id, **kw)
    opts = make_opts(seed=1, rng_mode=RNG_MT, window=window)
    ref = oracle_mod.OracleScene(world.to_scene_desc()).render(cam.camera_desc(), opts, threads=1)
    got = cam.render_frame(seed=1, rng_mode=RNG_MT, window=window, count_detail=True)
    print("MT fixed point after %d passes" % cam.renderer().last_mt_passes())
    if window:  # compare the strip only: pixels outside it are not rendered by either side
        x0, y0, x1, y1 = window
        for f in (ref, got):
            f.rgba, f.rgb, f.hit = f.rgba[y0:y1, x0:x1], f.rgb[y0:y1, x0:x1], f.hit[y0:y1, x0:x1]
    check(ref, got, True)
    assert got.stats["adaptive_pixels"] == ref.stats["adaptive_pixels"]
    assert got.stats["mc_rays"] == ref.stats["mc_rays"]
    ctr = cam.render_frame(seed=1, window=window)
    if window:
        ctr.rgb = ctr.rgb[y0:y1, x0:x1]
    assert not np.array_equal(ctr.rgb, got.rgb)  # a different stream than the counter RNG


def _tiny_world(objects, lights):
    from raytracing_rb_b200 import World
    return World({"max_distance": 10000, "soft_shadow_exponent": 2, "lights": lights, "world_objects": objects})


@pytest.mark.parametrize("precision", [PREC_STRICT, PREC_FAST64])
@pytest.mark.parametrize("case", ["empty_world", "no_lights", "one_pixel", "ragged_37x19", "max_below_pre", "behind_camera"])
def test_edge_cases_match_oracle(oracle_mod, case, precision):
    """Empty and ragged inputs: no objects, no lights (every hit falls through to the Monte-Carlo branch and emits
    no colour, ray_tracer.rb:124-142), a 1x1 frame, a frame that is not a multiple of the 32-pixel super-tile or
    the 8x4 warp block, max_sample_times < pre_sample_times (empty extra loop, camera.rb:89-93 still rescales),
    and a scene entirely behind the camera."""
    from raytracing_rb_b200 import Camera, scenes
    _, cdoc = scenes.build(3, width=64, height=36)
    objs = [scenes.ground(), scenes.matte("a", (5, 0, -0.3), 0.7, (1, 0.5, 0.3)), scenes.glass("b", (4, 1.2, -0.6), 0.4)]
    lights = [scenes.light([5, -4, 4], 0.8)]
    if case == "empty_world":
        objs = []
    elif case == "no_lights":
        lights = []
        cdoc = dict(cdoc, monte_carlo_diffusion_times=2, trace_depth=3)
    elif case == "one_pixel":
        cdoc = dict(cdoc, width=1, height=1)
    elif case == "ragged_37x19":
        cdoc = dict(cdoc, width=37, height=19)
    elif case == "max_below_pre":
        cdoc = dict(cdoc, pre_sample_times=4, max_sample_times=2, variant_threshold=0.0)
    elif case == "behind_camera":
        objs = [scenes.matte("a", (-5, 0, 0), 1.0, (1, 1, 1))]
    world = _tiny_world(objs, lights)
    cam = Camera(world, cdoc)
    ref = oracle_mod.OracleScene(world.to_scene_desc()).render(cam.camera_desc(), make_opts(seed=11))
    got = cam.render_frame(seed=11, precision=precision, count_detail=True)
    check(ref, got, precision == PREC_STRICT)
    assert got.stats["samples"] == ref.stats["samples"] > 0
    if case == "empty_world":
        assert got.stats["hits"] == 0 and not got.rgba[..., :3].any() and (got.hit == -1).all()
    if case == "no_lights":
        assert got.stats["mc_rays"] == ref.stats["mc_rays"] > 0 and got.stats["local_shaded"] == 0
    if case == "max_below_pre":
        assert got.stats["adaptive_pixels"] == cdoc["width"] * cdoc["height"]  # variance >= 0.0 always


@pytest.mark.parametrize("config_id,kw,spp_hi", [
    (4, dict(width=160, height=90), 512),   # soft shadows, 16 spp, Monte-Carlo diffuse rays
    (3, dict(width=160, height=90), 256),   # depth 8 through the aperture, 4 spp
    (1, {}, 256),                           # reference default scene, adaptive 3..10 spp
])
def test_stochastic_configs_psnr_vs_high_spp_reference(oracle_mod, config_id, kw, spp_hi):
    """BASELINE.json tier 3: the stochastic configs, rendered on the GPU at their configured sample counts, reach
    PSNR >= 40 dB against a high-spp render of the reference algorithm (the CPU oracle, a different seed)."""
    from helpers_rtrb import psnr_u8
    from raytracing_rb_b200 import Camera, World, scenes
    wdoc, cdoc = scenes.build(config_id, **kw)
    world = World(wdoc)
    got = Camera(world, cdoc).render_frame(seed=1, want_rgb=False, want_hit=False)
    hi_doc = dict(cdoc, pre_sample_times=spp_hi, max_sample_times=spp_hi)
    ref = oracle_mod.OracleScene(world.to_scene_desc()).render(Camera(world, hi_doc).camera_desc(), make_opts(seed=7),
                                                              want_rgb=False, want_hit=False)
    p = psnr_u8(got.rgba, ref.rgba)
    print("config %d: PSNR %.2f dB (GPU at configured spp vs oracle at %d spp)" % (config_id, p, spp_hi))
    assert p >= 40.0


def test_more_spheres_than_the_filter_can_index(oracle_mod):
    """The BVH filter packs survivor indices into 16 bits; a scene with more than 65 536 spheres must fall back to
    the reference's own scan instead of truncating indices (latent in round 1: the guard sat at 2^20).  Small
    spheres on a fine grid, so that most primary rays have a survivor with a high index."""
    from raytracing_rb_b200 import Camera, World, scenes
    rs = np.random.RandomState(3)
    n = 66000
    objs = [scenes.ground()]
    gy, gx = np.meshgrid(np.linspace(-8, 8, 250), np.linspace(30, 3, 264))  # far rows first: the near spheres get the high indices
    for k, (x, y) in enumerate(zip(gx.ravel()[:n], gy.ravel()[:n])):
        r = 0.02 + 0.01 * rs.uniform()
        objs.append(scenes.matte("m%d" % k, (float(x), float(y), -1 + r), r, (0.9, 0.5, 0.4)))
    w = World({"max_distance": 10000, "soft_shadow_exponent": 2, "lights": [scenes.light([5, -4, 4], 0.0)],
               "world_objects": objs})
    _, cdoc = scenes.build(2, width=48, height=27)
    cam = Camera(w, dict(cdoc, trace_depth=2))
    ref = oracle_mod.OracleScene(w.to_scene_desc()).render(cam.camera_desc(), make_opts(seed=1))
    got = cam.render_frame(seed=1, precision=PREC_FAST64, count_detail=True)
    assert (got.hit > 65536).sum() > 0, "the test needs primary hits on high-index spheres"
    check(ref, got, False)


@pytest.mark.parametrize("seed", range(8))
def test_lean_scene_kernels_match_the_generic_path(oracle_mod, seed):
    """Scenes with ONE light of radius exactly 0, no textures and soft_shadow_exponent 2 run depth-1 frames on kernels
    compiled without the code such a scene cannot reach (rtrb_trace_fast_d1lean.cu: light loops, pow, texture lookup,
    the penumbra branch of Sphere#cover_area).  They must reproduce STRICT bit for bit and the oracle's frame, also
    with the camera inside a sphere, spheres cut by planes, a glassy plane, 1 and 3 samples per pixel and the adaptive
    pass; a light radius of 1e-300 or a second light must fall back to the generic kernels with the same result."""
    from raytracing_rb_b200 import Camera, World, scenes
    rs = np.random.RandomState(100 + seed)
    objs = [scenes.ground()]
    if seed % 3 == 1:
        w2 = scenes.wall(14)
        for k in ("texture_file_path", "texture_horizontal_scale", "texture_vertical_scale"):
            w2["properties"].pop(k)
        w2["properties"].update(refractive_rate=1.3, refractive_attenuation=[0.2, 0.2, 0.2], diffuse_rate=[0.4, 0.4, 0.4])
        objs.append(w2)
    for k in range(int(rs.randint(0, 20))):
        r = float(rs.uniform(0.1, 1.2))
        c = (float(rs.uniform(1.5, 12)), float(rs.uniform(-5, 5)), float(rs.uniform(-1.2, 1.0)))
        objs.append(scenes.glass("g%d" % k, c, r) if k % 3 == 0 else scenes.matte("m%d" % k, c, r, rs.uniform(0.3, 1, 3)))
    if seed == 5:
        objs.append(scenes.glass("around the camera", (0.2, 0.1, 0.0), 1.5))
    lpos = [float(rs.uniform(2, 9)), float(rs.uniform(-5, 5)), float(rs.uniform(0.5, 6))]
    variants = [("lean", [scenes.light(lpos, 0.0)])]
    if seed == 0:
        variants += [("tiny radius", [scenes.light(lpos, 1e-300)]), ("two lights", [scenes.light(lpos, 0.0), scenes.light([3, 2, 5], 0.0)])]
    _, cdoc = scenes.build(2, width=96, height=54)
    if seed % 2 == 1:
        cdoc = dict(cdoc, pre_sample_times=3, max_sample_times=7, variant_threshold=1e-5, aperture_radius=0.002)
    for label, lights in variants:
        world = World({"max_distance": 10000, "soft_shadow_exponent": 2, "lights": lights, "world_objects": objs})
        cam = Camera(world, cdoc)
        ref = oracle_mod.OracleScene(world.to_scene_desc()).render(cam.camera_desc(), make_opts(seed=seed))
        a = cam.render_frame(seed=seed, precision=PREC_STRICT, count_detail=True)
        b = cam.render_frame(seed=seed, precision=PREC_FAST64, count_detail=True)
        c = cam.render_frame(seed=seed, precision=PREC_FAST64, count_detail=False)
        assert np.array_equal(a.rgb, b.rgb) and np.array_equal(a.rgba, b.rgba) and np.array_equal(a.hit, b.hit), label
        assert np.array_equal(b.rgba, c.rgba) and np.array_equal(b.hit, c.hit), label
        assert ref.stats["status"] == b.stats["status"], label
        frac, maxdiff, ndiff = compare_u8(b.rgba, ref.rgba)
        assert ndiff == 0 and np.array_equal(b.hit, ref.hit), (label, ndiff, maxdiff)
        for k in ("samples", "rays", "shadow_queries", "hits", "local_shaded", "lit_lights", "adaptive_pixels", "status"):
            assert a.stats[k] == b.stats[k] == ref.stats[k], (label, k)
        assert c.stats["rays"] == b.stats["rays"] and c.stats["shadow_queries"] == b.stats["shadow_queries"]
