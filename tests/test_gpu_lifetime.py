"""Renderer teardown: renderers created, used and destroyed over and over must give back all of their device memory.
Each round goes through every call that allocates: the framebuffers and caches of a windowed frame, the pipeline
slots of submit / submit_png, the PNG encoder's scratch, the ray calls' control block, staging buffer and lens table,
and the RTRB_RNG_MT draw stream."""
import pytest

from raytracing_rb_b200 import Camera, Renderer, World, _abi, make_opts, png_max_bytes, scenes

pytestmark = pytest.mark.gpu

ROUNDS = 10
MARGIN = 64 << 20  # bytes of free device memory a round trip may cost (allocator granularity); see the footprint check


def use_renderer(world, cam, bufs, close=True):
    r = Renderer(world.to_scene_desc(), 0)
    cd = cam.camera_desc()
    W, H = cd.width, cd.height
    fr = r.render(cd, make_opts(seed=3, window=(40, 24, W - 40, H - 24)))
    assert fr.hit[0, 0] == -3 and fr.hit[H // 2, W // 2] != -3
    stats, code = r.wait(r.submit(cd, bufs["rgba"], make_opts(seed=3)))
    assert code == _abi.RTRB_OK and stats["samples"] == W * H
    png, _, code = r.wait_png(r.submit_png(cd, bufs["png"], make_opts(seed=3, pixel_format=_abi.FMT_RGB8)))
    assert code == _abi.RTRB_OK and png[:8] == b"\x89PNG\r\n\x1a\n"
    assert r.encode_png(W, H, _abi.FMT_RGBA8)[:8] == png[:8]
    rays, keys = r.camera_rays(cd, seed=3)
    rgb, hit, stats, _ = r.trace_rays(rays, keys=keys)
    assert rgb.shape == (W * H, 3) and stats["samples"] == W * H
    assert len(r.intersect_rays(rays)) == W * H
    r.render(cd, make_opts(seed=3, rng_mode=_abi.RNG_MT, window=(0, 0, 16, 16)), want_rgb=False, want_hit=False)
    assert r.last_mt_passes() >= 1
    if not close:
        return r
    r.close()


def test_destroyed_renderers_give_back_their_device_memory():
    import torch
    wdoc, cdoc = scenes.build(2)
    world = World(wdoc)
    cam = Camera(world, cdoc)
    bufs = {"rgba": torch.zeros((cam.height, cam.width, 4), dtype=torch.uint8).pin_memory().numpy(),
            "png": torch.zeros(png_max_bytes(cam.width, cam.height), dtype=torch.uint8).pin_memory().numpy()}
    use_renderer(world, cam, bufs)  # warm-up: context, modules and driver pools
    free_start = torch.cuda.mem_get_info(0)[0]
    r = use_renderer(world, cam, bufs, close=False)
    footprint = free_start - torch.cuda.mem_get_info(0)[0]
    r.close()
    for _ in range(ROUNDS - 1):
        use_renderer(world, cam, bufs)
    leaked = free_start - torch.cuda.mem_get_info(0)[0]
    print("renderer footprint %.1f MB, free memory lost over %d rounds %.1f MB" % (footprint / 2**20, ROUNDS,
                                                                                  leaked / 2**20))
    assert footprint > 4 * MARGIN  # the margin is far below what one leaked renderer would cost
    assert leaked < MARGIN
