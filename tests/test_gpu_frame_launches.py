"""Kernel launches per call (rtrb_launch_count, which bench.py reports): rtrb_render_device in each way render_at is
finished (in the trace kernel's thread, in its CTA, from the sample buffer), the hit prefill of a windowed frame, and
the passes of a progressive frame."""
import pytest

from raytracing_rb_b200 import Camera, World, make_opts, scenes, PREC_FAST64, PREC_STRICT
from raytracing_rb_b200._lib import lib

pytestmark = pytest.mark.gpu


def camera(config, **overrides):
    """A small camera of config 1 (adaptive 3 / 10 samples, depth 4) or config 2 (depth 1, 1 spp)."""
    w, c = scenes.build(config)
    world = World(w)
    return Camera(world, dict(c, width=64, height=36, **overrides))


def launches(call):
    before = lib().rtrb_launch_count()
    call()
    return lib().rtrb_launch_count() - before


FRAMES = {  # name: (config, camera overrides, options, launches)
    "in_thread": (2, {}, dict(precision=PREC_FAST64), 1),                         # trace
    "in_cta": (1, dict(pre_sample_times=4), dict(precision=PREC_FAST64), 3),      # trace, extra trace, extra resolve
    "sample_buffer": (1, {}, dict(precision=PREC_STRICT), 4),                     # ... and the resolve
    "windowed": (2, {}, dict(precision=PREC_FAST64, window=(5, 3, 40, 30)), 2),  # in_thread + the hit prefill
}


@pytest.mark.parametrize("name", sorted(FRAMES))
def test_render_device_launches(name):
    config, overrides, opts, want = FRAMES[name]
    cam = camera(config, **overrides)
    cd = cam.camera_desc()
    if name in ("in_cta", "sample_buffer"):
        assert cd.max_sample_times > cd.pre_sample_times  # extra samples for the adaptive pixels
    r = cam.renderer()
    o = make_opts(seed=1, **opts)
    r.render_device(cd, o)  # warm-up
    for want_stats in (True, False):
        assert launches(lambda: r.render_device(cd, o, want_stats=want_stats)) == want, (name, want_stats)


@pytest.mark.parametrize("precision", [PREC_STRICT, PREC_FAST64])
@pytest.mark.parametrize("extra", [True, False])
def test_progressive_pass_launches(precision, extra):
    cam = camera(1) if extra else camera(1, max_sample_times=3)
    cd = cam.camera_desc()
    assert (cd.pre_sample_times, cd.max_sample_times > cd.pre_sample_times) == (3, extra)
    r = cam.renderer()
    box = []
    assert launches(lambda: box.append(r.progressive(cd, make_opts(seed=1, precision=precision)))) == 0
    p = box[0]
    try:
        assert launches(lambda: p.pass_to(1)) == 2  # pass, preview resolve
        assert launches(lambda: p.pass_to(2)) == 2
        # final: pass and resolve, then with extra samples the extra trace and extra resolve
        assert launches(lambda: p.pass_to(3)) == (4 if extra else 2)
    finally:
        p.close()
