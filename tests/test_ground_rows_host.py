"""Host checks of the ground certificates of the depth-1 linear-filter kernels (rtrb_ground_rows in
raytracing_rb_b200/csrc/rtrb_cull_tables.h).  A ground tile whose camera candidate mask is empty sends its camera rays
straight to the exact test of the scene's one plane, so for every pixel of every certified tile the kernels' own FP32
filter must send that plane to the exact test, or frames, hit ids or counters would change.

The builder is compiled with g++ from tests/ground_rows_harness.cpp into a temporary directory.  For every pixel of a
certified tile the test forms the primary ray as lens_ray does (FP64) and the kernels' FP32 cull ray, and evaluates
classify_plane in FP32: it must not reject the plane, and its lo must not exceed max_distance_f.  rcp.approx /
rsqrt.approx are taken at both ends of a 2^-21 relative error band."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np
import pytest

from test_tile_rows_host import APPROX, EPS, LIGHT, Frame, cull_dirs, f32, fma, light_record, plane_record

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
SOURCES = (os.path.join(HERE, "ground_rows_harness.cpp"), os.path.join(ROOT, "raytracing_rb_b200", "csrc", "rtrb_cull_tables.h"))
COLS = 128


@pytest.fixture(scope="module")
def G():
    h = hashlib.sha256(b"".join(open(p, "rb").read() for p in SOURCES)).hexdigest()[:16]
    so = os.path.join(tempfile.gettempdir(), "rtrb_ground_rows_%s_%d.so" % (h, os.getuid()))
    if not os.path.isfile(so):
        tmp = so + ".%d.tmp" % os.getpid()
        subprocess.check_call(["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-o", tmp, SOURCES[0]])
        os.replace(tmp, so)
    L = C.CDLL(so)
    dp = C.POINTER(C.c_double)
    args = [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_float, dp, dp, dp, dp, dp, C.c_double, C.c_double,
            C.c_double, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
    L.rtrb_test_ground_rows.argtypes = args
    L.rtrb_test_ground_rows_seconds.argtypes = [C.c_int] + args
    L.rtrb_test_ground_rows_seconds.restype = C.c_double
    return L


def dp(a):
    return np.ascontiguousarray(a, np.float64).ctypes.data_as(C.POINTER(C.c_double))


def max_distance_f(d):
    return np.nextafter(f32(d), f32(np.inf)) if f32(d) < d else f32(d)


def certify(G, fr, planes, light, max_distance=10000.0, iters=0):
    pl = np.ascontiguousarray(np.concatenate(planes), np.float32)
    lr = np.ascontiguousarray(np.array(light[0] if light else [0] * 5, np.float32))
    tile_rows, rows = np.zeros((COLS, 4), np.uint8), np.zeros((COLS, 2), np.uint8)
    args = (pl.ctypes.data, len(planes), lr.ctypes.data, light[1] if light else 0, 1 if light else 0,
            float(max_distance_f(max_distance)), dp(fr.pos), dp(fr.focal), dp(fr.left), dp(fr.up_n), dp(fr.front), fr.D,
            fr.rw, fr.rh, fr.W, fr.H, tile_rows.ctypes.data, rows.ctypes.data)
    G.rtrb_test_ground_rows(*args)
    sec = G.rtrb_test_ground_rows_seconds(iters, *args) if iters else 0.0
    return tile_rows, rows, sec


def plane_sent_to_exact(a, p, o, d, mdf):
    """classify_plane(...) != 0 and lo <= max_distance_f for every ray of d, rcp.approx at both ends of its band."""
    den = fma(a[2], d[:, 2], fma(a[1], d[:, 1], f32(a[0] * d[:, 0])))
    rx, ry, rz = f32(p[0] - o[0]), f32(p[1] - o[1]), f32(p[2] - o[2])
    num = fma(rz, a[2], fma(ry, a[1], f32(rx * a[0])))
    mo = f32(max(abs(o[0]), abs(o[1]), abs(o[2])))
    e_num = f32(f32(f32(16.0) * EPS) * a[3]) * f32(p[3] + mo)
    e_den = f32(f32(16.0) * EPS) * a[3]
    grazing = ~(np.abs(den) > f32(16.0) * e_den)
    ok = np.ones(len(d), bool)
    with np.errstate(all="ignore"):
        for e in APPROX:
            inv = f32(f32(1.0) / den) * f32(e)
            t = f32(num * inv)
            e_t = f32(f32(f32(e_num + f32(np.abs(t) * e_den)) * np.abs(inv)) * f32(1.1)) + f32(f32(8.0) * EPS) * np.abs(t)
            lo = np.fmax(f32(t - e_t), f32(0.0))
            lo = np.where(np.isnan(lo), f32(0.0), lo)
            ok &= grazing | (~(f32(t + e_t) < f32(0.0)) & (lo <= mdf))
    return ok


def check(G, fr, planes, light, max_distance=10000.0):
    """Every pixel of every certified tile satisfies its certificate.  Returns the number of ground tiles."""
    tile_rows, rows, _ = certify(G, fr, planes, light, max_distance)
    n_ground = 0
    mdf = max_distance_f(max_distance)
    for c in range(min(COLS, (fr.W + 31) // 32)):
        g0, g1 = (int(v) for v in rows[c])
        if g1 <= g0:
            continue
        assert len(planes) == 1
        assert tile_rows[c][2] <= g0 and g1 <= tile_rows[c][3] and g1 <= (fr.H + 31) // 32, (rows[c], tile_rows[c])
        n_ground += g1 - g0
        X, Y = np.meshgrid(np.arange(32 * c, min(32 * c + 32, fr.W)), np.arange(32 * g0, min(32 * g1, fr.H)), indexing="ij")
        fd, o = fr.rays(X.ravel(), Y.ravel())
        for d in cull_dirs(fd):
            bad = ~plane_sent_to_exact(planes[0][:4], planes[0][4:], o, d, mdf)
            assert not bad.any(), "column %d rows %s: plane not sent to the exact test at %s" % (c, rows[c], np.argwhere(bad)[:3])
    return n_ground


GROUND = plane_record((0.0, 0.0, -1.0), (0.0, 0.0, 1.0))


def test_headline_frame_certifies_the_ground(G):
    """Config 2's camera at 1080p: every row below the horizon is ground in every column, and the certificates hold."""
    fr = Frame((0, 0, 0), (1, 0, 0), (0, 0, 1), 1920, 1080)
    n_ground = check(G, fr, [GROUND], LIGHT)
    assert n_ground >= 0.45 * 60 * 34, n_ground
    _, _, sec = certify(G, fr, [GROUND], LIGHT, iters=20000)
    print("ground tiles %d of %d; rtrb_tile_rows + rtrb_ground_rows at 1920x1080: %.2f us per frame"
          % (n_ground, 60 * 34, sec * 1e6))


DOWN = ((0, 0, 0), (1, 0, -0.35), (0, 0, 1))
CASES = {  # camera (pos, front, up), planes, light, max_distance
    "low_light": (DOWN, [GROUND], light_record((-2.0, 3.0, -0.7), 3.0), 10000.0),
    "light_overhead": (DOWN, [GROUND], light_record((4.0, 0.1, 9.0), 3.0), 10000.0),
    "light_in_view": (DOWN, [GROUND], light_record((4.0, 0.0, -0.9), 10.0), 10000.0),
    "tilted_plane": (DOWN, [plane_record((0, 0, -1.2), (0.15, -0.1, 1.0))], LIGHT, 10000.0),
    "two_planes": (DOWN, [GROUND, plane_record((30.0, 0, 0), (-1.0, 0, 0))], LIGHT, 10000.0),
    "below_the_plane": (((0, 0, -3), (1, 0, 0.4), (0, 0, 1)), [GROUND], LIGHT, 10000.0),
    "max_distance_cut": (DOWN, [GROUND], LIGHT, 4.5),
    "rolled": (((0, 0, 0), (1, 0, -0.3), (0, 0.5, 1)), [GROUND], LIGHT, 10000.0),
    "upside_down": (((0, 0, 0), (1, 0, -0.3), (0, 0, -1)), [GROUND], LIGHT, 10000.0),
    "far_horizon": (((0, 0, 40), (1, 0, -0.08), (0, 0, 1)), [GROUND], LIGHT, 10000.0),
    "no_light": (DOWN, [GROUND], None, 10000.0),
}


@pytest.mark.parametrize("case", sorted(CASES))
def test_certified_tiles_hold_for_every_pixel(G, case):
    (pos, front, up), planes, light, md = CASES[case]
    n_ground = check(G, Frame(pos, front, up, 320, 200), planes, light, md)
    if case == "two_planes":
        assert n_ground == 0
    if case in ("low_light", "rolled", "upside_down", "below_the_plane"):
        assert n_ground > 0


def test_fuzzed_cameras(G):
    rng = np.random.default_rng(7)
    for _ in range(24):
        pos = rng.uniform(-3, 3, 3)
        front = rng.normal(size=3)
        up = rng.normal(size=3)
        W, Hh = int(rng.integers(40, 360)), int(rng.integers(40, 260))
        plane = plane_record(tuple(rng.uniform(-2, 2, 3) - np.array([0, 0, 3.0])), tuple(rng.normal(0, 0.3, 3) + np.array([0, 0, 1.0])))
        light = light_record(tuple(rng.uniform(-10, 10, 3)), float(rng.uniform(1, 40)))
        md = float(rng.choice([10000.0, rng.uniform(2, 20)]))
        check(G, Frame(pos, front, up, W, Hh, rw=float(rng.uniform(0.005, 0.02)), rh=float(rng.uniform(0.005, 0.02))),
              [plane], light, md)
