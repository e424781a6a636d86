"""Host checks of the tile certificates of the depth-1 linear-filter kernels (rtrb_tile_rows in
raytracing_rb_b200/csrc/rtrb_cull_tables.h).  A certified tile skips the plane filter, the highlight filter or (with an
empty candidate mask) the whole trace, so every primary ray of every certified tile must get the outcome the
certificate states from the kernels' own FP32 filters, or frames, hit ids or counters would change.

The builder is compiled with g++ from tests/tile_rows_harness.cpp into a temporary directory.  For every pixel of a
certified tile the test forms the primary ray as lens_ray does (FP64), the kernels' FP32 cull ray, and evaluates
classify_plane and highlight_match_fast in FP32.  Their rcp.approx / rsqrt.approx results are taken at both ends of a
2^-21 relative error band (wider than the documented error), and the claim must hold at both."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
SOURCES = (os.path.join(HERE, "tile_rows_harness.cpp"), os.path.join(ROOT, "raytracing_rb_b200", "csrc", "rtrb_cull_tables.h"))
EPS = np.float32(2.0 ** -24)
APPROX = (1.0 - 2.0 ** -21, 1.0 + 2.0 ** -21)
f32 = np.float32


@pytest.fixture(scope="module")
def H():
    h = hashlib.sha256(b"".join(open(p, "rb").read() for p in SOURCES)).hexdigest()[:16]
    so = os.path.join(tempfile.gettempdir(), "rtrb_tile_rows_%s_%d.so" % (h, os.getuid()))
    if not os.path.isfile(so):
        tmp = so + ".%d.tmp" % os.getpid()
        subprocess.check_call(["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-o", tmp, SOURCES[0]])
        os.replace(tmp, so)
    L = C.CDLL(so)
    dp = C.POINTER(C.c_double)
    args = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int, dp, dp, dp, dp, dp, C.c_double, C.c_double, C.c_double,
            C.c_int, C.c_int, C.c_void_p]
    L.rtrb_test_tile_rows.argtypes = args
    L.rtrb_test_tile_rows_seconds.argtypes = [C.c_int] + args
    L.rtrb_test_tile_rows_seconds.restype = C.c_double
    return L


def normalize(a):
    a = np.asarray(a, np.float64)
    return a / np.sqrt(a[0] * a[0] + a[1] * a[1] + a[2] * a[2])


def fma(a, b, c):
    return f32(np.float64(a) * np.float64(b) + np.float64(c))


def plane_record(point, front):
    """rtrb_api.cu's cull_pl pair: (n, |n|_1 rounded up), (P, |P|_inf rounded up)."""
    n1 = np.nextafter(f32(sum(abs(x) for x in front)), f32(np.inf))
    pm = np.nextafter(f32(max(abs(x) for x in point)), f32(np.inf))
    return np.array([front[0], front[1], front[2], n1, point[0], point[1], point[2], pm], np.float32)


def light_record(pos, angle_deg):
    thr = angle_deg / 180.0 * np.pi
    pm = np.nextafter(f32(max(abs(x) for x in pos)), f32(np.inf))
    c = np.cos(thr)
    return [f32(pos[0]), f32(pos[1]), f32(pos[2]), pm, f32(c * c)], (1 if 1e-4 < thr < 1.5 else 0)


class Frame:
    def __init__(self, pos, front, up, W, Hh, image_distance=0.01714573877962683, focal_distance=0.017, rw=0.016, rh=0.009):
        self.pos, self.front, self.up = (np.asarray(a, np.float64) for a in (pos, front, up))
        self.left = normalize(np.cross(self.up, self.front))
        self.up_n = normalize(self.up)
        front_n = normalize(self.front)
        self.retina_center = self.pos - front_n * image_distance
        od = focal_distance * image_distance / (image_distance - focal_distance)
        self.focal = self.pos + front_n * od
        self.W, self.H, self.D, self.rw, self.rh = W, Hh, image_distance, rw, rh

    def rows(self, L, planes, lights):
        pl = np.ascontiguousarray(np.concatenate(planes) if planes else np.zeros(8, np.float32), np.float32)
        lr = np.ascontiguousarray(np.array([l[0] for l in lights] or [[0] * 5], np.float32))
        md = np.ascontiguousarray(np.array([l[1] for l in lights] or [0], np.int32))
        out = np.zeros((L.rtrb_test_tile_cols(), 4), np.uint8)
        dp = lambda a: np.ascontiguousarray(a, np.float64).ctypes.data_as(C.POINTER(C.c_double))
        self.args = (pl.ctypes.data, len(planes), lr.ctypes.data, md.ctypes.data, len(lights), dp(self.pos), dp(self.focal),
                     dp(self.left), dp(self.up_n), dp(self.front), self.D, self.rw, self.rh, self.W, self.H, out.ctypes.data)
        self.keep = (pl, lr, md, out)
        L.rtrb_test_tile_rows(*self.args)
        return out

    def rays(self, X, Y):
        """lens_ray (pinhole) in FP64, then make_cull_ray's FP32 direction before normalisation and its origin."""
        sx = 2.0 * (X / self.W - 0.5) * self.rw
        sy = 2 * (Y / self.H - 0.5) * self.rh
        rp = (self.retina_center[None, :] + self.left[None, :] * sx[:, None]) + self.up_n[None, :] * sy[:, None]
        rf = self.pos[None, :] - rp
        t = ((self.focal[None, :] - rp) @ self.front) / (rf @ self.front)
        rd = (rp + rf * t[:, None]) - self.pos[None, :]
        return rd.astype(np.float32), self.pos.astype(np.float32)


def cull_dirs(fd):
    """make_cull_ray's unit directions, rsqrt.approx at both ends of its error band."""
    s = fma(fd[:, 2], fd[:, 2], fma(fd[:, 1], fd[:, 1], f32(fd[:, 0] * fd[:, 0])))
    out = []
    for e in APPROX:
        inv = f32(f32(1.0) / np.sqrt(s)) * f32(e)
        out.append((fd * inv[:, None]).astype(np.float32))
    return out


def plane_rejects(a, p, o, d):
    """classify_plane(...) == 0 for every ray of d, rcp.approx at both ends of its band."""
    den = fma(a[2], d[:, 2], fma(a[1], d[:, 1], f32(a[0] * d[:, 0])))
    rx, ry, rz = f32(p[0] - o[0]), f32(p[1] - o[1]), f32(p[2] - o[2])
    num = fma(rz, a[2], fma(ry, a[1], f32(rx * a[0])))
    mo = f32(max(abs(o[0]), abs(o[1]), abs(o[2])))
    e_num = f32(f32(f32(16.0) * EPS) * a[3]) * f32(p[3] + mo)
    e_den = f32(f32(16.0) * EPS) * a[3]
    ok = np.abs(den) > f32(16.0) * e_den
    for e in APPROX:
        inv = f32(f32(1.0) / den) * f32(e)
        t = f32(num * inv)
        e_t = f32(f32(f32(e_num + f32(np.abs(t) * e_den)) * np.abs(inv)) * f32(1.1)) + f32(f32(8.0) * EPS) * np.abs(t)
        ok &= f32(t + e_t) < f32(0.0)
    return ok


def no_highlight(lt, o, d):
    """highlight_match_fast returns false at its FP32 test for every ray of d."""
    (px, py, pz, pmax, cos2), mode = lt
    ax, ay, az = f32(px - o[0]), f32(py - o[1]), f32(pz - o[2])
    ret = fma(az, d[:, 2], fma(ay, d[:, 1], f32(ax * d[:, 0])))
    a2 = fma(az, az, fma(ay, ay, f32(ax * ax)))
    mo = f32(max(abs(o[0]), abs(o[1]), abs(o[2])))
    ea = f32(f32(8.0) * EPS) * f32(pmax + mo)
    ok = np.full(len(d), mode == 1)
    for e in APPROX:
        c2 = f32(f32(ret * ret) * f32(f32(f32(1.0) / a2) * f32(e)))
        rho = f32(8.0) * f32(ea * f32(f32(f32(1.0) / np.sqrt(a2)) * f32(e)) + f32(8.0) * EPS)
        tol = fma(rho, rho, f32(2.0) * rho)
        ok &= (rho < f32(0.25)) & (f32(c2 + tol) < cos2)
    return ok


def check(L, fr, planes, lights):
    """Every pixel of every certified tile satisfies its certificate.  Returns the share of sky tiles in the frame."""
    rows = fr.rows(L, planes, lights)
    W, Hh = fr.W, fr.H
    sky_tiles, tiles = 0, ((W + 31) // 32) * ((Hh + 31) // 32)
    for c in range(min(rows.shape[0], (W + 31) // 32)):
        s0, s1, h0, h1 = (int(v) for v in rows[c])
        for (r0, r1, sky) in ((s0, s1, True), (h0, h1, False)):
            if r1 <= r0:
                continue
            assert r1 <= (Hh + 31) // 32, rows[c]
            if sky:
                sky_tiles += r1 - r0
            xs = np.arange(32 * c, min(32 * c + 32, W))
            ys = np.arange(32 * r0, min(32 * r1, Hh))
            X, Y = np.meshgrid(xs, ys, indexing="ij")
            fd, o = fr.rays(X.ravel(), Y.ravel())
            for d in cull_dirs(fd):
                for lt in lights:
                    bad = ~no_highlight(lt, o, d)
                    assert not bad.any(), "column %d rows %s: highlight not ruled out at %s" % (c, rows[c], np.argwhere(bad)[:3])
                if sky:
                    for pr in planes:
                        bad = ~plane_rejects(pr[:4], pr[4:], o, d)
                        assert not bad.any(), "column %d rows %s: plane kept at %s" % (c, rows[c], np.argwhere(bad)[:3])
    return sky_tiles / tiles


GROUND = plane_record((0.0, 0.0, -1.0), (0.0, 0.0, 1.0))
LIGHT = light_record((5.0, -4.0, 4.0), 3.0)


def test_headline_frame_certifies_the_sky(H):
    """Config 2's camera: the rows above the horizon are sky in every column, and the certificates hold."""
    fr = Frame((0, 0, 0), (1, 0, 0), (0, 0, 1), 1920, 1080)
    share = check(H, fr, [GROUND], [LIGHT])
    assert share > 0.4, share
    n = 20000
    sec = H.rtrb_test_tile_rows_seconds(n, *fr.args)
    print("rtrb_tile_rows at 1920x1080, one plane and one light: %.2f us per frame" % (sec * 1e6))


CAMERAS = [  # (pos, front, up): rolled, upside down, under the ground plane, looking at the light, off-axis and high
    ((0.0, 0.0, 0.0), (1.0, 0.0, 0.0), (0.0, 0.5, 1.0)),
    ((0.0, 0.0, 0.0), (1.0, 0.0, 0.0), (0.0, 0.0, -1.0)),
    ((0.0, 0.0, -3.0), (1.0, 0.0, 0.4), (0.0, 0.0, 1.0)),
    ((0.0, 0.0, 0.0), (5.0, -4.0, 4.0), (0.0, 0.0, 1.0)),
    ((2.0, 3.0, 40.0), (1.0, 1.0, -0.2), (0.1, 0.0, 1.0)),
    ((0.0, 0.0, -0.99), (1.0, 0.0, 0.001), (0.0, 0.0, 1.0)),  # just above the plane, looking along it
]
PLANE_SETS = [
    [],
    [GROUND],
    [GROUND, plane_record((0.0, 0.0, 30.0), (0.0, 0.0, -1.0))],                                 # floor and ceiling
    [GROUND, plane_record((50.0, 0.0, 0.0), (-1.0, 0.2, 0.0)), plane_record((0, 9, 0), (0.3, -1.0, 0.1))],
]
LIGHT_SETS = [[], [LIGHT], [LIGHT, light_record((20.0, 1.0, 0.5), 10.0)], [light_record((5.0, 0.0, 0.0), 0.001)]]


@pytest.mark.parametrize("cam", range(len(CAMERAS)))
@pytest.mark.parametrize("scene", range(len(PLANE_SETS)))
def test_certified_tiles_hold_for_every_pixel(H, cam, scene):
    pos, front, up = CAMERAS[cam]
    fr = Frame(pos, front, up, 320, 200)
    check(H, fr, PLANE_SETS[scene], LIGHT_SETS[(cam + scene) % len(LIGHT_SETS)])


def test_fuzzed_cameras(H):
    rng = np.random.default_rng(5)
    for _ in range(12):
        pos = rng.uniform(-5, 5, 3)
        front = rng.normal(size=3)
        up = rng.normal(size=3)
        W, Hh = int(rng.integers(40, 400)), int(rng.integers(40, 300))
        planes = [plane_record(tuple(rng.uniform(-4, 4, 3)), tuple(rng.normal(size=3))) for _ in range(int(rng.integers(0, 4)))]
        lights = [light_record(tuple(rng.uniform(-20, 20, 3)), float(rng.uniform(1, 40))) for _ in range(int(rng.integers(0, 3)))]
        check(H, Frame(pos, front, up, W, Hh, rw=float(rng.uniform(0.005, 0.02)), rh=float(rng.uniform(0.005, 0.02))), planes,
              lights)


def test_no_certificates_without_bounds(H):
    """Degenerate cameras, a light at the camera, and a light whose filter never decides certify nothing."""
    for fr, lights in ((Frame((0, 0, 0), (0, 0, 0), (0, 0, 1), 64, 64), [LIGHT]),
                       (Frame((0, 0, 0), (1, 0, 0), (0, 0, 1), 64, 64, focal_distance=0.02), [LIGHT]),
                       (Frame((5.0, -4.0, 4.0), (1, 0, 0), (0, 0, 1), 64, 64), [LIGHT]),
                       (Frame((0, 0, 0), (1, 0, 0), (0, 0, 1), 64, 64), [light_record((5.0, 0.0, 0.0), 120.0)])):
        assert not fr.rows(H, [GROUND], lights).any()
