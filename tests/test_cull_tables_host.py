"""Host checks of the candidate masks of the depth-1 linear-filter kernels (raytracing_rb_b200/csrc/rtrb_cull_tables.h):
every sphere whose apex test can keep a ray must be in that ray's candidate mask, or the kernels' survivor masks
(and with them counters, status bits and frames) would change.

The builders are compiled with g++ from tests/cull_tables_harness.cpp into a temporary directory.  The apex tables are
built here as rtrb_api.cu's apex_entry builds them; the rays are the pixels' primary rays (lens_ray in FP64, then the
kernels' FP32 normalisation) and dense sets of probe directions from the light.  A sphere counts as kept when the FP64
apex condition holds with a slack of 2^-20: (V . u)^2 >= Kq - 2^-20 |V|^2."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
SOURCES = (os.path.join(HERE, "cull_tables_harness.cpp"), os.path.join(ROOT, "raytracing_rb_b200", "csrc", "rtrb_cull_tables.h"))
SLACK = 2.0 ** -20
EPS = 2.0 ** -24


@pytest.fixture(scope="module")
def H():
    h = hashlib.sha256(b"".join(open(p, "rb").read() for p in SOURCES)).hexdigest()[:16]
    so = os.path.join(tempfile.gettempdir(), "rtrb_cull_tables_%s_%d.so" % (h, os.getuid()))
    if not os.path.isfile(so):
        tmp = so + ".%d.tmp" % os.getpid()
        subprocess.check_call(["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-o", tmp, SOURCES[0]])
        os.replace(tmp, so)
    L = C.CDLL(so)
    dims = (C.c_int * 3)()
    L.rtrb_test_cull_dims(dims)
    L.dims = tuple(dims)
    dp = C.POINTER(C.c_double)
    L.rtrb_test_camera_masks.argtypes = [C.c_void_p, C.c_int, dp, dp, dp, dp, dp, C.c_double, C.c_double, C.c_double,
                                         C.c_int, C.c_int, C.c_void_p, C.c_void_p]
    L.rtrb_test_light_masks.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
    return L


def apex_table(A, rho, centres, radii, m_scale):
    """rtrb_api.cu apex_entry for every sphere: (C - A as float, Kq rounded down; NaN Kq -> -inf)."""
    tab = np.zeros((len(radii), 4), np.float32)
    for k, (c, r) in enumerate(zip(centres, radii)):
        v = np.asarray(c, np.float64) - np.asarray(A, np.float64)
        v2 = float(v[0] * v[0] + v[1] * v[1] + v[2] * v[2])
        vlen = np.sqrt(v2)
        rp = abs(r) + rho + 96.0 * EPS * (m_scale + vlen) + 8.0 * EPS * vlen
        kq = v2 - (rp * rp + 32.0 * EPS * v2)
        with np.errstate(over="ignore", invalid="ignore"):
            kf = np.float32(kq)
        if float(kf) > kq:
            kf = np.nextafter(kf, np.float32(-np.inf))
        if kq != kq:
            kf = np.float32(-np.inf)
        tab[k] = (np.float32(v[0]), np.float32(v[1]), np.float32(v[2]), kf)
    return tab


def kept(tab, u):
    """[rays, spheres] bool: the FP64 apex condition with slack, u = the kernels' FP32 unit directions [rays, 3]."""
    u = u.astype(np.float64)
    with np.errstate(invalid="ignore", over="ignore"):
        uh = u / np.linalg.norm(u, axis=1, keepdims=True)
        V = tab[:, :3].astype(np.float64)
        b = uh @ V.T
        kq = tab[:, 3].astype(np.float64)
        keep = ~(b * b < kq[None, :] - SLACK * (V * V).sum(1)[None, :])  # NaN keeps, like the kernels' test
    return keep


def f32_unit(d):
    f = d.astype(np.float32)
    with np.errstate(divide="ignore", invalid="ignore"):
        inv = np.float32(1.0) / np.sqrt((f * f).sum(1, dtype=np.float32))
    return f * inv[:, None]


def normalize(a):
    a = np.asarray(a, np.float64)
    return a / np.sqrt(a[0] * a[0] + a[1] * a[1] + a[2] * a[2])


def camera_case(H, centres, radii, pos, front, up, W, Hh, image_distance=1.0, focal_distance=0.5, rw=0.8, rh=0.45):
    pos, front, up = (np.asarray(a, np.float64) for a in (pos, front, up))
    left = normalize(np.cross(up, front))
    front_n, up_n = normalize(front), normalize(up)
    retina_center = pos - front_n * image_distance
    od = focal_distance * image_distance / (image_distance - focal_distance)
    focal = pos + front_n * od
    n = len(radii)
    m_scene = max([np.float32(max(abs(c[0]), abs(c[1]), abs(c[2])) + abs(r)) for c, r in zip(centres, radii)] + [0.0])
    cm = max(abs(pos[0]), abs(pos[1]), abs(pos[2]))
    tab = apex_table(pos, 0.0, centres, radii, float(m_scene) + cm) if n else np.zeros((0, 4), np.float32)
    ntx, nty, _ = H.dims
    tx, ty = np.zeros(ntx, np.uint32), np.zeros(nty, np.uint32)
    dp = lambda a: np.ascontiguousarray(a, np.float64).ctypes.data_as(C.POINTER(C.c_double))
    H.rtrb_test_camera_masks(np.ascontiguousarray(tab).ctypes.data if n else None, n, dp(pos), dp(focal), dp(left), dp(up_n),
                             dp(front), image_distance, rw, rh, W, Hh, tx.ctypes.data, ty.ctypes.data)
    # every pixel's primary ray, as lens_ray forms it (pinhole)
    xs = 2.0 * (np.arange(W) / W - 0.5) * rw
    ys = 2 * (np.arange(Hh) / Hh - 0.5) * rh
    X, Y = np.meshgrid(np.arange(W), np.arange(Hh), indexing="ij")
    sx, sy = xs[X.ravel()], ys[Y.ravel()]
    rp = (retina_center[None, :] + left[None, :] * sx[:, None]) + up_n[None, :] * sy[:, None]
    rf = pos[None, :] - rp
    t = ((focal[None, :] - rp) @ front) / (rf @ front)
    target = rp + rf * t[:, None]
    rd = target - pos[None, :]
    if n == 0:
        assert not tx.any() and not ty.any()
        return 0
    keep = kept(tab, f32_unit(rd))
    cand = tx[np.minimum(X.ravel() >> 5, ntx - 1)] & ty[np.minimum(Y.ravel() >> 5, nty - 1)]
    bits = (cand[:, None] >> np.arange(n, dtype=np.uint32)[None, :]) & 1
    missing = keep & (bits == 0)
    assert not missing.any(), "pixels %s miss spheres %s" % (np.argwhere(missing)[:5, 0], np.argwhere(missing)[:5, 1])
    if n < 32:
        assert not (cand >> np.uint32(n)).any(), "bits beyond the spheres"
    return float(np.unpackbits(cand.view(np.uint8)).sum()) / len(cand)


def light_case(H, centres, radii, L, rng, extra_dirs=None):
    n = len(radii)
    tab = apex_table(L, 0.0, centres, radii, 10.0 + max(abs(x) for x in L)) if n else np.zeros((0, 4), np.float32)
    _, _, N = H.dims
    m = np.zeros((3, 2, N), np.uint32)
    H.rtrb_test_light_masks(np.ascontiguousarray(tab).ctypes.data if n else None, n, m.ctypes.data)
    if n == 0:
        assert not m.any()
        return 0
    dirs = [rng.normal(size=(40000, 3))]
    for k in range(n):  # directions aimed at and just around each sphere, both ways along the line
        v = tab[k, :3].astype(np.float64)
        off = rng.normal(size=(3000, 3)) * (abs(radii[k]) * rng.uniform(0.0, 1.3, size=(3000, 1)))
        dirs += [v[None, :] + off, -(v[None, :] + off)]
    # cube-edge directions: two components of equal magnitude
    e = rng.normal(size=(6000, 3))
    e[:, 1] = np.sign(e[:, 1]) * np.abs(e[:, 0])
    e[2000:4000, 2] = np.sign(e[2000:4000, 2]) * np.abs(e[2000:4000, 0])
    dirs.append(e)
    if extra_dirs is not None:
        dirs.append(extra_dirs)
    u = f32_unit(np.concatenate(dirs))
    keep = kept(tab, u)
    # the kernels' bin lookup (light_survivors_of), in FP32
    ax, ay, az = np.abs(u[:, 0]), np.abs(u[:, 1]), np.abs(u[:, 2])
    a = np.where((ax >= ay) & (ax >= az), 0, np.where(ay >= az, 1, 2))
    idx = np.arange(len(u))
    wa, wb, wc = u[idx, a], u[idx, (a + 1) % 3], u[idx, (a + 2) % 3]
    with np.errstate(divide="ignore", invalid="ignore"):
        inv = np.float32(1.0) / wa
        s, t = wb * inv, wc * inv
        ok = (np.abs(s) <= 2) & (np.abs(t) <= 2)
        i = np.clip(np.where(ok, ((s + np.float32(1)) * np.float32(N / 2)), 0).astype(np.int64), 0, N - 1)
        j = np.clip(np.where(ok, ((t + np.float32(1)) * np.float32(N / 2)), 0).astype(np.int64), 0, N - 1)
    cand = np.where(ok, m[a, 0, i] & m[a, 1, j], np.uint32(0xffffffff))
    bits = (cand[:, None] >> np.arange(n, dtype=np.uint32)[None, :]) & 1
    missing = keep & (bits == 0)
    assert not missing.any(), "directions %s miss spheres %s" % (u[np.argwhere(missing)[:3, 0]], np.argwhere(missing)[:3, 1])
    return int(keep.sum())


def random_spheres(rng, n, spread=6.0, rmin=0.1, rmax=1.5):
    return [tuple(rng.uniform(-spread, spread, 3)) for _ in range(n)], list(rng.uniform(rmin, rmax, n))


CAMERAS = [  # (pos, front, up)
    ((0.0, 1.0, -8.0), (0.0, 0.0, 1.0), (0.0, 1.0, 0.0)),
    ((3.0, 2.0, 5.0), (-0.3, -0.2, -1.0), (0.0, 1.0, 0.0)),        # up not perpendicular to front
    ((0.5, 0.5, 0.5), (1.0, 0.3, 0.2), (0.3, 1.0, -0.4)),          # inside the sphere cloud: spheres behind and around
    ((0.0, 0.0, 0.0), (0.0, -1.0, 0.01), (0.0, 0.0, 1.0)),
]


@pytest.mark.parametrize("n", [0, 1, 5, 16, 32])
@pytest.mark.parametrize("cam", range(len(CAMERAS)))
def test_camera_masks_hold_every_kept_sphere(H, n, cam):
    rng = np.random.default_rng(100 * n + cam)
    centres, radii = random_spheres(rng, n)
    pos, front, up = CAMERAS[cam]
    camera_case(H, centres, radii, pos, front, up, 192, 108)


def test_camera_masks_enclosing_and_behind(H):
    pos, front, up = CAMERAS[0]
    centres = [pos, (0.0, 1.0, -12.0), (0.0, 1.0, -8.5), (5.0, 1.0, -8.0), (0.0, 1.0, 20.0), (0.3, 1.2, -7.0)]
    radii = [2.0, 1.0, 0.4, 1.0, 3.0, 0.2]  # around the camera, behind it, just behind, beside, ahead, near
    camera_case(H, centres, radii, pos, front, up, 160, 90)
    camera_case(H, centres, radii, pos, front, up, 160, 90, image_distance=-1.0)
    camera_case(H, centres, radii, pos, front, up, 160, 90, rw=-0.8)


@pytest.mark.parametrize("W,Hh", [(4400, 24), (24, 2700)])
def test_camera_masks_frames_over_the_cap(H, W, Hh):
    rng = np.random.default_rng(W + Hh)
    centres, radii = random_spheres(rng, 12)
    pos, front, up = CAMERAS[0]
    camera_case(H, centres, radii, pos, front, up, W, Hh)


def test_camera_masks_are_tight_on_the_headline_scene(H):
    """Config 2's frame: the masks must actually cull (most tiles need a few spheres, not all 16)."""
    from raytracing_rb_b200 import _abi
    from helpers_rtrb import load_scene
    world, cam = load_scene(2)
    desc = world.to_scene_desc().desc
    sph = [(tuple(o.point), o.radius) for o in (desc.objects[i] for i in range(desc.n_objects)) if o.type == _abi.OBJ_SPHERE]
    assert len(sph) == 16
    c = cam.camera_desc()
    mean_cand = camera_case(H, [s[0] for s in sph], [s[1] for s in sph], tuple(c.position), tuple(c.front), tuple(c.up), c.width,
                         c.height, c.image_distance, c.focal_distance, c.retina_width, c.retina_height)
    assert mean_cand < 1.0, mean_cand


@pytest.mark.parametrize("n", [0, 1, 7, 16, 32])
def test_light_masks_hold_every_kept_sphere(H, n):
    rng = np.random.default_rng(7 + n)
    centres, radii = random_spheres(rng, n)
    light_case(H, centres, radii, (0.3, 8.0, -2.0), rng)


def test_light_masks_light_inside_on_and_across_faces(H):
    rng = np.random.default_rng(3)
    L = (1.0, 2.0, 3.0)
    centres = [L, (1.0, 2.0 + 0.5, 3.0), (4.0, 5.0, 6.0), (4.0, -1.0, 6.0), (-2.0, 5.0, 0.0), (1.0, 2.0, 9.0), (5.0, 2.0, 3.0)]
    radii = [0.5, 0.5, 1.0, 1.0, 1.0, 2.5, 0.01]  # enclosing the light, light on its surface, on cube edges / corners
    light_case(H, centres, radii, L, rng)


def test_light_masks_are_tight(H):
    rng = np.random.default_rng(11)
    centres, radii = random_spheres(rng, 16, rmax=0.6)
    tab = apex_table((0.0, 20.0, 0.0), 0.0, centres, radii, 30.0)
    _, _, N = H.dims
    m = np.zeros((3, 2, N), np.uint32)
    H.rtrb_test_light_masks(np.ascontiguousarray(tab).ctypes.data, 16, m.ctypes.data)
    pop = np.vectorize(lambda v: bin(int(v)).count("1"))(m[1])
    assert pop.mean() < 6, pop  # the light looks down on the cloud along +-y
