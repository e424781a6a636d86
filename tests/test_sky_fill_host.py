"""Host checks of the sky-fill layout of depth-1 frames (rtrb_sky_fill in raytracing_rb_b200/csrc/rtrb_cull_tables.h).
The fill CTAs store the tiles of each super-tile row's sky run without tracing, and the trace CTAs find their tile from
the per-row prefix of traced tiles, so every tile of a run must be one the kernels' sky branch would store (inside its
column's sky rows, empty candidate mask), and the kernels' mapping of trace and fill items must reach every tile of the
frame exactly once.

The builder is compiled with g++ from tests/sky_fill_harness.cpp into a temporary directory.  The sky rows come from
rtrb_tile_rows on real cameras (tests/test_tile_rows_host.py); the candidate masks are fuzzed, with adversarial ones that
split a row's sky tiles.  The device mapping (sky_fill_row and its two callers in rtrb_trace.cuh) is restated here."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np
import pytest

from test_tile_rows_host import GROUND, LIGHT, Frame, H, light_record, plane_record  # noqa: F401 (H: fixture)

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
SOURCES = (os.path.join(HERE, "sky_fill_harness.cpp"), os.path.join(ROOT, "raytracing_rb_b200", "csrc", "rtrb_cull_tables.h"))
TX, TY = 128, 80  # RTRB_CAM_TX, RTRB_CAM_TY


@pytest.fixture(scope="module")
def S():
    h = hashlib.sha256(b"".join(open(p, "rb").read() for p in SOURCES)).hexdigest()[:16]
    so = os.path.join(tempfile.gettempdir(), "rtrb_sky_fill_%s_%d.so" % (h, os.getuid()))
    if not os.path.isfile(so):
        tmp = so + ".%d.tmp" % os.getpid()
        subprocess.check_call(["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-o", tmp, SOURCES[0]])
        os.replace(tmp, so)
    L = C.CDLL(so)
    args = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
    L.rtrb_test_sky_fill.argtypes = args
    L.rtrb_test_sky_fill_seconds.argtypes = [C.c_int] + args
    L.rtrb_test_sky_fill_seconds.restype = C.c_double
    return L


def build(S, tx, ty, rows, stx, sty):
    tx, ty = np.ascontiguousarray(tx, np.uint32), np.ascontiguousarray(ty, np.uint32)
    rows = np.ascontiguousarray(rows, np.uint8)
    run = np.zeros((TY, 2), np.uint8)
    before = np.zeros(TY, np.uint16)
    args = (tx.ctypes.data, ty.ctypes.data, rows.ctypes.data, stx, sty, run.ctypes.data, before.ctypes.data)
    n = S.rtrb_test_sky_fill(*args)
    return n, run, before, (tx, ty, rows, run, before, args)


def row(i, sty, before):
    """sky_fill_row: the last row r < sty with before(r) <= i (the kernels' binary search finds the same)."""
    return max(r for r in range(sty) if before(r) <= i)


def device_tiles(n_sky, run, before, stx, sty):
    """The tiles the trace CTAs (decode_traced_pixel) and the fill CTAs (store_sky_tiles) take, in launch order."""
    traced = stx * sty - n_sky
    a, b = run[:, 0].astype(int), run[:, 1].astype(int)
    out = []
    for k in range(traced):
        r = row(k, sty, lambda r: int(before[r]))
        c = k - int(before[r])
        out.append((c if c < a[r] else c + b[r] - a[r], r, "trace"))
    for i in range(n_sky):
        sky_before = lambda r: r * stx - int(before[r])
        r = row(i, sty, sky_before)
        out.append((a[r] + i - sky_before(r), r, "fill"))
    return out


def check(S, tx, ty, rows, stx, sty):
    """Runs are sky tiles with empty masks, and the device mapping enumerates every tile exactly once."""
    n, run, before, _ = build(S, tx, ty, rows, stx, sty)
    if sty > TY or stx * sty > 0xFFFF:
        assert n == 0 and not run.any()
        return n
    for r in range(sty):
        a, b = int(run[r, 0]), int(run[r, 1])
        assert a <= b <= min(stx, TX), (r, a, b)
        for c in range(a, b):
            assert rows[c][0] <= r < rows[c][1], (c, r, rows[c])
            assert tx[c] & ty[r] == 0, (c, r)
    assert not run[sty:].any()
    seen = {}
    for c, r, kind in device_tiles(n, run, before, stx, sty):
        assert 0 <= c < stx and 0 <= r < sty, (c, r, kind)
        assert (c, r) not in seen, (c, r, kind, seen[(c, r)])
        seen[(c, r)] = kind
        assert (kind == "fill") == (run[r, 0] <= c < run[r, 1]), (c, r, kind)
    assert len(seen) == stx * sty
    return n


def masks(rng, kind, sty):
    tx = np.zeros(TX, np.uint32)
    ty = np.zeros(TY, np.uint32)
    if kind == "random":
        tx[:] = rng.integers(0, 2 ** 32, TX, dtype=np.uint64) * (rng.random(TX) < 0.3)
        ty[:] = rng.integers(0, 2 ** 32, TY, dtype=np.uint64) * (rng.random(TY) < 0.3)
    elif kind == "split":  # spheres in some columns of some rows cut those rows' sky tiles in two, unequal parts
        tx[[c for c in range(TX) if c % 9 == 4 or c == 17]] = 1
        ty[[r for r in range(TY) if r % 7 == 3 or r == sty // 3]] = 1
    elif kind == "all":
        tx[:] = 1
        ty[:] = 1
    return tx, ty


CAMERAS = [  # (pos, front, up): config 2's, rolled, upside down, under the plane, looking down at the ground
    ((0.0, 0.0, 0.0), (1.0, 0.0, 0.0), (0.0, 0.0, 1.0)),
    ((0.0, 0.0, 0.0), (1.0, 0.0, 0.0), (0.0, 0.5, 1.0)),
    ((0.0, 0.0, 0.0), (1.0, 0.0, 0.0), (0.0, 0.0, -1.0)),
    ((0.0, 0.0, -3.0), (1.0, 0.0, 0.4), (0.0, 0.0, 1.0)),
    ((0.0, 0.0, 0.0), (-1.0, 0.0, 1.0), (1.0, 0.0, 1.0)),
    ((0.0, 0.0, 0.0), (1.0, 0.0, -1.0), (1.0, 0.0, 1.0)),
]
SIZES = [(1920, 1080), (333, 250), (31, 17), (4096, 2160), (97, 1000), (5000, 300), (64, 3000)]


@pytest.mark.parametrize("kind", ["none", "random", "split", "all"])
@pytest.mark.parametrize("cam", range(len(CAMERAS)))
def test_runs_are_sky_and_tiles_map_once(H, S, cam, kind):
    rng = np.random.default_rng(cam * 7 + len(kind))
    pos, front, up = CAMERAS[cam]
    for W, Hh in SIZES:
        fr = Frame(pos, front, up, W, Hh)
        rows = fr.rows(H, [GROUND], [LIGHT])
        stx, sty = (W + 31) // 32, (Hh + 31) // 32
        tx, ty = masks(rng, kind, sty)
        n = check(S, tx, ty, rows, stx, sty)
        if kind == "all":
            assert n == 0


def test_split_sky_rows_keep_the_longest_run(S):
    stx, sty = 20, 3
    rows = np.zeros((TX, 4), np.uint8)
    rows[:stx, 0], rows[:stx, 1] = 0, 3
    rows[1, 0] = 1  # column 1 is not sky in row 0
    tx, ty = np.zeros(TX, np.uint32), np.zeros(TY, np.uint32)
    tx[[6, 9]] = 1
    ty[[0, 2]] = 1  # rows 0 and 2: columns [0, 6), [7, 9), [10, 20) (row 0 also loses column 1); row 1: all 20
    n, run, _, _ = build(S, tx, ty, rows, stx, sty)
    assert [tuple(run[r]) for r in range(sty)] == [(10, 20), (0, 20), (10, 20)]
    assert n == 10 + 20 + 10
    check(S, tx, ty, rows, stx, sty)


def test_fuzzed_layouts(S):
    """Arbitrary sky rows and masks, including frames past the tables' limits."""
    rng = np.random.default_rng(11)
    for _ in range(300):
        stx, sty = int(rng.integers(1, 140)), int(rng.integers(1, 100))
        rows = np.zeros((TX, 4), np.uint8)
        r0 = rng.integers(0, min(sty, 255) + 1, TX)
        r1 = r0 + rng.integers(0, min(sty, 255) + 1, TX)
        rows[:, 0], rows[:, 1] = r0, np.minimum(r1, min(sty, 255))
        tx, ty = masks(rng, str(rng.choice(["none", "random", "split"])), sty)
        check(S, tx, ty, rows, stx, sty)


def test_host_cost(H, S):
    fr = Frame((0.0, 0.0, 0.0), (1.0, 0.0, 0.0), (0.0, 0.0, 1.0), 1920, 1080)
    rows = fr.rows(H, [GROUND], [LIGHT])
    tx, ty = masks(np.random.default_rng(0), "random", 34)
    _, _, _, keep = build(S, tx, ty, rows, 60, 34)
    sec = S.rtrb_test_sky_fill_seconds(20000, *keep[-1])
    print("rtrb_sky_fill at 1920x1080: %.3f us per frame" % (sec * 1e6))
