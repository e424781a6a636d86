"""bench.py's contract pieces that need no GPU: both arms describe the workload with the SAME `config` object
(VERDICT r1: the driver's `same_config` check), the reference arm runs here on the host cores and prints one JSON line
with every key the contract names, and the helper that names the dispatched kernel instantiation follows
rtrb_trace_fast.cu's dispatch."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402


def test_config_record_is_the_workload_only_and_identical_for_both_arms():
    world, cdoc, name = bench.workload(2)
    a = bench.config_record(name, cdoc)
    b = bench.config_record(name, dict(cdoc))
    assert a == b and set(a) >= {"workload", "width", "height", "pre_sample_times", "trace_depth", "rng", "l2"}
    assert (a["width"], a["height"], a["pre_sample_times"], a["trace_depth"]) == (1920, 1080, 1, 1)
    assert not any(k in a for k in ("model", "global_batch", "seq_len"))  # no ML vocabulary in `config`


def test_kernel_name_follows_the_dispatch():
    from raytracing_rb_b200 import Camera
    for cid, klass, want in ((2, "lean", "rtrb_fast_lean::trace_pre_fast_kernel<1,false,false>"),
                             (1, "one_light", "rtrb_fast_l1::trace_pre_tree_kernel<10,false,false>"),
                             (3, "one_light", "rtrb_fast_l1n::trace_pre_tree_kernel<10,false,false>"),
                             (4, "one_light", "rtrb_fast_l1::trace_pre_tree_kernel<10,false,false>"),
                             (5, "one_light", "rtrb_fast_l1n::trace_pre_tree_kernel<10,false,true>")):
        world, cdoc, _ = bench.workload(cid)
        cd = Camera(world, cdoc).camera_desc()
        n_sph = sum(1 for o in world.world_objects if type(o).__name__ in ("Sphere", "Box"))
        assert bench.scene_class(world) == klass
        assert bench.kernel_name(cd, n_sph, klass) == want


def test_kernel_names_exist_in_the_library():
    """Every name bench.kernel_name gives for configs 1-5, with the linear filter and with the BVH, is a kernel of the
    built library (bench.py reports it as the kernel that ran)."""
    import re
    import shutil
    from raytracing_rb_b200 import Camera, _lib
    if not os.path.exists(_lib.LIB_PATH) or shutil.which("cuobjdump") is None:
        pytest.skip("needs the built library and cuobjdump")
    out = subprocess.run(["cuobjdump", "-res-usage", _lib.LIB_PATH], capture_output=True, text=True, check=True).stdout
    functions = set(re.findall(r"Function (\S+):", out))
    for cid in range(1, 6):
        world, cdoc, _ = bench.workload(cid)
        cd = Camera(world, cdoc).camera_desc()
        for n_sph in (0, 33):  # linear filter, BVH
            name = bench.kernel_name(cd, n_sph, bench.scene_class(world))
            ns, fn, cap, detail, bvh = re.fullmatch(r"(\w+)::(\w+)<(\d+),(true|false),(true|false)>", name).groups()
            mangled = "_ZN%d%s%d%sILi%sELb%dELb%dEEEv11FrameParams" % (len(ns), ns, len(fn), fn, cap, detail == "true",
                                                                        bvh == "true")
            assert mangled in functions, name


def test_cpu_window_is_a_centred_full_height_strip():
    assert bench.cpu_window(1920, 1080, 1.0, 16) == (0, 0, 1920, 1080)
    assert bench.cpu_window(1920, 1080, 0.25, 16) == (720, 0, 1200, 1080)
    assert bench.cpu_window(3840, 2160, 8.0 / 3840.0, 16) == (1916, 0, 1924, 2160)
    assert bench.cpu_window(192, 108, 0.0, 8) == (95, 0, 96, 108)  # never empty


def test_algorithmic_flops_uses_the_survey_constants():
    s = dict.fromkeys(("rays", "sphere_tests", "sphere_accepts", "plane_tests", "plane_accepts", "hits", "lit_lights",
                       "local_shaded", "texel_fetches", "shadow_queries", "cover_sphere", "cover_sphere_full",
                       "cover_sphere_penumbra", "cover_plane", "cover_plane_accepts", "samples"), 0)
    s.update(rays=1, sphere_tests=16, sphere_accepts=1, plane_tests=1, plane_accepts=1, hits=1, samples=1)
    # SURVEY 8d: 7 + 15*20 + 44 + 29 + (82 + 2) + (60 + 2)
    assert bench.algorithmic_flops(s) == 7 + 15 * 20 + 44 + 29 + 84 + 62


def test_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference` on a small workload: rank 0 prints ONE JSON line (impl, metric, unit, value, config,
    cpu_baseline with kind/cores/sample, e2e with zero copy bytes); another rank prints nothing and exits 0."""
    env = dict(os.environ, RANK="0", WORLD_SIZE="1")
    out = subprocess.check_output([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--config", "1",
                                   "--steps", "2", "--warmup", "1"], env=env, cwd=ROOT, timeout=300).decode()
    lines = [l for l in out.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "Mrays/s" and d["unit"] == "Mrays/s" and d["higher_is_better"] is True
    assert d["steps"] == 2 and d["warmup"] == 1 and d["value"] > 0 and d["dtype"] == "f64" and d["vs_baseline"] is None
    world, cdoc, name = bench.workload(1)
    assert d["config"] == bench.config_record(name, cdoc)          # what the GPU arm prints for the same --config
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["run"]["frames_rendered_per_step"] == 1.0
    env["RANK"], env["WORLD_SIZE"] = "1", "2"
    out = subprocess.check_output([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--config", "1",
                                   "--steps", "1", "--warmup", "0"], env=env, cwd=ROOT, timeout=120).decode()
    assert out.strip() == ""


def test_dump_outputs_writes_the_last_step_frames(tmp_path):
    """`--dump-outputs DIR` (reference arm here): float32 pixel values of the last timed step's frame with their
    (frame, y, x), at most 64 MB, identical from run to run with the same arguments."""
    from raytracing_rb_b200 import Camera, make_opts
    from oracle import oracle
    dumps = []
    for k in range(2):
        out = tmp_path / ("d%d" % k)
        subprocess.check_call([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--config", "1",
                               "--steps", "1", "--warmup", "0", "--cpu-fraction", "0.25", "--dump-outputs", str(out)],
                              cwd=ROOT, timeout=300, stdout=subprocess.DEVNULL)
        dumps.append({n: np.load(out / (n + ".npy")) for n in ("frames_sample", "frames_sample_index")})
        assert sum(f.stat().st_size for f in out.iterdir()) <= 64 << 20
    for d in dumps:
        assert all(a.dtype == np.float32 for a in d.values())
        assert np.array_equal(d["frames_sample"], dumps[0]["frames_sample"])
        assert np.array_equal(d["frames_sample_index"], dumps[0]["frames_sample_index"])
    world, cdoc, _ = bench.workload(1)
    cd = Camera(world, cdoc).camera_desc()
    win = bench.cpu_window(cd.width, cd.height, 0.25, 1)
    want = oracle.OracleScene(world.to_scene_desc()).render(cd, make_opts(seed=1, window=win)).rgba
    vals, where = dumps[0]["frames_sample"], dumps[0]["frames_sample_index"].astype(np.int64)
    assert vals.shape == (cd.height * (win[2] - win[0]), 3) and (where[:, 0] == 0).all()
    assert where[:, 2].min() == win[0] and where[:, 2].max() == win[2] - 1  # x in the full frame
    assert np.array_equal(vals, want[where[:, 1], where[:, 2], :3].astype(np.float32))


@pytest.mark.gpu
@pytest.mark.parametrize("pixel_format", ["rgb8", "rgba8"])
def test_gpu_arm_dump_outputs_are_the_frames_of_the_last_step(tmp_path, pixel_format):
    """`--dump-outputs DIR` on the CUDA arm: the frame slots read back after the timed steps, cut to each frame's
    bytes in either pixel format, must give the pixels a direct render of the same batch cameras gives."""
    from raytracing_rb_b200 import PREC_FAST64, Renderer, _abi, make_opts
    B = 3
    subprocess.check_call([sys.executable, os.path.join(ROOT, "bench.py"), "--small", "--steps", "2", "--warmup", "1",
                           "--frames-per-step", str(B), "--pixel-format", pixel_format, "--headline-only",
                           "--sustained-seconds", "0", "--dump-outputs", str(tmp_path)],
                          cwd=ROOT, timeout=600, stdout=subprocess.DEVNULL)
    vals = np.load(tmp_path / "frames_sample.npy")
    where = np.load(tmp_path / "frames_sample_index.npy").astype(np.int64)
    world, cdoc, _ = bench.workload(2, small=True)
    cams = bench.batch_cameras(world, cdoc, B)
    W, H = cams[0].width, cams[0].height
    assert vals.dtype == np.float32 and vals.shape == (B * H * W, 3)  # small enough to be dumped whole
    r = Renderer(world.to_scene_desc(), 0)
    fmt = _abi.FMT_RGB8 if pixel_format == "rgb8" else _abi.FMT_RGBA8
    for f in range(B):
        want = r.render(cams[f], make_opts(seed=1, precision=PREC_FAST64, pixel_format=fmt),
                        want_rgb=False, want_hit=False).rgba
        m = where[:, 0] == f
        assert m.sum() == H * W
        assert np.array_equal(vals[m], want[where[m, 1], where[m, 2], :3].astype(np.float32)), f
    r.close()


def test_gpu_arm_fails_loudly_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "1"], cwd=ROOT,
                       capture_output=True, timeout=300)
    assert p.returncode != 0 and b"no CPU fallback" in p.stderr + p.stdout
