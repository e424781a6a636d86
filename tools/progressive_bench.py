"""Progressive frames (DESIGN.md §14) against one-shot frames on one GPU -> profiles/progressive.json (or --out).

  - config 5 at 3840x2160 / 64 spp and config 3 at 1920x1080 / 4 spp (FAST64): the device time of every pass of the
    doubling schedule (1, 2, 4, ... samples per pixel; the first pass is the 1-spp preview), the whole progressive
    frame (sum of its passes) and the one-shot frame, each from the CUDA events of the library's stats (device_ms of a
    pass covers that pass only); plus the host time from rtrb_progressive_create to the first preview's return;
  - config 1 (the reference's default camera: adaptive 3 / 10, Monte-Carlo rays) the same way.
Every shape is warmed up first; the one-shot and the progressive frame alternate, --reps times each, and the median is
reported with the spread.  The final progressive frame is checked against the one-shot frame byte for byte.  The card's
name and power limit are read in the same run."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from raytracing_rb_b200 import Camera, World, _abi, make_opts, progressive_schedule, scenes  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, power, clock = [s.strip() for s in q.split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def spread(v):
    v = sorted(v)
    return {"median": float(np.median(v)), "min": float(v[0]), "max": float(v[-1])}


def measure(label, wdoc, cdoc, reps):
    world = World(wdoc)
    cam = Camera(world, cdoc)
    r = cam.renderer()
    cd = cam.camera_desc()
    opts = make_opts(seed=1, precision=_abi.PREC_FAST64, skip_outputs=_abi.SKIP_RGB | _abi.SKIP_HIT)
    sched = progressive_schedule(cd.pre_sample_times)
    W, H = cd.width, cd.height

    def oneshot():
        stats, _ = r.render_device(cd, opts)
        return stats["device_ms"]

    def progressive():
        t0 = time.perf_counter()
        p = r.progressive(cd, opts)
        passes, first_host = [], None
        try:
            for e in sched:
                stats, _ = p.pass_to(e)
                if first_host is None:
                    first_host = (time.perf_counter() - t0) * 1e3
                passes.append(stats["device_ms"])
            frame = p.download(want_rgb=False, want_hit=False).rgba
        finally:
            p.close()
        return passes, first_host, frame

    oneshot()
    _, _, final = progressive()  # warm-up of every shape
    ref = np.empty_like(final)
    _lib_download(r, ref)
    one, prog, first_host = [], [], []
    per_pass = [[] for _ in sched]
    for _ in range(reps):
        one.append(oneshot())
        passes, fh, _ = progressive()
        prog.append(sum(passes))
        first_host.append(fh)
        for k, ms in enumerate(passes):
            per_pass[k].append(ms)
    ratio = float(np.median(prog) / np.median(one))
    return {"config": label, "width": W, "height": H, "pre_sample_times": cd.pre_sample_times,
            "max_sample_times": cd.max_sample_times, "trace_depth": cd.trace_depth, "schedule": sched, "reps": reps,
            "oneshot_device_ms": spread(one), "progressive_device_ms": spread(prog),
            "progressive_over_oneshot": ratio,
            "passes_device_ms": [dict(samples_end=e, **spread(v)) for e, v in zip(sched, per_pass)],
            "first_preview_device_ms": spread(per_pass[0]), "first_preview_host_ms_from_create": spread(first_host),
            "final_equals_oneshot": bool(np.array_equal(final, ref))}


def _lib_download(r, out):
    from raytracing_rb_b200._lib import check, lib
    check(lib().rtrb_download(r.handle, out.ctypes.data, None, None))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "progressive.json"))
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    res = {"gpu": card(), "precision": "FAST64", "outputs": "8-bit RGBA frame only (skip_outputs = RGB | HIT)",
           "runs": []}
    w5, c5 = scenes.build(5)
    w3, c3 = scenes.build(3)
    w1, c1 = scenes.build(1)
    for label, w, c in (("config5 3840x2160 64 spp", w5, c5), ("config3 1920x1080 4 spp", w3, c3),
                        ("config1 192x108 adaptive 3/10", w1, c1)):
        run = measure(label, w, c, args.reps)
        print(json.dumps(run), flush=True)
        res["runs"].append(run)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
