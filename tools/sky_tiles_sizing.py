"""Trace-kernel time of the headline world (config 2, 1920x1080, depth 1, 1 spp) seen from three cameras: the
workload's own, one pitched up so that every pixel is sky (misses everything), and one pitched down so that every
pixel is the ground plane.  With the hit-id shares of config 2 this sizes what skipping the sky tiles can gain.

  python tools/sky_tiles_sizing.py --out DIR/sky_sizing.json [name=path/to/librtrb_b200.so ...]

Each library (RTRB_B200_LIB; none given = the in-tree build) runs in its own process.  Per camera: the median over
--frames frames of render_device's trace_ms and device_ms (CUDA events inside the library), the L2 flushed by a
256 MiB write before every frame, the frames in the benchmark's format (RGB8 into a device buffer, no FP64 / hit-id
outputs).  The card's name and power limit are recorded with the numbers."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

SNIPPET = r"""
import json, statistics, sys, copy
sys.path.insert(0, %(root)r)
import torch
from raytracing_rb_b200 import Camera, World, Renderer, make_opts, scenes, PREC_FAST64
from raytracing_rb_b200 import _abi
w, c = scenes.build(2)
world = World(copy.deepcopy(w))
cams = {"config2": dict(c),
        "all_sky": dict(c, front=[-1.0, 0.0, 1.0], up=[1.0, 0.0, 1.0]),      # 45 deg up, away from the light
        "all_ground": dict(c, front=[1.0, 0.0, -1.0], up=[1.0, 0.0, 1.0])}   # 45 deg down
r = Renderer(world.to_scene_desc(), 0)
W, H = c["width"], c["height"]
fb = r.framebuffer_ptr(W, H)
flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
out = {}
for name, cd in cams.items():
    cam = Camera(world, cd).camera_desc()
    o = make_opts(seed=1, precision=PREC_FAST64, rgba_device_out=fb, skip_outputs=_abi.SKIP_RGB | _abi.SKIP_HIT,
                  pixel_format=_abi.FMT_RGB8)
    for _ in range(20):
        r.render_device(cam, o)
    tr, dv = [], []
    for _ in range(%(frames)d):
        flush.zero_()
        torch.cuda.synchronize()  # the flush runs on torch's stream, the frame on the renderer's non-blocking one
        st, _ = r.render_device(cam, o)
        tr.append(st["trace_ms"]); dv.append(st["device_ms"])
    st, _ = r.render_device(cam, make_opts(seed=1, precision=PREC_FAST64, count_detail=True))
    f = r.render(cam, make_opts(seed=1, precision=PREC_FAST64))
    out[name] = {"trace_ms_median": statistics.median(tr), "trace_ms_min": min(tr), "trace_ms_max": max(tr),
                 "device_ms_median": statistics.median(dv), "miss_share": float((f.hit < 0).mean()),
                 "ground_share": float((f.hit == 0).mean()), "exact_tests": st.get("exact_tests")}
print("SIZING " + json.dumps(out))
"""


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--frames", type=int, default=200)
    ap.add_argument("builds", nargs="*", help="name=path/to/librtrb_b200.so")
    a = ap.parse_args()
    builds = [tuple(b.split("=", 1)) for b in a.builds] or [("tree", "")]
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    res = {"gpu": smi[0] if smi else None, "frames": a.frames, "builds": {}}
    for name, lib in builds:
        env = dict(os.environ)
        if lib:
            env["RTRB_B200_LIB"] = lib
        p = subprocess.run([sys.executable, "-c", SNIPPET % {"root": ROOT, "frames": a.frames}], cwd=ROOT, env=env,
                           capture_output=True, text=True, timeout=900)
        line = [l for l in p.stdout.splitlines() if l.startswith("SIZING ")]
        if p.returncode != 0 or not line:
            raise RuntimeError("sizing failed for %s:\n%s\n%s" % (name, p.stdout[-2000:], p.stderr[-2000:]))
        res["builds"][name] = json.loads(line[-1][7:])
        print(name, json.dumps(res["builds"][name], indent=1), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
