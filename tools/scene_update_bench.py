"""Cost of rtrb_scene_update (DESIGN.md §13) on one GPU -> profiles/scene_update.json (or --out).

  - one update that moves every sphere, and one update with an unchanged scene (the library's no-op): host time of the
    call and device time of what it queues (CUDA events around it on a stream of its own), for the config-2 world, the
    config-5 world (1 026 objects, BVH) and the 66 000-sphere scene of test_more_spheres_than_the_filter_can_index;
  - World.to_scene_desc() host time of the same worlds (what Camera.renderer() pays before every frame);
  - animated sequences through rtrb_submit / rtrb_wait (four frames in flight), every sphere moved every frame: 200
    config-2 frames at 1920x1080, and config 5 at 480x270, 4 spp; each against the same frames without an update and
    against destroy + create per frame.
Scene descriptors are flattened before the timed loops, so the sequences time the library, not the Python mirror.
The card's name and power limit are read in the same run."""
import argparse
import copy
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from raytracing_rb_b200 import Camera, Renderer, World, _abi, make_opts, scenes  # noqa: E402


def moved(wdoc, f):
    w = copy.deepcopy(wdoc)
    for o in w["world_objects"]:
        if o["type"] == "Sphere":
            c = o["properties"]["center"]
            o["properties"]["center"] = [c[0] + 0.01 * (f % 50), c[1] - 0.005 * (f % 50), c[2]]
    return w


def big_world():
    rs = np.random.RandomState(3)
    n = 66000
    objs = [scenes.ground()]
    gy, gx = np.meshgrid(np.linspace(-8, 8, 250), np.linspace(30, 3, 264))
    for k, (x, y) in enumerate(zip(gx.ravel()[:n], gy.ravel()[:n])):
        r = 0.02 + 0.01 * rs.uniform()
        objs.append(scenes.matte("m%d" % k, (float(x), float(y), -1 + r), r, (0.9, 0.5, 0.4)))
    return {"max_distance": 10000, "soft_shadow_exponent": 2, "lights": [scenes.light([5, -4, 4], 0.0)],
            "world_objects": objs}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def single_update(wdoc, reps):
    """Host and device ms of an update that moves every sphere, and of a no-op update."""
    import torch
    s = torch.cuda.Stream()
    descs = [World(moved(wdoc, f)).to_scene_desc() for f in range(2)]
    r = Renderer(descs[0], 0)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    out = {}
    for name, pick in (("move_every_sphere", lambda i: descs[(i + 1) % 2]), ("no_op", lambda i: descs[0])):
        if name == "no_op":
            r.update(descs[0], stream=s)
        host, dev = [], []
        for i in range(reps):
            h = pick(i)
            torch.cuda.synchronize()
            e0.record(s)
            t = time.perf_counter()
            r.update(h, stream=s)
            host.append((time.perf_counter() - t) * 1e3)
            e1.record(s)
            torch.cuda.synchronize()
            dev.append(e0.elapsed_time(e1))
        out[name] = {"host_ms_median": float(np.median(host)), "device_ms_median": float(np.median(dev)), "reps": reps}
    r.close()
    w = World(copy.deepcopy(wdoc))
    t = time.perf_counter()
    for _ in range(max(1, reps // 4)):
        w.to_scene_desc()
    out["to_scene_desc_host_ms"] = (time.perf_counter() - t) * 1e3 / max(1, reps // 4)
    out["objects"] = len(wdoc["world_objects"])
    return out


def sequence(wdoc, cdoc, n):
    """Frames/s of n submitted frames: updated every frame, no update, destroy + create per frame."""
    import torch
    cam = Camera(World(copy.deepcopy(wdoc)), cdoc).camera_desc()
    descs = [World(moved(wdoc, f)).to_scene_desc() for f in range(n)]
    opts = make_opts(seed=1, pixel_format=_abi.FMT_RGB8)
    bufs = [torch.zeros((cam.height, cam.width, 3), dtype=torch.uint8).pin_memory().numpy() for _ in range(4)]
    res = {}

    def pipelined(r, update):
        tickets = []
        t = time.perf_counter()
        for f in range(n):
            if len(tickets) == 4:
                r.wait(tickets.pop(0))
            if update:
                r.update(descs[f])
            tickets.append(r.submit(cam, bufs[f % 4], opts))
        for tk in tickets:
            r.wait(tk)
        return time.perf_counter() - t

    r = Renderer(descs[0], 0)
    pipelined(r, True)  # warm-up: modules, slots, staging
    res["updated_every_frame_s"] = pipelined(r, True)
    res["no_update_s"] = pipelined(r, False)
    r.close()
    m = max(10, n // 4)
    t = time.perf_counter()
    for f in range(m):
        rr = Renderer(descs[f], 0)
        rr.wait(rr.submit(cam, bufs[0], opts))
        rr.close()
    res["destroy_create_per_frame_s"] = (time.perf_counter() - t) * n / m
    res["destroy_create_frames_timed"] = m
    res["frames"] = n
    res["frame_ms_updated"] = res["updated_every_frame_s"] * 1e3 / n
    res["frame_ms_no_update"] = res["no_update_s"] * 1e3 / n
    res["frame_ms_destroy_create"] = res["destroy_create_per_frame_s"] * 1e3 / n
    res["update_overhead_ms_per_frame"] = res["frame_ms_updated"] - res["frame_ms_no_update"]
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "scene_update.json"))
    ap.add_argument("--frames", type=int, default=200)
    ap.add_argument("--reps", type=int, default=40)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("scene_update_bench needs a CUDA device")
    w2, c2 = scenes.build(2)
    w5, c5 = scenes.build(5, width=480, height=270, spp=4)
    result = {"card": card(), "torch_device": torch.cuda.get_device_name(0)}
    result["single_update"] = {"config2": single_update(w2, a.reps), "config5": single_update(w5, a.reps),
                               "spheres_66000": single_update(big_world(), 6)}
    result["sequence"] = {"config2_1920x1080": sequence(w2, c2, a.frames),
                          "config5_480x270_4spp": sequence(w5, c5, max(20, a.frames // 4))}
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result, indent=1))


if __name__ == "__main__":
    main()
