"""A/B of library builds on the headline workload (config 2, depth-1 frames in 16-frame steps), alternating builds
round by round in one job, plus a cross-build check of what the builds compute.

  python tools/cull_tables_ab.py --out DIR/cull_tables.json --rounds 5 parent=path/to/lib.so new=path/to/lib.so ...

Every round runs `bench.py --gpus 1 --steps 20 --warmup 5 --headline-only --sustained-seconds 0` once per build
(RTRB_B200_LIB selects the library) and keeps its headline `value` (Mrays/s), ms per step and e2e value.  Then each build
renders config 2 at 1920x1080 and a few depth-1 fuzz frames with full counters, and the JSON records whether frames,
hit ids and every counter (the FAST64 refine count `exact_tests` included) agree with the first build's.  The card's
name and power limit are recorded with the numbers."""
import argparse
import hashlib
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

STATS_SNIPPET = r"""
import hashlib, json, sys, copy
sys.path.insert(0, %(root)r); sys.path.insert(0, %(root)r + "/tests")
import numpy as np
from raytracing_rb_b200 import Camera, World, Renderer, make_opts, scenes, PREC_FAST64
out = {}
def rec(name, wdoc, cdoc):
    world = World(copy.deepcopy(wdoc))
    cam = Camera(world, copy.deepcopy(cdoc)).camera_desc()
    r = Renderer(world.to_scene_desc(), 0)
    for detail in (False, True):
        f = r.render(cam, make_opts(seed=5, precision=PREC_FAST64, count_detail=detail))
        st = {k: v for k, v in f.stats.items() if k not in ("device_ms", "trace_ms")}
        out["%%s/detail=%%d" %% (name, detail)] = {"rgba": hashlib.sha256(f.rgba.tobytes()).hexdigest(),
            "hit": hashlib.sha256(f.hit.tobytes()).hexdigest(), "code": int(f.code), "stats": st}
    r.close()
w, c = scenes.build(2)
rec("config2", w, c)
import test_gpu_fuzz as fz
for seed in range(12):
    wd, cd = fz.random_scene(seed)
    cd = dict(cd, trace_depth=1, pre_sample_times=1, max_sample_times=1, aperture_radius=0.0)
    rec("fuzz%%d" %% seed, wd, cd)
print("STATS " + json.dumps(out))
"""


def bench_once(lib):
    env = dict(os.environ, RTRB_B200_LIB=lib)
    p = subprocess.run([sys.executable, "bench.py", "--gpus", "1", "--steps", "20", "--warmup", "5", "--headline-only",
                        "--sustained-seconds", "0"], cwd=ROOT, env=env, capture_output=True, text=True, timeout=900)
    line = [l for l in p.stdout.splitlines() if l.startswith("{")]
    if p.returncode != 0 or not line:
        raise RuntimeError("bench failed for %s:\n%s\n%s" % (lib, p.stdout[-2000:], p.stderr[-2000:]))
    return json.loads(line[-1])


def stats_of(lib):
    env = dict(os.environ, RTRB_B200_LIB=lib)
    p = subprocess.run([sys.executable, "-c", STATS_SNIPPET % {"root": ROOT}], cwd=ROOT, env=env, capture_output=True,
                       text=True, timeout=900)
    line = [l for l in p.stdout.splitlines() if l.startswith("STATS ")]
    if p.returncode != 0 or not line:
        raise RuntimeError("stats failed for %s:\n%s\n%s" % (lib, p.stdout[-2000:], p.stderr[-2000:]))
    return json.loads(line[-1][6:])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("builds", nargs="+", help="name=path/to/librtrb_b200.so")
    a = ap.parse_args()
    builds = [tuple(b.split("=", 1)) for b in a.builds]
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    res = {"gpu": smi[0] if smi else None, "command": "bench.py --gpus 1 --steps 20 --warmup 5 --headline-only "
           "--sustained-seconds 0, builds alternating within each round", "rounds": []}
    for r in range(a.rounds):
        row = {}
        for name, lib in builds:
            j = bench_once(lib)
            row[name] = {"value": j["value"], "ms_per_step": j["ms_per_step"], "e2e": j["e2e"]["value"]}
            print("round %d %-10s %.1f Mrays/s" % (r, name, j["value"]), flush=True)
        res["rounds"].append(row)
    summ = {}
    for name, _ in builds:
        v = [row[name]["value"] for row in res["rounds"]]
        summ[name] = {"median": statistics.median(v), "min": min(v), "max": max(v)}
    base = builds[0][0]
    for name, _ in builds:
        summ[name]["vs_%s" % base] = summ[name]["median"] / summ[base]["median"] - 1.0
    res["summary"] = summ
    st = {name: stats_of(lib) for name, lib in builds}
    res["same_outputs_and_counters_as_%s" % base] = {name: st[name] == st[base] for name, _ in builds}
    diffs = {}
    for name, _ in builds:
        for k in st[base]:
            if st[name].get(k) != st[base][k]:
                diffs.setdefault(name, []).append(k)
    res["differing_frames"] = diffs
    res["config2_counters"] = st[base]["config2/detail=1"]["stats"]
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res["summary"], indent=1))
    print("same outputs/counters:", res["same_outputs_and_counters_as_%s" % base], diffs)


if __name__ == "__main__":
    main()
