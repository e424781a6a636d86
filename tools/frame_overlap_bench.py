"""Per-frame fixed cost of the headline workload (config 2: 1920x1080, depth 1, 1 spp; bench.py's 16-frame steps) with
and without frame overlap (RTRB_FRAME_OVERLAP, read when a renderer is created), A/B in one process, and writes
profiles/frame_overlap.json (or --out).  Records the GPU's name and power limit in the same run.

  (a) host enqueue time per frame: perf_counter around 16 render_device(want_stats=False) calls, no synchronise
      (if this approaches the device time per frame, the step is paced by the host, not by the device);
  (b) device time per 16-frame step: bench.py's workload, cameras, frame slots and 256 MiB L2 flush between steps,
      CUDA events on the launch stream; the arms alternate round by round;
  (c) the trace kernel alone: the library's CUDA events around one launch (render_device with stats), cold L2;
  (d) a torch.profiler run of its own: the gaps between consecutive trace kernels of a step (negative = overlap);
  (e) overlap on, plus a timing event recorded on the stream after every frame: does an event between two
      overlapping frames keep the second one from starting under the first one's tail?
(b)/16 - (c) is what a frame costs beyond its kernel.  The frames of the last step of every arm must be byte-identical.

python tools/frame_overlap_bench.py [--out profiles/frame_overlap.json] [--steps 20] [--rounds 5]"""
import argparse
import hashlib
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

KERNEL = "trace_pre_fast_kernel"


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, power, clock = [s.strip() for s in q.split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "frame_overlap.json"))
    ap.add_argument("--steps", type=int, default=20, help="timed steps per arm and round")
    ap.add_argument("--rounds", type=int, default=5, help="rounds of the alternating arms")
    ap.add_argument("--frames", type=int, default=16, help="frames per step (bench.py's --frames-per-step)")
    args = ap.parse_args()
    import numpy as np
    import torch
    from torch.profiler import ProfilerActivity, profile
    import bench
    from raytracing_rb_b200 import Renderer, _abi, make_opts

    if not torch.cuda.is_available():
        raise SystemExit("frame_overlap_bench needs a CUDA device")
    B = args.frames
    world, cdoc, name = bench.workload(2)
    cams = bench.batch_cameras(world, cdoc, B)
    W, H = cams[0].width, cams[0].height
    slot_bytes = W * H * 4
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    arms = {}
    for arm, env in (("off", "0"), ("on", "1")):
        os.environ["RTRB_FRAME_OVERLAP"] = env
        r = Renderer(world.to_scene_desc(), 0)
        base = r.framebuffer_ptr(W, H * B)
        opts = [make_opts(seed=1, stream=stream.cuda_stream, rgba_device_out=base + f * slot_bytes,
                          skip_outputs=_abi.SKIP_RGB | _abi.SKIP_HIT, pixel_format=_abi.FMT_RGB8) for f in range(B)]
        arms[arm] = (r, opts)
    os.environ.pop("RTRB_FRAME_OVERLAP")
    st, _ = arms["off"][0].render_device(cams[0], arms["off"][1][0])
    rays_per_frame = st["rays"] + st["shadow_queries"]

    def step(arm, event_after=None):
        r, opts = arms[arm]
        for f in range(B):
            r.render_device(cams[f], opts[f], want_stats=False)
            if event_after is not None:
                event_after.record(stream)

    def timed_steps(arm, n, event_after=None):
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n)]
        for k in range(n):
            flush.zero_()
            ev[k][0].record(stream)
            step(arm, event_after)
            ev[k][1].record(stream)
        torch.cuda.synchronize()
        return [a.elapsed_time(b) for a, b in ev]

    for arm in arms:
        for _ in range(5):
            step(arm)
    torch.cuda.synchronize()

    res = {"gpu": gpu_info(), "workload": name, "size": [W, H], "frames_per_step": B, "steps_per_round": args.steps,
           "rounds": args.rounds, "rays_per_frame": rays_per_frame,
           "l2": "256 MiB write between timed steps, as bench.py", "arms": {}}

    # (a) host enqueue
    enqueue = {}
    for arm in arms:
        per = []
        for _ in range(20):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            step(arm)
            per.append((time.perf_counter() - t0) / B * 1e6)
            torch.cuda.synchronize()
        enqueue[arm] = statistics.median(per)

    # (b) device time per step, arms alternating; (e) overlap on with an event after every frame
    ev_between = torch.cuda.Event(enable_timing=True)
    steps = {"off": [], "on": [], "on_event_between_frames": []}
    round_medians = {k: [] for k in steps}
    for _ in range(args.rounds):
        for arm in ("off", "on", "on_event_between_frames"):
            ms = timed_steps("on" if arm != "off" else "off", args.steps,
                             ev_between if arm == "on_event_between_frames" else None)
            steps[arm] += ms
            round_medians[arm].append(statistics.median(ms))

    # frames of the last step of each arm, byte for byte
    digests = {}
    for arm in arms:
        r, _ = arms[arm]
        step(arm)
        torch.cuda.synchronize()
        got = np.zeros((H * B, W, 4), np.uint8)
        r.framebuffer_download(W, H * B, got)
        digests[arm] = hashlib.sha256(got.reshape(B, slot_bytes)[:, :W * H * 3].tobytes()).hexdigest()

    # (c) the kernel alone
    kernel = {}
    for arm in arms:
        r, opts = arms[arm]
        tr, dev = [], []
        for f in range(B):
            flush.zero_()
            torch.cuda.synchronize()
            st, _ = r.render_device(cams[f], opts[f])
            tr.append(st["trace_ms"] * 1e3)
            dev.append(st["device_ms"] * 1e3)
        kernel[arm] = {"trace_us_mean": statistics.mean(tr), "trace_us_median": statistics.median(tr),
                       "device_us_median": statistics.median(dev)}

    # (d) profiler: gaps between consecutive trace kernels inside a step
    gaps = {}
    for arm in arms:
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(4):
                flush.zero_()
                step(arm)
            torch.cuda.synchronize()
        with tempfile.TemporaryDirectory() as d:
            path = os.path.join(d, "trace.json")
            prof.export_chrome_trace(path)
            with open(path) as f:
                trace = json.load(f)
        ks = sorted((e for e in trace.get("traceEvents", []) if e.get("cat") == "kernel"), key=lambda e: e["ts"])
        g, durs, run = [], [], []
        for e in ks:
            if KERNEL in e["name"]:
                durs.append(e["dur"])
                if run:
                    g.append(e["ts"] - (run[-1]["ts"] + run[-1]["dur"]))
                run.append(e)
            else:
                run = []  # the L2 flush separates steps
        gaps[arm] = {"kernels": len(durs), "kernel_us_median": statistics.median(durs) if durs else None,
                     "gap_us_median": statistics.median(g) if g else None, "gap_us_min": min(g) if g else None,
                     "gap_us_max": max(g) if g else None,
                     "note": "start of trace kernel i+1 minus end of kernel i within a step; negative = the two overlap"}

    for arm in steps:
        ms = steps[arm]
        k = "on" if arm != "off" else "off"
        rec = {"step_ms_median": statistics.median(ms), "step_ms_mean": statistics.mean(ms),
               "round_medians_ms": round_medians[arm],
               "round_spread": (max(round_medians[arm]) - min(round_medians[arm])) / statistics.median(round_medians[arm]),
               "frame_us": statistics.median(ms) / B * 1e3,
               "mrays_s": rays_per_frame * B / (statistics.mean(ms) * 1e-3) / 1e6}
        if arm in arms:
            rec.update(enqueue_us_per_frame=enqueue[arm], kernel=kernel[arm], profiler=gaps[arm],
                       frames_sha256=digests[arm],
                       beyond_kernel_us_per_frame=rec["frame_us"] - kernel[arm]["trace_us_mean"])
        res["arms"][arm] = rec
    res["frames_equal"] = digests["on"] == digests["off"]
    res["speedup_on_vs_off"] = res["arms"]["off"]["step_ms_median"] / res["arms"]["on"]["step_ms_median"]
    res["speedup_on_event_between_vs_off"] = (res["arms"]["off"]["step_ms_median"] /
                                              res["arms"]["on_event_between_frames"]["step_ms_median"])
    print(json.dumps(res, indent=1))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
