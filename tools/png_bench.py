"""Measures the device PNG encoder (rtrb_encode_png / rtrb_submit_png, Camera.render_png) on one GPU and writes
profiles/png_encode.json (or --out).  Records the GPU's name and power limit in the same run.

  - encode device time: sum of the encoder's kernels per encode from torch.profiler over --encodes back-to-back
    encodes of the same frame (L2-warm: the 6.2 MB frame, the scratch and the file stay resident in the 126 MB L2),
    plus the CUDA-event time of the blocking call that also brings the file to the host;
  - PNG bytes against the raw filtered stream and host zlib levels 1 and 6 of the same stream;
  - wall time of Camera.render_cuda(path) against Camera.render_png(path) (median of --reps, after a warm-up);
  - frames/s of submit_png/wait_png against RGB8 submit/wait, 3 frames in flight, pinned buffers (bench.py's e2e);
  - the encoder's zero-copy store of the file into mapped host memory (png_publish_kernel) against cudaMemcpyAsync
    device-to-pinned-host copies of the same byte count.

python tools/png_bench.py [--out profiles/png_encode.json]"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time
import zlib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, power, clock = [s.strip() for s in q.split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def idat_payload(png):
    import struct
    pos, out = 8, []
    while pos < len(png):
        n, = struct.unpack(">I", png[pos:pos + 4])
        if png[pos + 4:pos + 8] == b"IDAT":
            out.append(png[pos + 8:pos + 8 + n])
        pos += 12 + n
    return zlib.decompress(b"".join(out))


def kernel_us(prof, prefix):
    """Summed device time (us) of kernels whose name contains `prefix`, by kernel."""
    out = {}
    for e in prof.events():
        if e.device_type.name == "CUDA" and prefix in e.name:
            key = e.name.split("png_")[1].split("_kernel")[0] if "png_" in e.name else e.name
            out[key] = out.get(key, 0.0) + e.device_time
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "png_encode.json"))
    ap.add_argument("--encodes", type=int, default=200)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--frames", type=int, default=600)
    args = ap.parse_args()
    import torch
    from torch.profiler import ProfilerActivity, profile
    from raytracing_rb_b200 import Camera, World, _abi, make_opts, png_max_bytes, scenes

    if not torch.cuda.is_available():
        raise SystemExit("png_bench needs a CUDA device")
    res = {"gpu": gpu_info(), "segment_bytes": _abi.PNG_SEGMENT_BYTES, "configs": {}}

    cams = {}
    for cid in (2, 3):
        wdoc, cdoc = scenes.build(cid, width=1920, height=1080)
        cam = Camera(World(wdoc), cdoc)
        cams[cid] = cam
        r, cd = cam.renderer(), cam.camera_desc()
        W, H = cd.width, cd.height
        r.render_device(cd, make_opts(seed=1, pixel_format=_abi.FMT_RGB8, skip_outputs=3))
        png = r.encode_png(W, H)
        for _ in range(5):
            assert r.encode_png(W, H) == png
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(args.encodes):
                r.encode_png(W, H)
            torch.cuda.synchronize()
        per = {k: v / args.encodes for k, v in kernel_us(prof, "png_").items()}
        dev_us = sum(per.values())
        s = torch.cuda.Stream()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(s):
            e0.record(s)
            for _ in range(args.encodes):
                r.encode_png(W, H, stream=s.cuda_stream)
            e1.record(s)
        e1.synchronize()
        call_us = e0.elapsed_time(e1) * 1e3 / args.encodes
        filtered = idat_payload(png)
        raw = len(filtered)
        rec = {"size": [W, H], "png_bytes": len(png), "filtered_bytes": raw, "png_max_bytes": png_max_bytes(W, H),
               "zlib1_bytes": len(zlib.compress(filtered, 1)), "zlib6_bytes": len(zlib.compress(filtered, 6)),
               "encode_device_us": dev_us, "encode_kernels_us": per,
               "encode_input_GBps": raw / (dev_us * 1e-6) / 1e9,
               "encode_png_call_us": call_us,
               "l2_state": "warm: frame, scratch and file resident in L2 (back-to-back encodes of one frame)"}
        t0 = time.perf_counter()
        zlib.compress(filtered, 6)
        rec["host_zlib6_ms_one_core"] = (time.perf_counter() - t0) * 1e3
        rec["png_over_zlib1"] = rec["png_bytes"] / rec["zlib1_bytes"]
        res["configs"]["config%d" % cid] = rec
        print(json.dumps({"config": cid, **rec}), flush=True)

    # wall time of the two file paths on config 2
    cam = cams[2]
    with tempfile.TemporaryDirectory() as d:
        a, b = os.path.join(d, "cuda.png"), os.path.join(d, "dev.png")
        cam.render_cuda(a)
        cam.render_png(b)
        ta, tb = [], []
        for _ in range(args.reps):
            t0 = time.perf_counter(); cam.render_cuda(a); ta.append(time.perf_counter() - t0)
            t0 = time.perf_counter(); cam.render_png(b); tb.append(time.perf_counter() - t0)
        res["file_wall_ms"] = {"render_cuda": statistics.median(ta) * 1e3, "render_png": statistics.median(tb) * 1e3,
                               "speedup": statistics.median(ta) / statistics.median(tb),
                               "render_cuda_bytes": os.path.getsize(a), "render_png_bytes": os.path.getsize(b),
                               "reps": args.reps, "config": "config2 1920x1080"}
    print(json.dumps(res["file_wall_ms"]), flush=True)

    # pipelined frame sequences on config 2
    r, cd = cam.renderer(), cam.camera_desc()
    W, H = cd.width, cd.height
    eo = make_opts(seed=1, pixel_format=_abi.FMT_RGB8)

    def run(submit, wait, bufs):
        wait(submit(bufs[0]))
        torch.cuda.synchronize()
        t0, pending = time.perf_counter(), []
        for i in range(args.frames):
            if len(pending) == 3:
                wait(pending.pop(0))
            pending.append(submit(bufs[i % 3]))
        for t in pending:
            wait(t)
        return args.frames / (time.perf_counter() - t0)

    rgb_bufs = [torch.empty((H, W, 3), dtype=torch.uint8).pin_memory().numpy() for _ in range(3)]
    png_bufs = [torch.empty(png_max_bytes(W, H), dtype=torch.uint8).pin_memory().numpy() for _ in range(3)]
    fps = {"submit_rgb8": [], "submit_png": []}
    for _ in range(2):  # alternate the two arms
        fps["submit_rgb8"].append(run(lambda b: r.submit(cd, b, eo), r.wait, rgb_bufs))
        fps["submit_png"].append(run(lambda b: r.submit_png(cd, b, eo), r.wait_png, png_bufs))
    res["pipelined_frames_per_s"] = {k: max(v) for k, v in fps.items()}
    res["pipelined_frames_per_s"].update(all_runs=fps, frames=args.frames, in_flight=3,
                                         d2h_bytes_per_frame={"submit_rgb8": W * H * 3,
                                                              "submit_png": res["configs"]["config2"]["png_bytes"]})
    print(json.dumps(res["pipelined_frames_per_s"]), flush=True)

    # zero-copy store of the file vs cudaMemcpyAsync of the same byte count
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for i in range(20):
            r.wait_png(r.submit_png(cd, png_bufs[i % 3], eo))
    pub_us = kernel_us(prof, "png_publish").get("publish", 0.0) / 20
    rates = {}
    for name, n in (("config2", res["configs"]["config2"]["png_bytes"]), ("config3", res["configs"]["config3"]["png_bytes"])):
        dev = torch.empty(n, dtype=torch.uint8, device="cuda")
        host = torch.empty(n, dtype=torch.uint8).pin_memory()
        host.copy_(dev, non_blocking=True)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(100):
            host.copy_(dev, non_blocking=True)
        e1.record()
        e1.synchronize()
        us = e0.elapsed_time(e1) * 1e3 / 100
        rates[name] = {"bytes": n, "memcpy_async_us": us, "memcpy_async_GBps": n / (us * 1e-6) / 1e9}
    n2 = res["configs"]["config2"]["png_bytes"]
    rates["config2"].update(zero_copy_store_us=pub_us, zero_copy_store_GBps=n2 / (pub_us * 1e-6) / 1e9 if pub_us else None)
    rates["config3"].update(zero_copy_store_us="not measured", zero_copy_store_GBps="not measured")
    res["file_to_host"] = rates
    print(json.dumps(rates), flush=True)

    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
