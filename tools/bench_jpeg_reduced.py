"""12 MP camera-sized JPEG files to pose records at 1, 1/2, 1/4 and 1/8 scale: host decode (ImageStream(reduce=d) ->
BatchPipeline) vs GPU decode (ImageStream(reduce=d, decode="gpu") -> BatchPipeline(jpeg=True, reduce=d)), alternated on the
same files with the records of both paths compared in the same run.

Inputs: seeded synthetic 4032 x 3024 photos (oracle.synth's smooth generator upscaled from 1008 x 756, rolled per file), q90
4:2:0, in three sets: "smooth", "noisy" (Gaussian noise, sigma 8, as a sensor leaves it; about 4x the bytes) and "noisy444"
(the same at 4:4:4).  The network is C2's (MobileNetV1 101, OS16, batch 64) at 513 x 385: the 4:3 frame scaled to 513 wide
(the same network input at every scale, so only the decode and the resize input change with d).

For every (set, d): files -> records images/s of both paths, host CPU seconds per file (getrusage, whole process), pinned host
bytes per stream slot, H2D bytes per batch, the files the GPU path left to cv2 (host fallbacks), the device time of one
pn_jpeg_decode_scaled per batch (CUDA events over many launches) and its per-kernel shares (torch.profiler, a run of its own).
Prints one JSON object (and writes it with --out), with the card's name and power limit.

    python tools/bench_jpeg_reduced.py [--out FILE] [--rounds 2] [--files 192] [--sets smooth,noisy,noisy444] [--reduce 1,2,4,8]
"""
import argparse
import concurrent.futures
import json
import os
import re
import resource
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (os.path.join(ROOT, "posenet-pytorch_b200"), ROOT):
    if p not in sys.path:
        sys.path.insert(0, p)

import cv2  # noqa: E402
import numpy as np  # noqa: E402
import torch  # noqa: E402

import posenet  # noqa: E402
from oracle import synth  # noqa: E402  (input generator only)

H, W = 3024, 4032
SETS = {"smooth": (0, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_420), "noisy": (8, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_420),
        "noisy444": (8, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_444)}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                        str(torch.cuda.current_device())], capture_output=True, text=True)
    return q.stdout.strip() or torch.cuda.get_device_name()


def make_files(d, kind, n):
    sigma, samp = SETS[kind]
    base = [cv2.resize(synth.smooth_image(H // 4, W // 4, 900 + s), (W, H), interpolation=cv2.INTER_CUBIC) for s in range(4)]
    params = [cv2.IMWRITE_JPEG_QUALITY, 90, cv2.IMWRITE_JPEG_SAMPLING_FACTOR, samp]

    def write(i):
        img = np.roll(base[i % 4], 7 * i, axis=1)
        if sigma:
            rng = np.random.default_rng(i)
            img = np.clip(img + rng.normal(0, sigma, img.shape), 0, 255).astype(np.uint8)
        p = os.path.join(d, "%s_%04d.jpg" % (kind, i))
        cv2.imwrite(p, img, params)
        return p

    with concurrent.futures.ThreadPoolExecutor(os.cpu_count()) as ex:
        return list(ex.map(write, range(n)))


def pinned_bytes(stream):
    b = stream._bufs[0].numel()
    if stream.decode == "gpu":
        e = stream._enc[0]
        b += e.arena.numel() + e.descs.numel()
    return b


def run_path(pipe, paths, batch, reduce, gpu, keep_records):
    stream = posenet.ImageStream(paths, batch=batch, reduce=reduce, decode="gpu" if gpu else "cv2")
    h2d, host = [], 0

    def items():
        for b, _ in stream.batches():
            if gpu:
                rows = sum(b.shapes[i][0] * b.shapes[i][1] * 3 if b.shapes[i] else pipe.h * pipe.w * 3 for i in b.host_rows)
                h2d.append(b.used + b.descs.numel() + rows)
            else:
                h2d.append(b.numel())
            yield b

    r0 = resource.getrusage(resource.RUSAGE_SELF)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    recs = []
    for r in pipe.run(items(), copy=keep_records):
        if keep_records:
            recs.append(r[:4])
        if gpu:
            assert (r[-1] >= 0).all(), r[-1]
            host += int((r[-1] == 1).sum())
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    r1 = resource.getrusage(resource.RUSAGE_SELF)
    cpu = (r1.ru_utime - r0.ru_utime) + (r1.ru_stime - r0.ru_stime)
    res = dict(images_per_s=len(paths) / dt, cpu_s_per_file=cpu / len(paths), h2d_bytes_per_batch=float(np.mean(h2d)),
               pinned_bytes_per_slot=pinned_bytes(stream))
    if gpu:
        res["host_fallbacks"] = host
    return res, recs


def decode_kernels_ms(pipe, reps=10):
    """Device time per batch of each pn_jpeg_decode_scaled launch (torch.profiler, a run of its own, kernels summed by name)."""
    from torch.profiler import ProfilerActivity, profile
    s = pipe.slots[0]
    with torch.cuda.stream(pipe.compute):
        s["dec"].decode(s["x"], pipe.h * pipe.w * 3)
        pipe.compute.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(reps):
                s["dec"].decode(s["x"], pipe.h * pipe.w * 3)
            pipe.compute.synchronize()
    out = {}
    for e in prof.key_averages():
        name = re.search(r"(\w+_kernel)", e.key)
        if name:
            out[name.group(1)] = round(out.get(name.group(1), 0.0) + e.device_time_total / 1000.0 / reps, 4)
    total = sum(out.values())
    return {k: {"ms": v, "share": round(v / total, 4)} for k, v in sorted(out.items(), key=lambda kv: -kv[1])}


def decode_ms(pipe, reps=20):
    s = pipe.slots[0]
    with torch.cuda.stream(pipe.compute):
        for _ in range(3):
            s["dec"].decode(s["x"], pipe.h * pipe.w * 3)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(pipe.compute)
        for _ in range(reps):
            s["dec"].decode(s["x"], pipe.h * pipe.w * 3)
        e1.record(pipe.compute)
        pipe.compute.synchronize()
    assert (s["dec"].status == 0).all()
    return e0.elapsed_time(e1) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--files", type=int, default=192)
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--sets", default="smooth,noisy,noisy444")
    ap.add_argument("--reduce", default="1,2,4,8")
    args = ap.parse_args()
    torch.cuda.set_device(0)
    batch, mid, os_ = args.batch, 101, 16
    out = {"metric": "12 MP JPEG files to pose records at 1/d, host (cv2 IMREAD_REDUCED_COLOR_d) vs GPU decode",
           "card": card(), "host_cores": os.cpu_count(), "file_size": [H, W], "model": mid, "output_stride": os_, "batch": batch,
           "workloads": {}}
    tmp = tempfile.mkdtemp()
    torch.manual_seed(0)
    model = posenet.MobileNetV1(mid, output_stride=os_).cuda().set_compute_dtype("bf16")
    for kind in args.sets.split(","):
        paths = make_files(tmp, kind, args.files)
        for d in (int(x) for x in args.reduce.split(",")):
            h, w = -(-H // d), -(-W // d)
            sf = 513.0 / w
            kw = dict(depth=2, max_pose_detections=10, min_pose_score=0.25, scale_factor=sf)
            host_pipe = posenet.BatchPipeline(model, batch, h, w, **kw)
            gpu_pipe = posenet.BatchPipeline(model, batch, h, w, jpeg=True, reduce=d, **kw)
            run_path(host_pipe, paths[:batch], batch, d, False, False)                          # warm-up
            run_path(gpu_pipe, paths[:batch], batch, d, True, False)
            res = {"host": [], "gpu": []}
            same = None
            for r in range(args.rounds):
                keep = r == 0
                hr, rh = run_path(host_pipe, paths, batch, d, False, keep)
                gr, rg = run_path(gpu_pipe, paths, batch, d, True, keep)
                res["host"].append(hr)
                res["gpu"].append(gr)
                if keep:
                    same = len(rh) == len(rg) and all(all(np.array_equal(a, b) for a, b in zip(x, y)) for x, y in zip(rh, rg))
                    assert same, "%s at 1/%d: the GPU decode's records differ from cv2's" % (kind, d)
            wl = {"reduce": d, "frame": [h, w], "network_input": [gpu_pipe.th, gpu_pipe.tw], "files": len(paths),
                  "bytes_per_file": float(np.mean([os.path.getsize(p) for p in paths])), "records_identical": bool(same),
                  "gpu_decode_ms_per_batch": round(decode_ms(gpu_pipe), 4),
                  "gpu_decode_kernels_ms_per_batch": decode_kernels_ms(gpu_pipe)}
            for k in ("host", "gpu"):
                wl[k] = {m: [round(x[m], 6) for x in res[k]] for m in res[k][0]}
                wl[k]["images_per_s_median"] = float(np.median(wl[k]["images_per_s"]))
            wl["speedup"] = round(wl["gpu"]["images_per_s_median"] / wl["host"]["images_per_s_median"], 4)
            out["workloads"]["%s_r%d" % (kind, d)] = wl
            print(kind, d, json.dumps(wl), flush=True)
            if args.out:                                                 # each workload as it completes
                write(args.out, out)
            del host_pipe, gpu_pipe
            torch.cuda.empty_cache()
        for p in paths:
            os.remove(p)
    print(json.dumps(out))
    if args.out:
        write(args.out, out)


def write(path, out):
    os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
    with open(path, "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
