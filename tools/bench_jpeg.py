"""JPEG files to pose records: host decode (ImageStream -> BatchPipeline) vs GPU decode (ImageStream(decode="gpu") ->
BatchPipeline(jpeg=True)), alternated three times each on the same files.

Workloads: C2 (512 files of 513 x 513, q90, bench_ingest.py's generator; MobileNetV1 101, OS16, batch 64), C2 again with noisy
q95 4:4:4 files (photographs compress worse than the smooth synthetic frames), C3 (1280 x 720 q90 frames; model 50, OS8, batch 32).
For each path: files -> records images/s, host CPU seconds per file (getrusage, whole process), H2D bytes per batch, bytes per
file; for the GPU path also the device time of one pn_jpeg_decode per batch (CUDA events over many launches).  Both paths'
records are compared for equality in the same run.  Prints one JSON object (and writes it with --out), with the card's name
and power limit.

    python tools/bench_jpeg.py [--out FILE] [--rounds 3]
"""
import argparse
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


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                        str(torch.cuda.current_device())], capture_output=True, text=True)
    return q.stdout.strip() or torch.cuda.get_device_name()


def make_files(d, kind, n):
    paths = []
    if kind == "c2":
        base = [synth.smooth_image(513, 513, s) for s in range(16)]           # bench_ingest.py's generator
        imgs = lambda i: np.roll(base[i % 16], i, axis=1)
        params = [cv2.IMWRITE_JPEG_QUALITY, 90]
    elif kind == "c2_noisy":
        rng = np.random.default_rng(0)
        base = [rng.integers(0, 256, (513, 513, 3), dtype=np.uint8) for _ in range(16)]
        imgs = lambda i: np.roll(base[i % 16], i, axis=1)
        params = [cv2.IMWRITE_JPEG_QUALITY, 95, cv2.IMWRITE_JPEG_SAMPLING_FACTOR, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_444]
    else:
        base = [synth.smooth_image(720, 1280, 50 + s) for s in range(8)]
        imgs = lambda i: np.roll(base[i % 8], 3 * i, axis=1)
        params = [cv2.IMWRITE_JPEG_QUALITY, 90]
    for i in range(n):
        p = os.path.join(d, "%s_%04d.jpg" % (kind, i))
        cv2.imwrite(p, imgs(i), params)
        paths.append(p)
    return paths


def run_path(pipe, paths, batch, gpu, keep_records):
    stream = posenet.ImageStream(paths, batch=batch, decode="gpu" if gpu else "cv2")
    h2d = []

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
            assert (r[-1][r[-1] != 1] == 0).all(), r[-1]
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    r1 = resource.getrusage(resource.RUSAGE_SELF)
    cpu = (r1.ru_utime - r0.ru_utime) + (r1.ru_stime - r0.ru_stime)
    return dict(images_per_s=len(paths) / dt, cpu_s_per_file=cpu / len(paths), h2d_bytes_per_batch=float(np.mean(h2d))), recs


def decode_kernels_ms(pipe, reps=10):
    """Device time per batch of each pn_jpeg_decode launch (torch.profiler, a run of its own, kernels summed by name)."""
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
    return out


def decode_ms(pipe, reps=50):
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
    return e0.elapsed_time(e1) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--rounds", type=int, default=3)
    args = ap.parse_args()
    torch.cuda.set_device(0)
    out = {"metric": "JPEG files to pose records, host vs GPU decode", "card": card(), "host_cores": os.cpu_count(),
           "workloads": {}}
    tmp = tempfile.mkdtemp()
    table = {"c2": (512, 64, 513, 513, 101, 16), "c2_noisy": (512, 64, 513, 513, 101, 16), "c3": (256, 32, 720, 1280, 50, 8)}
    for name, (n, batch, H, W, mid, os_) in table.items():
        paths = make_files(tmp, name, n)
        torch.manual_seed(0)
        model = posenet.MobileNetV1(mid, output_stride=os_).cuda().set_compute_dtype("bf16")
        kw = dict(depth=2, max_pose_detections=10, min_pose_score=0.25)
        host_pipe = posenet.BatchPipeline(model, batch, H, W, **kw)
        gpu_pipe = posenet.BatchPipeline(model, batch, H, W, jpeg=True, **kw)
        run_path(host_pipe, paths[:2 * batch], batch, False, False)                        # warm-up
        run_path(gpu_pipe, paths[:2 * batch], batch, True, False)
        res = {"host": [], "gpu": []}
        same = None
        for r in range(args.rounds):
            keep = r == 0
            h, rh = run_path(host_pipe, paths, batch, False, keep)
            g, rg = run_path(gpu_pipe, paths, batch, True, keep)
            res["host"].append(h)
            res["gpu"].append(g)
            if keep:
                same = all(all(np.array_equal(a, b) for a, b in zip(x, y)) for x, y in zip(rh, rg)) and len(rh) == len(rg)
        w = {"files": n, "batch": batch, "frame": [H, W], "model": mid, "output_stride": os_,
             "bytes_per_file": float(np.mean([os.path.getsize(p) for p in paths])), "records_identical": bool(same),
             "gpu_decode_ms_per_batch": decode_ms(gpu_pipe), "gpu_decode_kernels_ms_per_batch": decode_kernels_ms(gpu_pipe)}
        for k in ("host", "gpu"):
            w[k] = {m: [round(x[m], 6) for x in res[k]] for m in res[k][0]}
            w[k]["images_per_s_median"] = float(np.median(w[k]["images_per_s"]))
        w["speedup"] = w["gpu"]["images_per_s_median"] / w["host"]["images_per_s_median"]
        out["workloads"][name] = w
        print(name, json.dumps(w), flush=True)
        for p in paths:
            os.remove(p)
        del host_pipe, gpu_pipe, model
        torch.cuda.empty_cache()
    print(json.dumps(out))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
