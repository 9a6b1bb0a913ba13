"""Directories of progressive JPEG files to pose records: progressive="cv2" (every file decoded by cv2 on the host thread pool)
vs progressive="gpu" (pn_jpeg_parse_progressive + the device decode), both through ImageStream(decode="gpu") ->
BatchPipeline(jpeg=True), alternated on the same files with the records of both arms compared in the same run.

Workloads (all files progressive, cv2's jpeg_simple_progression at q90 4:2:0):
  c2     512 files of 513 x 513 (smooth synthetic frames); MobileNetV1 101, OS16, batch 64, full-size decode
  12mp   96 files of 4032 x 3024 (bench_jpeg_reduced.py's smooth photos); the same network at 513 x 385, decoded at 1/4
For each: files -> records images/s of both arms, host CPU seconds per file, the device time of one decode per batch (CUDA
events) and its per-kernel shares (torch.profiler, a run of its own; progressive_kernel is the entropy stage).  Then the same
per-kernel split for a batch of BASELINE c2 files, where progressive_kernel only checks each descriptor's kind, and
tools/bench_jpeg.py --rounds 2 in a subprocess for the baseline rates.  Prints one JSON object (and writes it with --out),
with the card's name and power limit and the host's core count.

    python tools/bench_jpeg_progressive.py [--out FILE] [--rounds 3] [--skip-baseline]
"""
import argparse
import json
import os
import resource
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (os.path.join(ROOT, "posenet-pytorch_b200"), ROOT, os.path.join(ROOT, "tools")):
    if p not in sys.path:
        sys.path.insert(0, p)

import cv2  # noqa: E402
import numpy as np  # noqa: E402
import torch  # noqa: E402

import posenet  # noqa: E402
from oracle import synth  # noqa: E402  (input generator only)
from bench_jpeg_reduced import card, decode_kernels_ms, decode_ms, write  # noqa: E402

PROG = [cv2.IMWRITE_JPEG_QUALITY, 90, cv2.IMWRITE_JPEG_PROGRESSIVE, 1]


def make_files(d, kind, n, progressive=True):
    params = PROG if progressive else PROG[:2]
    if kind == "c2":
        base = [synth.smooth_image(513, 513, 500 + s) for s in range(8)]
    else:
        base = [cv2.resize(synth.smooth_image(756, 1008, 900 + s), (4032, 3024), interpolation=cv2.INTER_CUBIC) for s in range(4)]
    paths = []
    for i in range(n):
        p = os.path.join(d, "%s_%s_%04d.jpg" % (kind, "p" if progressive else "b", i))
        cv2.imwrite(p, np.roll(base[i % len(base)], 7 * i, axis=1), params)
        paths.append(p)
    return paths


def run_arm(pipe, paths, batch, reduce, progressive, keep_records):
    stream = posenet.ImageStream(paths, batch=batch, reduce=reduce, decode="gpu", progressive=progressive)
    r0 = resource.getrusage(resource.RUSAGE_SELF)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    recs, host = [], 0
    for r, nv in zip(pipe.run((b for b, _ in stream.batches()), copy=keep_records), stream.valid_counts()):
        if keep_records:
            recs.append(r[:4])
        assert (r[-1] >= 0).all(), r[-1]
        host += int((r[-1][:nv] == 1).sum())            # rows past the last file are skipped (status 1) in both arms
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    r1 = resource.getrusage(resource.RUSAGE_SELF)
    cpu = (r1.ru_utime - r0.ru_utime) + (r1.ru_stime - r0.ru_stime)
    return dict(images_per_s=len(paths) / dt, cpu_s_per_file=cpu / len(paths), host_decodes=host), recs


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--skip-baseline", action="store_true")
    args = ap.parse_args()
    torch.cuda.set_device(0)
    batch, mid, os_ = 64, 101, 16
    out = {"metric": "progressive JPEG files to pose records: progressive='cv2' (host) vs 'gpu'", "card": card(),
           "host_cores": os.cpu_count(), "model": mid, "output_stride": os_, "batch": batch, "workloads": {}}
    tmp = tempfile.mkdtemp()
    torch.manual_seed(0)
    model = posenet.MobileNetV1(mid, output_stride=os_).cuda().set_compute_dtype("bf16")
    for kind, n, reduce, (H, W) in (("c2", 512, 1, (513, 513)), ("12mp", 96, 4, (3024, 4032))):
        paths = make_files(tmp, kind, n)
        h, w = -(-H // reduce), -(-W // reduce)
        kw = dict(depth=2, max_pose_detections=10, min_pose_score=0.25, scale_factor=513.0 / w)
        pipe = posenet.BatchPipeline(model, batch, h, w, jpeg=True, reduce=reduce, **kw)     # the stream's default arena
        for prog in ("cv2", "gpu"):                                                          # warm-up
            run_arm(pipe, paths[:batch], batch, reduce, prog, False)
        res = {"cv2": [], "gpu": []}
        same = None
        for r in range(args.rounds):
            keep = r == 0
            for prog in ("cv2", "gpu") if r % 2 == 0 else ("gpu", "cv2"):
                x, recs = run_arm(pipe, paths, batch, reduce, prog, keep)
                res[prog].append(x)
                if keep:
                    res[prog + "_recs"] = recs
            if keep:
                a, b = res.pop("cv2_recs"), res.pop("gpu_recs")
                same = len(a) == len(b) and all(all(np.array_equal(u, v) for u, v in zip(x, y)) for x, y in zip(a, b))
                assert same, "%s: the GPU decode's records differ from cv2's" % kind
        wl = {"reduce": reduce, "file_size": [H, W], "frame": [h, w], "files": n,
              "bytes_per_file": float(np.mean([os.path.getsize(p) for p in paths])), "records_identical": bool(same),
              "gpu_decode_ms_per_batch": round(decode_ms(pipe), 4), "gpu_decode_kernels_ms_per_batch": decode_kernels_ms(pipe)}
        for k in ("cv2", "gpu"):
            wl[k] = {m: [round(x[m], 6) for x in res[k]] for m in res[k][0]}
            wl[k]["images_per_s_median"] = float(np.median(wl[k]["images_per_s"]))
        assert max(wl["gpu"]["host_decodes"]) == 0 and min(wl["cv2"]["host_decodes"]) == n
        wl["speedup"] = round(wl["gpu"]["images_per_s_median"] / wl["cv2"]["images_per_s_median"], 4)
        out["workloads"][kind] = wl
        print(kind, json.dumps(wl), flush=True)
        if args.out:
            write(args.out, out)
        if kind == "c2":                    # the same decode of baseline files: what the extra launch costs them
            base = make_files(tmp, kind, batch, progressive=False)
            run_arm(pipe, base, batch, 1, "gpu", False)
            out["baseline_c2_decode_kernels_ms_per_batch"] = decode_kernels_ms(pipe)
            out["baseline_c2_decode_ms_per_batch"] = round(decode_ms(pipe), 4)
            for p in base:
                os.remove(p)
        del pipe
        torch.cuda.empty_cache()
        for p in paths:
            os.remove(p)
    if not args.skip_baseline:
        r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "bench_jpeg.py"), "--rounds", "2"], capture_output=True,
                           text=True)
        assert r.returncode == 0, r.stderr[-2000:]
        out["bench_jpeg"] = json.loads(r.stdout.strip().splitlines()[-1])
    if args.out:
        write(args.out, out)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
