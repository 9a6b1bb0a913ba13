"""A phone's photo directory to pose records: 12 MP JPEG files of which half are portraits stored as landscape scans with EXIF
orientation 6 (and some 3 and 8), decoded by cv2 (ImageStream(mixed=True) -> BatchPipeline(mixed=True)), by the GPU with the
default routing (rotated files decoded by cv2 on the host: ImageStream(decode="gpu")), and by the GPU with orientation="gpu"
(rotated files decoded and rotated on the device).  The three arms are alternated on the same files and their records compared.

Inputs: the smooth set of tools/bench_jpeg_reduced.py (seeded synthetic 4032 x 3024 photos, q90 4:2:0) with an Exif APP1 segment
after SOI: orientation 6 on every odd file, 3 on files 2 mod 8, 8 on files 4 mod 8, 1 otherwise.  The stream is mixed (portraits
and landscapes), its frames at most 4032 x 4032 at 1/d; the network is MobileNetV1 101, OS16, at 513 x 513.

For every d: images/s per arm, host-decoded files per arm, host CPU seconds per file, and the device time of color_kernel (the
only launch the orientation changes) per batch of the same file tagged 1, 3 and 6 (torch.profiler, a run of its own).  Prints one
JSON object (and writes it with --out), with the card's name and power limit.

    python tools/bench_jpeg_orient.py [--out FILE] [--rounds 2] [--files 128] [--batch 32] [--reduce 1,4]
"""
import argparse
import json
import os
import re
import resource
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (os.path.join(ROOT, "posenet-pytorch_b200"), ROOT, os.path.join(ROOT, "tools")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import posenet  # noqa: E402
from posenet import jpeg as pj  # noqa: E402
from bench_jpeg_reduced import H, W, card, make_files  # noqa: E402


def exif(o):
    tiff = b"MM\x00*\x00\x00\x00\x08\x00\x01\x01\x12\x00\x03\x00\x00\x00\x01" + o.to_bytes(2, "big") + bytes(6)
    return b"\xff\xe1" + (len(tiff) + 8).to_bytes(2, "big") + b"Exif\0\0" + tiff


def orientation_of(i):
    return 6 if i % 2 else 3 if i % 8 == 2 else 8 if i % 8 == 4 else 1


def tag_files(paths):
    for i, p in enumerate(paths):
        with open(p, "rb") as f:
            b = f.read()
        with open(p, "wb") as f:
            f.write(b[:2] + exif(orientation_of(i)) + b[2:])


def run_arm(pipe, paths, batch, side, reduce, arm, keep):
    kw = dict(height=side, width=side, mixed=True, reduce=reduce)
    if arm != "cv2":
        kw.update(decode="gpu", orientation="gpu" if arm == "gpu_oriented" else "cv2")
    stream = posenet.ImageStream(paths, batch=batch, **kw)
    r0 = resource.getrusage(resource.RUSAGE_SELF)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    recs, status = [], []
    for r in pipe.run(((b, sh) for b, _, sh in stream.batches()), copy=keep):
        if keep:
            recs.append(r[:4])
        if arm != "cv2":
            status.append(r[-1])
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    r1 = resource.getrusage(resource.RUSAGE_SELF)
    cpu = (r1.ru_utime - r0.ru_utime) + (r1.ru_stime - r0.ru_stime)
    status = np.concatenate(status)[:len(paths)] if status else None   # rows past the last file are skipped (1)
    assert status is None or (status >= 0).all(), status
    return dict(images_per_s=len(paths) / dt, cpu_s_per_file=cpu / len(paths),
                host_decoded_files=len(paths) if status is None else int((status == 1).sum())), recs


def color_kernel_ms(path, batch, side, reduce, reps=10):
    """Device time per batch of color_kernel decoding `batch` copies of one file tagged 1, 3 and 6 (and of the whole decode)."""
    from torch.profiler import ProfilerActivity, profile
    with open(path, "rb") as f:
        raw = f.read()
    body = raw[2 + len(exif(1)):]                  # the file without its Exif segment
    out = {}
    dec = pj.Decoder(batch, batch * (len(body) + 64), side, side, reduce=reduce)
    frames = torch.empty((batch, side * side * 3), dtype=torch.uint8, device="cuda")
    for o in (1, 3, 6):
        b = raw[:2] + exif(o) + body
        descs = []
        for i in range(batch):
            d = pj.parse(b, orientation="gpu")
            assert d.kind == 0 and (d.orientation or 1) == o
            d.file_offset = i * len(b)
            descs.append(d)
        dec.arena[:batch * len(b)].copy_(torch.from_numpy(np.frombuffer(b * batch, np.uint8).copy()))
        dec.descs.copy_(torch.from_numpy(pj.desc_bytes(descs)))
        dec.decode(frames, side * side * 3)
        torch.cuda.synchronize()
        assert (dec.status == 0).all()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(reps):
                dec.decode(frames, side * side * 3)
            torch.cuda.synchronize()
        ms = {}
        for e in prof.key_averages():
            name = re.search(r"(\w+_kernel)", e.key)
            if name:
                ms[name.group(1)] = ms.get(name.group(1), 0.0) + e.device_time_total / 1000.0 / reps
        out["orientation_%d" % o] = {"color_kernel_ms": round(ms["color_kernel"], 4), "decode_ms": round(sum(ms.values()), 4)}
    base = out["orientation_1"]["color_kernel_ms"]
    for o in (3, 6):
        out["orientation_%d" % o]["color_vs_orientation_1"] = round(out["orientation_%d" % o]["color_kernel_ms"] / base, 4)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--files", type=int, default=128)
    ap.add_argument("--batch", type=int, default=32)
    ap.add_argument("--reduce", default="1,4")
    args = ap.parse_args()
    torch.cuda.set_device(0)
    batch, mid, os_ = args.batch, 101, 16
    out = {"metric": "12 MP phone directory (half EXIF-rotated) to pose records: cv2 vs GPU decode, default routing vs "
                     "orientation='gpu'", "card": card(), "host_cores": os.cpu_count(), "file_size": [H, W], "model": mid,
           "output_stride": os_, "batch": batch, "orientations": {str(o): sum(orientation_of(i) == o for i in range(args.files))
                                                                 for o in (1, 3, 6, 8)}, "workloads": {}}
    tmp = tempfile.mkdtemp()
    torch.manual_seed(0)
    model = posenet.MobileNetV1(mid, output_stride=os_).cuda().set_compute_dtype("bf16")
    paths = make_files(tmp, "smooth", args.files)
    tag_files(paths)
    arms = ("cv2", "gpu_default", "gpu_oriented")
    for d in (int(x) for x in args.reduce.split(",")):
        side = -(-max(H, W) // d)
        kw = dict(depth=2, max_pose_detections=10, min_pose_score=0.25, mixed=True, scale_factor=513.0 / side)
        pipes = {"cv2": posenet.BatchPipeline(model, batch, side, side, **kw)}
        pipes["gpu_default"] = pipes["gpu_oriented"] = posenet.BatchPipeline(model, batch, side, side, jpeg=True, reduce=d, **kw)
        for a in arms:                                                     # warm-up
            run_arm(pipes[a], paths[:batch], batch, side, d, a, False)
        res = {a: [] for a in arms}
        same = None
        for r in range(args.rounds):
            recs = {}
            for a in (arms if r % 2 == 0 else arms[::-1]):
                m, recs[a] = run_arm(pipes[a], paths, batch, side, d, a, r == 0)
                res[a].append(m)
            if r == 0:
                same = all(len(recs[a]) == len(recs["cv2"]) and all(all(np.array_equal(x, y) for x, y in zip(p, q))
                                                                    for p, q in zip(recs[a], recs["cv2"])) for a in arms[1:])
                assert same, "1/%d: the GPU arms' records differ from cv2's" % d
        wl = {"reduce": d, "frame_capacity": [side, side], "network_input": [pipes["cv2"].th, pipes["cv2"].tw], "files": len(paths),
              "bytes_per_file": float(np.mean([os.path.getsize(p) for p in paths])), "records_identical": bool(same),
              "color_kernel_per_batch": color_kernel_ms(paths[0], batch, side, d)}
        for a in arms:
            wl[a] = {m: [round(x[m], 6) for x in res[a]] for m in res[a][0]}
            wl[a]["images_per_s_median"] = float(np.median(wl[a]["images_per_s"]))
        wl["oriented_vs_default"] = round(wl["gpu_oriented"]["images_per_s_median"] / wl["gpu_default"]["images_per_s_median"], 4)
        wl["oriented_vs_cv2"] = round(wl["gpu_oriented"]["images_per_s_median"] / wl["cv2"]["images_per_s_median"], 4)
        out["workloads"]["smooth_r%d" % d] = wl
        print(d, json.dumps(wl), flush=True)
        if args.out:
            write(args.out, out)
        del pipes
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
