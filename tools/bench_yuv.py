"""YUV video frames into BatchPipeline (yuv=code, converted on the GPU by pn_yuv_to_bgr) vs BGR frames, at C3.

C3 is bench.py's webcam workload: MobileNetV1-50, 1280x720 frames resized to 721x1281 on the GPU, OS8, batch 32, bf16.  Arms:
  - bgr:  the existing path, pinned uint8 BGR batches (3 B/px over PCIe);
  - i420, nv12, yuy2: pinned batches in cv2's layout of that code (1.5 / 1.5 / 2 B/px), converted in the step's graph.
Every arm is fed the same seeded frames (the 4:2:2 batch repeats each chroma row over its row pair, so all arms convert to the
same BGR frames) and the records of all arms must be identical.  The arms are timed in turn, --rounds times over.

Per arm: end-to-end images/s (copies overlapped, CUDA graphs, results read in place like bench.py), H2D bytes per batch, the
conversion kernel's device time per batch (CUDA events over --reps launches, rotating over enough buffers that the working set
exceeds L2) with its bytes/s against a device-to-device copy of the same traffic timed the same way in the same run, and the host's
cv2.cvtColor time per frame on 1 and 16 threads (the work the device path takes off the host).  Prints one JSON object (and
writes it with --out), with the card's name and power limit.

    python tools/bench_yuv.py [--out FILE] [--steps 60] [--rounds 3] [--reps 200]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (os.path.join(ROOT, "posenet-pytorch_b200"), ROOT):
    if p not in sys.path:
        sys.path.insert(0, p)

import cv2  # noqa: E402
import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench  # noqa: E402  (the workload table and decode settings)

ARMS = {"bgr": None, "i420": cv2.COLOR_YUV2BGR_I420, "nv12": cv2.COLOR_YUV2BGR_NV12, "yuy2": cv2.COLOR_YUV2BGR_YUY2}
L2_BYTES = 126 << 20


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                        str(torch.cuda.current_device())], capture_output=True, text=True)
    return q.stdout.strip() or torch.cuda.get_device_name()


def make_batches(n_batches, batch, H, W, seed=1234):
    """Seeded random planes per batch -> {arm: [pinned host batch]}; the bgr arm holds cv2's conversion of the I420 frames."""
    rng = np.random.default_rng(seed)
    out = {a: [] for a in ARMS}
    for _ in range(n_batches):
        Y = rng.integers(0, 256, (batch, H, W), dtype=np.uint8)
        U = rng.integers(0, 256, (batch, H // 2, W // 2), dtype=np.uint8)
        V = rng.integers(0, 256, (batch, H // 2, W // 2), dtype=np.uint8)
        i420 = np.concatenate([Y.reshape(batch, -1), U.reshape(batch, -1), V.reshape(batch, -1)], 1).reshape(batch, H * 3 // 2, W)
        nv12 = np.concatenate([Y, np.stack([U, V], -1).reshape(batch, H // 2, W)], 1)
        U2, V2 = np.repeat(U, 2, 1), np.repeat(V, 2, 1)
        yuy2 = np.stack([Y[:, :, 0::2], U2, Y[:, :, 1::2], V2], -1).reshape(batch, H, W, 2)
        bgr = np.stack([cv2.cvtColor(f, cv2.COLOR_YUV2BGR_I420) for f in i420])
        for a, arr in (("bgr", bgr), ("i420", i420), ("nv12", nv12), ("yuy2", yuy2)):
            out[a].append(torch.from_numpy(np.ascontiguousarray(arr)).pin_memory())
    return out


def rotating_ms(launch, n_sets, reps):
    """Device ms per call of launch(k) over reps calls, k cycling over n_sets buffer sets (CUDA events)."""
    for k in range(n_sets):
        launch(k)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(reps):
        launch(i % n_sets)
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / reps


def kernel_and_copy(code, batch, H, W, reps):
    from posenet import yuv
    layout = yuv.layout_of(code)
    src_bytes = batch * int(np.prod(yuv.frame_shape(layout, H, W)))
    dst_bytes = batch * H * W * 3
    traffic = src_bytes + dst_bytes
    n_sets = max(2, -(-2 * L2_BYTES // traffic))                 # the rotation's working set is at least twice L2
    srcs = [torch.randint(0, 256, (src_bytes,), dtype=torch.uint8, device="cuda") for _ in range(n_sets)]
    dsts = [torch.empty((batch, H, W, 3), dtype=torch.uint8, device="cuda") for _ in range(n_sets)]
    conv_ms = rotating_ms(lambda k: yuv.convert(srcs[k], batch, H, W, layout, dsts[k]), n_sets, reps)
    half = traffic // 2                                          # a copy of traffic / 2 bytes reads and writes `traffic` bytes
    a = [torch.empty(half, dtype=torch.uint8, device="cuda") for _ in range(n_sets)]
    b = [torch.empty(half, dtype=torch.uint8, device="cuda") for _ in range(n_sets)]
    copy_ms = rotating_ms(lambda k: b[k].copy_(a[k]), n_sets, reps)
    del srcs, dsts, a, b
    torch.cuda.empty_cache()
    return {"kernel_ms_per_batch": conv_ms, "bytes_per_batch": traffic, "kernel_GBps": traffic / conv_ms / 1e6,
            "d2d_copy_ms_same_traffic": copy_ms, "d2d_copy_GBps": traffic / copy_ms / 1e6,
            "share_of_copy": copy_ms / conv_ms, "buffer_sets_rotated": n_sets}


def host_cvt_ms(frames, code, threads, n=64):
    cv2.setNumThreads(threads)
    cv2.cvtColor(frames[0], code)
    t0 = time.perf_counter()
    for i in range(n):
        cv2.cvtColor(frames[i % len(frames)], code)
    return (time.perf_counter() - t0) / n * 1e3


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--steps", type=int, default=60)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--reps", type=int, default=200)
    args = ap.parse_args()
    import posenet
    torch.cuda.set_device(0)
    mid, _, _, os_, batch, desc = bench.WORKLOADS["c3"]
    H, W = bench.SOURCE_SIZE["c3"]
    res = {"card": card(), "workload": desc, "frames": "%d x %dx%d" % (batch, H, W), "host_cores": os.cpu_count(),
           "gpus_visible": torch.cuda.device_count(), "arms": {}}
    torch.manual_seed(0)
    model = posenet.MobileNetV1(mid, output_stride=os_).cuda().set_compute_dtype("bf16")
    host = make_batches(4, batch, H, W)
    pipes = {a: posenet.BatchPipeline(model, batch, H, W, depth=2, output_stride=os_, yuv=code, **bench.DECODE_KW)
             for a, code in ARMS.items()}
    # identical records: every arm over the same frames
    recs = {a: list(pipes[a].run(host[a])) for a in ARMS}
    for a in ARMS:
        for got, ref in zip(recs[a], recs["bgr"]):
            assert all(np.array_equal(x, y) for x, y in zip(got, ref)), "records of arm %s differ from the BGR arm" % a
    res["records_identical"] = True
    res["poses_per_image"] = float(np.mean([(r[0] > 0).sum(1).mean() for r in recs["bgr"]]))
    ips = {a: [] for a in ARMS}
    for _ in range(args.rounds):                                 # arms alternated, each round timing every arm once
        for a in ARMS:
            pipe = pipes[a]
            for _ in pipe.run(host[a][:2], copy=False):
                pass
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in pipe.run((host[a][i % len(host[a])] for i in range(args.steps)), copy=False):
                pass
            ips[a].append(batch * args.steps / (time.perf_counter() - t0))
    for a, code in ARMS.items():
        r = {"images_per_s": ips[a], "images_per_s_median": float(np.median(ips[a])),
             "h2d_bytes_per_batch": int(pipes[a].h2d_bytes_per_batch)}
        if code is not None:
            r["conversion"] = kernel_and_copy(code, batch, H, W, args.reps)
            frames = host[a][0].numpy()
            r["host_cvtColor_ms_per_frame"] = {"1_thread": host_cvt_ms(frames, code, 1), "16_threads": host_cvt_ms(frames, code, 16)}
        res["arms"][a] = r
        print(json.dumps({a: r}), flush=True)
    res["multi_gpu"] = "not measured: this script runs on one GPU (%d visible)" % torch.cuda.device_count()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
