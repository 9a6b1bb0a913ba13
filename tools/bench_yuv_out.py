"""Drawn frames out of BatchPipeline as YUV (yuv_out=code, converted on the GPU by pn_bgr_to_yuv) vs as BGR converted on the host.

Workloads (bench.py's models, weights, decode settings and seeded noise frames; overlay drawn at (0.25, 0.25) with
source_coords):
  - C3: MobileNetV1-50, 32 frames of 1280x720 resized to 721x1281 on the GPU, OS8;
  - C2: MobileNetV1-101 at 513x513, OS16, batch 64.  cv2 converts only even sizes, so the frames here are 512x512 (resized to
    the same 513x513 network input on the GPU), in every arm.
Arms, each handing the caller I420 / YUY2 frames a video sink takes:
  - bgr_host_i420: overlay pipeline returning BGR frames (3 B/px device-to-host), then cv2.cvtColor(COLOR_BGR2YUV_I420) of every
    frame on a pool of 16 host threads while the next batch runs;
  - i420, yuy2: BatchPipeline(yuv_out=code): the step's graph converts the drawn frames, 1.5 / 2 B/px device-to-host.
The arms are timed in turn, --rounds times over (median reported).  Every arm's bytes are checked against each other first: the
records of all arms, and each YUV arm's frames against cv2.cvtColor of the BGR arm's frames.

Also: D2H bytes per step (from shapes, records included); at C3 the conversion kernel's device time per batch (CUDA events over
--reps launches, rotating over enough buffers that the working set exceeds L2) with its bytes/s against a device-to-device copy of
the same traffic timed the same way in the same run; and host cv2.cvtColor ms per frame on 1 and 16 threads.  Prints one JSON
object (and writes it with --out), with the card's name and power limit.

    python tools/bench_yuv_out.py [--out FILE] [--steps 120] [--rounds 3] [--reps 200] [--workloads c3,c2]
"""
import argparse
import concurrent.futures
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

THR = (0.25, 0.25)                     # image_demo.py:53
ARMS = {"bgr_host_i420": None, "i420": cv2.COLOR_BGR2YUV_I420, "yuy2": cv2.COLOR_BGR2YUV_YUY2}
FRAMES = {"c3": (720, 1280), "c2": (512, 512)}
HOST_THREADS = 16
L2_BYTES = 126 << 20


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                        str(torch.cuda.current_device())], capture_output=True, text=True)
    return q.stdout.strip() or torch.cuda.get_device_name()


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
    layout = yuv.layout_of_output(code)
    shape = yuv.frame_shape(layout, H, W)
    traffic = batch * H * W * 3 + batch * int(np.prod(shape))
    n_sets = max(2, -(-2 * L2_BYTES // traffic))                 # the rotation's working set is at least twice L2
    srcs = [torch.randint(0, 256, (batch, H, W, 3), dtype=torch.uint8, device="cuda") for _ in range(n_sets)]
    dsts = [torch.empty((batch,) + shape, dtype=torch.uint8, device="cuda") for _ in range(n_sets)]
    conv_ms = rotating_ms(lambda k: yuv.convert_out(srcs[k], batch, H, W, layout, dsts[k]), n_sets, reps)
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


def host_convert(pool, frames):
    """The BGR arm's host step: every frame of a batch to I420 on the pool (cv2 releases the GIL)."""
    return list(pool.map(lambda f: cv2.cvtColor(f, cv2.COLOR_BGR2YUV_I420), frames))


def run_arm(pipe, arm, batches, pool, copy):
    """Yields what the caller gets per batch: (records..., I420 / YUY2 frames)."""
    for r in pipe.run(batches, copy=copy):
        yield r[:4] + (host_convert(pool, r[4]),) if arm == "bgr_host_i420" else r


def workload(name, args, pool):
    import posenet
    mid, _, _, os_, batch, desc = bench.WORKLOADS[name]
    H, W = FRAMES[name]
    torch.manual_seed(0)
    model = posenet.MobileNetV1(mid, output_stride=os_).cuda().set_compute_dtype("bf16")
    rng = np.random.default_rng(1234)
    host = [torch.from_numpy(rng.integers(0, 256, (batch, H, W, 3), dtype=np.uint8)).pin_memory() for _ in range(4)]
    pipes = {a: posenet.BatchPipeline(model, batch, H, W, depth=2, output_stride=os_, source_coords=True, overlay=THR,
                                      yuv_out=code, **bench.DECODE_KW) for a, code in ARMS.items()}
    res = {"desc": desc, "frames": "%d x %dx%d" % (batch, H, W), "arms": {}}
    # identical bytes: the records of every arm, and each YUV arm's frames against cv2 of the BGR frames
    ref = list(pipes["bgr_host_i420"].run(host))
    got = {a: list(run_arm(pipes[a], a, host, pool, True)) for a in ARMS}
    same = True
    for a, code in ARMS.items():
        for g, r in zip(got[a], ref):
            same &= all(np.array_equal(x, y) for x, y in zip(g[:4], r[:4]))
            same &= np.array_equal(np.stack(g[4]), np.stack([cv2.cvtColor(f, code or cv2.COLOR_BGR2YUV_I420) for f in r[4]]))
    res["bytes_identical"] = bool(same)
    res["poses_per_image"] = float(np.mean([(r[0] > 0).sum(1).mean() for r in ref]))
    del ref, got
    ips = {a: [] for a in ARMS}
    for _ in range(args.rounds):                                 # arms alternated, each round timing every arm once
        for a in ARMS:
            for _ in run_arm(pipes[a], a, host[:2], pool, False):
                pass
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in run_arm(pipes[a], a, (host[i % len(host)] for i in range(args.steps)), pool, False):
                pass
            ips[a].append(batch * args.steps / (time.perf_counter() - t0))
    frames = host[0].numpy()
    for a, code in ARMS.items():
        r = {"images_per_s": ips[a], "images_per_s_median": float(np.median(ips[a])),
             "d2h_bytes_per_step": int(pipes[a].d2h_bytes_per_batch)}
        if code is not None and name == "c3":
            r["conversion"] = kernel_and_copy(code, batch, H, W, args.reps)
        cc = code or cv2.COLOR_BGR2YUV_I420
        r["host_cvtColor_ms_per_frame"] = {"1_thread": host_cvt_ms(frames, cc, 1), "16_threads": host_cvt_ms(frames, cc, 16)}
        res["arms"][a] = r
    cv2.setNumThreads(1)
    del pipes, model, host
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--steps", type=int, default=120)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--reps", type=int, default=200)
    ap.add_argument("--workloads", default="c3,c2")
    args = ap.parse_args()
    torch.cuda.set_device(0)
    res = {"card": card(), "threshold": THR, "host_cores": os.cpu_count(), "host_threads_bgr_arm": HOST_THREADS,
           "gpus_visible": torch.cuda.device_count(), "workloads": {}}
    cv2.setNumThreads(1)                                         # the BGR arm's parallelism is the pool's
    with concurrent.futures.ThreadPoolExecutor(HOST_THREADS) as pool:
        for name in args.workloads.split(","):
            res["workloads"][name] = workload(name, args, pool)
            print(json.dumps({name: res["workloads"][name]}), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
