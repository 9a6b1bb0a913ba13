"""Pose overlays on the GPU (pn_draw_poses) vs cv2 on the host, and what drawing costs end to end.

For the bench workloads C2 / C3 / C4 (bench.py's models, seeds and frames; C3 draws on the 1280x720 source frames):
  - device time of one draw launch per batch (CUDA events), with the bench's decoded records and with synthetic crowds of
    10 to 50 people per image;
  - host time of posenet.draw_skel_and_kp for the same records, on one core and on all cores (one process per core; the
    helper's Python part holds the GIL, so threads do not scale);
  - images/s of BatchPipeline with and without overlay (copies overlapped, CUDA graphs, results read in place like bench.py).
Prints one JSON object (and writes it with --out), with the card's name and power limit.

    python tools/bench_overlay.py [--out FILE] [--steps 30] [--host-images 64]
"""
import argparse
import concurrent.futures
import json
import multiprocessing
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

import bench  # noqa: E402  (the workload table, decode settings and input seeds)

THR = (0.25, 0.25)                     # image_demo.py:53


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                        str(torch.cuda.current_device())], capture_output=True, text=True)
    return q.stdout.strip() or torch.cuda.get_device_name()


def crowd(rng, n, people, P, H, W):
    ps = np.zeros((n, P))
    ps[:, :people] = np.sort(rng.uniform(0.3, 1, (n, people)))[:, ::-1]
    ks = rng.uniform(0, 1, (n, P, 17))
    centre = np.stack([rng.uniform(0, H, (n, P, 1)), rng.uniform(0, W, (n, P, 1))], -1)
    kc = centre + rng.normal(0, min(H, W) / 10, (n, P, 17, 2))          # people of about a fifth of the frame
    return ps, ks, kc


def device_ms(frames_dev, recs, reps):
    import posenet
    work = frames_dev.clone()
    for _ in range(3):
        posenet.draw_skel_and_kp_batch(work, *recs, *THR)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    total = 0.0
    for _ in range(reps):                                                 # fresh frames each time (the draw blends in place)
        work.copy_(frames_dev)
        e0.record()
        posenet.draw_skel_and_kp_batch(work, *recs, *THR)
        e1.record()
        e1.synchronize()
        total += e0.elapsed_time(e1)
    return total / reps


_HOST = None                           # (frames, records) inherited by the forked workers


def _draw_one(i):
    import posenet
    frames, (ps, ks, kc) = _HOST
    i %= frames.shape[0]
    posenet.draw_skel_and_kp(frames[i].copy(), ps[i], ks[i], kc[i], *THR)


def host_ms(frames, recs, n_img, procs):
    """Wall time per image of draw_skel_and_kp over n_img images, in this process or in `procs` forked ones."""
    global _HOST
    _HOST = (frames, tuple(r.cpu().numpy() for r in recs))
    cv2.setNumThreads(1)
    _draw_one(0)
    if procs == 1:
        t0 = time.perf_counter()
        for i in range(n_img):
            _draw_one(i)
        return (time.perf_counter() - t0) / n_img * 1e3
    with concurrent.futures.ProcessPoolExecutor(procs, mp_context=multiprocessing.get_context("fork")) as ex:
        list(ex.map(_draw_one, range(procs)))                          # workers up and warm
        t0 = time.perf_counter()
        list(ex.map(_draw_one, range(n_img), chunksize=max(1, n_img // (4 * procs))))
        return (time.perf_counter() - t0) / n_img * 1e3


def e2e(model, batch, sh, sw, os_, host, steps, overlay):
    import posenet
    pipe = posenet.BatchPipeline(model, batch, sh, sw, depth=2, output_stride=os_, source_coords=overlay is not None,
                                 overlay=overlay, **bench.DECODE_KW)
    for _ in pipe.run(host[:2]):
        pass
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in pipe.run((host[i % len(host)] for i in range(steps)), copy=False):
        pass
    return batch * steps / (time.perf_counter() - t0), pipe.d2h_bytes_per_batch


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--host-images", type=int, default=64)
    ap.add_argument("--workloads", default="c2,c3,c4")
    args = ap.parse_args()
    import posenet
    torch.cuda.set_device(0)
    res = {"card": card(), "threshold": THR, "cores": os.cpu_count(), "workloads": {}}
    for name in args.workloads.split(","):
        mid, H, W, os_, batch, desc = bench.WORKLOADS[name]
        sh, sw = bench.SOURCE_SIZE.get(name, (H, W))
        torch.manual_seed(0)
        model = posenet.MobileNetV1(mid, output_stride=os_).cuda().set_compute_dtype("bf16")
        rng = np.random.default_rng(1234)
        host = [torch.from_numpy(rng.integers(0, 256, (batch, sh, sw, 3), dtype=np.uint8)).pin_memory() for _ in range(4)]
        frames = host[0].numpy()
        frames_dev = host[0].cuda()
        x, scale = posenet.resize_u8_gpu(frames_dev, 1.0, os_) if (sh, sw) != (H, W) else (frames_dev, np.ones(2))
        ps, ks, kc, _, counts = posenet.decode_multiple_poses_batch(*model.forward_u8(x), output_stride=os_, **bench.DECODE_KW)
        kc = kc * torch.as_tensor(scale, device=kc.device)
        recs = (ps, ks, kc)
        r = {"desc": desc, "frames": "%d x %dx%d" % (batch, sh, sw), "bench_records": {
            "poses_per_image": float(counts.float().mean()), "device_ms_per_batch": device_ms(frames_dev, recs, args.reps),
            "host_ms_per_image_1core": host_ms(frames, recs, args.host_images, 1),
            "host_ms_per_image_all_cores": host_ms(frames, recs, args.host_images * 8, os.cpu_count())}}
        for people in (10, 20, 30, 50):
            cr = crowd(np.random.default_rng(people), batch, people, 50, sh, sw)
            crd = tuple(torch.as_tensor(a, device="cuda") for a in cr)
            r["crowd_%d" % people] = {"device_ms_per_batch": device_ms(frames_dev, crd, args.reps),
                                      "host_ms_per_image_1core": host_ms(frames, crd, args.host_images, 1),
                                      "host_ms_per_image_all_cores": host_ms(frames, crd, args.host_images * 8, os.cpu_count())}
        for key, ov in (("pipeline_plain", None), ("pipeline_overlay", THR)):
            ips, d2h = e2e(model, batch, sh, sw, os_, host, args.steps, ov)
            r[key] = {"images_per_s": ips, "d2h_bytes_per_step": int(d2h)}
        res["workloads"][name] = r
        print(json.dumps({name: r}), flush=True)
        del model, host, frames_dev
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
