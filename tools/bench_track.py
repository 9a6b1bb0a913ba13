"""Pose tracking and keypoint smoothing on the GPU (PoseTracker / BatchPipeline(track=...), pn_track_poses,
pn_smooth_keypoints): what they cost on the device and end to end, and what the same work costs on the host.

  - kernel: pn_track_poses device time per batch, CUDA events around --reps replays of a CUDA graph holding one call, on
    seeded synthetic records of moving people (P = 10, bench.py's max_pose_detections): a C3 batch of 32 frames (1280x720
    coordinates) and a C4 batch of 512 (257x257), each with its rows on 1 stream (a single video: the frames run one after
    another in one warp) and on 32 streams (rows round-robin).  The ids of every timed configuration are first checked against
    the numpy oracle (tests/trackref.py) over a few batches.
  - smoothing kernel: pn_smooth_keypoints (One Euro, PoseTracker(smoothing=OneEuro())) device time per batch, the same four
    configurations with the oracle's ids of those records, CUDA events around --reps replays of a graph holding one call (in
    place: each replay is one more frame of every stream, every detection an update).  The coordinates are first checked
    bit for bit against the numpy oracle (tests/smoothref.py) over a few batches.
  - end to end: C3 (bench.py's workload: MobileNetV1-50, 32 frames of 1280x720 resized to 721x1281 on the GPU, OS8, bf16,
    bench.py's decode settings, source_coords) images/s from BGR frames to records with and without track= (all rows one
    stream), the two arms alternated --rounds times (medians reported).  The arms' records are checked to be identical, and
    the track= arm's ids against the oracle fed with those records.  A third arm, track= with smoothing, is alternated with
    them; its records are checked against the smoothing oracle fed with the track= arm's records and ids.
  - host: the numpy oracles' time per frame on the C3 records, one thread: the per-frame cost a Python tracker (and a Python
    One Euro filter) between result() and the next submit() would put on the host.
Prints one JSON object (and writes it with --out), with the card's name and power limit.

    python tools/bench_track.py [--out FILE] [--reps 2000] [--steps 120] [--rounds 3]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (os.path.join(ROOT, "posenet-pytorch_b200"), ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench  # noqa: E402  (the workload table and decode settings)
from smoothref import SmoothOracle  # noqa: E402
from trackref import Oracle, synth_stream  # noqa: E402

P = bench.DECODE_KW["max_pose_detections"]
KERNEL_CASES = {"c3": (32, 720.0), "c4": (512, 257.0)}     # batch, frame size the synthetic people live in


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                        str(torch.cuda.current_device())], capture_output=True, text=True)
    return q.stdout.strip() or torch.cuda.get_device_name()


def records(batch, n_streams, size, n_batches, seed):
    """n_batches batches of rows round-robin over n_streams synthetic streams of moving people."""
    rng = np.random.default_rng(seed)
    per = -(-batch * n_batches // n_streams)
    recs = [synth_stream(rng, per, 8, P, 30, size=size) for _ in range(n_streams)]
    sid = np.arange(batch, dtype=np.int32) % n_streams
    out, cursor = [], [0] * n_streams
    for _ in range(n_batches):
        rows = []
        for s in sid:
            rows.append(tuple(a[cursor[s]] for a in recs[s]))
            cursor[s] += 1
        out.append(tuple(np.stack([r[j] for r in rows]) for j in range(3)))
    return out, sid


def kernel_case(batch, size, n_streams, reps):
    import posenet
    batches, sid = records(batch, n_streams, size, 8, seed=batch + n_streams)
    tracker = posenet.PoseTracker(n_streams)
    ref = Oracle(n_streams)
    dev = [torch.from_numpy(a).cuda() for a in batches[0]]
    sid_d = torch.from_numpy(sid).cuda()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=side):
        ids = tracker.update(*dev, sid_d)
    torch.cuda.current_stream().wait_stream(side)
    same = True
    for b in batches:                                            # ids against the oracle first
        for d, h in zip(dev, b):
            d.copy_(torch.from_numpy(h))
        g.replay()
        same &= bool(np.array_equal(ids.cpu().numpy(), ref.batch(*b, sid)))
    for _ in range(20):
        g.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        g.replay()
    e1.record()
    e1.synchronize()
    ms = e0.elapsed_time(e1) / reps
    det = float(np.mean([(b[0] > 0).sum(1).mean() for b in batches]))
    return {"us_per_batch": ms * 1e3, "ids_match_oracle": same, "detections_per_frame": det, "replays": reps}


def smooth_kernel_case(batch, size, n_streams, reps):
    import posenet
    batches, sid = records(batch, n_streams, size, 8, seed=batch + n_streams)
    tr = Oracle(n_streams)
    ids = [tr.batch(*b, sid) for b in batches]
    tracker = posenet.PoseTracker(n_streams, smoothing=posenet.OneEuro())
    ref = SmoothOracle(n_streams, **tracker.smoothing._asdict())
    kc_d = torch.from_numpy(batches[0][2]).cuda()
    ids_d = torch.from_numpy(ids[0]).cuda()
    sid_d = torch.from_numpy(sid).cuda()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=side):
        tracker.launch_smooth(ids_d, kc_d, sid_d)
    torch.cuda.current_stream().wait_stream(side)
    same = True
    for b, i in zip(batches, ids):                               # coordinates against the oracle first, bit for bit
        kc_d.copy_(torch.from_numpy(b[2]))
        ids_d.copy_(torch.from_numpy(i))
        g.replay()
        same &= bool(np.array_equal(kc_d.cpu().numpy().view(np.int64), ref.batch(i, b[2], sid).view(np.int64)))
    for _ in range(20):
        g.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        g.replay()
    e1.record()
    e1.synchronize()
    ms = e0.elapsed_time(e1) / reps
    det = float((ids[-1] > 0).sum(1).mean())
    return {"us_per_batch": ms * 1e3, "coords_match_oracle": same, "filtered_poses_per_frame": det, "replays": reps}


def end_to_end(args):
    import posenet
    mid, _, _, os_, batch, desc = bench.WORKLOADS["c3"]
    H, W = bench.SOURCE_SIZE["c3"]
    torch.manual_seed(0)
    model = posenet.MobileNetV1(mid, output_stride=os_).cuda().set_compute_dtype("bf16")
    rng = np.random.default_rng(1234)
    host = [torch.from_numpy(rng.integers(0, 256, (batch, H, W, 3), dtype=np.uint8)).pin_memory() for _ in range(4)]
    streams = [0] * batch
    tracker = posenet.PoseTracker(1)
    smoother = posenet.PoseTracker(1, smoothing=posenet.OneEuro())
    kw = dict(depth=2, output_stride=os_, source_coords=True, **bench.DECODE_KW)
    pipes = {"plain": posenet.BatchPipeline(model, batch, H, W, **kw),
             "track": posenet.BatchPipeline(model, batch, H, W, track=tracker, **kw),
             "track_smooth": posenet.BatchPipeline(model, batch, H, W, track=smoother, **kw)}
    items = {"plain": lambda hb: hb, "track": lambda hb: (hb, None, streams), "track_smooth": lambda hb: (hb, None, streams)}
    ref = list(pipes["plain"].run(host))
    got = list(pipes["track"].run(items["track"](hb) for hb in host))
    smoothed = list(pipes["track_smooth"].run(items["track_smooth"](hb) for hb in host))
    oracle = Oracle(1, min_part_score=bench.DECODE_KW["score_threshold"])
    smooth_oracle = SmoothOracle(1, **smoother.smoothing._asdict())
    same = all(all(np.array_equal(a, b) for a, b in zip(g[:4], r)) for g, r in zip(got, ref))
    ids_ok = all(np.array_equal(g[4], oracle.batch(r[0], r[1], r[2], streams)) for g, r in zip(got, ref))
    smooth_ok = all(np.array_equal(m[4], g[4]) and all(np.array_equal(m[j], g[j]) for j in (0, 1, 3)) and
                    np.array_equal(m[2].view(np.int64), smooth_oracle.batch(g[4], g[2], streams).view(np.int64))
                    for m, g in zip(smoothed, got))
    res = {"desc": desc, "frames": "%d x %dx%d, one stream" % (batch, H, W), "records_identical": bool(same),
           "ids_match_oracle": bool(ids_ok), "smoothed_coords_match_oracle": bool(smooth_ok),
           "poses_per_image": float(np.mean([(r[0] > 0).sum(1).mean() for r in ref]))}
    ips = {a: [] for a in pipes}
    for _ in range(args.rounds):                                 # arms alternated, each round timing each arm once
        for a, pipe in pipes.items():
            for _ in pipe.run(items[a](hb) for hb in host[:2]):
                pass
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in pipe.run((items[a](host[i % len(host)]) for i in range(args.steps)), copy=False):
                pass
            ips[a].append(batch * args.steps / (time.perf_counter() - t0))
    for a in pipes:
        res[a] = {"images_per_s": ips[a], "images_per_s_median": float(np.median(ips[a])),
                  "d2h_bytes_per_step": int(pipes[a].d2h_bytes_per_batch)}
    res["oracle_records"] = ref
    return res


def host_oracle_ms(recs, n_frames=2000):
    oracle = Oracle(1)
    ps, ks, kc = (np.concatenate([r[j] for r in recs]) for j in range(3))
    t0 = time.perf_counter()
    n = 0
    while n < n_frames:
        for i in range(len(ps)):
            oracle.frame(0, ps[i], ks[i], kc[i])
            n += 1
    return (time.perf_counter() - t0) / n * 1e3


def host_smooth_oracle_ms(recs, n_frames=2000):
    """The smoothing oracle alone, on the tracker oracle's ids of the records."""
    ps, ks, kc = (np.concatenate([r[j] for r in recs]) for j in range(3))
    ids = Oracle(1).batch(ps, ks, kc, [0] * len(ps))
    oracle = SmoothOracle(1)
    t0 = time.perf_counter()
    n = 0
    while n < n_frames:
        for i in range(len(ps)):
            oracle.frame(0, ids[i], kc[i])
            n += 1
    return (time.perf_counter() - t0) / n * 1e3


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--reps", type=int, default=2000)
    ap.add_argument("--steps", type=int, default=120)
    ap.add_argument("--rounds", type=int, default=3)
    args = ap.parse_args()
    torch.cuda.set_device(0)
    res = {"card": card(), "host_cores": os.cpu_count(), "P": P, "kernel": {}, "smooth_kernel": {}}
    for name, (batch, size) in KERNEL_CASES.items():
        for n_streams in (1, 32):
            key = "%s_batch%d_%dstream%s" % (name, batch, n_streams, "s" if n_streams > 1 else "")
            res["kernel"][key] = kernel_case(batch, size, n_streams, args.reps)
            print(json.dumps({key: res["kernel"][key]}), flush=True)
            res["smooth_kernel"][key] = smooth_kernel_case(batch, size, n_streams, args.reps)
            print(json.dumps({"smooth_" + key: res["smooth_kernel"][key]}), flush=True)
    e2e = end_to_end(args)
    recs = e2e.pop("oracle_records")
    res["c3_end_to_end"] = e2e
    print(json.dumps({"c3_end_to_end": e2e}), flush=True)
    res["host_oracle_ms_per_frame"] = {"c3_records": host_oracle_ms(recs),
                                       "synthetic_8_people": host_oracle_ms(records(32, 1, 720.0, 4, 7)[0])}
    res["host_smooth_oracle_ms_per_frame"] = {"c3_records": host_smooth_oracle_ms(recs),
                                              "synthetic_8_people": host_smooth_oracle_ms(records(32, 1, 720.0, 4, 7)[0])}
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
