"""PNG files of the drawn frames on the GPU (pn_png_encode) vs cv2.imencode(".png") on the host, and what encoding costs end to
end.

For the bench workloads C2 / C3 / C4 (bench.py's models and decode settings; C3 draws on the 1280x720 source frames), with the
records the bench model decodes drawn at 0.25 / 0.25 (image_demo.py:53) on smooth synthetic frames (oracle/synth.py), encoded as
cv2 does without params.  Smooth synthetic frames compress far better under Z_RLE than photographs do (which come close to
their raw size), so the file bytes and D2H figures here are a lower end:
  - device time of one pn_png_encode per batch (CUDA events over many calls) and each kernel's share (torch.profiler, a run of
    its own);
  - cv2.imencode(".png") per image on one host core and over all cores (a thread pool: cv2 releases the GIL);
  - images/s from pinned batches: BatchPipeline(overlay) + cv2.imencode(".png") of every frame on a thread pool, against
    BatchPipeline(overlay, encode=[], encode_ext=".png"), and the D2H bytes per batch of both.  Both paths' files are asserted
    identical.
Prints one JSON object (and writes it with --out), with the card's name and power limit.

    python tools/bench_png_encode.py [--out FILE] [--steps 20]
"""
import argparse
import concurrent.futures
import json
import os
import re
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
from oracle import synth  # noqa: E402  (input generator only)

THR = (0.25, 0.25)
EXT = ".png"


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                        str(torch.cuda.current_device())], capture_output=True, text=True)
    return q.stdout.strip() or torch.cuda.get_device_name()


def device_ms(enc, frames_dev, stride, reps):
    for _ in range(3):
        enc.encode(frames_dev, stride)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        enc.encode(frames_dev, stride)
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / reps


def kernel_shares(enc, frames_dev, stride, reps=10):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            enc.encode(frames_dev, stride)
        torch.cuda.synchronize()
    t = {}
    for e in prof.key_averages():
        m = re.search(r"(\w+_kernel)(<\w+>)?\(", e.key)
        if m:
            name = m.group(1) + (m.group(2) or "")
            t[name] = t.get(name, 0.0) + e.device_time_total
    total = sum(t.values()) or 1.0
    return {k: {"ms_per_call": v / reps / 1e3, "share": v / total} for k, v in sorted(t.items(), key=lambda kv: -kv[1])}


def host_ms(frames, n_img, threads):
    cv2.setNumThreads(1)
    enc = lambda i: cv2.imencode(EXT, frames[i % len(frames)])[1]
    enc(0)
    t0 = time.perf_counter()
    if threads == 1:
        for i in range(n_img):
            enc(i)
    else:
        with concurrent.futures.ThreadPoolExecutor(threads) as ex:
            list(ex.map(enc, range(n_img)))
    return (time.perf_counter() - t0) / n_img * 1e3


def e2e(model, batch, sh, sw, os_, resize, host, steps, device_encode, pool):
    """images/s over `steps` steps and the D2H bytes of the last one; the host arm encodes every returned batch on `pool` while
    the GPU runs on.  Also returns the last batch's files."""
    import posenet
    pipe = posenet.BatchPipeline(model, batch, sh, sw, depth=2, output_stride=os_, source_coords=resize, overlay=THR,
                                 **(dict(encode=[], encode_ext=EXT) if device_encode else {}), **bench.DECODE_KW)

    def host_files(frames):
        return list(pool.map(lambda f: cv2.imencode(EXT, f)[1].tobytes(), frames))
    for r in pipe.run(host[:2]):
        pass
    torch.cuda.synchronize()
    pending, last = [], None
    outer = concurrent.futures.ThreadPoolExecutor(2)                   # hands each batch to the pool, off this thread
    t0 = time.perf_counter()
    for r in pipe.run((host[i % len(host)] for i in range(steps)), copy=False):
        if device_encode:
            last = r[4]
        else:
            pending.append(outer.submit(host_files, r[4].copy()))
            if len(pending) > 2:
                last = pending.pop(0).result()
    for f in pending:
        last = f.result()
    dt = time.perf_counter() - t0
    outer.shutdown()
    d2h = pipe.nrec * 8 + 8 * (batch + 1) + pipe.last_file_bytes if device_encode else pipe.d2h_bytes_per_batch
    return batch * steps / dt, int(d2h), last


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--host-images", type=int, default=64)
    ap.add_argument("--workloads", default="c2,c3,c4")
    args = ap.parse_args()
    import posenet
    from posenet import png as pp
    torch.cuda.set_device(0)
    cores = os.cpu_count()
    res = {"card": card(), "threshold": THR, "params": "cv2 defaults (SUB filter, zlib level 1, Z_RLE)", "cores": cores, "workloads": {}}
    pool = concurrent.futures.ThreadPoolExecutor(cores)
    for name in args.workloads.split(","):
        mid, H, W, os_, batch, desc = bench.WORKLOADS[name]
        sh, sw = bench.SOURCE_SIZE.get(name, (H, W))
        torch.manual_seed(0)
        model = posenet.MobileNetV1(mid, output_stride=os_).cuda().set_compute_dtype("bf16")
        base = [synth.smooth_image(sh, sw, s) for s in range(8)]
        host = [torch.from_numpy(np.stack([np.roll(base[(k + i) % 8], 7 * i, axis=1) for i in range(batch)])).pin_memory()
                for k in range(4)]
        frames_dev = host[0].cuda()
        x, scale = posenet.resize_u8_gpu(frames_dev, 1.0, os_) if (sh, sw) != (H, W) else (frames_dev, np.ones(2))
        ps, ks, kc, _, counts = posenet.decode_multiple_poses_batch(*model.forward_u8(x), output_stride=os_, **bench.DECODE_KW)
        kc = kc * torch.as_tensor(scale, device=kc.device)
        posenet.draw_skel_and_kp_batch(frames_dev, ps, ks, kc, *THR)
        drawn = frames_dev.cpu().numpy()
        enc = pp.Encoder(batch, sh, sw)
        stride = sh * sw * 3
        r = {"desc": desc, "frames": "%d x %dx%d" % (batch, sh, sw), "poses_per_image": float(counts.float().mean()),
             "device_ms_per_batch": device_ms(enc, frames_dev, stride, args.reps),
             "kernels": kernel_shares(enc, frames_dev, stride)}
        files = enc.files()
        assert files == [cv2.imencode(EXT, f)[1].tobytes() for f in drawn]
        r["file_bytes_per_image"] = float(np.mean([len(f) for f in files]))
        r["raw_bytes_per_image"] = stride
        r["host_ms_per_image_1core"] = host_ms(drawn, args.host_images, 1)
        r["host_ms_per_image_all_cores"] = host_ms(drawn, args.host_images * 8, cores)
        ips_h, d2h_h, files_h = e2e(model, batch, sh, sw, os_, (sh, sw) != (H, W), host, args.steps, False, pool)
        ips_d, d2h_d, files_d = e2e(model, batch, sh, sw, os_, (sh, sw) != (H, W), host, args.steps, True, pool)
        assert files_h == files_d, "device and host files differ"
        r["pipeline_overlay_host_encode"] = {"images_per_s": ips_h, "d2h_bytes_per_step": d2h_h}
        r["pipeline_overlay_device_encode"] = {"images_per_s": ips_d, "d2h_bytes_per_step": d2h_d}
        r["identical_bytes"] = True
        res["workloads"][name] = r
        print(json.dumps({name: r}), flush=True)
        del model, host, frames_dev, enc
        torch.cuda.empty_cache()
    pool.shutdown()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
