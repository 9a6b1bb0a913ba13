"""bench.py -- images/sec of the PoseNet hot path (backbone + heads + multi-pose decode).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload c2|c3|c4] [--dump-outputs DIR]

One "step" = one pass of  uint8 images -> (fused preprocess) stem -> 13 separable blocks -> heads ->
part candidates -> greedy decode  over one batch.  Default workload = BASELINE.json configs[1]:
MobileNetV1 model 101, 513x513, output stride 16, batch 64 per GPU, bf16, random-init weights, synthetic images.
Rank 0 prints ONE JSON line (see the keys below); with ``--dump-outputs DIR`` it also writes the pose records of the last
timed step to ``DIR/*.npy`` (inputs and weights are seeded, so two builds can be compared output for output).
``--impl reference`` times the reference's own CPU code on the host
cores instead: the unmodified reference package byte-compiled into ``oracle/_ref`` by ``oracle/make_ref.py``
(``cpu_baseline.kind`` "reference"), or, when that build is absent, the oracle port (``kind`` "port": torch-CPU fp32
convs + numpy float64 decode).  Both arms print the same ``config`` dict; how each arm batches the workload is in ``run``.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "posenet-pytorch_b200")
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)          # `oracle` (checker / CPU arm).  The product arm adds PKG; the reference arm adds oracle/_ref:
                                      # both packages are called `posenet`, so a process imports exactly one of them.

import numpy as np  # noqa: E402
import torch  # noqa: E402

WORKLOADS = {
    # name: (model, H, W, output_stride, batch per GPU, description)
    "c2": (101, 513, 513, 16, 64, "MobileNetV1-101 513x513 OS16 batch 64/GPU bf16 (BASELINE configs[1])"),
    "c3": (50, 721, 1281, 8, 32, "MobileNetV1-50 1280x720 frames -> 721x1281 (cv2-exact GPU resize inside the step) OS8 batch 32/GPU bf16 "
                                  "(BASELINE configs[2])"),
    "c4": (75, 257, 257, 32, 512, "MobileNetV1-75 257x257 OS32 batch 512/GPU bf16 (BASELINE configs[3])"),
}
SOURCE_SIZE = {"c3": (720, 1280)}          # frames arrive at webcam resolution (utils.py:51-55) and are resized on the GPU
METRIC = "images/sec (backbone+decode)"
DECODE_KW = dict(max_pose_detections=10, score_threshold=0.5, nms_radius=20, min_pose_score=0.25)  # benchmark.py:37-44


def workload_config(name):
    """The `config` object of the JSON line -- identical for the product arm and the reference arm (what is computed);
    how an arm batches it (64 images per launch chain on the GPU, one image at a time on the host like benchmark.py:32-44)
    is reported separately under `run`."""
    mid, H, W, os_, batch, desc = WORKLOADS[name]
    sh, sw = SOURCE_SIZE.get(name, (H, W))
    return {"workload": desc, "model": "mobilenet_v1_%03d" % mid, "network_input": "%dx%d" % (H, W), "source_frames": "%dx%d" % (sh, sw),
            "output_stride": os_, "decode": DECODE_KW, "weights": "random-init (torch default init, seed 0)",
            "images": "synthetic uint8 noise, seeded"}


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return dict(hbm=d["hbm_gbs"], bf16_burst=d["bf16_tflops"], bf16_sustained=d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                    src="measured")
    return dict(hbm=6650.0, bf16_burst=1590.0, bf16_sustained=1400.0, src="fallback")   # B200_PROFILING.md


def bind_to_gpu_numa_node(index):
    """Pin this process to the CPUs NVML reports as local to the GPU, so that the pinned host batches of the end-to-end leg are
    allocated on the GPU's NUMA node and the H2D copies of 8 ranks do not all cross the socket interconnect.  Best effort."""
    try:
        import pynvml
        pynvml.nvmlInit()
        visible = os.environ.get("CUDA_VISIBLE_DEVICES")
        phys = int(visible.split(",")[index]) if visible and all(v.strip().isdigit() for v in visible.split(",")) else index
        h = pynvml.nvmlDeviceGetHandleByIndex(phys)
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
        cpus = {64 * i + b for i, w in enumerate(words) for b in range(64) if (int(w) >> b) & 1}
        before = set(os.sched_getaffinity(0))
        cpus &= before
        if cpus:
            os.sched_setaffinity(0, cpus)
            return "gpu-local cpus (%d of %d)" % (len(cpus), len(before)), before
    except Exception:
        pass
    return "unchanged", None


class ClockSampler(threading.Thread):
    """SM clock and throttle reasons sampled DURING the timed region.  NVML is polled in-process (a reading takes
    ~0.1 ms, so even a 15 ms timed region holds dozens); `nvidia-smi` (one reading per ~100 ms) is the fallback
    when the NVML binding is missing."""
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], threading.Event()     # rows: (t, sm_mhz, reason flags)
        self.max_mhz, self.source, self.window = None, "nvidia-smi", None
        try:
            import pynvml
            pynvml.nvmlInit()
            visible = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(visible.split(",")[index]) if visible and all(v.strip().isdigit() for v in visible.split(",")) else index
            self.h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.nv = pynvml
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.bits = [pynvml.nvmlClocksEventReasonHwSlowdown, pynvml.nvmlClocksEventReasonHwThermalSlowdown,
                         pynvml.nvmlClocksEventReasonSwThermalSlowdown, pynvml.nvmlClocksEventReasonSwPowerCap]
            self.source = "nvml"
            self._read()                                         # first NVML query is slow (~10 ms): pay for it here
        except Exception:
            self.nv = None

    def _read(self):
        if self.nv is not None:
            mhz = float(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM))
            mask = int(self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
            return mhz, [bool(mask & b) for b in self.bits]
        out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=5).stdout.strip()
        c = [x.strip() for x in out.split(",")]
        self.max_mhz = float(c[1])
        return float(c[0]), [x.lower().startswith("active") for x in c[2:6]]

    def sample_now(self):
        """One reading from the calling thread (the main thread calls this right after enqueueing the timed steps, while
        the GPU is still executing them, so that even a few-millisecond region holds a reading)."""
        try:
            mhz, flags = self._read()
            self.rows.append((time.perf_counter(), mhz, flags))
        except Exception:
            pass

    def run(self):
        while not self.stop_flag.is_set():
            self.sample_now()
            self.stop_flag.wait(0.0005 if self.nv is not None else 0.2)

    def summary(self):
        """`window` = (t0, t1) host times bracketing the timed region (set by the caller): readings inside it are
        counted separately; the median and the reasons come from the readings inside the window when there are any."""
        self.stop_flag.set()
        self.join(timeout=6)
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["clock query unavailable"], "samples": 0}
        inside = [r for r in self.rows if self.window and self.window[0] <= r[0] <= self.window[1]]
        use = inside or self.rows
        sm = sorted(r[1] for r in use)
        reasons = [n for i, n in enumerate(self.NAMES) if any(r[2][i] for r in use)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_min_mhz": sm[0], "sm_max_mhz": self.max_mhz, "reasons": reasons,
                "samples": len(self.rows), "samples_in_timed_region": len(inside), "source": self.source}


# ------------------------------------------------------------------------------------------ reference arm
def cpu_reference_run(workload, images_per_step, steps, warmup):
    """The reference's path on the host cores, one image at a time like benchmark.py:32-44 (plus the pre-processing of :29):
    utils._process_input (utils.py:13-26) -> MobileNetV1.forward (mobilenet_v1.py:156-162, torch CPU fp32) ->
    decode_multiple_poses (decode_multi.py:61-148).  Runs the reference's OWN code from oracle/_ref when that build exists
    (kind "reference"), the oracle port otherwise (kind "port").  Must be called in a process that has not imported the
    product package (both are named `posenet`)."""
    from oracle import make_ref, synth
    mid, H, W, os_, _, _ = WORKLOADS[workload]
    sh, sw = SOURCE_SIZE.get(workload, (H, W))
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    imgs = [synth.noise_image(sh, sw, s) for s in range(4)]
    if make_ref.available():
        assert "posenet" not in sys.modules, "the reference arm needs a process that has not imported the product package"
        sys.path.insert(0, make_ref.IMPORT_PATH)
        import posenet as ref
        import posenet.decode_multi as ref_dm
        assert os.path.realpath(ref.__file__).startswith(os.path.realpath(make_ref.REF_DIR)), ref.__file__
        torch.manual_seed(0)
        model = ref.MobileNetV1(mid, output_stride=os_)          # load_model minus the checkpoint file: default init, seeded
        kind, how = "reference", "unmodified reference package (oracle/_ref, byte-compiled by oracle/make_ref.py)"

        def one(i):
            x, _, _ = ref.utils._process_input(imgs[i % len(imgs)], 1.0, os_)                     # benchmark.py:29
            with torch.no_grad():
                heat, off, fwd, bwd = model(torch.Tensor(x))                                       # benchmark.py:33-36
                return ref_dm.decode_multiple_poses(heat.squeeze(0), off.squeeze(0), fwd.squeeze(0), bwd.squeeze(0),
                                                    output_stride=os_, max_pose_detections=DECODE_KW["max_pose_detections"],
                                                    min_pose_score=DECODE_KW["min_pose_score"])   # benchmark.py:37-44
    else:
        from oracle import decode as odec, net as onet, preprocess as opre
        sd = onet.init_params(mid, seed=0)
        kind, how = "port", "oracle port (oracle/_ref not built here)"

        def one(i):
            x, _, _ = opre.process_input(imgs[i % len(imgs)], 1.0, os_)
            heads = onet.forward(sd, mid, os_, torch.from_numpy(x))
            return odec.decode_multiple_poses(*[t.squeeze(0).numpy() for t in heads], os_, **DECODE_KW)

    for i in range(warmup):
        one(i)
    t0 = time.perf_counter()
    for s in range(steps):
        for i in range(images_per_step):
            one(s * images_per_step + i)
    dt = time.perf_counter() - t0
    return dict(value=steps * images_per_step / dt, ms_per_step=dt / steps * 1e3, cores=cores, kind=kind,
                sample="%d steps x %d images, one image per call (benchmark.py:32-44), %s: cv2 preprocess + torch-CPU fp32 forward + "
                       "numpy f64 decode, %d torch threads" % (steps, images_per_step, how, cores))


REF_IMAGES_PER_STEP = 4


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    r = cpu_reference_run(args.workload, images_per_step=REF_IMAGES_PER_STEP, steps=args.steps, warmup=args.warmup)
    line = {"impl": "reference", "metric": METRIC, "value": r["value"], "unit": "images/sec", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["ms_per_step"], "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args.workload),
            "run": {"images_per_step": REF_IMAGES_PER_STEP, "batch": 1, "device": "host cpu", "threads": r["cores"]},
            "cpu_baseline": {"value": r["value"], "unit": "images/sec", "cores": r["cores"], "kind": r["kind"], "sample": r["sample"]},
            "e2e": {"value": r["value"], "unit": "images/sec", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def cpu_baseline_subprocess(workload, steps=3, warmup=1):
    """cpu_baseline of the product line: the reference arm in a fresh process (this one has imported the product `posenet`)."""
    try:
        out = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--workload", workload, "--steps", str(steps),
                              "--warmup", str(warmup)], capture_output=True, text=True, timeout=900,
                             env={k: v for k, v in os.environ.items() if k not in ("RANK", "LOCAL_RANK", "WORLD_SIZE")})
        line = json.loads(out.stdout.strip().splitlines()[-1])
        return line["cpu_baseline"]
    except Exception as e:                                           # the product line must not die with its baseline leg
        return {"value": None, "unit": "images/sec", "cores": os.cpu_count(), "kind": "unavailable", "sample": "failed: %r" % (e,)}


# ------------------------------------------------------------------------------------------ B200 arm
def layer_costs(model, n, H, W):
    """Algorithmic bytes / flops per launch (SURVEY 8(d)): depthwise bytes = (in + out pixels) * C * 2 (+ weights),
    pointwise flops = 2 M K N and bytes = (M K + M N + K N) * 2."""
    rows, h, w = [], H, W
    for L in model._layers:
        s, d = L["stride"], L["rate"]
        pad = ((s - 1) + 2 * d) // 2
        ho, wo = (h + 2 * pad - 2 * d - 1) // s + 1, (w + 2 * pad - 2 * d - 1) // s + 1
        m = n * ho * wo
        if L["block_id"] == 0:
            rows.append(("stem", n * h * w * 3 + m * L["outp"] * 2, 2 * 27 * m * L["outp"]))
        else:
            c = L["inp"]
            rows.append(("dw%d" % L["block_id"], (n * h * w + m) * c * 2 + 40 * c, 18 * m * c))
            rows.append(("pw%d" % L["block_id"], (m * c + m * L["outp"] + c * L["outp"]) * 2, 2 * m * c * L["outp"]))
            # fused block: input read once, output written once, the depthwise intermediate never leaves the SM
            rows.append(("sep%d" % L["block_id"], (n * h * w * c + m * L["outp"] + c * L["outp"]) * 2 + 40 * c,
                         18 * m * c + 2 * m * c * L["outp"]))
        h, w = ho, wo
    m = n * h * w
    c = model._layers[-1]["outp"]
    rows.append(("heads", (m * c + 128 * c) * 2 + m * 115 * 4, 2 * m * c * 115))
    # candidates read the heatmap (17 h w fp32); the greedy decode touches at most all four head maps
    rows.append(("candidates+decode", m * 17 * 4 + m * 115 * 4, 0))
    return rows, (h, w)


def per_kernel_times(model, imgs_list, reps=5):
    """Device time of every launch of one forward, measured IN SITU: pn_plan_profile enqueues the same
    launches as a normal forward with a CUDA event between consecutive kernels on the launching stream
    (so each kernel sees the cache state its producer left).  Median over `reps` forwards; plus the
    candidate + decode kernels timed the same way around the public decode call."""
    import posenet
    n, H, W, _ = imgs_list[0].shape
    plan = model._plan(n, H, W, True)
    heads = [torch.empty((n, ch, plan.out_h, plan.out_w), dtype=torch.float32, device=imgs_list[0].device) for ch in (17, 34, 32, 32)]
    runs = []
    for r in range(reps + 1):
        runs.append(plan.profile(imgs_list[r % len(imgs_list)], heads))
    runs = runs[1:]
    times = {name: sorted(run[i][1] for run in runs)[reps // 2] for i, (name, _) in enumerate(runs[0])}
    # candidates + decode: replayed from a CUDA graph (as in the step), so that the host time between the two launches of an
    # eager call does not count as device time
    ws, dec = {}, []
    posenet.decode_multiple_poses_batch(*heads, output_stride=model.output_stride, workspace=ws, **DECODE_KW)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        posenet.decode_multiple_poses_batch(*heads, output_stride=model.output_stride, workspace=ws, **DECODE_KW)
    for r in range(reps + 1):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        g.replay()
        e1.record()
        torch.cuda.synchronize()
        dec.append(e0.elapsed_time(e1))
    times["candidates+decode"] = sorted(dec[1:])[reps // 2]
    return times


def h2d_ceiling(host_batches, dev, world, reps=6):
    """What the host can feed: plain pinned-host -> device copies of the SAME buffers the end-to-end leg submits, nothing else
    running, every rank at once (barrier, CUDA events, max over ranks).  Returns aggregate GB/s over all ranks."""
    dst = [torch.empty_like(h, device=dev) for h in host_batches[:2]]
    st = torch.cuda.Stream(dev)

    def burst(n):
        with torch.cuda.stream(st):
            for i in range(n):
                dst[i % 2].copy_(host_batches[i % len(host_batches)], non_blocking=True)
    burst(2)
    st.synchronize()
    if world > 1:
        torch.distributed.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.cuda.stream(st):
        e0.record(st)
    burst(reps)
    with torch.cuda.stream(st):
        e1.record(st)
    st.synchronize()
    ms = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms], device=dev)
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        ms = float(t)
    return world * reps * host_batches[0].numel() / (ms * 1e-3) / 1e9


DUMP_NAMES = ("pose_scores", "keypoint_scores", "keypoint_coords", "pose_offsets", "pose_counts")   # decode_multiple_poses_batch
DUMP_LIMIT = 64 << 20


def dump_outputs(out_dir, outputs):
    """Write the records of one step as ``out_dir/<name>.npy`` (float64, first axis = image).  Above DUMP_LIMIT bytes only a
    fixed, seeded sample of images is written, and their batch indices go to ``image_index.npy``."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = [t.numpy().astype(np.float64) for t in outputs]
    n = arrays[0].shape[0]
    per_image = sum(a.nbytes for a in arrays) // n
    if n * per_image > DUMP_LIMIT:
        index = np.sort(np.random.default_rng(0).choice(n, DUMP_LIMIT // (per_image + 8), replace=False))
        arrays = [a[index] for a in arrays]
        np.save(os.path.join(out_dir, "image_index.npy"), index.astype(np.float64))
    for name, a in zip(DUMP_NAMES, arrays):
        np.save(os.path.join(out_dir, name + ".npy"), a)


def run_b200(args):
    if PKG not in sys.path:
        sys.path.insert(0, PKG)
    import posenet
    from posenet import _native as nat
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    affinity, all_cpus = bind_to_gpu_numa_node(local)            # before any pinned allocation (first touch decides the NUMA node)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    mid, H, W, os_, batch, desc = WORKLOADS[args.workload]
    if args.batch:
        batch = args.batch
    torch.manual_seed(0)
    model = posenet.MobileNetV1(mid, output_stride=os_).cuda().set_compute_dtype("bf16")   # default torch init, seeded
    model.set_fused(not args.unfused)
    n_sets = 4                                                   # rotate inputs: 4 x 50 MB u8 > 126 MB L2
    rng = np.random.default_rng(1234 + rank)
    sh, sw = SOURCE_SIZE.get(args.workload, (H, W))
    host = [torch.from_numpy(rng.integers(0, 256, (batch, sh, sw, 3), dtype=np.uint8)).pin_memory() for _ in range(n_sets)]
    imgs = [h.to(dev) for h in host]
    resized = torch.empty((batch, H, W, 3), dtype=torch.uint8, device=dev) if (sh, sw) != (H, W) else None
    ws = {}

    def step(x):
        if resized is not None:                                  # P1's resize stage, bit-exact with cv2 (pn_resize_u8)
            x, _ = posenet.resize_u8_gpu(x, 1.0, os_, out=resized)
        heads = model.forward_u8(x)
        return posenet.decode_multiple_poses_batch(*heads, output_stride=os_, workspace=ws, **DECODE_KW)

    # ---- device-resident throughput: one CUDA graph per input set
    for x in imgs:
        step(x)
    torch.cuda.synchronize()
    graphs = []
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for x in imgs:
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=side):
                out = step(x)
            graphs.append((g, out))
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    for i in range(args.warmup):
        graphs[i % n_sets][0].replay()
    barrier()
    sampler = ClockSampler(local)
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_begin = time.perf_counter()
    e0.record()
    for i in range(args.steps):
        graphs[i % n_sets][0].replay()
    e1.record()
    if sampler.nv is not None:
        sampler.sample_now()                                     # the replays above are still executing
    barrier()
    sampler.window = (t_begin, time.perf_counter())
    ms = e0.elapsed_time(e1)
    last_step = [t.cpu() for t in graphs[(args.steps - 1) % n_sets][1]] if args.dump_outputs and rank == 0 else None
    # the nvidia-smi fallback answers in ~100 ms and the timed region can be shorter than that: keep the SAME load running
    # (untimed) until the sampler has at least 5 readings; NVML readings (~0.1 ms each) land inside the timed region
    t_extra = time.perf_counter()
    i = 0
    while len(sampler.rows) < 5 and time.perf_counter() - t_extra < 3.0:
        graphs[i % n_sets][0].replay()
        i += 1
        if i % 8 == 0:
            torch.cuda.synchronize()
    torch.cuda.synchronize()
    clocks = sampler.summary()
    if not clocks.get("samples_in_timed_region"):
        clocks["note"] = "no reading fell inside the timed region; these were taken under the same graph replays, untimed"
    if world > 1:
        t = torch.tensor([ms], device=dev)
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        ms = float(t)
    value = world * batch * args.steps / (ms / 1e3)

    # ---- sustained leg: the SAME graph replays for >= `--sustain` seconds (the timed region above is a 0.03 s burst at the boost
    # clock; MEASURED_PEAKS.json shows this pool settling to a lower SM clock under a seconds-long load).  Device-timed, max over
    # ranks, with its own clock / throttle-reason samples.
    sustained = None
    if args.sustain > 0:
        barrier()
        s_sampler = ClockSampler(local)
        s_sampler.start()
        chunk = max(8, int(0.25 / (ms / args.steps / 1e3)))           # ~0.25 s of replays between host synchronisations
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t_s = time.perf_counter()
        s0.record()
        n_rep = 0
        while time.perf_counter() - t_s < args.sustain:
            for _ in range(chunk):
                graphs[n_rep % n_sets][0].replay()
                n_rep += 1
            torch.cuda.current_stream().synchronize()
        s1.record()
        torch.cuda.synchronize()
        s_sampler.window = (t_s, time.perf_counter())
        s_ms = s0.elapsed_time(s1)
        s_clk = s_sampler.summary()
        rate = batch * n_rep / (s_ms / 1e3)                            # this rank's images/s over its own window
        if world > 1:
            t = torch.tensor([rate], device=dev)
            torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MIN)
            rate = float(t)                                           # slowest rank x world: ranks run the same load independently
        sustained = {"value": round(world * rate, 1), "unit": "images/sec", "seconds": round(s_ms / 1e3, 2), "steps": n_rep,
                     "ms_per_step": round(s_ms / n_rep, 4), "vs_burst": round(world * rate / value, 4),
                     "clocks": {k: s_clk.get(k) for k in ("sm_mhz", "sm_min_mhz", "sm_max_mhz", "reasons", "samples_in_timed_region")}}

    # ---- end to end through the public API (posenet.BatchPipeline): every step copies ITS pinned host uint8 batch to the
    # device, runs model + decode, and copies ITS pose records back to pinned host memory; the copies of neighbouring
    # steps overlap the kernels (2 slots in flight), nothing is cached across steps.
    e2e_steps = 1 if args.skip_e2e else args.steps
    pipe = posenet.BatchPipeline(model, batch, sh, sw, depth=args.depth, output_stride=os_, gather=world > 1, **DECODE_KW)
    for rec in pipe.run(host[i % n_sets] for i in range(1 if args.skip_e2e else max(3, args.warmup))):
        pass
    barrier()
    t0 = time.perf_counter()
    for rec in pipe.run((host[i % n_sets] for i in range(e2e_steps)), copy=False):
        pass
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([e2e_s], device=dev)
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        e2e_s = float(t)
    e2e = {"value": world * batch * e2e_steps / e2e_s, "unit": "images/sec", "h2d_bytes_per_step": int(pipe.h2d_bytes_per_batch),
           "d2h_bytes_per_step": int(pipe.d2h_bytes_per_batch), "api": "posenet.BatchPipeline.run (depth %d)" % args.depth}
    if world > 1:
        # every step's pose records were all-gathered over NCCL inside the timed loop above (BatchPipeline(gather=True): each rank
        # ends the step holding the records of all `world` shards on its device, rank 0 reads all of them back to the host);
        # the collective's device time alone, for the record:
        e2e["gather"] = "all_gather_into_tensor of %d B per rank per step (NCCL, own stream), inside the timed loop; rank 0 reads all %d shards back" % (
            pipe.nrec * 8, world)
        e2e["gather_ms"] = round(pipe.time_gather(reps=20), 4)
    # the same step without overlap (one batch at a time, synchronous), for reference
    t0 = time.perf_counter()
    for i in range(e2e_steps):
        rec = pipe.result(pipe.submit(host[i % n_sets]), copy=False)
    e2e["value_serial"] = world * batch * e2e_steps / (time.perf_counter() - t0)
    del pipe
    if not args.skip_e2e:
        # the ceiling the host can feed: the same pinned batches, copies only, all ranks at once
        gbs = h2d_ceiling(host, dev, world)
        e2e["h2d_ceiling_gbs"] = round(gbs, 1)
        e2e["h2d_gbs"] = round(e2e["value"] * (host[0].numel() / batch) / 1e9, 1)
        e2e["frac_of_h2d_ceiling"] = round(e2e["h2d_gbs"] / gbs, 4)

    if rank != 0:
        return
    # ---- per-kernel roofline (rank 0, live CUDA events on the launching stream)
    pk = peaks()
    net_in = imgs
    if resized is not None:
        net_in = [posenet.resize_u8_gpu(x, 1.0, os_)[0] for x in imgs[:2]]
    times = per_kernel_times(model, net_in)
    costs, _ = layer_costs(model, batch, H, W)
    total_ms = sum(times.values())
    kernels = []
    for name, nbytes, flops in costs:
        if name not in times:
            continue                                             # fused plans have sepN, unfused dwN + pwN
        t = times[name] * 1e-3
        ai = flops / nbytes
        # each kernel is timed alone inside a 1.6 ms step at the boost clock: the burst bf16 peak is its denominator (and sets
        # the ridge); the sustained peak belongs to the sustained leg only
        tensor_bound = name.startswith(("pw", "sep", "heads")) and ai > pk["bf16_burst"] * 1e3 / pk["hbm"]
        kernels.append({"name": name, "ms": round(times[name], 4), "share": round(times[name] / total_ms, 4),
                        "gbs": round(nbytes / t / 1e9, 1), "tflops": round(flops / t / 1e12, 2),
                        "bound": "tensor" if tensor_bound else "hbm",
                        "frac": round((flops / t / 1e12) / pk["bf16_burst"] if tensor_bound else (nbytes / t / 1e9) / pk["hbm"], 4)})
    top = max(kernels, key=lambda k: k["ms"])
    # DRAM bytes per launch of that kernel from the committed `ncu --set full` capture of the same workload
    # (profiles/ncu_traffic.json: launch name -> dram__bytes_read.sum + dram__bytes_write.sum), null if not captured
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if os.path.exists(tpath):
        t = json.load(open(tpath))
        if t.get("workload") == args.workload and t.get("batch") == batch:
            traffic = t.get("dram_bytes", {}).get(top["name"])
    roofline = {"kernel": top["name"], "bound": top["bound"],
                "achieved": top["tflops"] if top["bound"] == "tensor" else top["gbs"],
                "peak": pk["bf16_burst"] if top["bound"] == "tensor" else pk["hbm"],
                "unit": "TFLOP/s" if top["bound"] == "tensor" else "GB/s", "frac": top["frac"], "traffic": traffic,
                "algorithmic_bytes": next(nb for nm, nb, _ in costs if nm == top["name"]),
                "peak_source": pk["src"] + (" (burst: the kernel is timed alone)" if top["bound"] == "tensor" else "")}
    if all_cpus:
        os.sched_setaffinity(0, all_cpus)                        # the CPU baseline gets every host core again
    cpu = cpu_baseline_subprocess(args.workload) if (world == 1 and not args.skip_cpu) else None
    launches = model.num_launches(batch, H, W, True) + 2 + (1 if resized is not None else 0)   # + candidates, decode (+ resize)
    line = {"metric": METRIC, "value": round(value, 1), "unit": "images/sec", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": round(ms / args.steps, 4), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": workload_config(args.workload),
            "run": {"batch_per_gpu": batch, "images_per_step": world * batch, "device": "B200 x %d" % world, "compute": "bf16 activations / fp32 accumulate",
                    "l2": "inputs rotate over %d batches (%d MB > 126 MB L2); per-step activation traffic >> L2" % (
                        n_sets, n_sets * host[0].numel() // 2 ** 20), "cuda_graph": True,
                    "fused_blocks": bool(model.fused_blocks), "cpu_affinity": affinity},
            "e2e": e2e, "gpu_launches": launches * args.steps, "clocks": clocks, "roofline": roofline,
            "kernels": kernels, "forward_ms_sum_of_kernels": round(total_ms, 3)}
    if sustained:
        line["sustained"] = sustained
        line["value_sustained"] = sustained["value"]
    if cpu:
        line["cpu_baseline"] = cpu
    if last_step is not None:
        dump_outputs(args.dump_outputs, last_step)
    print(json.dumps(line), flush=True)
    if world > 1:
        torch.distributed.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS))
    ap.add_argument("--batch", type=int, default=0, help="override the per-GPU batch (debug)")
    ap.add_argument("--skip-cpu", action="store_true", help="profiling runs: skip the cpu_baseline leg")
    ap.add_argument("--skip-e2e", action="store_true", help="profiling runs: skip the end-to-end leg")
    ap.add_argument("--sustain", type=float, default=3.0, help="seconds of back-to-back replays for the sustained leg (0: skip)")
    ap.add_argument("--depth", type=int, default=3, help="batches in flight in the end-to-end leg (BatchPipeline depth)")
    ap.add_argument("--unfused", action="store_true", help="run every block as depthwise + pointwise kernels (A/B against the fused blocks)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write rank 0's pose records of the last timed step to DIR/*.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs records the B200 arm only")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
