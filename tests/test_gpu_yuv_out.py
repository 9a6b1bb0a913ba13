"""Drawn frames converted to YUV on the GPU (pn_bgr_to_yuv) against cv2.cvtColor, byte for byte: bgr_to_yuv_batch over every
code and many frame sizes, the raw entry point with padded strides and guard bytes, graph replay, and BatchPipeline(overlay,
yuv_out=code) against cv2.cvtColor of the frames the same pipeline returns without yuv_out (alone, with yuv= input and with a
jpeg=True stream)."""
import ctypes as C

import cv2
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

import posenet  # noqa: E402
from posenet import _native as nat  # noqa: E402
from posenet import yuv  # noqa: E402
from oracle import net as onet  # noqa: E402
from oracle import synth  # noqa: E402
from test_yuv_out_cpu import OUT_CODES, OUT_LAYOUTS, SIZES, SIZES_422, code_of  # noqa: E402

DEV = "cuda"


def cv2_batch(frames, code):
    return np.stack([cv2.cvtColor(f, code) for f in frames])


@pytest.mark.parametrize("name", OUT_LAYOUTS)
def test_batch_matches_cv2(name):
    layout = OUT_CODES[name][0]
    rng = np.random.default_rng(300 + layout)
    sizes = SIZES + [(2 * int(rng.integers(1, 40)), 2 * int(rng.integers(1, 400))) for _ in range(6)]
    if layout > nat.YUV_NV21:
        sizes += SIZES_422
    for i, (h, w) in enumerate(sizes):
        frames = rng.integers(0, 256, (int(rng.integers(1, 5)), h, w, 3), dtype=np.uint8)
        ref = cv2_batch(frames, code_of(name))
        src = [frames, torch.from_numpy(frames), torch.from_numpy(frames).to(DEV)][i % 3]
        for a in OUT_CODES[name][1]:
            got = posenet.bgr_to_yuv_batch(src, getattr(cv2, a))
            assert got.is_cuda and got.shape == ref.shape and got.dtype == torch.uint8
            assert np.array_equal(got.cpu().numpy(), ref), (name, a, h, w)
    empty = posenet.bgr_to_yuv_batch(np.zeros((0, 4, 4, 3), np.uint8), code_of(name))
    assert empty.shape == (0,) + yuv.frame_shape(layout, 4, 4)


@pytest.mark.parametrize("name", OUT_LAYOUTS)
def test_raw_call_with_padded_strides_and_guard_bytes(name):
    """Frames further apart than their size, at odd offsets, with guard bytes around every frame: only the frames' YUV bytes
    change, and the source is only read."""
    layout = OUT_CODES[name][0]
    rng = np.random.default_rng(400 + layout)
    lib = nat.load()
    for n, h, w in [(3, 30, 262), (2, 18, 1282), (5, 2, 14), (2, 720, 1280)] + ([(3, 9, 258)] if layout > nat.YUV_NV21 else []):
        shape = yuv.frame_shape(layout, h, w)
        fb = int(np.prod(shape))
        ss, ds, G = 3 * h * w + 41, fb + 29, 4099                   # odd strides: every frame at another alignment
        src_h = rng.integers(0, 256, G + n * ss + G, dtype=np.uint8)
        dst_h = rng.integers(0, 256, G + n * ds + G, dtype=np.uint8)
        src, dst = torch.from_numpy(src_h).to(DEV), torch.from_numpy(dst_h).to(DEV)
        rc = lib.pn_bgr_to_yuv(C.c_void_p(src.data_ptr() + G + 5), n, h, w, ss, layout, C.c_void_p(dst.data_ptr() + G + 3), ds,
                               nat.stream_ptr())
        nat.check(rc, "pn_bgr_to_yuv")
        got = dst.cpu().numpy()
        assert np.array_equal(src.cpu().numpy(), src_h)
        expect = dst_h.copy()
        for i in range(n):
            f = src_h[G + 5 + i * ss:G + 5 + i * ss + 3 * h * w].reshape(h, w, 3)
            expect[G + 3 + i * ds:G + 3 + i * ds + fb] = cv2.cvtColor(f, code_of(name)).ravel()
        assert np.array_equal(got, expect), (name, n, h, w, int((got != expect).sum()))


def test_bad_arguments_return_err_arg():
    lib = nat.load()
    buf = torch.zeros(1 << 16, dtype=torch.uint8, device=DEV)
    p = C.c_void_p(buf.data_ptr())
    for layout in (nat.YUV_I420, nat.YUV_YUY2):
        fb = int(np.prod(yuv.frame_shape(layout, 8, 8)))
        bad = [(None, 1, 8, 8, 192, layout, p, fb), (p, 1, 8, 8, 192, layout, None, fb), (p, 1, 8, 7, 192, layout, p, fb),
               (p, 1, 8, 8, 192, 7, p, fb), (p, 1, 8, 8, 192, -1, p, fb), (p, 1, 8, 8, 192, nat.YUV_NV12, p, fb),
               (p, 1, 8, 8, 192, nat.YUV_NV21, p, fb), (p, 1, 8, 8, 191, layout, p, fb), (p, 1, 8, 8, 192, layout, p, fb - 1),
               (p, 0, 8, 8, 192, layout, p, fb), (p, 65536, 8, 8, 192, layout, p, fb), (p, 1, 0, 8, 192, layout, p, fb),
               (p, 1, 8, 0, 192, layout, p, fb), (p, 1, -2, 8, 192, layout, p, fb)]
        if layout == nat.YUV_I420:
            bad.append((p, 1, 7, 8, 192, layout, p, fb))
        for args in bad:
            assert lib.pn_bgr_to_yuv(*args, nat.stream_ptr()) == -1, args            # PN_ERR_ARG
    # odd heights of 4:2:2 are accepted
    assert lib.pn_bgr_to_yuv(p, 1, 7, 8, 168, nat.YUV_UYVY, C.c_void_p(buf.data_ptr() + 4096), 112, nat.stream_ptr()) == 0
    torch.cuda.synchronize()


@pytest.mark.parametrize("name", ["I420", "YUY2"])
def test_graph_capture_and_replay_with_new_frames(name):
    layout = OUT_CODES[name][0]
    rng = np.random.default_rng(500 + layout)
    n, h, w = 4, 180, 322
    src = torch.zeros((n, h, w, 3), dtype=torch.uint8, device=DEV)
    dst = torch.zeros((n,) + yuv.frame_shape(layout, h, w), dtype=torch.uint8, device=DEV)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        yuv.convert_out(src, n, h, w, layout, dst)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=s):
            yuv.convert_out(src, n, h, w, layout, dst)
    torch.cuda.current_stream().wait_stream(s)
    for _ in range(3):
        frames = rng.integers(0, 256, (n, h, w, 3), dtype=np.uint8)
        src.copy_(torch.from_numpy(frames))
        g.replay()
        assert np.array_equal(dst.cpu().numpy(), cv2_batch(frames, code_of(name)))


def model(os_):
    sd = onet.init_params(50, seed=5, scheme="scaled", gain=0.8)
    m = posenet.MobileNetV1(50, output_stride=os_)
    m.load_state_dict(sd)
    return m.cuda().set_compute_dtype("bf16")


def bgr_batches(n_batches, N, H, W):
    return [torch.from_numpy(np.stack([synth.smooth_image(H, W, 40 * b + i) for i in range(N)])).pin_memory()
            for b in range(n_batches)]


def check_against_bgr(ref, got, code, N):
    """Items of the yuv_out pipeline: the records of the BGR pipeline, and cv2's conversion of its drawn frames."""
    assert len(got) == len(ref) and any(r[0].max() > 0 for r in ref)
    for g, r in zip(got, ref):
        assert len(g) == len(r)
        for a, b in zip(g[:4], r[:4]):
            assert np.array_equal(a, b)
        assert g[4].shape[0] == N and np.array_equal(g[4], cv2_batch(r[4], code))
        for a, b in zip(g[5:], r[5:]):
            assert np.array_equal(a, b)


@pytest.mark.parametrize("name,N,H,W,os_", [(n, 2, 180, 322, 16) for n in OUT_LAYOUTS] +
                         [("YUY2", 2, 181, 322, 16), ("I420", 2, 720, 1280, 8), ("YUY2", 2, 720, 1280, 8)])
@pytest.mark.parametrize("use_graph", [True, False])
def test_pipeline_matches_cvtcolor_of_bgr_pipeline(name, N, H, W, os_, use_graph):
    m = model(os_)
    batches = bgr_batches(3, N, H, W)
    kw = dict(depth=2, output_stride=os_, use_graph=use_graph, source_coords=True, overlay=(0.1, 0.1), max_pose_detections=8,
              min_pose_score=0.05)
    ref_pipe = posenet.BatchPipeline(m, N, H, W, **kw)
    ref = list(ref_pipe.run(batches))
    pipe = posenet.BatchPipeline(m, N, H, W, yuv_out=code_of(name), **kw)
    fb = N * int(np.prod(yuv.frame_shape(OUT_CODES[name][0], H, W)))
    assert pipe.d2h_bytes_per_batch == ref_pipe.d2h_bytes_per_batch - 3 * N * H * W + fb
    check_against_bgr(ref, list(pipe.run(batches)), code_of(name), N)


@pytest.mark.parametrize("name", ["I420", "UYVY"])
def test_pipeline_video_in_video_out(name):
    """yuv= input (I420 video frames) and yuv_out= output in one pipeline."""
    N, H, W, os_ = 2, 180, 322, 16
    m = model(os_)
    bgr = bgr_batches(3, N, H, W)
    i420 = [torch.from_numpy(cv2_batch(b.numpy(), cv2.COLOR_BGR2YUV_I420)).pin_memory() for b in bgr]
    kw = dict(depth=2, output_stride=os_, source_coords=True, overlay=(0.1, 0.1), max_pose_detections=8, min_pose_score=0.05,
              yuv=cv2.COLOR_YUV2BGR_I420)
    ref = list(posenet.BatchPipeline(m, N, H, W, **kw).run(i420))
    got = list(posenet.BatchPipeline(m, N, H, W, yuv_out=code_of(name), **kw).run(i420))
    check_against_bgr(ref, got, code_of(name), N)


@pytest.mark.parametrize("reduce", [1, 2])
def test_pipeline_jpeg_stream(tmp_path, reduce):
    """ImageStream(decode="gpu") + BatchPipeline(jpeg=True, yuv_out=YUY2 / I420): 640 x 480 files (320 x 240 at 1/2), 19 of
    them, so the last batch has black rows."""
    paths = []
    for i in range(19):
        ok, buf = cv2.imencode(".jpg", synth.smooth_image(480, 640, 600 + i), [cv2.IMWRITE_JPEG_QUALITY, 90])
        assert ok
        p = tmp_path / ("img%03d.jpg" % i)
        p.write_bytes(buf.tobytes())
        paths.append(str(p))
    H, W = 480 // reduce, 640 // reduce
    m = model(16)
    kw = dict(depth=2, output_stride=16, min_pose_score=0.1, overlay=(0.1, 0.1), source_coords=True, jpeg=True, reduce=reduce)
    code = cv2.COLOR_BGR2YUV_YUY2 if reduce == 1 else cv2.COLOR_BGR2YUV_I420
    runs = []
    for extra in ({}, dict(yuv_out=code)):
        stream = posenet.ImageStream(paths, batch=8, height=H, width=W, decode="gpu", reduce=reduce)
        runs.append(list(posenet.BatchPipeline(m, 8, H, W, **kw, **extra).run(b for b, _ in stream.batches())))
    assert [int((g[-1] == 0).sum()) for g in runs[1]] == [8, 8, 3]
    check_against_bgr(runs[0], runs[1], code, 8)
