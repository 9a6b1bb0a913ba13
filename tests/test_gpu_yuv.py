"""YUV video frames converted to BGR on the GPU (pn_yuv_to_bgr) against cv2.cvtColor, byte for byte: yuv_to_bgr_batch over
every code and many frame sizes, the raw entry point with padded strides and guard bytes, and BatchPipeline(yuv=code) against a
BatchPipeline fed the cv2-converted BGR frames (records, drawn frames and encoded files identical)."""
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
from test_yuv_cpu import CODES, LAYOUTS, code_of, pack  # noqa: E402

DEV = "cuda"


def random_frames(name, n, h, w, rng):
    return rng.integers(0, 256, (n,) + yuv.frame_shape(CODES[name][0], h, w), dtype=np.uint8)


def cv2_batch(frames, code):
    return np.stack([cv2.cvtColor(f, code) for f in frames])


@pytest.mark.parametrize("name", LAYOUTS)
def test_batch_matches_cv2(name):
    layout = CODES[name][0]
    rng = np.random.default_rng(100 + layout)
    sizes = [(720, 1280), (2, 2), (2, 6), (10, 34), (16, 258), (18, 514), (34, 770), (6, 1030)]
    sizes += [(2 * int(rng.integers(1, 40)), 2 * int(rng.integers(1, 400))) for _ in range(6)]
    if layout > nat.YUV_NV21:
        sizes += [(1, 2), (9, 258), (17, 66)]                        # cv2 converts odd heights of 4:2:2
    for i, (h, w) in enumerate(sizes):
        frames = random_frames(name, int(rng.integers(1, 5)), h, w, rng)
        ref = cv2_batch(frames, code_of(name))
        src = [frames, torch.from_numpy(frames), torch.from_numpy(frames).to(DEV)][i % 3]
        for a in CODES[name][1]:
            got = posenet.yuv_to_bgr_batch(src, getattr(cv2, a))
            assert got.is_cuda and got.shape == ref.shape and got.dtype == torch.uint8
            assert np.array_equal(got.cpu().numpy(), ref), (name, a, h, w)
    assert posenet.yuv_to_bgr_batch(np.zeros((0,) + yuv.frame_shape(layout, 4, 4), np.uint8), code_of(name)).shape == (0, 4, 4, 3)


@pytest.mark.parametrize("name", LAYOUTS)
def test_raw_call_with_padded_strides_and_guard_bytes(name):
    """Frames further apart than their size, at odd offsets, with guard bytes around every frame: only the frames' BGR bytes
    change, and the source is only read."""
    layout = CODES[name][0]
    rng = np.random.default_rng(200 + layout)
    lib = nat.load()
    for n, h, w in [(3, 30, 262), (2, 18, 1282), (5, 2, 14)]:
        fb = int(np.prod(yuv.frame_shape(layout, h, w)))
        ss, ds, G = fb + 37, 3 * h * w + 53, 4099                   # odd strides: every frame at another alignment
        src_h = rng.integers(0, 256, G + n * ss + G, dtype=np.uint8)
        dst_h = rng.integers(0, 256, G + n * ds + G, dtype=np.uint8)
        src, dst = torch.from_numpy(src_h).to(DEV), torch.from_numpy(dst_h).to(DEV)
        rc = lib.pn_yuv_to_bgr(C.c_void_p(src.data_ptr() + G + 1), n, h, w, ss, layout, C.c_void_p(dst.data_ptr() + G + 3), ds,
                               nat.stream_ptr())
        nat.check(rc, "pn_yuv_to_bgr")
        got = dst.cpu().numpy()
        assert np.array_equal(src.cpu().numpy(), src_h)
        expect = dst_h.copy()
        for i in range(n):
            f = src_h[G + 1 + i * ss:G + 1 + i * ss + fb].reshape(yuv.frame_shape(layout, h, w))
            expect[G + 3 + i * ds:G + 3 + i * ds + 3 * h * w] = cv2.cvtColor(f, code_of(name)).ravel()
        assert np.array_equal(got, expect), (name, n, h, w, int((got != expect).sum()))
    # argument checks: nothing is launched
    buf = torch.zeros(1 << 16, dtype=torch.uint8, device=DEV)
    p = C.c_void_p(buf.data_ptr())
    fb = int(np.prod(yuv.frame_shape(layout, 8, 8)))
    bad = [(None, 1, 8, 8, fb, layout, p, 192), (p, 1, 8, 8, fb, layout, None, 192), (p, 1, 8, 7, fb, layout, p, 192),
           (p, 1, 8, 8, fb, 7, p, 192), (p, 1, 8, 8, fb, -1, p, 192), (p, 1, 8, 8, fb - 1, layout, p, 192),
           (p, 1, 8, 8, fb, layout, p, 191), (p, 0, 8, 8, fb, layout, p, 192), (p, 1, 0, 8, fb, layout, p, 192)]
    if layout <= nat.YUV_NV21:
        bad.append((p, 1, 7, 8, fb, layout, p, 192))
    for args in bad:
        assert lib.pn_yuv_to_bgr(*args, nat.stream_ptr()) == -1, args            # PN_ERR_ARG
    torch.cuda.synchronize()


def model(os_):
    sd = onet.init_params(50, seed=5, scheme="scaled", gain=0.8)
    m = posenet.MobileNetV1(50, output_stride=os_)
    m.load_state_dict(sd)
    return m.cuda().set_compute_dtype("bf16")


def video_batches(name, n_batches, N, H, W):
    """Seeded smooth frames in `name`'s layout (chroma of cv2's I420 with noise, repeated over row pairs for 4:2:2), and their
    cv2 conversion."""
    layout = CODES[name][0]
    rng = np.random.default_rng(H + W)
    yuv_b, bgr_b = [], []
    for b in range(n_batches):
        frames = []
        for i in range(N):
            i420 = cv2.cvtColor(synth.smooth_image(H, W, 30 * b + i), cv2.COLOR_BGR2YUV_I420)
            Y = i420[:H]
            U = i420[H:H + H // 4].reshape(H // 2, W // 2)
            V = i420[H + H // 4:].reshape(H // 2, W // 2)
            U, V = ((c.astype(np.int16) + rng.integers(-20, 21, c.shape)).clip(0, 255).astype(np.uint8) for c in (U, V))
            if layout > nat.YUV_NV21:
                U, V = np.repeat(U, 2, 0), np.repeat(V, 2, 0)
            frames.append(pack(name, Y, U, V))
        frames = np.stack(frames)
        yuv_b.append(torch.from_numpy(frames).pin_memory())
        bgr_b.append(torch.from_numpy(cv2_batch(frames, code_of(name))).pin_memory())
    return yuv_b, bgr_b


@pytest.mark.parametrize("name,N,H,W,os_", [(n, 2, 180, 322, 16) for n in LAYOUTS] +
                         [("I420", 2, 720, 1280, 8), ("NV12", 2, 720, 1280, 8), ("YUY2", 2, 720, 1280, 8)])
@pytest.mark.parametrize("use_graph", [True, False])
def test_pipeline_matches_bgr_pipeline(name, N, H, W, os_, use_graph):
    m = model(os_)
    yuv_b, bgr_b = video_batches(name, 3, N, H, W)
    kw = dict(depth=2, output_stride=os_, use_graph=use_graph, source_coords=True, overlay=(0.1, 0.1), max_pose_detections=8,
              min_pose_score=0.05)
    ref = list(posenet.BatchPipeline(m, N, H, W, **kw).run(bgr_b))
    pipe = posenet.BatchPipeline(m, N, H, W, yuv=code_of(name), **kw)
    assert pipe.h2d_bytes_per_batch == yuv_b[0].numel() < 3 * N * H * W
    got = list(pipe.run(yuv_b))
    assert len(got) == len(ref) and any(r[0].max() > 0 for r in ref)
    for g, r in zip(got, ref):
        assert len(g) == 5
        for a, b in zip(g, r):
            assert np.array_equal(a, b)
    if use_graph:
        ref = list(posenet.BatchPipeline(m, N, H, W, encode=[], **kw).run(bgr_b))
        got = list(posenet.BatchPipeline(m, N, H, W, encode=[], yuv=code_of(name), **kw).run(yuv_b))
        for g, r in zip(got, ref):
            for a, b in zip(g[:4], r[:4]):
                assert np.array_equal(a, b)
            assert g[4] == r[4] and len(g[4]) == N
