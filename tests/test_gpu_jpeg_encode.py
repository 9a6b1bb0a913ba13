"""JPEG files encoded on the GPU (pn_jpeg_encode) against cv2.imencode, byte for byte: imencode_batch on dense and mixed-size
batches, guard bytes past the packed output, graph replay, a round trip through imdecode_batch, and BatchPipeline(encode=...)
against cv2.imencode of the frames BatchPipeline(overlay=...) returns."""
import ctypes as C

import cv2
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

import posenet  # noqa: E402
from posenet import _native as nat  # noqa: E402
from posenet import jpeg as pj  # noqa: E402
from oracle import net as onet  # noqa: E402
from oracle import synth  # noqa: E402
from jpeg_corpus import corpus  # noqa: E402

DEV = "cuda"
S = cv2.IMWRITE_JPEG_SAMPLING_FACTOR


def ref(img, params):
    return cv2.imencode(".jpg", np.ascontiguousarray(img), params)[1].tobytes()


def model(os_=16):
    sd = onet.init_params(50, seed=5, scheme="scaled", gain=0.8)
    m = posenet.MobileNetV1(50, output_stride=os_)
    m.load_state_dict(sd)
    return m.cuda().set_compute_dtype("bf16")


@pytest.mark.parametrize("params", [[], [cv2.IMWRITE_JPEG_QUALITY, 100, S, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_444],
                                    [cv2.IMWRITE_JPEG_QUALITY, 50, S, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_411,
                                     cv2.IMWRITE_JPEG_RST_INTERVAL, 3],
                                    [cv2.IMWRITE_JPEG_QUALITY, 0, S, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_440],
                                    [cv2.IMWRITE_JPEG_QUALITY, 75, S, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_422,
                                     cv2.IMWRITE_JPEG_RST_INTERVAL, 1]])
def test_dense_batch(params):
    rng = np.random.default_rng(1)
    frames = np.stack([synth.smooth_image(257, 257, i) for i in range(5)] + [rng.integers(0, 256, (257, 257, 3), dtype=np.uint8)])
    got = posenet.imencode_batch(torch.from_numpy(frames).to(DEV), params)
    assert len(got) == len(frames)
    for i, f in enumerate(frames):
        assert got[i] == ref(f, params), i


def test_mixed_batch_with_empty_row():
    imgs = [img for img, params, _ in corpus(seed=5) if img.ndim == 3][:40] + [np.zeros((0, 0, 3), np.uint8)]
    imgs.insert(7, np.zeros((0, 0, 3), np.uint8))
    H, W = max(i.shape[0] for i in imgs), max(i.shape[1] for i in imgs)
    rows = torch.zeros((len(imgs), H * W * 3), dtype=torch.uint8)
    for k, im in enumerate(imgs):
        rows[k, :im.size] = torch.from_numpy(im.reshape(-1))
    params = [cv2.IMWRITE_JPEG_QUALITY, 90, cv2.IMWRITE_JPEG_RST_INTERVAL, 7]
    got = posenet.imencode_batch(rows.to(DEV), params, shapes=[im.shape[:2] for im in imgs])
    for k, im in enumerate(imgs):
        assert got[k] == (ref(im, params) if im.size else b""), k


def test_guard_bytes_and_frames_untouched():
    rng = np.random.default_rng(2)
    n, H, W = 4, 100, 130
    frames = torch.from_numpy(rng.integers(0, 256, (n, H, W, 3), dtype=np.uint8)).to(DEV)
    keep = frames.clone()
    enc = pj.Encoder(n, H, W, [cv2.IMWRITE_JPEG_QUALITY, 100, S, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_444])
    enc.out.fill_(0xA5)
    enc.encode(frames, H * W * 3)
    torch.cuda.synchronize()
    end = int(enc.offsets[-1])
    assert 0 < end < enc.out.numel()
    assert bool((enc.out[end:] == 0xA5).all())
    assert torch.equal(frames, keep)
    files = enc.files()
    for i in range(n):
        assert files[i] == ref(frames[i].cpu().numpy(), [cv2.IMWRITE_JPEG_QUALITY, 100, S, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_444])


def test_bound_is_checked():
    enc = pj.Encoder(2, 64, 64)
    frames = torch.zeros((2, 64, 64, 3), dtype=torch.uint8, device=DEV)
    with pytest.raises(nat.NativeError):
        nat.check(nat.load().pn_jpeg_encode(
            C.c_void_p(frames.data_ptr()), 2, 64, 64, 64 * 64 * 3, None, 95, 0x221111, 0, C.c_void_p(enc.out.data_ptr()),
            enc.capacity - 1, C.c_void_p(enc.offsets.data_ptr()), C.c_void_p(enc.ws.data_ptr()), enc.ws.numel(),
            nat.stream_ptr()), "pn_jpeg_encode")


def test_graph_replay_on_new_contents():
    n, H, W = 3, 120, 90
    params = [cv2.IMWRITE_JPEG_QUALITY, 85]
    frames = torch.zeros((n, H, W, 3), dtype=torch.uint8, device=DEV)
    enc = pj.Encoder(n, H, W, params)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        enc.encode(frames, H * W * 3)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        enc.encode(frames, H * W * 3)
    for seed in (3, 4):
        new = np.stack([synth.smooth_image(H, W, seed * 10 + i) for i in range(n)])
        frames.copy_(torch.from_numpy(new))
        g.replay()
        torch.cuda.synchronize()
        got = enc.files()
        assert got == [ref(f, params) for f in new]


def test_round_trip_through_device_decode():
    frames = np.stack([synth.smooth_image(513, 513, 40 + i) for i in range(3)])
    files = posenet.imencode_batch(torch.from_numpy(frames).to(DEV), [cv2.IMWRITE_JPEG_QUALITY, 90])
    dec, status = posenet.imdecode_batch(files)
    assert status.cpu().tolist() == [0, 0, 0]
    for k, f in enumerate(files):
        assert np.array_equal(dec[k].cpu().numpy(), cv2.imdecode(np.frombuffer(f, np.uint8), cv2.IMREAD_COLOR))


def _check_pipeline(got, plain, params, count):
    assert len(got) == len(plain)
    for g, p in zip(got, plain):
        for a, b in zip(g[:4], p[:4]):
            assert np.array_equal(a, b)
        frames = p[4]
        assert isinstance(g[4], list) and len(g[4]) == count
        for k in range(count):
            assert g[4][k] == ref(frames[k], params), k


@pytest.mark.parametrize("mode", ["dense", "mixed"])
def test_pipeline_encode(mode):
    mp, mk = 0.25, 0.25
    params = [cv2.IMWRITE_JPEG_QUALITY, 90]
    kw = dict(max_pose_detections=8, min_pose_score=0.05, depth=2, output_stride=16)
    m = model()
    if mode == "mixed":
        N, H, W = 3, 161, 200
        sizes = [[(129, 161), (100, 141), (161, 129)], [(64, 65), (150, 200)]]
        items = []
        for b, shp in enumerate(sizes):
            hb = torch.zeros((N, H * W * 3), dtype=torch.uint8)
            for i, (h, w) in enumerate(shp):
                hb[i, :h * w * 3] = torch.from_numpy(synth.smooth_image(h, w, 50 + 10 * b + i).reshape(-1))
            items.append((hb.pin_memory(), shp))
        kw.update(mixed=True, source_coords=True)
    else:
        N, H, W = 3, 129, 161
        items = [torch.from_numpy(np.stack([synth.smooth_image(H, W, 20 * b + i) for i in range(N)])).pin_memory() for b in range(3)]
    plain = list(posenet.BatchPipeline(m, N, H, W, overlay=(mp, mk), **kw).run(items))
    pipe = posenet.BatchPipeline(m, N, H, W, overlay=(mp, mk), encode=params, **kw)
    got = list(pipe.run(items))
    assert any(p[0].max() > 0 for p in plain)
    if mode == "mixed":
        for g, p, shp in zip(got, plain, sizes):
            _check_pipeline([g], [p], params, len(shp))
    else:
        _check_pipeline(got, plain, params, N)
    assert pipe.last_file_bytes > 0
    with pytest.raises(AssertionError):
        posenet.BatchPipeline(m, N, H, W, encode=params, **kw)          # encode needs overlay
    with pytest.raises(ValueError):
        posenet.BatchPipeline(m, N, H, W, overlay=(mp, mk), encode=[cv2.IMWRITE_JPEG_PROGRESSIVE, 1], **kw)


def test_pipeline_encode_jpeg_input(tmp_path):
    imgs = [synth.smooth_image(257, 257, 500 + i) for i in range(7)]
    paths = []
    for i, im in enumerate(imgs):
        p = tmp_path / ("f%02d.jpg" % i)
        p.write_bytes(ref(im, [cv2.IMWRITE_JPEG_QUALITY, 90]))
        paths.append(str(p))
    m = model()
    params = [cv2.IMWRITE_JPEG_QUALITY, 95]
    kw = dict(depth=2, output_stride=16, min_pose_score=0.1, overlay=(0.25, 0.25), jpeg=True)
    plain = list(posenet.BatchPipeline(m, 4, 257, 257, **kw).run(
        b for b, _ in posenet.ImageStream(paths, batch=4, decode="gpu").batches()))
    got = list(posenet.BatchPipeline(m, 4, 257, 257, encode=params, **kw).run(
        b for b, _ in posenet.ImageStream(paths, batch=4, decode="gpu").batches()))
    for g, p in zip(got, plain):
        assert np.array_equal(g[-1], p[-1])
    _check_pipeline(got, plain, params, 4)
