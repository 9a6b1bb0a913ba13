"""PNG files encoded on the GPU (pn_png_encode) against cv2.imencode(".png"), byte for byte: imencode_png_batch on dense and
mixed-size batches, guard bytes past the packed output, the capacity check, graph replay, cv2.imdecode of the files, and
BatchPipeline(encode=[], encode_ext=".png") against cv2.imencode of the frames BatchPipeline(overlay=...) returns."""
import ctypes as C

import cv2
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

import posenet  # noqa: E402
from posenet import _native as nat  # noqa: E402
from posenet import png as pp  # noqa: E402
from oracle import net as onet  # noqa: E402
from oracle import synth  # noqa: E402

DEV = "cuda"


def ref(img):
    return cv2.imencode(".png", np.ascontiguousarray(img))[1].tobytes()


def model(os_=16):
    sd = onet.init_params(50, seed=5, scheme="scaled", gain=0.8)
    m = posenet.MobileNetV1(50, output_stride=os_)
    m.load_state_dict(sd)
    return m.cuda().set_compute_dtype("bf16")


def _frames(h, w, seed):
    rng = np.random.default_rng(seed)
    noise = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
    quant = (rng.integers(0, 3, (h, w, 3)) * 127).astype(np.uint8)
    half = synth.smooth_image(h, w, seed)
    half[: h // 2] = noise[: h // 2]
    return [synth.smooth_image(h, w, seed + 1), noise, quant, np.full((h, w, 3), 9, np.uint8), half]


# 1080 x 1920 is 1520 tiles of 4096 filtered bytes: the per-image tile loops (carry, scan) run more than one 1024-wide round
@pytest.mark.parametrize("hw", [(1, 1), (5, 7), (3, 2000), (257, 257), (513, 513), (720, 1280), (1080, 1920)])
def test_dense_batch(hw):
    frames = np.stack(_frames(*hw, seed=hw[0]))
    got = posenet.imencode_png_batch(torch.from_numpy(frames).to(DEV))
    assert len(got) == len(frames)
    for i, f in enumerate(frames):
        assert got[i] == ref(f), i


def test_mixed_batch_with_empty_rows():
    sizes = [(1, 1), (1, 2), (2, 3), (13, 40), (100, 33), (0, 0), (64, 64), (200, 333), (40, 170), (0, 0), (150, 90)]
    imgs = []
    for k, (h, w) in enumerate(sizes):
        fr = _frames(max(h, 1), max(w, 1), k)[k % 5]
        imgs.append(fr[:h, :w])
    H, W = max(h for h, _ in sizes), max(w for _, w in sizes)
    rows = torch.zeros((len(imgs), H * W * 3), dtype=torch.uint8)
    for k, im in enumerate(imgs):
        rows[k, :im.size] = torch.from_numpy(np.ascontiguousarray(im).reshape(-1))
    got = posenet.imencode_png_batch(rows.to(DEV), shapes=sizes)
    for k, im in enumerate(imgs):
        assert got[k] == (ref(im) if im.size else b""), k


def test_guard_bytes_and_frames_untouched():
    rng = np.random.default_rng(2)
    n, H, W = 4, 100, 130
    frames = torch.from_numpy(rng.integers(0, 256, (n, H, W, 3), dtype=np.uint8)).to(DEV)
    keep = frames.clone()
    enc = pp.Encoder(n, H, W)
    enc.out.fill_(0xA5)
    enc.encode(frames, H * W * 3)
    torch.cuda.synchronize()
    end = int(enc.offsets[-1])
    assert 0 < end < enc.out.numel()
    assert bool((enc.out[end:] == 0xA5).all())
    assert torch.equal(frames, keep)
    files = enc.files()
    for i in range(n):
        assert files[i] == ref(frames[i].cpu().numpy())


def test_bound_is_checked():
    enc = pp.Encoder(2, 64, 64)
    frames = torch.zeros((2, 64, 64, 3), dtype=torch.uint8, device=DEV)
    with pytest.raises(nat.NativeError):
        nat.check(nat.load().pn_png_encode(
            C.c_void_p(frames.data_ptr()), 2, 64, 64, 64 * 64 * 3, None, C.c_void_p(enc.out.data_ptr()), enc.capacity - 1,
            C.c_void_p(enc.offsets.data_ptr()), C.c_void_p(enc.ws.data_ptr()), enc.ws.numel(), nat.stream_ptr()),
            "pn_png_encode")


def test_graph_replay_on_new_contents():
    n, H, W = 3, 120, 90
    frames = torch.zeros((n, H, W, 3), dtype=torch.uint8, device=DEV)
    enc = pp.Encoder(n, H, W)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        enc.encode(frames, H * W * 3)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        enc.encode(frames, H * W * 3)
    for seed in (3, 4):
        new = np.stack([_frames(H, W, seed * 10 + i)[(seed + i) % 5] for i in range(n)])
        frames.copy_(torch.from_numpy(new))
        g.replay()
        torch.cuda.synchronize()
        assert enc.files() == [ref(f) for f in new]


def test_files_decode_to_the_frames():
    frames = np.stack(_frames(513, 513, 40))
    files = posenet.imencode_png_batch(torch.from_numpy(frames).to(DEV))
    for k, f in enumerate(files):
        assert np.array_equal(cv2.imdecode(np.frombuffer(f, np.uint8), cv2.IMREAD_COLOR), frames[k])


def _check_pipeline(got, plain, count):
    assert len(got) == len(plain)
    for g, p in zip(got, plain):
        for a, b in zip(g[:4], p[:4]):
            assert np.array_equal(a, b)
        frames = p[4]
        assert isinstance(g[4], list) and len(g[4]) == count
        for k in range(count):
            assert g[4][k] == ref(frames[k]), k


@pytest.mark.parametrize("mode", ["dense", "mixed"])
def test_pipeline_encode_png(mode):
    mp, mk = 0.25, 0.25
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
    pipe = posenet.BatchPipeline(m, N, H, W, overlay=(mp, mk), encode=[], encode_ext=".png", **kw)
    got = list(pipe.run(items))
    assert any(p[0].max() > 0 for p in plain)
    if mode == "mixed":
        for g, p, shp in zip(got, plain, sizes):
            _check_pipeline([g], [p], len(shp))
    else:
        _check_pipeline(got, plain, N)
    assert pipe.last_file_bytes > 0
    with pytest.raises(ValueError):
        posenet.BatchPipeline(m, N, H, W, overlay=(mp, mk), encode=[cv2.IMWRITE_PNG_COMPRESSION, 1], encode_ext=".png", **kw)
    with pytest.raises(ValueError):
        posenet.BatchPipeline(m, N, H, W, overlay=(mp, mk), encode=[], encode_ext=".bmp", **kw)
    with pytest.raises(AssertionError):
        posenet.BatchPipeline(m, N, H, W, overlay=(mp, mk), encode_ext=".png", **kw)     # encode_ext needs encode


def test_pipeline_encode_png_jpeg_input(tmp_path):
    imgs = [synth.smooth_image(257, 257, 500 + i) for i in range(7)]
    paths = []
    for i, im in enumerate(imgs):
        p = tmp_path / ("f%02d.jpg" % i)
        p.write_bytes(cv2.imencode(".jpg", im, [cv2.IMWRITE_JPEG_QUALITY, 90])[1].tobytes())
        paths.append(str(p))
    m = model()
    kw = dict(depth=2, output_stride=16, min_pose_score=0.1, overlay=(0.25, 0.25), jpeg=True)
    plain = list(posenet.BatchPipeline(m, 4, 257, 257, **kw).run(
        b for b, _ in posenet.ImageStream(paths, batch=4, decode="gpu").batches()))
    got = list(posenet.BatchPipeline(m, 4, 257, 257, encode=[], encode_ext=".png", **kw).run(
        b for b, _ in posenet.ImageStream(paths, batch=4, decode="gpu").batches()))
    for g, p in zip(got, plain):
        assert np.array_equal(g[-1], p[-1])
    _check_pipeline(got, plain, 4)
