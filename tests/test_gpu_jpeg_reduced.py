"""JPEG files decoded on the GPU at 1/2, 1/4 and 1/8 (pn_jpeg_decode_scaled / imdecode_batch(reduce=d)) against
cv2.imdecode(IMREAD_REDUCED_COLOR_d), byte for byte, and ImageStream(reduce=d) + BatchPipeline(jpeg=True, reduce=d) against the
pipeline fed cv2's reduced frames."""
import ctypes as C

import cv2
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

import posenet  # noqa: E402
from jpeg_corpus import corpus  # noqa: E402
from oracle import net as onet  # noqa: E402
from oracle import synth  # noqa: E402
from posenet import _native as nat  # noqa: E402
from posenet import jpeg as pj  # noqa: E402

REDUCED = {1: cv2.IMREAD_COLOR, 2: cv2.IMREAD_REDUCED_COLOR_2, 4: cv2.IMREAD_REDUCED_COLOR_4, 8: cv2.IMREAD_REDUCED_COLOR_8}
TIFF6 = b"MM\x00\x2a\x00\x00\x00\x08\x00\x01\x01\x12\x00\x03\x00\x00\x00\x01\x00\x06\x00\x00\x00\x00\x00\x00"
APP1 = b"\xff\xe1" + (len(TIFF6) + 8).to_bytes(2, "big") + b"Exif\x00\x00" + TIFF6


def encode(img, params):
    ok, enc = cv2.imencode(".jpg", img, params)
    assert ok
    return enc.tobytes()


def check_batch(bufs, denom):
    out = posenet.imdecode_batch(bufs, reduce=denom)
    rows, status = out[0], out[1].cpu().numpy()
    shapes = out[2] if len(out) == 3 else [tuple(rows.shape[1:3])] * len(bufs)
    rows = rows.view(len(bufs), -1).cpu().numpy()
    for i, b in enumerate(bufs):
        ref = cv2.imdecode(np.frombuffer(b, np.uint8), REDUCED[denom])
        h, w = shapes[i]
        assert ref.shape[:2] == (h, w), (i, ref.shape, h, w)
        got = rows[i, :h * w * 3].reshape(h, w, 3)
        assert np.array_equal(got, ref), (i, denom, int(status[i]), h, w, int((got != ref).sum()))
    return status


@pytest.mark.parametrize("denom", [2, 4, 8])
def test_corpus_as_one_mixed_batch_reduced(denom):
    bufs = [encode(img, p) for img, p, _ in corpus(seed=5)]
    rng = np.random.default_rng(denom)
    bufs.append(encode(rng.integers(0, 256, (513, 513, 3), dtype=np.uint8),
                       [cv2.IMWRITE_JPEG_QUALITY, 95, cv2.IMWRITE_JPEG_SAMPLING_FACTOR, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_444]))
    status = check_batch(bufs, denom)
    assert (status == 0).all(), status


@pytest.mark.parametrize("denom", [2, 8])
def test_host_fallback_rows_reduced(denom):
    img = synth.smooth_image(90, 70, 8)
    prog = encode(img, [cv2.IMWRITE_JPEG_PROGRESSIVE, 1])
    png = cv2.imencode(".png", img)[1].tobytes()
    base = encode(img, [cv2.IMWRITE_JPEG_QUALITY, 80])
    rot = base[:2] + APP1 + base[2:]
    status = check_batch([base, prog, png, rot, base], denom)
    assert status.tolist() == [0, 1, 1, 1, 0]


def test_reduce_one_is_the_full_size_decode():
    """reduce=1 and the original entry point give the same bytes."""
    bufs = [encode(img, p) for img, p, _ in corpus(seed=7)][::3]
    a = posenet.imdecode_batch(bufs, reduce=1)
    descs = [pj.parse(b) for b in bufs]
    off = 0
    for d, b in zip(descs, bufs):
        d.file_offset = off
        off += len(b)
    H, W = max(d.height for d in descs), max(d.width for d in descs)
    arena = torch.from_numpy(np.frombuffer(b"".join(bufs), np.uint8).copy()).cuda()
    descs_t = torch.from_numpy(pj.desc_bytes(descs)).cuda()
    n = C.c_size_t()
    lib = nat.load()
    nat.check(lib.pn_jpeg_workspace(len(bufs), off, H, W, C.byref(n)), "pn_jpeg_workspace")
    ws = torch.empty(n.value, dtype=torch.uint8, device="cuda")
    rows = torch.empty((len(bufs), H * W * 3), dtype=torch.uint8, device="cuda")
    status = torch.empty(len(bufs), dtype=torch.int32, device="cuda")
    nat.check(lib.pn_jpeg_decode(C.c_void_p(arena.data_ptr()), off, C.c_void_p(descs_t.data_ptr()), len(bufs), H, W,
                                 C.c_void_p(rows.data_ptr()), H * W * 3, None, C.c_void_p(ws.data_ptr()), ws.numel(),
                                 C.c_void_p(status.data_ptr()), nat.stream_ptr()), "pn_jpeg_decode")
    assert (status == 0).all() and (a[1] == 0).all()
    shapes = a[2]
    for i, (h, w) in enumerate(shapes):
        assert torch.equal(a[0][i, :h * w * 3], rows[i, :h * w * 3]), i


@pytest.mark.parametrize("denom", [2, 4, 8])
def test_malformed_scans_reduced(denom):
    """Corrupt scans give status < 0 and a zero frame at the reduced size; no byte outside the frames is written and the arena
    is only read."""
    rng = np.random.default_rng(31 + denom)
    files = []
    for k in range(24):
        img = synth.smooth_image(int(rng.integers(8, 160)), int(rng.integers(8, 160)), 40 + k)
        samp = (cv2.IMWRITE_JPEG_SAMPLING_FACTOR_420, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_422, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_444)[k % 3]
        b = bytearray(encode(img, [cv2.IMWRITE_JPEG_QUALITY, 90, cv2.IMWRITE_JPEG_SAMPLING_FACTOR, samp] +
                             ([cv2.IMWRITE_JPEG_RST_INTERVAL, 2] if k % 4 == 0 else [])))
        d = pj.parse(bytes(b))
        lo, hi = d.scan_offset, len(b) - 2
        if k % 2:
            for _ in range(int(rng.integers(1, 4))):
                q = int(rng.integers(lo, hi))
                if b[q] != 0xFF and b[q - 1] != 0xFF:
                    b[q] ^= 1 << int(rng.integers(0, 8))
                    if b[q] == 0xFF:
                        b[q] = 0xFE
        else:
            b = b[:lo + int((hi - lo) * rng.uniform(0.1, 0.9))] + b"\xff\xd9"
        files.append(bytes(b))
    descs = [pj.parse(b) for b in files]
    assert all(d.kind == nat.JPEG_SUPPORTED for d in descs)
    sizes = [pj.reduced_size(d.height, d.width, denom) for d in descs]
    H, W = max(s[0] for s in sizes), max(s[1] for s in sizes)
    G = 4096
    arena = bytearray(G)
    for d, b in zip(descs, files):
        d.file_offset = len(arena)
        arena += b + bytes(G)
    arena_t = torch.frombuffer(bytearray(arena), dtype=torch.uint8).cuda()
    arena_before = arena_t.clone()
    n = len(files)
    stride = H * W * 3 + G
    frames = torch.full((n * stride + G,), 0xAB, dtype=torch.uint8, device="cuda")
    ws_n = C.c_size_t()
    lib = nat.load()
    nat.check(lib.pn_jpeg_workspace_scaled(n, len(arena), H, W, denom, C.byref(ws_n)), "pn_jpeg_workspace_scaled")
    ws = torch.empty(ws_n.value, dtype=torch.uint8, device="cuda")
    descs_t = torch.from_numpy(pj.desc_bytes(descs).copy()).cuda()
    status = torch.full((n,), 99, dtype=torch.int32, device="cuda")
    hw = torch.full((n, 2), -1, dtype=torch.int32, device="cuda")
    nat.check(lib.pn_jpeg_decode_scaled(C.c_void_p(arena_t.data_ptr()), len(arena), C.c_void_p(descs_t.data_ptr()), n, H, W,
                                        denom, C.c_void_p(frames.data_ptr()), stride, C.c_void_p(hw.data_ptr()),
                                        C.c_void_p(ws.data_ptr()), ws.numel(), C.c_void_p(status.data_ptr()), nat.stream_ptr()),
              "pn_jpeg_decode_scaled")
    st, fr, hw = status.cpu().numpy(), frames.cpu().numpy(), hw.cpu().numpy()
    assert torch.equal(arena_t, arena_before)
    assert (fr[n * stride:] == 0xAB).all()
    negative = 0
    for i, ((h, w), b) in enumerate(zip(sizes, files)):
        row = fr[i * stride:(i + 1) * stride]
        npx = h * w * 3
        assert (row[npx:] == 0xAB).all(), i
        if st[i] == 0:
            assert np.array_equal(row[:npx].reshape(h, w, 3), cv2.imdecode(np.frombuffer(b, np.uint8), REDUCED[denom])), i
            assert tuple(hw[i]) == (h, w)
        else:
            assert st[i] < 0 and (row[:npx] == 0).all() and tuple(hw[i]) == (0, 0), (i, st[i])
            negative += 1
    assert negative >= n // 2, st


def test_graph_replay_on_new_files():
    """A decode captured in a CUDA graph replays on new file contents: the launch geometry depends only on the capacity."""
    denom, batch = 4, 6
    rng = np.random.default_rng(5)

    def files(seed):
        out = []
        for k in range(batch):
            h, w = int(rng.integers(100, 400)), int(rng.integers(100, 400))
            s = (cv2.IMWRITE_JPEG_SAMPLING_FACTOR_420, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_422, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_444)[k % 3]
            out.append(encode(synth.smooth_image(h, w, seed + k), [cv2.IMWRITE_JPEG_QUALITY, 90, cv2.IMWRITE_JPEG_SAMPLING_FACTOR, s]))
        return out

    H = W = 100
    dec = pj.Decoder(batch, batch * 400 * 400, H, W, reduce=denom)
    frames = torch.zeros((batch, H * W * 3), dtype=torch.uint8, device="cuda")
    hw = torch.zeros((batch, 2), dtype=torch.int32, device="cuda")

    def load(bufs):
        descs, off = [], 0
        for b in bufs:
            d = pj.parse(b)
            d.file_offset = off
            off += len(b)
            descs.append(d)
        dec.arena[:off].copy_(torch.from_numpy(np.frombuffer(b"".join(bufs), np.uint8).copy()))
        dec.descs.copy_(torch.from_numpy(pj.desc_bytes(descs)))

    load(files(0))
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        dec.decode(frames, H * W * 3, hw)
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        dec.decode(frames, H * W * 3, hw)
    for seed in (100, 200):
        bufs = files(seed)
        load(bufs)
        g.replay()
        torch.cuda.synchronize()
        assert (dec.status == 0).all()
        fr, sz = frames.cpu().numpy(), hw.cpu().numpy()
        for i, b in enumerate(bufs):
            ref = cv2.imdecode(np.frombuffer(b, np.uint8), REDUCED[denom])
            h, w = sz[i]
            assert (h, w) == ref.shape[:2]
            assert np.array_equal(fr[i, :h * w * 3].reshape(h, w, 3), ref), (seed, i)


# ---- ImageStream + BatchPipeline ----------------------------------------------------------------------------------------------------
def decode_encoded(enc, h, w):
    """The frames of one EncodedBatch as BatchPipeline(jpeg=True) would decode them (device decode + host rows)."""
    dec = pj.Decoder(enc.batch, enc.arena.numel(), h, w, reduce=enc.reduce)
    dec.arena[:enc.used].copy_(enc.arena[:enc.used])
    dec.descs.copy_(enc.descs)
    x = torch.zeros((enc.batch, h * w * 3), dtype=torch.uint8, device="cuda")
    raw = enc.raw.view(enc.batch, -1)
    for i in enc.host_rows:
        x[i].copy_(raw[i])
    dec.decode(x, h * w * 3)
    return x.cpu().numpy(), dec.status.cpu().numpy()


def _write(tmp_path, imgs, params_of):
    paths = []
    for i, img in enumerate(imgs):
        p = tmp_path / ("img%03d.jpg" % i)
        p.write_bytes(params_of(i, img))
        paths.append(str(p))
    return paths


@pytest.mark.parametrize("denom", [2, 4, 8])
def test_stream_frames_cv2_and_gpu_identical(tmp_path, denom):
    imgs = [synth.smooth_image(300 + 7 * i, 410 - 5 * i, 500 + i) for i in range(7)]
    paths = _write(tmp_path, imgs, lambda i, im: encode(im, [cv2.IMWRITE_JPEG_QUALITY, 90]) if i != 3
                   else encode(im, [cv2.IMWRITE_JPEG_PROGRESSIVE, 1]))
    H, W = pj.reduced_size(400, 420, denom)
    ref = posenet.ImageStream(paths, batch=4, height=H, width=W, mixed=True, reduce=denom)
    got = posenet.ImageStream(paths, batch=4, height=H, width=W, mixed=True, reduce=denom, decode="gpu")
    for (rb, rn, rsh), (enc, gn, gsh) in zip(ref.batches(), got.batches()):
        assert rn == gn and rsh == gsh
        fr, st = decode_encoded(enc, H, W)
        rows = rb.view(4, -1).numpy()
        for i, (h, w) in enumerate(rsh):
            assert np.array_equal(fr[i, :h * w * 3], rows[i, :h * w * 3]), i
        assert all(s in (0, 1) for s in st[:gn])


def model(os_=16):
    sd = onet.init_params(50, seed=5, scheme="scaled", gain=0.8)
    m = posenet.MobileNetV1(50, output_stride=os_)
    m.load_state_dict(sd)
    return m.cuda().set_compute_dtype("bf16")


def _same(a, b):
    assert len(a) == len(b)
    for ra, rb in zip(a, b):
        assert len(ra) == len(rb)
        for x, y in zip(ra, rb):
            if isinstance(x, list):
                assert len(x) == len(y) and all(np.array_equal(u, v) for u, v in zip(x, y))
            else:
                assert np.array_equal(x, y)


def test_pipeline_dense_reduced_c2_shapes(tmp_path):
    """1026 x 1026 photos at 1/2: 513 x 513 frames, the C2 shape.  Records and drawn frames equal the cv2-reduced pipeline's."""
    imgs = [synth.smooth_image(1026, 1026, 700 + i) for i in range(11)]
    paths = _write(tmp_path, imgs, lambda i, im: encode(im, [cv2.IMWRITE_JPEG_QUALITY, 90]))
    m = model()
    kw = dict(depth=2, output_stride=16, min_pose_score=0.1, overlay=(0.1, 0.1))
    ref_stream = posenet.ImageStream(paths, batch=4, reduce=2)
    assert (ref_stream.height, ref_stream.width) == (513, 513)
    ref = list(posenet.BatchPipeline(m, 4, 513, 513, **kw).run(b for b, _ in ref_stream.batches()))
    stream = posenet.ImageStream(paths, batch=4, reduce=2, decode="gpu")
    pipe = posenet.BatchPipeline(m, 4, 513, 513, jpeg=True, reduce=2, **kw)
    got = list(pipe.run(b for b, _ in stream.batches()))
    assert [int((g[-1] == 0).sum()) for g in got] == [4, 4, 3]
    _same(ref, [g[:-1] for g in got])
    with pytest.raises(AssertionError):                               # a stream at another scale is refused
        other = posenet.ImageStream(paths, batch=4, height=257, width=257, reduce=4, decode="gpu")
        list(pipe.run(b for b, _ in other.batches()))


def test_pipeline_mixed_reduced_with_host_files_overlay_encode(tmp_path):
    """Different sizes at 1/4 with progressive and EXIF-rotated files among them, source_coords, overlay and JPEG encode of the
    drawn reduced frames: the files written equal the cv2-reduced pipeline's."""
    rng = np.random.default_rng(4)
    imgs = [synth.smooth_image(int(rng.integers(400, 1200)), int(rng.integers(400, 1200)), 800 + i) for i in range(10)]

    def enc(i, im):
        if i % 5 == 1:
            return encode(im, [cv2.IMWRITE_JPEG_PROGRESSIVE, 1])
        if i % 5 == 3:
            b = encode(im, [cv2.IMWRITE_JPEG_QUALITY, 85])
            return b[:2] + APP1 + b[2:]
        return encode(im, [cv2.IMWRITE_JPEG_QUALITY, 90, cv2.IMWRITE_JPEG_SAMPLING_FACTOR,
                           (cv2.IMWRITE_JPEG_SAMPLING_FACTOR_420, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_422)[i % 2]])
    paths = _write(tmp_path, imgs, enc)
    m = model()
    kw = dict(depth=2, output_stride=16, min_pose_score=0.1, mixed=True, source_coords=True, overlay=(0.1, 0.1),
              encode=[cv2.IMWRITE_JPEG_QUALITY, 90])
    ref_stream = posenet.ImageStream(paths, batch=4, height=300, width=300, mixed=True, reduce=4)
    ref = list(posenet.BatchPipeline(m, 4, 300, 300, **kw).run((b, sh) for b, _, sh in ref_stream.batches()))
    stream = posenet.ImageStream(paths, batch=4, height=300, width=300, mixed=True, reduce=4, decode="gpu")
    got = list(posenet.BatchPipeline(m, 4, 300, 300, jpeg=True, reduce=4, arena_bytes=stream.arena_bytes, **kw).run(
        (b, sh) for b, _, sh in stream.batches()))
    status = np.concatenate([g[-1][:4] for g in got])[:len(paths)]
    assert status.tolist() == [1 if i % 5 in (1, 3) else 0 for i in range(len(paths))]
    _same(ref, [g[:-1] for g in got])
