"""Baseline JPEG files decoded on the GPU (pn_jpeg_decode / posenet.imdecode_batch) against cv2.imdecode, byte for byte, and
ImageStream(decode="gpu") + BatchPipeline(jpeg=True) against ImageStream() + BatchPipeline(): identical pose records and
overlay frames."""
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


def encode(img, params):
    ok, enc = cv2.imencode(".jpg", img, params)
    assert ok
    return enc.tobytes()


def check_batch(bufs):
    out = posenet.imdecode_batch(bufs)
    rows, status = out[0], out[1].cpu().numpy()
    shapes = out[2] if len(out) == 3 else [tuple(rows.shape[1:3])] * len(bufs)
    rows = rows.view(len(bufs), -1).cpu().numpy()
    for i, b in enumerate(bufs):
        ref = cv2.imdecode(np.frombuffer(b, np.uint8), cv2.IMREAD_COLOR)
        h, w = shapes[i]
        assert ref.shape[:2] == (h, w)
        got = rows[i, :h * w * 3].reshape(h, w, 3)
        assert np.array_equal(got, ref), (i, int(status[i]), h, w, int((got != ref).sum()))
    return status


def test_corpus_as_one_mixed_batch():
    bufs = [encode(img, p) for img, p, _ in corpus(seed=5)]
    status = check_batch(bufs)
    assert (status == 0).all(), status


def test_long_scans_and_stuffed_bytes():
    """Noisy q95-q100 scans span thousands of subsequences and are dense in stuffed 0xFF bytes."""
    rng = np.random.default_rng(21)
    bufs = []
    for (h, w), q, s in (((513, 513), 95, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_444), ((720, 1280), 100, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_420),
                         ((1024, 768), 98, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_422)):
        bufs.append(encode(rng.integers(0, 256, (h, w, 3), dtype=np.uint8), [cv2.IMWRITE_JPEG_QUALITY, q,
                                                                             cv2.IMWRITE_JPEG_SAMPLING_FACTOR, s]))
    assert max(len(b) for b in bufs) * 8 > 2000 * 1024
    assert min(b.count(b"\xff\x00") for b in bufs) > 500
    bufs.append(encode(synth.smooth_image(1, 1, 3), [cv2.IMWRITE_JPEG_QUALITY, 90]))               # shorter than one subsequence
    bufs.append(encode(synth.smooth_image(64, 96, 4), [cv2.IMWRITE_JPEG_RST_INTERVAL, 1]))        # one MCU per restart interval
    assert (check_batch(bufs) == 0).all()


def test_host_fallback_rows():
    img = synth.smooth_image(90, 70, 8)
    prog = encode(img, [cv2.IMWRITE_JPEG_PROGRESSIVE, 1])
    png = cv2.imencode(".png", img)[1].tobytes()
    base = encode(img, [cv2.IMWRITE_JPEG_QUALITY, 80])
    status = check_batch([base, prog, png, base])
    assert status.tolist() == [0, 1, 1, 0]


def test_malformed_scans_are_flagged_and_nothing_outside_is_written():
    rng = np.random.default_rng(31)
    files = []
    for k in range(24):
        img = synth.smooth_image(int(rng.integers(8, 120)), int(rng.integers(8, 120)), 40 + k)
        b = bytearray(encode(img, [cv2.IMWRITE_JPEG_QUALITY, 90] + ([cv2.IMWRITE_JPEG_RST_INTERVAL, 2] if k % 3 == 0 else [])))
        d = pj.parse(bytes(b))
        lo, hi = d.scan_offset, len(b) - 2
        if k % 2:                                                          # flipped bits inside the scan
            for _ in range(int(rng.integers(1, 4))):
                q = int(rng.integers(lo, hi))
                if b[q] != 0xFF and b[q - 1] != 0xFF:
                    b[q] ^= 1 << int(rng.integers(0, 8))
                    if b[q] == 0xFF:
                        b[q] = 0xFE
        else:                                                              # scan cut short, the EOI kept
            b = b[:lo + int((hi - lo) * rng.uniform(0.1, 0.9))] + b"\xff\xd9"
        files.append(bytes(b))
    descs = [pj.parse(b) for b in files]
    assert all(d.kind == nat.JPEG_SUPPORTED for d in descs)
    H = max(d.height for d in descs)
    W = max(d.width for d in descs)
    G = 4096                                                               # guard bytes around every row and past the arena
    offs, arena = [], bytearray(G)
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
    nat.check(lib.pn_jpeg_workspace(n, len(arena), H, W, C.byref(ws_n)), "pn_jpeg_workspace")
    ws = torch.empty(ws_n.value, dtype=torch.uint8, device="cuda")
    descs_t = torch.from_numpy(pj.desc_bytes(descs).copy()).cuda()
    status = torch.full((n,), 99, dtype=torch.int32, device="cuda")
    hw = torch.full((n, 2), -1, dtype=torch.int32, device="cuda")
    nat.check(lib.pn_jpeg_decode(C.c_void_p(arena_t.data_ptr()), len(arena), C.c_void_p(descs_t.data_ptr()), n, H, W,
                                 C.c_void_p(frames.data_ptr()), stride, C.c_void_p(hw.data_ptr()), C.c_void_p(ws.data_ptr()),
                                 ws.numel(), C.c_void_p(status.data_ptr()), nat.stream_ptr()), "pn_jpeg_decode")
    st, fr, hw = status.cpu().numpy(), frames.cpu().numpy(), hw.cpu().numpy()
    assert torch.equal(arena_t, arena_before)
    assert (fr[n * stride:] == 0xAB).all()
    negative = 0
    for i, (d, b) in enumerate(zip(descs, files)):
        row = fr[i * stride:(i + 1) * stride]
        npx = d.height * d.width * 3
        assert (row[npx:] == 0xAB).all(), i
        if st[i] == 0:                                                     # still a valid stream: then it is cv2's image
            assert np.array_equal(row[:npx].reshape(d.height, d.width, 3), cv2.imdecode(np.frombuffer(b, np.uint8), 1)), i
            assert tuple(hw[i]) == (d.height, d.width)
        else:
            assert st[i] < 0 and (row[:npx] == 0).all() and tuple(hw[i]) == (0, 0), (i, st[i])
            negative += 1
    assert negative >= n // 2, st


def model(os_=16):
    sd = onet.init_params(50, seed=5, scheme="scaled", gain=0.8)
    m = posenet.MobileNetV1(50, output_stride=os_)
    m.load_state_dict(sd)
    return m.cuda().set_compute_dtype("bf16")


def _write(tmp_path, imgs, params_of):
    paths = []
    for i, img in enumerate(imgs):
        p = tmp_path / ("img%03d.jpg" % i)
        p.write_bytes(params_of(i, img))
        paths.append(str(p))
    return paths


def _same(a, b):
    assert len(a) == len(b)
    for ra, rb in zip(a, b):
        for x, y in zip(ra, rb):
            if isinstance(x, list):
                assert all(np.array_equal(u, v) for u, v in zip(x, y))
            else:
                assert np.array_equal(x, y)


def test_stream_pipeline_uniform_c2_shapes(tmp_path):
    """C2 shapes (513 x 513 files, OS16), overlay drawn: the records and frames of the GPU decode equal the cv2 path's."""
    imgs = [synth.smooth_image(513, 513, 200 + i) for i in range(19)]
    paths = _write(tmp_path, imgs, lambda i, im: encode(im, [cv2.IMWRITE_JPEG_QUALITY, 90]))
    m = model()
    kw = dict(depth=2, output_stride=16, min_pose_score=0.1, overlay=(0.1, 0.1))
    ref_stream = posenet.ImageStream(paths, batch=8)
    ref = list(posenet.BatchPipeline(m, 8, 513, 513, **kw).run(b for b, _ in ref_stream.batches()))
    stream = posenet.ImageStream(paths, batch=8, decode="gpu")
    got = list(posenet.BatchPipeline(m, 8, 513, 513, jpeg=True, **kw).run(b for b, _ in stream.batches()))
    assert [int((g[-1] == 0).sum()) for g in got] == [8, 8, 3]
    _same(ref, [g[:-1] for g in got])


def test_stream_pipeline_mixed_sizes_and_host_files(tmp_path):
    """A directory of different sizes, with progressive and EXIF-rotated files among the baseline ones (status 1 rows)."""
    rng = np.random.default_rng(4)
    imgs = [synth.smooth_image(int(rng.integers(100, 400)), int(rng.integers(100, 400)), 300 + i) for i in range(14)]
    tiff = b"MM\x00\x2a\x00\x00\x00\x08\x00\x01\x01\x12\x00\x03\x00\x00\x00\x01\x00\x06\x00\x00\x00\x00\x00\x00"
    app1 = b"\xff\xe1" + (len(tiff) + 8).to_bytes(2, "big") + b"Exif\x00\x00" + tiff

    def enc(i, im):
        if i % 5 == 1:
            return encode(im, [cv2.IMWRITE_JPEG_PROGRESSIVE, 1])
        if i % 5 == 3:
            b = encode(im, [cv2.IMWRITE_JPEG_QUALITY, 85])
            return b[:2] + app1 + b[2:]
        return encode(im, [cv2.IMWRITE_JPEG_QUALITY, 90, cv2.IMWRITE_JPEG_SAMPLING_FACTOR,
                           (cv2.IMWRITE_JPEG_SAMPLING_FACTOR_420, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_444)[i % 2]])
    paths = _write(tmp_path, imgs, enc)
    m = model()
    kw = dict(depth=2, output_stride=16, min_pose_score=0.1, mixed=True, source_coords=True, overlay=(0.1, 0.1))
    ref_stream = posenet.ImageStream(paths, batch=6, height=400, width=400, mixed=True)
    ref = list(posenet.BatchPipeline(m, 6, 400, 400, **kw).run((b, sh) for b, _, sh in ref_stream.batches()))
    stream = posenet.ImageStream(paths, batch=6, height=400, width=400, mixed=True, decode="gpu")
    got = list(posenet.BatchPipeline(m, 6, 400, 400, jpeg=True, **kw).run((b, sh) for b, _, sh in stream.batches()))
    status = np.concatenate([g[-1][:6] for g in got])[:len(paths)]
    assert status.tolist() == [1 if i % 5 in (1, 3) else 0 for i in range(len(paths))]
    _same(ref, [g[:-1] for g in got])


def test_stream_unreadable_file_raises(tmp_path):
    p = tmp_path / "missing.jpg"
    good = tmp_path / "good.jpg"
    good.write_bytes(encode(synth.smooth_image(40, 40, 1), [cv2.IMWRITE_JPEG_QUALITY, 90]))
    stream = posenet.ImageStream([str(good), str(p)], batch=2, decode="gpu")
    with pytest.raises(IOError):
        list(stream.batches())
