"""EXIF-rotated JPEG files decoded and rotated on the GPU (orientation="gpu": pn_jpeg_parse_oriented + pn_jpeg_decode_scaled)
against cv2.imdecode / cv2.imread, which rotate them, byte for byte: batches, the raw ABI, graph replay, and ImageStream +
BatchPipeline against the pipeline fed cv2's frames."""
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


def exif(o, le=False):
    bo = "little" if le else "big"
    tiff = (b"II*\x00" if le else b"MM\x00*") + (8).to_bytes(4, bo) + (1).to_bytes(2, bo) + (0x0112).to_bytes(2, bo) + \
        (3).to_bytes(2, bo) + (1).to_bytes(4, bo) + o.to_bytes(2, bo) + b"\0\0" + bytes(4)
    payload = b"Exif\0\0" + tiff
    return b"\xff\xe1" + (len(payload) + 2).to_bytes(2, "big") + payload


def rotate(buf, o, le=False):
    return buf[:2] + exif(o, le) + buf[2:]


def encode(img, params):
    ok, enc = cv2.imencode(".jpg", img, params)
    assert ok
    return enc.tobytes()


def check_batch(bufs, denom, orientation="gpu"):
    out = posenet.imdecode_batch(bufs, reduce=denom, orientation=orientation)
    rows, status = out[0], out[1].cpu().numpy()
    shapes = out[2] if len(out) == 3 else [tuple(rows.shape[1:3])] * len(bufs)
    rows = rows.view(len(bufs), -1)
    for i, b in enumerate(bufs):
        ref = cv2.imdecode(np.frombuffer(b, np.uint8), REDUCED[denom])
        h, w = shapes[i]
        assert ref.shape[:2] == (h, w), (i, ref.shape, h, w)
        got = rows[i, :h * w * 3].cpu().numpy().reshape(h, w, 3)
        assert np.array_equal(got, ref), (i, denom, int(status[i]), h, w, int((got != ref).sum()))
    return status


@pytest.mark.parametrize("denom", [1, 2, 4, 8])
def test_corpus_every_orientation_as_one_batch(denom):
    bufs = []
    for k, (img, p, _) in enumerate(corpus(seed=5)):
        base = encode(img, p)
        bufs += [rotate(base, o, le=(k + o) % 2 == 1) for o in range(1, 9)]
    status = check_batch(bufs, denom)
    assert (status == 0).all(), np.nonzero(status)[0][:20]


def test_default_routing_keeps_rotated_files_on_the_host():
    base = encode(synth.smooth_image(90, 70, 8), [cv2.IMWRITE_JPEG_QUALITY, 85])
    bufs = [rotate(base, o) for o in range(1, 9)]
    for denom in (1, 4):
        assert check_batch(bufs, denom, orientation="cv2").tolist() == [0] + [1] * 7
        assert check_batch(bufs, denom).tolist() == [0] * 8


@pytest.mark.parametrize("denom", [1, 4])
def test_raw_abi_capacity_and_guard_bytes(denom):
    """max_h != max_w; rotated files whose frame just fits, one that fits only unrotated (a descriptor error) and an orientation
    past 8 (a descriptor error): every frame is written at its oriented size, nothing outside the frames, the arena only read."""
    MH, MW = 40, 96
    rng = np.random.default_rng(denom)

    def jpeg(h, w, k):
        s = (cv2.IMWRITE_JPEG_SAMPLING_FACTOR_420, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_422, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_444)[k % 3]
        return encode(rng.integers(0, 256, (h, w, 3), dtype=np.uint8) if k % 2 else synth.smooth_image(h, w, 90 + k),
                      [cv2.IMWRITE_JPEG_QUALITY, 90, cv2.IMWRITE_JPEG_SAMPLING_FACTOR, s])

    full_h, full_w = MH * denom, MW * denom
    cases = [(jpeg(full_h, full_w, 0), 1, "ok"), (jpeg(full_w, full_h, 1), 6, "ok"), (jpeg(full_w, full_h, 2), 5, "ok"),
             (jpeg(full_w - 3, full_h - 1, 3), 7, "ok"), (jpeg(full_w, full_h, 4), 8, "ok"), (jpeg(full_h, full_w, 5), 3, "ok"),
             (jpeg(full_h, full_w - 5, 6), 2, "ok"), (jpeg(full_h, full_w, 7), 6, "err"), (jpeg(17, 23, 8), 4, "bad")]
    files = [rotate(b, o) for b, o, _ in cases]
    descs = [pj.parse(b, orientation="gpu") for b in files]
    assert all(d.kind == nat.JPEG_SUPPORTED for d in descs)
    descs[-1].orientation = 9
    G = 4096
    arena = bytearray(G)
    for d, b in zip(descs, files):
        d.file_offset = len(arena)
        arena += b + bytes(G)
    arena_t = torch.frombuffer(bytearray(arena), dtype=torch.uint8).cuda()
    arena_before = arena_t.clone()
    n = len(files)
    stride = MH * MW * 3 + G
    frames = torch.full((n * stride + G,), 0xAB, dtype=torch.uint8, device="cuda")
    ws_n = C.c_size_t()
    lib = nat.load()
    nat.check(lib.pn_jpeg_workspace_scaled(n, len(arena), MH, MW, denom, C.byref(ws_n)), "pn_jpeg_workspace_scaled")
    ws = torch.empty(ws_n.value, dtype=torch.uint8, device="cuda")
    descs_t = torch.from_numpy(pj.desc_bytes(descs).copy()).cuda()
    status = torch.full((n,), 99, dtype=torch.int32, device="cuda")
    hw = torch.full((n, 2), -1, dtype=torch.int32, device="cuda")
    nat.check(lib.pn_jpeg_decode_scaled(C.c_void_p(arena_t.data_ptr()), len(arena), C.c_void_p(descs_t.data_ptr()), n, MH, MW,
                                        denom, C.c_void_p(frames.data_ptr()), stride, C.c_void_p(hw.data_ptr()),
                                        C.c_void_p(ws.data_ptr()), ws.numel(), C.c_void_p(status.data_ptr()), nat.stream_ptr()),
              "pn_jpeg_decode_scaled")
    st, fr, hw = status.cpu().numpy(), frames.cpu().numpy(), hw.cpu().numpy()
    assert torch.equal(arena_t, arena_before)
    assert (fr[n * stride:] == 0xAB).all()
    for i, ((_, o, kind), b) in enumerate(zip(cases, files)):
        row = fr[i * stride:(i + 1) * stride]
        if kind == "ok":
            ref = cv2.imdecode(np.frombuffer(b, np.uint8), REDUCED[denom])
            h, w = ref.shape[:2]
            assert st[i] == 0 and tuple(hw[i]) == (h, w), (i, st[i], hw[i], ref.shape)
            assert np.array_equal(row[:h * w * 3].reshape(h, w, 3), ref), (i, o)
            assert (row[h * w * 3:] == 0xAB).all(), i
        else:
            assert st[i] == -1 and tuple(hw[i]) == (0, 0), (i, st[i])                          # PN_JPEG_ERR_DESC
            assert (row == 0xAB).all(), i


def test_graph_replay_with_other_orientations():
    """A decode captured in a CUDA graph replays on new files in other orientations: the launch geometry depends only on the
    capacity, not on the orientations."""
    denom, batch = 2, 8
    rng = np.random.default_rng(6)

    def files(seed, orients):
        out = []
        for k, o in enumerate(orients):
            h, w = int(rng.integers(60, 200)), int(rng.integers(60, 200))
            s = (cv2.IMWRITE_JPEG_SAMPLING_FACTOR_420, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_422)[k % 2]
            out.append(rotate(encode(synth.smooth_image(h, w, seed + k), [cv2.IMWRITE_JPEG_QUALITY, 90,
                                                                         cv2.IMWRITE_JPEG_SAMPLING_FACTOR, s]), o))
        return out

    H = W = 100
    dec = pj.Decoder(batch, batch * 200 * 200, H, W, reduce=denom)
    frames = torch.zeros((batch, H * W * 3), dtype=torch.uint8, device="cuda")
    hw = torch.zeros((batch, 2), dtype=torch.int32, device="cuda")

    def load(bufs):
        descs, off = [], 0
        for b in bufs:
            d = pj.parse(b, orientation="gpu")
            d.file_offset = off
            off += len(b)
            descs.append(d)
        dec.arena[:off].copy_(torch.from_numpy(np.frombuffer(b"".join(bufs), np.uint8).copy()))
        dec.descs.copy_(torch.from_numpy(pj.desc_bytes(descs)))

    load(files(0, [1] * batch))
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        dec.decode(frames, H * W * 3, hw)
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        dec.decode(frames, H * W * 3, hw)
    for seed, orients in ((100, range(1, 9)), (200, [6, 6, 3, 8, 5, 1, 7, 2])):
        bufs = files(seed, list(orients))
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


@pytest.mark.parametrize("denom,encode_params", [(1, None), (4, [cv2.IMWRITE_JPEG_QUALITY, 90])])
def test_pipeline_mixed_rotated_directory(tmp_path, denom, encode_params):
    """A phone directory: landscapes, portraits stored with orientation 6, some 3 and 8 files, and a progressive one.  Records,
    drawn frames and written files of ImageStream(orientation="gpu") + BatchPipeline(jpeg=True) equal the cv2 stream's."""
    rng = np.random.default_rng(9 + denom)
    size = (360, 480) if denom == 1 else (900, 1200)
    orients = [1, 6, 6, 3, 1, 8, 6, 1, 6, 5]
    paths = []
    for i, o in enumerate(orients):
        img = synth.smooth_image(size[0] - int(rng.integers(0, 40)), size[1] - int(rng.integers(0, 40)), 900 + i)
        params = [cv2.IMWRITE_JPEG_QUALITY, 90, cv2.IMWRITE_JPEG_SAMPLING_FACTOR,
                  (cv2.IMWRITE_JPEG_SAMPLING_FACTOR_420, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_422)[i % 2]]
        if i == 7:
            params = [cv2.IMWRITE_JPEG_PROGRESSIVE, 1]
        p = tmp_path / ("img%03d.jpg" % i)
        p.write_bytes(rotate(encode(img, params), o, le=i % 3 == 0))
        paths.append(str(p))
    side = -(-max(size) // denom)
    m = model()
    kw = dict(depth=2, output_stride=16, min_pose_score=0.1, mixed=True, source_coords=True, overlay=(0.1, 0.1))
    if encode_params is not None:
        kw["encode"] = encode_params
    ref_stream = posenet.ImageStream(paths, batch=4, height=side, width=side, mixed=True, reduce=denom)
    ref = list(posenet.BatchPipeline(m, 4, side, side, **kw).run((b, sh) for b, _, sh in ref_stream.batches()))
    stream = posenet.ImageStream(paths, batch=4, height=side, width=side, mixed=True, reduce=denom, decode="gpu",
                                 orientation="gpu")
    extra = dict(reduce=denom, arena_bytes=stream.arena_bytes) if denom > 1 else {}
    pipe = posenet.BatchPipeline(m, 4, side, side, jpeg=True, **extra, **kw)
    got = list(pipe.run((b, sh) for b, _, sh in stream.batches()))
    status = np.concatenate([g[-1][:4] for g in got])[:len(paths)]
    assert status.tolist() == [1 if i == 7 else 0 for i in range(len(paths))]
    _same(ref, [g[:-1] for g in got])
    # the default routing: the rotated files are cv2's (status 1), the records the same
    old = posenet.ImageStream(paths, batch=4, height=side, width=side, mixed=True, reduce=denom, decode="gpu")
    got_old = list(pipe.run((b, sh) for b, _, sh in old.batches()))
    status = np.concatenate([g[-1][:4] for g in got_old])[:len(paths)]
    assert status.tolist() == [0 if o == 1 and i != 7 else 1 for i, o in enumerate(orients)]
    _same(ref, [g[:-1] for g in got_old])


def test_dense_stream_refuses_a_mix_like_cv2(tmp_path):
    base = encode(synth.smooth_image(64, 96, 2), [cv2.IMWRITE_JPEG_QUALITY, 90])
    paths = []
    for i, o in enumerate((1, 3, 6)):
        p = tmp_path / ("f%d.jpg" % i)
        p.write_bytes(rotate(base, o))
        paths.append(str(p))
    for kw in (dict(decode="gpu", orientation="gpu"), dict()):
        with pytest.raises(ValueError):
            list(posenet.ImageStream(paths, batch=3, **kw).batches())
    enc, n = next(posenet.ImageStream(paths[:2], batch=2, decode="gpu", orientation="gpu").batches())
    assert enc.host_rows == [] and enc.shapes[:n] == [(64, 96)] * 2
