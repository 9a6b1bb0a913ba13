"""Progressive JPEG files decoded on the GPU (progressive="gpu": pn_jpeg_parse_progressive + pn_jpeg_decode_scaled) against
cv2.imdecode / cv2.imread byte for byte: batches at every scale and orientation, mixed batches, malformed entropy data with guard
bytes, graph replay, and ImageStream + BatchPipeline against the pipeline fed cv2's frames."""
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
PROG = [cv2.IMWRITE_JPEG_PROGRESSIVE, 1]


def rotate(buf, o):
    """The file with an Exif APP1 segment of orientation o after its SOI."""
    tiff = b"MM\x00*" + (8).to_bytes(4, "big") + (1).to_bytes(2, "big") + (0x0112).to_bytes(2, "big") + (3).to_bytes(2, "big") + \
        (1).to_bytes(4, "big") + o.to_bytes(2, "big") + b"\0\0" + bytes(4)
    payload = b"Exif\0\0" + tiff
    return buf[:2] + b"\xff\xe1" + (len(payload) + 2).to_bytes(2, "big") + payload + buf[2:]


def encode(img, params):
    ok, enc = cv2.imencode(".jpg", img, params)
    assert ok
    return enc.tobytes()


def check_batch(bufs, denom, orientation="cv2", progressive="gpu"):
    out = posenet.imdecode_batch(bufs, reduce=denom, orientation=orientation, progressive=progressive)
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
def test_corpus_as_one_batch(denom):
    bufs = [encode(img, p + PROG) for img, p, _ in corpus(seed=11)]
    status = check_batch(bufs, denom)
    assert (status == 0).all(), np.nonzero(status)[0][:20]


@pytest.mark.parametrize("denom", [1, 4])
def test_rotated_progressive_files(denom):
    bufs = []
    for k, (img, p, _) in enumerate(corpus(seed=12)[::6]):
        base = encode(img, p + PROG)
        bufs += [rotate(base, o) for o in range(1, 9)]
    assert (check_batch(bufs, denom, orientation="gpu") == 0).all()
    assert check_batch(bufs, denom).tolist() == [0 if i % 8 == 0 else 1 for i in range(len(bufs))]


def test_mixed_batch_statuses():
    """Baseline, progressive, PNG and progressive cut short after a scan (EOI kept: an incomplete script, which cv2 decodes with
    block smoothing): 0 / 0 / 1 / 1; with progressive="cv2" the progressive file is cv2's."""
    img = synth.smooth_image(120, 90, 4)
    base, prog = encode(img, [cv2.IMWRITE_JPEG_QUALITY, 90]), encode(img, [cv2.IMWRITE_JPEG_QUALITY, 90] + PROG)
    png = cv2.imencode(".png", img)[1].tobytes()
    last = nat.JpegScan.from_buffer_copy(pj.parse(prog, progressive="gpu")[1], C.sizeof(nat.JpegScans) + 6 * C.sizeof(nat.JpegScan))
    bufs = [base, prog, png, prog[:last.end] + b"\xff\xd9"]
    for denom in (1, 2):
        assert check_batch(bufs, denom).tolist() == [0, 0, 1, 1]
        assert check_batch(bufs, denom, progressive="cv2").tolist() == [0, 1, 1, 1]


def test_malformed_entropy_data_and_guard_bytes():
    """Corrupt entropy-coded data or a wrong RST marker gives a status < 0 and a zero frame; a broken scan table or an MCU layout
    other than the parser's (a permuted one, one without a component) is a descriptor error that leaves its frame untouched;
    nothing outside the frames is written and the arena is only read."""
    rng = np.random.default_rng(3)
    MH, MW, G = 96, 128, 4096
    files, descs, expect = [], [], []
    for k in range(12):
        h, w = int(rng.integers(40, MH)), int(rng.integers(40, MW))
        img = rng.integers(0, 256, (h, w, 3), dtype=np.uint8) if k % 2 else synth.smooth_image(h, w, 30 + k)
        params = [cv2.IMWRITE_JPEG_QUALITY, 90] + PROG + ([cv2.IMWRITE_JPEG_RST_INTERVAL, 2] if k % 3 == 0 else [])
        buf = bytearray(encode(img, params))
        d, table = pj.parse(bytes(buf), progressive="gpu")
        scans = [nat.JpegScan.from_buffer_copy(table, C.sizeof(nat.JpegScans) + i * C.sizeof(nat.JpegScan)) for i in range(10)]
        kind = "ok"
        if k in (1, 4, 7):                  # garbage in the middle of the last (largest) scan: bad codes or a length error
            s = scans[-1]
            for q in range(s.start + (s.end - s.start) // 3, s.start + (s.end - s.start) // 2):
                buf[q] = int(rng.integers(0, 255))
            kind = "err"
        elif k == 3:                        # RST1 of the first scan renumbered RST3
            q = bytes(buf).index(b"\xff\xd1", scans[0].start)
            assert q < scans[0].end
            buf[q + 1] = 0xD3
            kind = "rst"
        elif k == 10:                       # 4:2:0 MCU table permuted: chroma first (each entry still in range)
            d.mcu_comp[:6] = [1, 2, 0, 0, 0, 0]
            d.mcu_bx[:6] = [0, 0, 0, 1, 0, 1]
            d.mcu_by[:6] = [0, 0, 0, 0, 1, 1]
            kind = "desc"
        elif k == 11:                       # Cr left out of the MCU table (a second Cb block in its place)
            d.mcu_comp[5] = 1
            kind = "desc"
        elif k == 5:                        # a scan range outside the file
            t = bytearray(table)
            nat.JpegScan.from_buffer(t, C.sizeof(nat.JpegScans)).end = len(buf) + 10
            table = bytes(t)
            kind = "desc"
        elif k == 8:                        # a scan in the same wave as the one it refines
            t = bytearray(table)
            nat.JpegScan.from_buffer(t, C.sizeof(nat.JpegScans) + 9 * C.sizeof(nat.JpegScan)).wave = 1
            table = bytes(t)
            kind = "desc"
        files.append((bytes(buf), table))
        descs.append(d)
        expect.append(kind)
    arena = bytearray(G)
    for d, (b, t) in zip(descs, files):
        d.file_offset = len(arena)
        arena += b + bytes(pj.align8(len(b)) - len(b)) + t
        arena += bytes(G - len(arena) % 8)
    arena_t = torch.frombuffer(bytearray(arena), dtype=torch.uint8).cuda()
    before = arena_t.clone()
    n, stride = len(files), MH * MW * 3 + G
    frames = torch.full((n * stride + G,), 0xAB, dtype=torch.uint8, device="cuda")
    ws_n = C.c_size_t()
    lib = nat.load()
    nat.check(lib.pn_jpeg_workspace(n, len(arena), MH, MW, C.byref(ws_n)), "pn_jpeg_workspace")
    ws = torch.empty(ws_n.value, dtype=torch.uint8, device="cuda")
    descs_t = torch.from_numpy(pj.desc_bytes(descs).copy()).cuda()
    status = torch.full((n,), 99, dtype=torch.int32, device="cuda")
    nat.check(lib.pn_jpeg_decode(C.c_void_p(arena_t.data_ptr()), len(arena), C.c_void_p(descs_t.data_ptr()), n, MH, MW,
                                 C.c_void_p(frames.data_ptr()), stride, None, C.c_void_p(ws.data_ptr()), ws.numel(),
                                 C.c_void_p(status.data_ptr()), nat.stream_ptr()), "pn_jpeg_decode")
    st, fr = status.cpu().numpy(), frames.cpu().numpy()
    assert torch.equal(arena_t, before)
    assert (fr[n * stride:] == 0xAB).all()
    for i, ((b, _), kind) in enumerate(zip(files, expect)):
        row = fr[i * stride:(i + 1) * stride]
        ref = cv2.imdecode(np.frombuffer(b, np.uint8), cv2.IMREAD_COLOR)
        h, w = descs[i].height, descs[i].width
        if kind == "ok":
            assert st[i] == 0 and np.array_equal(row[:h * w * 3].reshape(h, w, 3), ref), (i, st[i])
        elif kind in ("err", "rst"):
            assert st[i] < 0 and (row[:h * w * 3] == 0).all(), (i, st[i])
            assert kind == "err" or st[i] == -3, (i, st[i])                                   # PN_JPEG_ERR_RESTART
        else:
            assert st[i] == -1 and (row == 0xAB).all(), (i, st[i])
        if kind != "desc":
            assert (row[h * w * 3:] == 0xAB).all(), i


def test_graph_replay_with_new_files():
    denom, batch, H, W = 2, 6, 100, 100
    rng = np.random.default_rng(8)

    def files(seed):
        out = []
        for k in range(batch):
            h, w = int(rng.integers(60, 200)), int(rng.integers(60, 200))
            p = [cv2.IMWRITE_JPEG_QUALITY, 70 + 5 * k] + (PROG if (seed + k) % 3 else [])
            out.append(encode(synth.smooth_image(h, w, seed + k), p))
        return out

    dec = pj.Decoder(batch, batch * 200 * 200 + batch * nat.JPEG_SCAN_TABLE_MAX, H, W, reduce=denom)
    frames = torch.zeros((batch, H * W * 3), dtype=torch.uint8, device="cuda")
    hw = torch.zeros((batch, 2), dtype=torch.int32, device="cuda")

    def load(bufs):
        descs, arena = [], bytearray()
        for b in bufs:
            d, t = pj.parse(b, progressive="gpu")
            d.file_offset = len(arena)
            arena += b + bytes(pj.align8(len(b)) - len(b)) + t
            arena += bytes(pj.align8(len(arena)) - len(arena))
            descs.append(d)
        dec.arena[:len(arena)].copy_(torch.frombuffer(arena, dtype=torch.uint8))
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
    for seed in (100, 201):
        bufs = files(seed)
        load(bufs)
        g.replay()
        torch.cuda.synchronize()
        assert (dec.status == 0).all()
        fr, sz = frames.cpu().numpy(), hw.cpu().numpy()
        for i, b in enumerate(bufs):
            ref = cv2.imdecode(np.frombuffer(b, np.uint8), REDUCED[denom])
            h, w = sz[i]
            assert (h, w) == ref.shape[:2] and np.array_equal(fr[i, :h * w * 3].reshape(h, w, 3), ref), (seed, i)


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
def test_pipeline_progressive_directory(tmp_path, denom, encode_params):
    """A web directory of progressive and baseline files of different sizes, one rotated: records, drawn frames and written files
    of ImageStream(progressive="gpu") + BatchPipeline(jpeg=True, mixed=True, source_coords=True) equal the cv2 stream's."""
    rng = np.random.default_rng(20 + denom)
    size = (360, 480) if denom == 1 else (900, 1200)
    paths = []
    for i in range(10):
        img = synth.smooth_image(size[0] - int(rng.integers(0, 40)), size[1] - int(rng.integers(0, 40)), 700 + i)
        params = [cv2.IMWRITE_JPEG_QUALITY, 90, cv2.IMWRITE_JPEG_SAMPLING_FACTOR,
                  (cv2.IMWRITE_JPEG_SAMPLING_FACTOR_420, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_444)[i % 2]]
        if i % 4 != 3:
            params += PROG
        if i == 5:
            params += [cv2.IMWRITE_JPEG_RST_INTERVAL, 4]
        buf = encode(img, params)
        p = tmp_path / ("img%03d.jpg" % i)
        p.write_bytes(rotate(buf, 6) if i == 2 else buf)
        paths.append(str(p))
    side = -(-max(size) // denom)
    m = model()
    kw = dict(depth=2, output_stride=16, min_pose_score=0.1, mixed=True, source_coords=True, overlay=(0.1, 0.1))
    if encode_params is not None:
        kw["encode"] = encode_params
    ref_stream = posenet.ImageStream(paths, batch=4, height=side, width=side, mixed=True, reduce=denom)
    ref = list(posenet.BatchPipeline(m, 4, side, side, **kw).run((b, sh) for b, _, sh in ref_stream.batches()))
    stream = posenet.ImageStream(paths, batch=4, height=side, width=side, mixed=True, reduce=denom, decode="gpu",
                                 orientation="gpu", progressive="gpu")
    pipe = posenet.BatchPipeline(m, 4, side, side, jpeg=True, reduce=denom, arena_bytes=stream.arena_bytes, **kw)
    got = list(pipe.run((b, sh) for b, _, sh in stream.batches()))
    status = np.concatenate([g[-1][:4] for g in got])[:len(paths)]
    assert status.tolist() == [0] * len(paths)
    _same(ref, [g[:-1] for g in got])


def test_pipeline_progressive_yuv_out(tmp_path):
    """BatchPipeline(jpeg=True, overlay=..., yuv_out=I420) fed progressive and baseline files by ImageStream(progressive="gpu"):
    records and YUV frames equal those of the same pipeline fed cv2's frames."""
    paths = []
    for i in range(10):
        params = [cv2.IMWRITE_JPEG_QUALITY, 90] + (PROG if i % 3 else [])
        p = tmp_path / ("img%03d.jpg" % i)
        p.write_bytes(encode(synth.smooth_image(480, 640, 800 + i), params))
        paths.append(str(p))
    m = model()
    kw = dict(depth=2, output_stride=16, min_pose_score=0.1, source_coords=True, overlay=(0.1, 0.1),
              yuv_out=cv2.COLOR_BGR2YUV_I420)
    ref_stream = posenet.ImageStream(paths, batch=4, height=480, width=640)
    ref = list(posenet.BatchPipeline(m, 4, 480, 640, **kw).run(b for b, _ in ref_stream.batches()))
    stream = posenet.ImageStream(paths, batch=4, height=480, width=640, decode="gpu", progressive="gpu")
    got = list(posenet.BatchPipeline(m, 4, 480, 640, jpeg=True, **kw).run(b for b, _ in stream.batches()))
    assert np.concatenate([g[-1] for g in got])[:len(paths)].tolist() == [0] * len(paths)
    assert any(r[0].max() > 0 for r in ref)
    _same(ref, [g[:-1] for g in got])
