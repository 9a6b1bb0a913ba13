"""Baseline JPEG decode on the GPU, bit-exact with ``cv2.imdecode(buf, cv2.IMREAD_COLOR)`` (``pn_jpeg_parse`` / ``pn_jpeg_decode``)
and, at 1/2, 1/4, 1/8, with ``cv2.IMREAD_REDUCED_COLOR_*`` (``pn_jpeg_decode_scaled``), and encode, bit-exact with ``cv2.imencode(".jpg", frame, params)`` (``pn_jpeg_encode``).

    frames, status = posenet.imdecode_batch(buffers)                  # files of one size: CUDA uint8 [N, h, w, 3]
    rows, status, shapes = posenet.imdecode_batch(buffers)            # sizes differ: row i holds frame i at its own size
    frames, status = posenet.imdecode_batch(buffers, reduce=4)        # at 1/4 (cv2.IMREAD_REDUCED_COLOR_4), ceil(h/4) x ceil(w/4)
    out = posenet.imdecode_batch(buffers, orientation="gpu")          # EXIF-rotated files (phone portraits) rotated on the GPU too

``status[i]``: 0 decoded on the GPU, 1 decoded by cv2 on the host (progressive, arithmetic-coded, 12-bit, CMYK / RGB-coded or
truncated files, EXIF-rotated ones unless ``orientation="gpu"``, anything the parser does not know) and uploaded, < 0 the file's
entropy-coded data is malformed: its frame is zeros (cv2 decodes such files with a warning; its recovery is not reproduced).

    files = posenet.imencode_batch(frames, [cv2.IMWRITE_JPEG_QUALITY, 90])   # list of bytes, one per frame"""
import ctypes as C

import cv2
import numpy as np
import torch

from posenet import _native as nat
from posenet.imencode import encode_files


REDUCE_FLAGS = {1: cv2.IMREAD_COLOR, 2: cv2.IMREAD_REDUCED_COLOR_2, 4: cv2.IMREAD_REDUCED_COLOR_4,
                8: cv2.IMREAD_REDUCED_COLOR_8}


def imread_flag(reduce):
    """The cv2 imread / imdecode flag of a ``reduce`` factor (1, 2, 4 or 8); ValueError for any other."""
    if isinstance(reduce, bool) or reduce not in REDUCE_FLAGS:
        raise ValueError("reduce=%r: the decoders scale by 1, 2, 4 or 8 (cv2.IMREAD_REDUCED_COLOR_*)" % (reduce,))
    return REDUCE_FLAGS[reduce]


def reduced_size(h, w, reduce):
    """The frame size of an h x w JPEG file decoded at 1 / reduce: ceil(h / reduce) x ceil(w / reduce)."""
    return -(-int(h) // reduce), -(-int(w) // reduce)


ORIENTATIONS = ("cv2", "gpu")


def parser(orientation):
    """The C parser of an ``orientation`` option: "cv2" (EXIF-rotated files are cv2's, on the host) -> pn_jpeg_parse, "gpu" (files
    whose EXIF orientation is certain are rotated by the GPU decode, as cv2.imread rotates them) -> pn_jpeg_parse_oriented."""
    if orientation not in ORIENTATIONS:
        raise ValueError("orientation=%r: 'cv2' (rotated files decoded on the host) or 'gpu'" % (orientation,))
    lib = nat.load()
    return lib.pn_jpeg_parse_oriented if orientation == "gpu" else lib.pn_jpeg_parse


def frame_size(desc, reduce):
    """The frame a SUPPORTED descriptor decodes to at 1 / reduce: the reduced size, transposed for EXIF orientations 5..8."""
    h, w = reduced_size(desc.height, desc.width, reduce)
    return (w, h) if 5 <= desc.orientation <= 8 else (h, w)


def parse(buf, orientation="cv2"):
    """pn_jpeg_parse (``orientation="gpu"``: pn_jpeg_parse_oriented) on the bytes of one file: a ``_native.JpegDesc`` (``kind``
    JPEG_SUPPORTED / JPEG_HOST, ``why``, ``orientation``)."""
    fn = parser(orientation)
    a = np.frombuffer(buf, np.uint8) if not isinstance(buf, np.ndarray) else np.ascontiguousarray(buf, np.uint8).reshape(-1)
    d = nat.JpegDesc()
    nat.check(fn(a.ctypes.data if a.size else C.c_void_p(1), a.size, C.byref(d)), "pn_jpeg_parse")
    return d


def desc_bytes(descs):
    """The descriptors as one uint8 array (what pn_jpeg_decode reads from device memory)."""
    arr = (nat.JpegDesc * len(descs))(*descs)
    return np.frombuffer(bytes(arr), np.uint8).copy()


class Decoder:
    """Device buffers for ``pn_jpeg_decode_scaled`` at a fixed capacity: ``batch`` files of together at most ``arena_bytes``
    bytes, decoded at 1 / ``reduce`` to frames of at most ``max_h`` x ``max_w`` (files up to ``reduce * max_h`` x
    ``reduce * max_w``).  ``decode`` enqueues on the current stream."""

    def __init__(self, batch, arena_bytes, max_h, max_w, device=None, reduce=1):
        imread_flag(reduce)
        self.batch, self.arena_bytes, self.max_h, self.max_w = int(batch), int(arena_bytes), int(max_h), int(max_w)
        self.reduce = int(reduce)
        dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        n = C.c_size_t()
        nat.check(nat.load().pn_jpeg_workspace_scaled(self.batch, self.arena_bytes, self.max_h, self.max_w, self.reduce, C.byref(n)),
                  "pn_jpeg_workspace_scaled")
        self.ws = torch.empty(n.value, dtype=torch.uint8, device=dev)
        self.arena = torch.empty(self.arena_bytes, dtype=torch.uint8, device=dev)
        self.descs = torch.empty(self.batch * C.sizeof(nat.JpegDesc), dtype=torch.uint8, device=dev)
        self.status = torch.empty(self.batch, dtype=torch.int32, device=dev)

    def decode(self, frames, frame_stride, frame_hw=None):
        """Enqueue pn_jpeg_decode_scaled of ``self.arena`` / ``self.descs`` (filled by the caller) into ``frames``."""
        nat.check(nat.load().pn_jpeg_decode_scaled(
            C.c_void_p(self.arena.data_ptr()), self.arena_bytes, C.c_void_p(self.descs.data_ptr()), self.batch, self.max_h,
            self.max_w, self.reduce, C.c_void_p(frames.data_ptr()), int(frame_stride),
            C.c_void_p(frame_hw.data_ptr()) if frame_hw is not None else None, C.c_void_p(self.ws.data_ptr()), self.ws.numel(),
            C.c_void_p(self.status.data_ptr()), nat.stream_ptr()), "pn_jpeg_decode_scaled")


def imdecode_batch(buffers, device=None, reduce=1, orientation="cv2"):
    """Decode the JPEG files in ``buffers`` (bytes / uint8 arrays) on the GPU.  Returns ``(frames, status)`` when all frames
    share one size (frames: CUDA uint8 [N, h, w, 3]), else ``(rows, status, shapes)``: rows is CUDA uint8 [N, H * W * 3] (H x W
    the largest frame) with frame i stored contiguously from the start of row i, shapes the list of (h_i, w_i).  status: CUDA
    int32 [N].  Files cv2 cannot decode at all raise ValueError.

    ``reduce`` (1, 2, 4 or 8; anything else is a ValueError): decode at 1 / reduce, frame i equal to ``cv2.imdecode(buf,
    cv2.IMREAD_REDUCED_COLOR_<reduce>)`` -- ceil(h / reduce) x ceil(w / reduce) for JPEG files, scaled in the DCT domain.  Rows
    cv2 decodes on the host (status 1: progressive, EXIF-rotated, PNG, ...) are cv2's reduced decode too.

    ``orientation``: "cv2" (default) leaves files with an EXIF orientation other than 1 to cv2 on the host; "gpu" decodes those
    whose orientation is certain on the GPU, flipped / rotated as cv2 does (frame i is then the rotated frame, w x h for
    orientations 5..8; the rest stay cv2's).  Anything else is a ValueError."""
    flag = imread_flag(reduce)
    parser(orientation)
    nat.require_device()
    bufs = [np.frombuffer(b, np.uint8) if not isinstance(b, np.ndarray) else np.ascontiguousarray(b, np.uint8).reshape(-1)
            for b in buffers]
    assert bufs, "no buffers"
    descs, host_imgs, shapes = [], {}, []
    offset = 0
    for i, b in enumerate(bufs):
        d = parse(b, orientation)
        if d.kind == nat.JPEG_SUPPORTED:
            d.file_offset = offset
            offset += b.size
            shapes.append(frame_size(d, reduce))
        else:
            img = cv2.imdecode(b, flag)
            if img is None:
                raise ValueError("buffer %d is not an image cv2 can decode" % i)
            host_imgs[i] = img
            shapes.append(img.shape[:2])
        descs.append(d)
    H, W = max(s[0] for s in shapes), max(s[1] for s in shapes)
    dec = Decoder(len(bufs), max(offset, 1), H, W, device, reduce)
    dev = dec.arena.device
    if offset:
        arena = torch.from_numpy(np.concatenate([b for b, d in zip(bufs, descs) if d.kind == nat.JPEG_SUPPORTED]))
        dec.arena[:offset].copy_(arena.pin_memory(), non_blocking=True)
    dec.descs.copy_(torch.from_numpy(desc_bytes(descs)).pin_memory(), non_blocking=True)
    rows = torch.empty((len(bufs), H * W * 3), dtype=torch.uint8, device=dev)
    for i, img in host_imgs.items():
        rows[i, :img.size].copy_(torch.from_numpy(img.reshape(-1)))
    dec.decode(rows, H * W * 3)
    status = dec.status.clone()
    if all(s == shapes[0] for s in shapes):
        return rows.view(len(bufs), H, W, 3), status
    return rows, status, shapes



# ---- encode: pn_jpeg_encode_bound / pn_jpeg_encode -----------------------------------------------------------------------------------
SAMPLINGS = (0x411111, 0x221111, 0x211111, 0x121111, 0x111111)     # cv2.IMWRITE_JPEG_SAMPLING_FACTOR_411 .. _444


def encode_options(params=()):
    """(quality, sampling, restart_interval) of a cv2 ``imencode`` params list, with cv2's defaults (95, 4:2:0, none) and its
    clamping of the quality to 0..100.  ValueError for anything the device encoder does not do (optimised tables, progressive,
    separate luma / chroma quality, other formats' flags): the caller can use cv2 for those."""
    params = [int(p) for p in params]
    if len(params) % 2:
        raise ValueError("imencode params are (flag, value) pairs: %r" % (params,))
    quality, sampling, rst = 95, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_420, 0
    for flag, value in zip(params[::2], params[1::2]):
        if flag == cv2.IMWRITE_JPEG_QUALITY:
            quality = min(max(value, 0), 100)
        elif flag == cv2.IMWRITE_JPEG_SAMPLING_FACTOR:
            if value not in SAMPLINGS:
                raise ValueError("IMWRITE_JPEG_SAMPLING_FACTOR 0x%x is not one of cv2's five" % value)
            sampling = value
        elif flag == cv2.IMWRITE_JPEG_RST_INTERVAL:
            rst = min(max(value, 0), 65535)
        elif flag in (cv2.IMWRITE_JPEG_OPTIMIZE, cv2.IMWRITE_JPEG_PROGRESSIVE) and value == 0:
            pass
        else:
            raise ValueError("imencode param %d = %d is not supported on the device (use cv2.imencode)" % (flag, value))
    return quality, sampling, rst


def encode_bound(h, w, sampling=cv2.IMWRITE_JPEG_SAMPLING_FACTOR_420, restart_interval=0):
    """pn_jpeg_encode_bound: the largest file an h x w frame can encode to."""
    n = C.c_int64()
    nat.check(nat.load().pn_jpeg_encode_bound(int(h), int(w), int(sampling), int(restart_interval), C.byref(n)),
              "pn_jpeg_encode_bound")
    return n.value


class Encoder:
    """Device buffers for ``pn_jpeg_encode`` at a fixed capacity: ``batch`` frames of at most ``max_h`` x ``max_w``, encoded with
    the cv2 ``params``.  ``encode`` enqueues on the current stream; file i is then ``out[offsets[i]:offsets[i + 1]]``."""

    def __init__(self, batch, max_h, max_w, params=(), device=None):
        self.quality, self.sampling, self.rst = encode_options(params)
        self.batch, self.max_h, self.max_w = int(batch), int(max_h), int(max_w)
        dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        n = C.c_size_t()
        nat.check(nat.load().pn_jpeg_encode_workspace(self.batch, self.max_h, self.max_w, self.sampling, self.rst, C.byref(n)),
                  "pn_jpeg_encode_workspace")
        self.ws = torch.empty(n.value, dtype=torch.uint8, device=dev)
        self.capacity = self.batch * encode_bound(self.max_h, self.max_w, self.sampling, self.rst)
        self.out = torch.empty(self.capacity, dtype=torch.uint8, device=dev)
        self.offsets = torch.zeros(self.batch + 1, dtype=torch.int64, device=dev)

    def encode(self, frames, frame_stride, frame_hw=None):
        """Enqueue pn_jpeg_encode of ``frames`` (frame i from byte ``i * frame_stride``; ``frame_hw``: CUDA int32 [batch, 2]
        per-frame sizes, or None for max_h x max_w everywhere) into ``self.out`` / ``self.offsets``."""
        nat.check(nat.load().pn_jpeg_encode(
            C.c_void_p(frames.data_ptr()), self.batch, self.max_h, self.max_w, int(frame_stride),
            C.c_void_p(frame_hw.data_ptr()) if frame_hw is not None else None, self.quality, self.sampling, self.rst,
            C.c_void_p(self.out.data_ptr()), self.capacity, C.c_void_p(self.offsets.data_ptr()), C.c_void_p(self.ws.data_ptr()),
            self.ws.numel(), nat.stream_ptr()), "pn_jpeg_encode")

    def files(self):
        """Synchronise and copy the files of the last ``encode`` back (the bytes in use only): a list of ``bytes``, one per
        frame."""
        off = self.offsets.cpu().numpy()
        data = self.out[:int(off[-1])].cpu().numpy()
        return [data[off[i]:off[i + 1]].tobytes() for i in range(self.batch)]


def imencode_batch(frames, params=(), shapes=None):
    """Encode every frame on the GPU; returns a list of ``bytes``, file i equal to ``cv2.imencode(".jpg", frame_i, params)[1]``.
    ``frames``: CUDA uint8 [N, h, w, 3] (BGR), or with ``shapes`` the rows [N, H * W * 3] and sizes ``imdecode_batch`` returns
    (frame i stored contiguously from the start of row i at its own size; a (0, 0) frame gives an empty file).  ``params``: cv2's
    flat list; IMWRITE_JPEG_QUALITY, _SAMPLING_FACTOR and _RST_INTERVAL, and OPTIMIZE / PROGRESSIVE at 0.  Anything else raises
    ValueError (see ``encode_options``)."""
    encode_options(params)
    return encode_files(Encoder, frames, params, shapes)
