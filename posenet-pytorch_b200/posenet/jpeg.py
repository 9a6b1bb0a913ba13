"""Baseline JPEG decode on the GPU, bit-exact with ``cv2.imdecode(buf, cv2.IMREAD_COLOR)`` (``pn_jpeg_parse`` / ``pn_jpeg_decode``).

    frames, status = posenet.imdecode_batch(buffers)                  # files of one size: CUDA uint8 [N, h, w, 3]
    rows, status, shapes = posenet.imdecode_batch(buffers)            # sizes differ: row i holds frame i at its own size

``status[i]``: 0 decoded on the GPU, 1 decoded by cv2 on the host (progressive, arithmetic-coded, 12-bit, CMYK / RGB-coded,
EXIF-rotated or truncated files, anything the parser does not know) and uploaded, < 0 the file's entropy-coded data is
malformed: its frame is zeros (cv2 decodes such files with a warning; its recovery is not reproduced)."""
import ctypes as C

import cv2
import numpy as np
import torch

from posenet import _native as nat


def parse(buf):
    """pn_jpeg_parse on the bytes of one file: a ``_native.JpegDesc`` (``kind`` JPEG_SUPPORTED / JPEG_HOST, ``why``)."""
    a = np.frombuffer(buf, np.uint8) if not isinstance(buf, np.ndarray) else np.ascontiguousarray(buf, np.uint8).reshape(-1)
    d = nat.JpegDesc()
    nat.check(nat.load().pn_jpeg_parse(a.ctypes.data if a.size else C.c_void_p(1), a.size, C.byref(d)), "pn_jpeg_parse")
    return d


def desc_bytes(descs):
    """The descriptors as one uint8 array (what pn_jpeg_decode reads from device memory)."""
    arr = (nat.JpegDesc * len(descs))(*descs)
    return np.frombuffer(bytes(arr), np.uint8).copy()


class Decoder:
    """Device buffers for ``pn_jpeg_decode`` at a fixed capacity: ``batch`` files of together at most ``arena_bytes`` bytes,
    none larger than ``max_h`` x ``max_w``.  ``decode`` enqueues on the current stream."""

    def __init__(self, batch, arena_bytes, max_h, max_w, device=None):
        self.batch, self.arena_bytes, self.max_h, self.max_w = int(batch), int(arena_bytes), int(max_h), int(max_w)
        dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        n = C.c_size_t()
        nat.check(nat.load().pn_jpeg_workspace(self.batch, self.arena_bytes, self.max_h, self.max_w, C.byref(n)), "pn_jpeg_workspace")
        self.ws = torch.empty(n.value, dtype=torch.uint8, device=dev)
        self.arena = torch.empty(self.arena_bytes, dtype=torch.uint8, device=dev)
        self.descs = torch.empty(self.batch * C.sizeof(nat.JpegDesc), dtype=torch.uint8, device=dev)
        self.status = torch.empty(self.batch, dtype=torch.int32, device=dev)

    def decode(self, frames, frame_stride, frame_hw=None):
        """Enqueue pn_jpeg_decode of ``self.arena`` / ``self.descs`` (filled by the caller) into ``frames``."""
        nat.check(nat.load().pn_jpeg_decode(
            C.c_void_p(self.arena.data_ptr()), self.arena_bytes, C.c_void_p(self.descs.data_ptr()), self.batch, self.max_h,
            self.max_w, C.c_void_p(frames.data_ptr()), int(frame_stride),
            C.c_void_p(frame_hw.data_ptr()) if frame_hw is not None else None, C.c_void_p(self.ws.data_ptr()), self.ws.numel(),
            C.c_void_p(self.status.data_ptr()), nat.stream_ptr()), "pn_jpeg_decode")


def imdecode_batch(buffers, device=None):
    """Decode the JPEG files in ``buffers`` (bytes / uint8 arrays) on the GPU.  Returns ``(frames, status)`` when all frames
    share one size (frames: CUDA uint8 [N, h, w, 3]), else ``(rows, status, shapes)``: rows is CUDA uint8 [N, H * W * 3] (H x W
    the largest frame) with frame i stored contiguously from the start of row i, shapes the list of (h_i, w_i).  status: CUDA
    int32 [N].  Files cv2 cannot decode at all raise ValueError."""
    nat.require_device()
    bufs = [np.frombuffer(b, np.uint8) if not isinstance(b, np.ndarray) else np.ascontiguousarray(b, np.uint8).reshape(-1)
            for b in buffers]
    assert bufs, "no buffers"
    descs, host_imgs, shapes = [], {}, []
    offset = 0
    for i, b in enumerate(bufs):
        d = parse(b)
        if d.kind == nat.JPEG_SUPPORTED:
            d.file_offset = offset
            offset += b.size
            shapes.append((d.height, d.width))
        else:
            img = cv2.imdecode(b, cv2.IMREAD_COLOR)
            if img is None:
                raise ValueError("buffer %d is not an image cv2 can decode" % i)
            host_imgs[i] = img
            shapes.append(img.shape[:2])
        descs.append(d)
    H, W = max(s[0] for s in shapes), max(s[1] for s in shapes)
    dec = Decoder(len(bufs), max(offset, 1), H, W, device)
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

