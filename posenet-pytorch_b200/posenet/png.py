"""PNG encode on the GPU, bit-exact with ``cv2.imencode(".png", frame)`` (``pn_png_encode``).

    files = posenet.imencode_png_batch(frames)                           # list of bytes, one per frame

cv2 writes PNG without params with libpng's SUB filter on every row and zlib's fastest level with the run-length strategy; that
is what the device reproduces.  Any PNG flag (compression level, strategy, filter, bilevel, buffer size) makes cv2 choose
adaptive filters and a different deflate: such params raise ValueError, and the caller can use cv2 for them."""
import ctypes as C

import torch

from posenet import _native as nat
from posenet.imencode import encode_files


def encode_options(params=()):
    """Check a cv2 ``imencode`` params list for the device encoder: only the empty list (cv2's defaults) is accepted."""
    params = [int(p) for p in params]
    if params:
        raise ValueError("imencode params %r are not supported by the PNG device encoder (use cv2.imencode)" % (params,))
    return ()


def encode_bound(h, w):
    """pn_png_encode_bound: the largest file an h x w frame can encode to."""
    n = C.c_int64()
    nat.check(nat.load().pn_png_encode_bound(int(h), int(w), C.byref(n)), "pn_png_encode_bound")
    return n.value


class Encoder:
    """Device buffers for ``pn_png_encode`` at a fixed capacity: ``batch`` frames of at most ``max_h`` x ``max_w``.  ``params``
    must be empty (see ``encode_options``).  ``encode`` enqueues on the current stream; file i is then
    ``out[offsets[i]:offsets[i + 1]]``.  The same interface as ``posenet.jpeg.Encoder``."""

    def __init__(self, batch, max_h, max_w, params=(), device=None):
        encode_options(params)
        self.batch, self.max_h, self.max_w = int(batch), int(max_h), int(max_w)
        dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        n = C.c_size_t()
        nat.check(nat.load().pn_png_encode_workspace(self.batch, self.max_h, self.max_w, C.byref(n)), "pn_png_encode_workspace")
        self.ws = torch.empty(n.value, dtype=torch.uint8, device=dev)
        self.capacity = self.batch * encode_bound(self.max_h, self.max_w)
        self.out = torch.empty(self.capacity, dtype=torch.uint8, device=dev)
        self.offsets = torch.zeros(self.batch + 1, dtype=torch.int64, device=dev)

    def encode(self, frames, frame_stride, frame_hw=None):
        """Enqueue pn_png_encode of ``frames`` (frame i from byte ``i * frame_stride``; ``frame_hw``: CUDA int32 [batch, 2]
        per-frame sizes, or None for max_h x max_w everywhere) into ``self.out`` / ``self.offsets``."""
        nat.check(nat.load().pn_png_encode(
            C.c_void_p(frames.data_ptr()), self.batch, self.max_h, self.max_w, int(frame_stride),
            C.c_void_p(frame_hw.data_ptr()) if frame_hw is not None else None, C.c_void_p(self.out.data_ptr()), self.capacity,
            C.c_void_p(self.offsets.data_ptr()), C.c_void_p(self.ws.data_ptr()), self.ws.numel(), nat.stream_ptr()),
            "pn_png_encode")

    def files(self):
        """Synchronise and copy the files of the last ``encode`` back (the bytes in use only): a list of ``bytes``, one per
        frame."""
        off = self.offsets.cpu().numpy()
        data = self.out[:int(off[-1])].cpu().numpy()
        return [data[off[i]:off[i + 1]].tobytes() for i in range(self.batch)]


def imencode_png_batch(frames, params=(), shapes=None):
    """Encode every frame on the GPU; returns a list of ``bytes``, file i equal to ``cv2.imencode(".png", frame_i, params)[1]``.
    ``frames``: CUDA uint8 [N, h, w, 3] (BGR), or with ``shapes`` the rows [N, H * W * 3] and sizes ``imdecode_batch`` returns
    (frame i stored contiguously from the start of row i at its own size; a (0, 0) frame gives an empty file).  ``params`` must
    be empty: anything else raises ValueError."""
    encode_options(params)
    return encode_files(Encoder, frames, params, shapes)
