"""Host image ingest in front of ``BatchPipeline`` (SURVEY 8(f) N2): decode image files on a thread pool straight into pinned
uint8 batches, so that file decoding, the host->device copy and the kernels of consecutive batches overlap.

The pixels are exactly what the reference feeds its network: ``cv2.imread`` (BGR uint8 HWC, ``posenet/utils.py:34-38``
``read_imgfile``); resizing / normalisation happen on the GPU (``pn_resize_u8`` + the stem), bit-exact with ``_process_input``.

    stream = posenet.ImageStream(paths, batch=64)                 # files sharing one frame size (camera / video frames)
    pipe = posenet.BatchPipeline(model, 64, stream.height, stream.width, min_pose_score=0.25)
    for (scores, kp_scores, kp_coords, offsets), n_valid in zip(pipe.run(b for b, _ in stream.batches()), stream.valid_counts()):
        ...

A directory of images of DIFFERENT sizes (``benchmark.py:24-29`` pre-processes every file at its own size):

    stream = posenet.ImageStream(paths, batch=64, height=720, width=1280, mixed=True)      # height x width: the largest frame
    pipe = posenet.BatchPipeline(model, 64, 720, 1280, mixed=True, source_coords=True, min_pose_score=0.25)
    for records in pipe.run((b, shapes) for b, _, shapes in stream.batches()):
        ...                                                       # coordinates already in each file's own pixel grid

JPEG files decoded on the GPU instead (``posenet.jpeg``; the records are identical, the host only reads and parses files):

    stream = posenet.ImageStream(paths, batch=64, decode="gpu")
    pipe = posenet.BatchPipeline(model, 64, stream.height, stream.width, jpeg=True, min_pose_score=0.25)
    for *records, status in pipe.run(b for b, _ in stream.batches()):
        ...                                                       # status[i]: 0 GPU, 1 decoded by cv2 on the host, < 0 malformed

Camera photos decoded at 1/2, 1/4 or 1/8 (``cv2.imread(path, cv2.IMREAD_REDUCED_COLOR_4)``; JPEG files scaled in the DCT domain,
without a full-size frame anywhere):

    stream = posenet.ImageStream(paths, batch=64, decode="gpu", reduce=4)        # height x width: the REDUCED frame size
    pipe = posenet.BatchPipeline(model, 64, stream.height, stream.width, jpeg=True, reduce=4, arena_bytes=stream.arena_bytes)
    ...                                                           # coordinates refer to the reduced frames

Phone photos with an EXIF orientation (portraits are stored as landscape scans with orientation 6) rotated on the GPU too, as
cv2.imread rotates them; a directory of portraits and landscapes has both frame orientations, so it is a mixed stream:

    stream = posenet.ImageStream(paths, batch=64, height=1008, width=1008, mixed=True, decode="gpu", reduce=4, orientation="gpu")
    pipe = posenet.BatchPipeline(model, 64, 1008, 1008, jpeg=True, mixed=True, reduce=4, arena_bytes=stream.arena_bytes,
                                 source_coords=True)

Progressive files (web images, CDN output) decoded on the GPU too; the pipeline is the same:

    stream = posenet.ImageStream(paths, batch=64, decode="gpu", progressive="gpu")
"""
import concurrent.futures
import ctypes as C
import os
import threading

import cv2
import numpy as np
import torch

from posenet import _native as nat
from posenet.jpeg import align8, check_progressive, frame_size, imread_flag, parse_progressive, parser


class EncodedBatch:
    """One batch of files as ``ImageStream(decode="gpu")`` hands it to ``BatchPipeline(jpeg=True)``: the bytes of the files the GPU
    decodes packed into a pinned byte arena (``arena[:used]``), their descriptors (``descs``, pinned uint8, one pn_jpeg_desc per
    row; rows the GPU does not decode are marked host), and the frames cv2 decoded on the host (``raw`` rows ``host_rows``).
    ``reduce``: the scale the frames are decoded at (1 / reduce), the stream's."""

    def __init__(self, arena, descs, raw, batch, reduce=1):
        self.arena, self.descs, self.raw, self.batch, self.reduce = arena, descs, raw, batch, reduce
        self.used = 0
        self.host_rows = []
        self.shapes = [None] * batch
        self.n_valid = 0
        self.lock = threading.Lock()

    def reset(self, n_valid):
        self.used = 0
        self.host_rows = []
        self.shapes = [None] * self.batch
        self.n_valid = n_valid
        host = nat.JpegDesc()
        host.kind = nat.JPEG_HOST
        self.descs.numpy()[:] = np.frombuffer(bytes((nat.JpegDesc * self.batch)(*([host] * self.batch))), np.uint8)


class ImageStream:
    def __init__(self, paths, batch, height=None, width=None, workers=None, slots=4, keep=2, pinned=None, mixed=False, decode="cv2",
                 reduce=1, arena_bytes=None, orientation="cv2", progressive="cv2"):
        """``mixed``: the files may have different sizes (each at most ``height`` x ``width``); a batch row then holds its frame
        contiguously at the frame's own size and ``batches()`` also yields the list of ``(h, w)`` -- the input format of a
        ``BatchPipeline(..., mixed=True)``, which resizes every frame on the GPU like ``_process_input`` (utils.py:13-26) does.

        ``slots`` batch buffers rotate.  A buffer handed out by ``batches()`` stays valid while the consumer takes ``keep``
        further batches and is decoded into again when it asks for the one after that; the remaining ``slots - 1 - keep``
        batches decode ahead on the thread pool.  ``BatchPipeline.run`` (depth d) copies batch i to the device asynchronously
        and only blocks on it after taking batch i + d, so ``keep >= d`` is what makes the reuse safe (defaults: d = 2).

        ``decode="gpu"``: the workers only read each file into the batch's pinned byte arena (``arena_bytes``, below) and parse
        its headers; ``batches()`` yields an ``EncodedBatch`` in place of the
        uint8 tensor, for a ``BatchPipeline(..., jpeg=True)`` to decode on the GPU.  Files the GPU does not decode (not baseline
        JPEG, EXIF-rotated unless ``orientation="gpu"``, ...; ``posenet.jpeg``) or that do not fit the arena's remaining space
        are decoded by cv2.imread into their row of a pinned side buffer.  Size checks and errors are those of ``decode="cv2"``.
        ``orientation="gpu"`` (with ``decode="gpu"`` only): files whose EXIF orientation is certain are decoded on the GPU and
        rotated there as cv2.imread rotates them (``pn_jpeg_parse_oriented``); shapes and size checks use the rotated size, so
        portraits and landscapes need ``mixed=True`` as with ``decode="cv2"``.
        ``progressive="gpu"`` (with ``decode="gpu"`` only): progressive files the GPU decodes (``pn_jpeg_parse_progressive``) go
        to the arena too, each file 8-byte aligned and followed by its scan table.  A worker reads and parses a file in buffers
        of its own and then takes exactly the space the file and its table need; a file and its table that do not fit the
        arena's remaining space are decoded by cv2.

        ``reduce`` (1, 2, 4 or 8): every file is decoded at 1 / reduce, as ``cv2.imread(path, cv2.IMREAD_REDUCED_COLOR_<reduce>)``
        does (JPEG files: ceil(h / reduce) x ceil(w / reduce), scaled in the DCT domain).  ``height`` / ``width`` are then the
        REDUCED frame size (taken from the first file read with that flag when not given), and size checks apply to it; pose
        coordinates downstream refer to the reduced frames.  With ``decode="gpu"`` the decode runs at that scale on the device.
        ``arena_bytes``: the pinned byte arena per batch of ``decode="gpu"`` (``self.arena_bytes``; a ``BatchPipeline`` needs a
        decoder arena at least as large).  Default: ``batch * height * width * 3`` at ``reduce=1``; otherwise ``batch *
        (reduce * height) * (reduce * width)``, room for full-size camera files of about a byte per pixel."""
        self.flag = imread_flag(reduce)
        self.reduce = int(reduce)
        self.paths = list(paths)
        assert self.paths, "no image files"
        self.batch = int(batch)
        assert not (mixed and (height is None or width is None)), "mixed=True needs the largest frame size (height, width)"
        if height is None or width is None:
            first = cv2.imread(self.paths[0], self.flag)
            if first is None:
                raise IOError("Image file not found or unreadable: %s" % self.paths[0])     # utils.py:36-37
            height, width = first.shape[:2]
        self.height, self.width = int(height), int(width)
        self.workers = workers or min(32, os.cpu_count() or 1)
        pinned = torch.cuda.is_available() if pinned is None else pinned
        self.mixed = bool(mixed)
        self.keep = int(keep)
        assert int(slots) >= self.keep + 2, "slots must be at least keep + 2 (one buffer in use, one decoding ahead)"
        self._bufs = []
        for _ in range(int(slots)):
            t = torch.zeros((self.batch, self.height, self.width, 3), dtype=torch.uint8)
            self._bufs.append(t.pin_memory() if pinned else t)
        self._views = [b.numpy() for b in self._bufs]
        self._shapes = [[None] * self.batch for _ in self._bufs]
        assert decode in ("cv2", "gpu"), "decode is 'cv2' or 'gpu'"
        self.decode = decode
        parser(orientation)
        if orientation == "gpu" and decode != "gpu":
            raise ValueError("orientation='gpu' rotates files in the GPU decode: it needs decode='gpu'")
        self.orientation = orientation
        check_progressive(progressive)
        if progressive == "gpu" and decode != "gpu":
            raise ValueError("progressive='gpu' decodes progressive files on the GPU: it needs decode='gpu'")
        self.progressive = progressive
        self._scratch = threading.local()        # progressive="gpu": each worker's file and scan-table buffers
        if arena_bytes is None:
            r = self.reduce
            arena_bytes = self._bufs[0].numel() if r == 1 else self.batch * (r * self.height) * (r * self.width)
        self.arena_bytes = int(arena_bytes)
        assert self.arena_bytes > 0, "arena_bytes must be positive"
        self._enc = []
        if decode == "gpu":
            for b in self._bufs:
                arena = torch.empty(self.arena_bytes, dtype=torch.uint8)
                descs = torch.empty(self.batch * C.sizeof(nat.JpegDesc), dtype=torch.uint8)
                self._enc.append(EncodedBatch(arena.pin_memory() if pinned else arena, descs.pin_memory() if pinned else descs, b,
                                              self.batch, self.reduce))

    def __len__(self):
        return (len(self.paths) + self.batch - 1) // self.batch

    def valid_counts(self):
        """Number of real images in every batch (the last one may be partial; its tail rows are zero images)."""
        n = len(self.paths)
        return [min(self.batch, n - i) for i in range(0, n, self.batch)]

    def _check_size(self, path, h, w):
        if self.mixed:
            if h > self.height or w > self.width:
                raise ValueError("%s is %dx%d, larger than the stream's %dx%d frames" % (path, w, h, self.width, self.height))
        elif (h, w) != (self.height, self.width):
            raise ValueError("%s is %dx%d, the stream carries %dx%d frames (mixed=True accepts different sizes)" % (
                path, w, h, self.width, self.height))

    def _load_encoded(self, path, enc, row):
        """Read one file into the arena and parse it; cv2 decodes it into its raw row when the GPU cannot."""
        if self.progressive == "gpu":
            return self._load_progressive(path, enc, row)
        try:
            with open(path, "rb") as f:
                size = os.fstat(f.fileno()).st_size
                with enc.lock:
                    off = enc.used
                    fits = off + size <= enc.arena.numel()
                    if fits:
                        enc.used += size
                view = enc.arena.numpy()[off:off + size] if fits else None
                n = f.readinto(memoryview(view)) if fits else -1
        except OSError:
            raise IOError("Image file not found or unreadable: %s" % path)
        if fits and n == size:
            d = nat.JpegDesc()
            nat.check(parser(self.orientation)(view.ctypes.data, size, C.byref(d)), "pn_jpeg_parse")
            if d.kind == nat.JPEG_SUPPORTED:
                self._place(path, enc, row, d, off)
                return
        self._load_host(path, enc, row)

    def _load_progressive(self, path, enc, row):
        """progressive="gpu": read and parse one file in this worker's scratch buffers, then take exactly the arena space it
        needs (8-byte aligned: the file, then its scan table at file_offset + align8(size)) and copy it there."""
        sc = self._scratch
        if not hasattr(sc, "table"):
            sc.table = np.zeros(nat.JPEG_SCAN_TABLE_MAX, np.uint8)
            sc.buf = np.zeros(0, np.uint8)
        try:
            with open(path, "rb") as f:
                size = os.fstat(f.fileno()).st_size
                if sc.buf.size < size:
                    sc.buf = np.zeros(max(size, 2 * sc.buf.size), np.uint8)
                view = sc.buf[:size]
                n = f.readinto(memoryview(view))
        except OSError:
            raise IOError("Image file not found or unreadable: %s" % path)
        if n == size:
            d, tb = parse_progressive(view, self.orientation, sc.table)
            if d.kind in (nat.JPEG_SUPPORTED, nat.JPEG_SUPPORTED_PROGRESSIVE):
                need = align8(size) + tb if d.kind == nat.JPEG_SUPPORTED_PROGRESSIVE else size
                with enc.lock:
                    off = align8(enc.used)
                    fits = off + need <= enc.arena.numel()
                    if fits:
                        enc.used = off + need
                if fits:
                    arena = enc.arena.numpy()
                    arena[off:off + size] = view
                    if d.kind == nat.JPEG_SUPPORTED_PROGRESSIVE:
                        arena[off + align8(size):off + need] = sc.table[:tb]
                    self._place(path, enc, row, d, off)
                    return
        self._load_host(path, enc, row)

    def _place(self, path, enc, row, d, off):
        """Record the descriptor of a file the GPU decodes, stored at arena offset ``off``."""
        h, w = frame_size(d, self.reduce)
        self._check_size(path, h, w)
        d.file_offset = off
        k = C.sizeof(nat.JpegDesc)
        enc.descs.numpy()[row * k:(row + 1) * k] = np.frombuffer(bytes(d), np.uint8)
        enc.shapes[row] = (h, w)

    def _load_host(self, path, enc, row):
        self._load(path, enc.raw.numpy()[row], enc.shapes, row)
        with enc.lock:
            enc.host_rows.append(row)

    def _load(self, path, dst, shapes, row):
        img = cv2.imread(path, self.flag)
        if img is None:
            raise IOError("Image file not found or unreadable: %s" % path)
        if self.mixed:
            if img.shape[0] > self.height or img.shape[1] > self.width:
                raise ValueError("%s is %dx%d, larger than the stream's %dx%d frames" % (path, img.shape[1], img.shape[0], self.width, self.height))
            dst.reshape(-1)[:img.size] = img.reshape(-1)             # the frame at its own size, contiguous at the start of the row
            shapes[row] = (img.shape[0], img.shape[1])
            return
        if img.shape != dst.shape:
            raise ValueError("%s is %dx%d, the stream carries %dx%d frames (mixed=True accepts different sizes)" % (
                path, img.shape[1], img.shape[0], self.width, self.height))
        dst[...] = img

    def batches(self):
        """Yields ``(uint8 tensor [batch, h, w, 3] (pinned when CUDA is available), n_valid)`` -- ``(tensor, n_valid, shapes)``
        for a mixed stream; decoding of the next ``slots - 1 - keep`` batches runs ahead on the thread pool."""
        n = len(self.paths)
        starts = list(range(0, n, self.batch))
        with concurrent.futures.ThreadPoolExecutor(max_workers=self.workers) as ex:
            def launch(bi):
                buf, shapes = self._views[bi % len(self._views)], self._shapes[bi % len(self._views)]
                lo = starts[bi]
                hi = min(n, lo + self.batch)
                if self.decode == "gpu":
                    enc = self._enc[bi % len(self._enc)]
                    enc.reset(hi - lo)
                    return [ex.submit(self._load_encoded, self.paths[i], enc, i - lo) for i in range(lo, hi)]
                if hi - lo < self.batch:
                    buf[hi - lo:] = 0
                return [ex.submit(self._load, self.paths[i], buf[i - lo], shapes, i - lo) for i in range(lo, hi)]
            ahead = len(self._bufs) - 1 - self.keep
            pending = {bi: launch(bi) for bi in range(min(ahead, len(starts)))}
            for bi in range(len(starts)):
                for f in pending.pop(bi):
                    f.result()                                   # re-raises decode errors
                nxt = bi + ahead
                # batch `nxt` decodes into the buffer handed out `keep + 1` batches ago: the consumer asking for batch `bi` is what
                # releases it, so its decode starts BEFORE the yield and overlaps the consumer's work on batch `bi`
                if nxt < len(starts):
                    pending[nxt] = launch(nxt)
                nv = min(self.batch, n - starts[bi])
                if self.decode == "gpu":
                    enc = self._enc[bi % len(self._enc)]
                    enc.host_rows.sort()
                    yield (enc, nv, list(enc.shapes[:nv])) if self.mixed else (enc, nv)
                elif self.mixed:
                    yield self._bufs[bi % len(self._bufs)], nv, list(self._shapes[bi % len(self._bufs)][:nv])
                else:
                    yield self._bufs[bi % len(self._bufs)], nv
