"""Streaming front end of the hot path: host uint8 batches in, host pose records out, with the
host->device copy of batch i+1 and the device->host copy of batch i-1 overlapping the kernels of
batch i (two copy engines + one compute stream, one CUDA graph per in-flight slot).

This is the batched form of what the reference's ``benchmark.py:32-44`` does per image
(``model(input)`` then ``decode_multiple_poses``): same results, no per-image synchronisation.

    pipe = posenet.BatchPipeline(model, batch=64, height=513, width=513, min_pose_score=0.25)
    for pose_scores, keypoint_scores, keypoint_coords, pose_offsets in pipe.run(batches):   # pinned uint8 [64,513,513,3]
        ...

Options on top of that (``overlay=`` draws the poses on the frames, ``encode=`` returns them as JPEG files, or as PNG files
with ``encode_ext=".png"``, ``jpeg=True`` takes JPEG files in, ``yuv=code`` video frames in YUV, ``yuv_out=code`` returns the drawn frames in YUV, ``track=PoseTracker(...)`` gives the poses of video streams track ids): ``source_coords=True`` maps the keypoint coordinates back to the submitted frames ON THE DEVICE
(``image_demo.py:50``), ``mixed=True`` accepts frames of different sizes in one batch (every file of a directory
pre-processed at its own size, ``benchmark.py:24-29``), ``gather=True`` all-gathers the records of every rank's shard over
NCCL inside the step (one process per GPU, ``posenet.sharding``).
"""
import ctypes as C

import numpy as np
import torch

from posenet import _native as nat
from posenet.constants import NUM_KEYPOINTS
from posenet.decode_multi import decode_multiple_poses_batch, split_pose_records


class BatchPipeline:
    def __init__(self, model, batch, height, width, depth=2, use_graph=True, output_stride=None, scale_factor=1.0,
                 source_coords=False, mixed=False, gather=False, group=None, overlay=None, jpeg=False, encode=None, encode_ext=".jpg",
                 reduce=1, arena_bytes=None, yuv=None, yuv_out=None, track=None, **decode_kw):
        """``height`` x ``width``: size of the uint8 frames handed to ``submit`` (``mixed=True``: the LARGEST frame; each
        frame of a batch then comes with its own size).  The network runs at ``valid_resolution(width * scale_factor,
        height * scale_factor)`` (utils.py:7-10); frames of any other size go through the bit-exact cv2 resize
        (``pn_resize_u8``) on the GPU in front of the stem -- inside the step's CUDA graph when all frames share one size.

        ``source_coords``: ``keypoint_coords *= (src_h / target_h, src_w / target_w)`` (image_demo.py:50, utils.py:19) applied to
        the record buffer on the device (``pn_scale_keypoint_coords``), per frame in mixed mode.
        ``gather``: with an initialised process group, every step ends with an all-gather of the ranks' record buffers (NCCL over
        NVLink) on its own stream -- the kernels of the next batch do not wait for it -- and rank 0 reads ALL ranks' records back
        (``result(..., gathered=True)``); the other ranks read back their own, as without ``gather``.
        ``overlay=(min_pose_score, min_part_score)``: the step also draws ``draw_skel_and_kp`` (image_demo.py:53) on the submitted
        frames at their own size, on the device (``pn_draw_poses``, bit-exact with cv2), and copies them back after the records;
        ``result`` then returns the frames as a fifth item.  Frames that are resized need ``source_coords=True`` (the overlay is
        drawn in their coordinates).  With ``gather``, the frames stay on their rank.
        ``jpeg``: ``submit`` takes the ``EncodedBatch`` of an ``ImageStream(..., decode="gpu")``.  The host-to-device copy carries
        the bytes of the files in use, their descriptors and the rows cv2 decoded on the host; ``pn_jpeg_decode`` writes the
        frames into the step's input buffer (same layout as the uint8 batches) on the compute stream, just before the step.
        ``result`` appends the int32 decode status ``[batch]`` as its last item (0 GPU, 1 host, < 0 malformed: a zero frame).
        ``reduce`` (with ``jpeg``; 1, 2, 4 or 8): the stream's ``reduce``.  The files are decoded at 1 / reduce
        (``pn_jpeg_decode_scaled``, bit-exact with ``cv2.imread(path, cv2.IMREAD_REDUCED_COLOR_<reduce>)``) and ``height`` x
        ``width`` are the reduced frame size.  Everything downstream -- resize, records, ``source_coords``, overlay, encode --
        works on the reduced frames: coordinates refer to them, not to the full-size files.  ``arena_bytes``: the decoder's
        byte arena, at least the stream's ``arena_bytes`` (default: what ``ImageStream`` allocates for the same batch, size and
        ``reduce``).  ``submit`` checks both against the ``EncodedBatch``.
        ``yuv``: a ``cv2.COLOR_YUV2BGR_*`` code of a 4:2:0 or 4:2:2 layout (I420 / IYUV, YV12, NV12, NV21, YUY2 / YUYV / YUNV,
        UYVY / Y422 / UYNV, YVYU).  ``submit`` then takes uint8 batches of video frames in cv2's input layout of that code
        (``[batch, h*3/2, w]`` or ``[batch, h, w, 2]``; ``height`` x ``width`` stay the BGR frame size, both even).  The host-to-device
        copy carries only those 1.5 or 2 bytes a pixel, and the step's first launch converts them into the BGR frames
        (``pn_yuv_to_bgr``, bit-exact with ``cv2.cvtColor(frame, yuv)``).  Everything downstream -- resize, records,
        ``source_coords``, overlay, encode, gather -- works on the converted frames.  Not with ``jpeg`` or ``mixed``.
        ``encode``: a cv2 ``imencode`` params list (``[]`` for cv2's defaults; needs ``overlay``).  The step's graph also encodes
        the drawn frames as JPEG files (``pn_jpeg_encode``, bit-exact with ``cv2.imencode(".jpg", frame, encode)``), and the
        in-graph device-to-host copy carries the files' offsets instead of the frames.  ``result`` copies exactly the bytes in use
        on a stream of its own (the offsets are only known on the host then) and returns a list of ``bytes`` as the fifth item
        instead of the frames: one per submitted frame in mixed mode, ``batch`` otherwise.  Params the device encoder does not
        do raise ValueError here.
        ``encode_ext``: ``".jpg"`` (the default) or ``".png"``: the files are then PNG (``pn_png_encode``, bit-exact with
        ``cv2.imencode(".png", frame)``; ``encode`` must be ``[]``).
        ``yuv_out``: a ``cv2.COLOR_BGR2YUV_*`` code of a layout cv2 writes (I420 / IYUV, YV12, YUY2 / YUYV / YUNV, UYVY / Y422 /
        UYNV, YVYU; needs ``overlay``), for handing the drawn frames to a video sink.  The step's graph converts the drawn frames
        right after drawing them (``pn_bgr_to_yuv``, bit-exact with ``cv2.cvtColor(frame, yuv_out)``), and the in-graph
        device-to-host copy carries only those 1.5 or 2 bytes a pixel.  ``result`` returns them as the fifth item instead of the
        BGR frames: uint8 ``[batch, h*3/2, w]`` (4:2:0) or ``[batch, h, w, 2]`` (4:2:2), cv2's layout.  ``height`` x ``width`` must
        be sizes cv2 converts (even width; even height for 4:2:0).  Works with ``yuv``, ``jpeg``, ``reduce``, ``source_coords`` and
        ``gather`` (the frames stay on their rank); not with ``encode`` (one output form per pipeline) or ``mixed`` (frames of
        their own, possibly odd, sizes).  ValueError otherwise.
        ``track``: a ``posenet.PoseTracker`` on the pipeline's device.  ``submit`` then takes ``streams=``, one stream id per
        row (-1: not tracked), which travel in the host-to-device copy with the batch; the step's graph runs ``pn_track_poses``
        on the records after the decode and after ``source_coords`` scaling (boxes in frame pixels then), before the overlay,
        and the device-to-host stream copies the ids back after the records.  ``result`` appends them as the last item, int64
        ``[batch, P]`` (after the decode status with ``jpeg``).  The tracker's ``min_part_score=None`` takes the decode's
        ``score_threshold``.  Works with every option but ``gather`` (each rank would hold its own tracks): ValueError.
        A tracker with ``smoothing=OneEuro(...)`` also runs ``pn_smooth_keypoints`` in the step's graph, right after the
        tracking: the keypoint coordinates of tracked rows are smoothed in place, so the returned records, the overlay, the
        ``encode`` files and the ``yuv_out`` frames carry the smoothed coordinates; ids, byte counts and ``result``'s items
        are as without it."""
        self.track = track
        if track is not None:
            from posenet.track import PoseTracker
            if not isinstance(track, PoseTracker):
                raise ValueError("track= takes a posenet.PoseTracker")
            if gather:
                raise ValueError("track= keeps the tracks on this rank: not with gather=True")
        self.yuv = None
        if yuv is not None:
            from posenet import yuv as yuv_mod
            self.yuv = yuv_mod.layout_of(yuv)
            if jpeg or mixed:
                raise ValueError("yuv= takes video frames of one size: not with jpeg=True or mixed=True")
            self.yuv_bytes = int(np.prod(yuv_mod.frame_shape(self.yuv, int(height), int(width))))
        self.yuv_out = None
        if yuv_out is not None:
            from posenet import yuv as yuv_mod
            self.yuv_out = yuv_mod.layout_of_output(yuv_out)
            if overlay is None:
                raise ValueError("yuv_out= converts the drawn frames: it needs overlay=")
            if encode is not None or mixed:
                raise ValueError("yuv_out= returns frames of one size as YUV: not with encode= or mixed=True")
            self.yuv_out_shape = yuv_mod.frame_shape(self.yuv_out, int(height), int(width))
        nat.require_device()
        assert depth >= 1
        self.model, self.batch, self.h, self.w = model, int(batch), int(height), int(width)
        from posenet.utils import valid_resolution
        self.os = output_stride or model.output_stride
        self.tw, self.th = valid_resolution(self.w * scale_factor, self.h * scale_factor, output_stride=self.os)
        self.mixed = bool(mixed)
        self.resize = self.mixed or (self.th, self.tw) != (self.h, self.w)
        self.scale = np.array([self.h / self.th, self.w / self.tw])           # utils.py:19, for mapping coordinates back
        self.source_coords = bool(source_coords)
        self.overlay = None if overlay is None else (float(overlay[0]), float(overlay[1]))
        assert self.overlay is None or self.source_coords or not self.resize, \
            "overlay on resized frames needs source_coords=True (the records must be in the frames' coordinates)"
        assert encode is None or self.overlay is not None, "encode= encodes the drawn frames: it needs overlay="
        self.encode = None if encode is None else list(encode)
        if encode_ext not in (".jpg", ".png"):
            raise ValueError("encode_ext %r: the device encoders write .jpg and .png" % (encode_ext,))
        self.encode_ext = encode_ext
        assert encode_ext == ".jpg" or self.encode is not None, "encode_ext= names the format of encode=: it needs encode="
        if self.encode is not None:
            from posenet import jpeg as jpeg_codec, png as png_codec
            codec = png_codec if encode_ext == ".png" else jpeg_codec
            codec.encode_options(self.encode)
            self.encoder = codec.Encoder
        self.decode_kw = dict(decode_kw)
        self.P = int(self.decode_kw.get("max_pose_detections", 10))
        dev = model._device()
        self.dev = dev
        if track is not None:
            if track.device != torch.device(dev):
                raise ValueError("the tracker's state is on %s, the pipeline runs on %s" % (track.device, dev))
            self.track_part_score = track.min_part_score if track.min_part_score is not None else \
                float(self.decode_kw.get("score_threshold", 0.5))
        self.world, self.rank, self.group = 1, 0, group
        if gather:
            import torch.distributed as dist
            assert dist.is_available() and dist.is_initialized(), "gather=True needs an initialised process group"
            self.world, self.rank = dist.get_world_size(group), dist.get_rank(group)
        self.gather = bool(gather) and self.world > 1
        with torch.cuda.device(dev):
            self.h2d, self.d2h, self.compute = torch.cuda.Stream(dev), torch.cuda.Stream(dev), torch.cuda.Stream(dev)
            self.collect_all = self.gather and self.rank == 0      # this rank's D2H copy carries every rank's records
            self.nrec = self.batch * self.P * (1 + 5 * NUM_KEYPOINTS)
            self.frame_shape = (self.h, self.w, 3) if self.yuv_out is None else self.yuv_out_shape     # of a returned frame
            nrec = self.nrec
            self.slots = []
            self._ws = {}
            for _ in range(depth):
                s = dict(x=torch.empty((self.batch, self.h, self.w, 3), dtype=torch.uint8, device=dev),
                         xr=torch.empty((self.batch, self.th, self.tw, 3), dtype=torch.uint8, device=dev) if self.resize else None,
                         rec=torch.zeros(nrec, dtype=torch.float64, device=dev),
                         rec_all=torch.zeros(self.world * nrec, dtype=torch.float64, device=dev) if self.gather else None,
                         rec_host=torch.zeros((self.world if self.collect_all else 1) * nrec, dtype=torch.float64).pin_memory(),
                         scales=torch.ones((self.batch, 2), dtype=torch.float64, device=dev) if self.mixed else None,
                         scales_host=torch.ones((self.batch, 2), dtype=torch.float64).pin_memory() if self.mixed else None,
                         frames_host=torch.empty((self.batch,) + self.frame_shape, dtype=torch.uint8).pin_memory()
                         if self.overlay and self.encode is None else None,
                         yuv_out=torch.empty((self.batch,) + self.yuv_out_shape, dtype=torch.uint8, device=dev)
                         if self.yuv_out is not None else None,
                         hw=torch.zeros((self.batch, 2), dtype=torch.int32, device=dev) if self.overlay and self.mixed else None,
                         hw_host=torch.zeros((self.batch, 2), dtype=torch.int32).pin_memory() if self.overlay and self.mixed else None,
                         yuv=torch.empty(self.batch * self.yuv_bytes, dtype=torch.uint8, device=dev) if self.yuv is not None else None,
                         shapes=None,
                         streams=torch.full((self.batch,), -1, dtype=torch.int32, device=dev) if track is not None else None,
                         streams_host=torch.full((self.batch,), -1, dtype=torch.int32).pin_memory() if track is not None else None,
                         ids=torch.empty((self.batch, self.P), dtype=torch.int64, device=dev) if track is not None else None,
                         ids_host=torch.empty((self.batch, self.P), dtype=torch.int64).pin_memory() if track is not None else None,
                         copied=torch.cuda.Event(), done=torch.cuda.Event(), out=torch.cuda.Event(), graph=None, busy=False)
                self.slots.append(s)
            self.jpeg = bool(jpeg)
            assert self.jpeg or (reduce == 1 and arena_bytes is None), "reduce= and arena_bytes= are for jpeg=True pipelines"
            if self.jpeg:
                from posenet.jpeg import Decoder, imread_flag
                imread_flag(reduce)
                self.reduce = int(reduce)
                r = self.reduce
                if arena_bytes is None:
                    arena_bytes = self.slots[0]["x"].numel() if r == 1 else self.batch * (r * self.h) * (r * self.w)
                for s in self.slots:
                    s["dec"] = Decoder(self.batch, int(arena_bytes), self.h, self.w, dev, r)
                    s["status_host"] = torch.zeros(self.batch, dtype=torch.int32).pin_memory()
                    s["h2d_bytes"] = 0
            if self.encode is not None:
                # the share of the frames' raw size the files take, for the estimates below: drawn frames at q95 4:2:0 are
                # 8-12 % as JPEG, smooth ones about 58 % as PNG (photographs more)
                self.file_share = 0.6 if encode_ext == ".png" else 0.1
                self.files_stream = torch.cuda.Stream(dev)             # result()'s copy of the packed files
                for s in self.slots:
                    s["enc"] = self.encoder(self.batch, self.h, self.w, self.encode, dev)
                    s["offsets_host"] = torch.zeros(self.batch + 1, dtype=torch.int64).pin_memory()
                    s["files_host"] = torch.empty(int(self.batch * self.h * self.w * 3 * min(2.5 * self.file_share, 1)),
                                                  dtype=torch.uint8).pin_memory()
            self.h2d_bytes_per_batch = self.slots[0]["x"].numel() if self.yuv is None else self.slots[0]["yuv"].numel()
            self.d2h_bytes_per_batch = (self.world if self.collect_all else 1) * nrec * 8
            if self.overlay and self.encode is None:
                self.d2h_bytes_per_batch += self.slots[0]["frames_host"].numel()   # mixed mode copies only the bytes in use
            elif self.encode is not None:
                # the offsets, plus the files: an estimate (file_share of the frames' raw size); result() copies exactly the
                # bytes in use and records them in last_file_bytes
                self.d2h_bytes_per_batch += 8 * (self.batch + 1) + int(self.slots[0]["x"].numel() * self.file_share)
            if track is not None:
                self.h2d_bytes_per_batch += self.slots[0]["streams"].numel() * 4
                self.d2h_bytes_per_batch += self.slots[0]["ids"].numel() * 8
                track.stream = self.compute                          # reset() is ordered with the steps
            self.last_file_bytes = 0
            # warm up (plans, workspaces) and capture one graph per slot on the compute stream
            self.compute.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(self.compute):
                for s in self.slots:
                    s["x"].zero_()
                    if self.yuv is not None:
                        s["yuv"].zero_()
                    if self.mixed:
                        s["xr"].zero_()
                    self._enqueue(s)
                self.compute.synchronize()
                if use_graph:
                    for s in self.slots:
                        g = torch.cuda.CUDAGraph()
                        with torch.cuda.graph(g, stream=self.compute):
                            self._enqueue(s)
                        s["graph"] = g
            self.compute.synchronize()
        self._next = 0

    def _enqueue(self, s):
        """The captured part of a step: (YUV -> BGR ->) (uniform resize ->) stem .. heads -> candidates -> greedy decode
        (-> coordinate scaling) (-> tracking (-> smoothing)) (-> overlay on the submitted frames (-> JPEG / PNG files | -> BGR -> YUV)))."""
        x = s["x"]
        lib = nat.load()
        if self.yuv is not None:
            from posenet.yuv import convert
            convert(s["yuv"], self.batch, self.h, self.w, self.yuv, x)
        if self.resize and not self.mixed:
            nat.check(lib.pn_resize_u8(x.data_ptr(), self.batch, self.h, self.w, self.th, self.tw, s["xr"].data_ptr(),
                                       nat.stream_ptr()), "pn_resize_u8")
        if self.resize:
            x = s["xr"]                                              # mixed: filled per frame by submit(), outside the graph
        heads = self.model.forward_u8(x)
        ps, ks, kc, ko, _ = decode_multiple_poses_batch(*heads, output_stride=self.os, workspace=self._ws, out=s["rec"], **self.decode_kw)
        if self.source_coords and (self.mixed or self.resize):
            nat.check(lib.pn_scale_keypoint_coords(C.c_void_p(kc.data_ptr()), self.batch, self.P * NUM_KEYPOINTS,
                                                   C.c_void_p(s["scales"].data_ptr()) if self.mixed else None,
                                                   float(self.scale[0]), float(self.scale[1]), nat.stream_ptr()),
                      "pn_scale_keypoint_coords")
        if self.track is not None:                                   # the warm-up's stream ids are all -1: the state stays
            self.track.launch(ps, ks, kc, s["streams"], s["ids"], self.track_part_score)
            if self.track.smoothing is not None:                     # the boxes and ids come from the raw coordinates
                self.track.launch_smooth(s["ids"], kc, s["streams"])
        if self.overlay:
            x = s["x"]
            nat.check(lib.pn_draw_poses(C.c_void_p(x.data_ptr()), self.batch, self.h, self.w, self.h * self.w * 3,
                                        C.c_void_p(s["hw"].data_ptr()) if self.mixed else None, C.c_void_p(ps.data_ptr()),
                                        C.c_void_p(ks.data_ptr()), C.c_void_p(kc.data_ptr()), self.P, self.overlay[0],
                                        self.overlay[1], nat.DRAW_KEYPOINTS | nat.DRAW_SKELETON, nat.stream_ptr()),
                      "pn_draw_poses")
            if self.encode is not None:
                s["enc"].encode(x, self.h * self.w * 3, s["hw"] if self.mixed else None)
            if self.yuv_out is not None:
                from posenet.yuv import convert_out
                convert_out(x, self.batch, self.h, self.w, self.yuv_out, s["yuv_out"])

    def _resize_mixed(self, s, shapes):
        """Per-frame cv2-exact resize of frames stored at their own size (row i of the slot's input buffer holds frame i
        contiguously: h_i * w_i * 3 bytes) into the network-sized batch; runs of equal-sized frames share a launch when
        they are also full-sized (then the rows are dense)."""
        lib, st = nat.load(), nat.stream_ptr()
        row = self.h * self.w * 3
        base_in, base_out = s["x"].data_ptr(), s["xr"].data_ptr()
        out_row = self.th * self.tw * 3
        i = 0
        while i < len(shapes):
            h, w = shapes[i]
            n = 1
            if (h, w) == (self.h, self.w):                           # dense rows: take the whole run at once
                while i + n < len(shapes) and tuple(shapes[i + n]) == (h, w):
                    n += 1
            nat.check(lib.pn_resize_u8(base_in + i * row, n, h, w, self.th, self.tw, base_out + i * out_row, st), "pn_resize_u8")
            i += n

    def _copy_encoded(self, s, enc, shapes):
        """H2D part of a jpeg=True step (on the h2d stream): file bytes in use, descriptors, host-decoded rows."""
        dec, x = s["dec"], s["x"].view(self.batch, -1)
        n = 0
        if enc.used:
            dec.arena[:enc.used].copy_(enc.arena[:enc.used], non_blocking=True)
            n += enc.used
        dec.descs.copy_(enc.descs, non_blocking=True)
        n += enc.descs.numel()
        raw = enc.raw.view(self.batch, -1)
        for i in enc.host_rows:
            used = shapes[i][0] * shapes[i][1] * 3 if self.mixed else x.shape[1]
            x[i, :used].copy_(raw[i, :used], non_blocking=True)
            n += used
        if not self.mixed and enc.n_valid < self.batch:
            x[enc.n_valid:].zero_()                                    # rows without a file decode as black frames
        s["h2d_bytes"] = n

    def submit(self, host_batch, shapes=None, streams=None):
        """Enqueue one batch (uint8 [batch,h,w,3], ideally pinned; with ``yuv``, the frames in cv2's YUV layout).  Returns a
        ticket for ``result``; if the slot is still in flight its previous result must have been collected.

        ``mixed=True``: ``host_batch`` is uint8 ``[batch, h*w*3]`` (or ``[batch,h,w,3]``) whose row i starts with frame i
        stored contiguously at its own size ``shapes[i] = (h_i, w_i)`` (``h_i <= h``, ``w_i <= w``); rows without a frame
        (``len(shapes) < batch``) decode as black frames.

        ``streams`` (``track=`` pipelines, required there): the stream id of every row, ``batch`` integers in
        -1..n_streams-1; ValueError otherwise."""
        s = self.slots[self._next]
        assert not s["busy"], "pipeline full: collect result() of the oldest ticket first"
        if self.track is None:
            if streams is not None:
                raise ValueError("streams= are for track= pipelines")
        else:
            if streams is None:
                raise ValueError("track=: pass streams=, the stream id of every row (-1: not tracked)")
            s["streams_host"].numpy()[:] = self.track.stream_ids(streams, self.batch)
        enc = None
        if self.jpeg:
            from posenet.ingest import EncodedBatch
            assert isinstance(host_batch, EncodedBatch), "jpeg=True: submit the EncodedBatch of an ImageStream(decode='gpu')"
            assert host_batch.batch == self.batch
            assert host_batch.reduce == self.reduce, \
                "the stream decodes at 1/%d, the pipeline at 1/%d (reduce=)" % (host_batch.reduce, self.reduce)
            assert host_batch.arena.numel() <= s["dec"].arena_bytes, \
                "the stream's arena (%d bytes) exceeds the decoder's (%d): pass arena_bytes=stream.arena_bytes" % (
                    host_batch.arena.numel(), s["dec"].arena_bytes)
            enc = host_batch
            if self.mixed and shapes is None:
                shapes = list(enc.shapes[:enc.n_valid])
        else:
            assert host_batch.numel() == (s["x"] if self.yuv is None else s["yuv"]).numel() and host_batch.dtype == torch.uint8
        if self.mixed:
            assert shapes is not None and len(shapes) <= self.batch, "mixed=True: pass the (h, w) of every frame"
            shapes = [(int(h), int(w)) for h, w in shapes]
            assert all(0 < h <= self.h and 0 < w <= self.w for h, w in shapes), "a frame exceeds the pipeline's %dx%d" % (self.h, self.w)
            sc = s["scales_host"]
            sc.fill_(1.0)
            for i, (h, w) in enumerate(shapes):
                sc[i, 0], sc[i, 1] = h / self.th, w / self.tw                     # utils.py:19, per frame
            if self.overlay:
                hw = s["hw_host"]
                hw.zero_()                                                        # rows without a frame are not drawn
                if shapes:
                    hw[:len(shapes)] = torch.tensor(shapes, dtype=torch.int32)
        else:
            assert shapes is None, "shapes are for mixed=True pipelines"
        s["shapes"] = shapes
        with torch.cuda.device(self.dev):
            with torch.cuda.stream(self.h2d):
                self.h2d.wait_event(s["done"])              # the previous use of this slot's input buffer has finished
                if self.overlay or self.jpeg:
                    self.h2d.wait_event(s["out"])           # ... and its drawn frames / decode status have been copied back
                if enc is not None:
                    self._copy_encoded(s, enc, shapes)
                    if self.mixed:
                        s["scales"].copy_(sc, non_blocking=True)
                elif self.mixed and shapes:
                    used = max(h * w * 3 for h, w in shapes)                      # one strided copy of the bytes in use
                    s["x"].view(self.batch, -1)[:len(shapes), :used].copy_(host_batch.view(self.batch, -1)[:len(shapes), :used],
                                                                          non_blocking=True)
                    s["scales"].copy_(sc, non_blocking=True)
                elif self.yuv is not None:
                    s["yuv"].copy_(host_batch.view(-1), non_blocking=True)
                elif not self.mixed:
                    s["x"].copy_(host_batch.view(s["x"].shape), non_blocking=True)
                if self.overlay and self.mixed:
                    s["hw"].copy_(s["hw_host"], non_blocking=True)
                if self.track is not None:
                    s["streams"].copy_(s["streams_host"], non_blocking=True)
                s["copied"].record(self.h2d)
            with torch.cuda.stream(self.compute):
                self.compute.wait_event(s["copied"])
                self.compute.wait_event(s["out"])           # the previous records of this slot have left the device
                if enc is not None:
                    s["dec"].decode(s["x"], self.h * self.w * 3)
                if self.mixed:
                    if len(shapes) < self.batch:
                        s["xr"][len(shapes):].zero_()
                    self._resize_mixed(s, shapes)
                if s["graph"] is not None:
                    s["graph"].replay()
                else:
                    self._enqueue(s)
                s["done"].record(self.compute)
            with torch.cuda.stream(self.d2h):
                self.d2h.wait_event(s["done"])
                if self.gather:                             # off the compute stream: the next batch's kernels do not wait for the peers
                    import torch.distributed as dist
                    dist.all_gather_into_tensor(s["rec_all"], s["rec"], group=self.group)
                s["rec_host"].copy_(s["rec_all"] if self.collect_all else s["rec"], non_blocking=True)
                if self.encode is not None:
                    s["offsets_host"].copy_(s["enc"].offsets, non_blocking=True)
                elif self.overlay and self.mixed and shapes:
                    used = max(h * w * 3 for h, w in shapes)
                    s["frames_host"].view(self.batch, -1)[:len(shapes), :used].copy_(s["x"].view(self.batch, -1)[:len(shapes), :used],
                                                                                   non_blocking=True)
                elif self.overlay and not self.mixed:
                    s["frames_host"].copy_(s["x"] if self.yuv_out is None else s["yuv_out"], non_blocking=True)
                if enc is not None:
                    s["status_host"].copy_(s["dec"].status, non_blocking=True)
                if self.track is not None:
                    s["ids_host"].copy_(s["ids"], non_blocking=True)
                s["out"].record(self.d2h)
        s["busy"] = True
        ticket = self._next
        self._next = (self._next + 1) % len(self.slots)
        return ticket

    def result(self, ticket, copy=True, source_coords=None, gathered=False):
        """Block until the ticket's records are on the host; returns the reference's 4-tuple for this rank's batch
        (numpy float64: [batch,P], [batch,P,17], [batch,P,17,2], [batch,P,17,2]).  With ``overlay``, a fifth item holds this
        rank's drawn frames: uint8 [batch,h,w,3] (with ``yuv_out``, in its YUV layout), or in mixed mode a list of [h_i,w_i,3] arrays, one per submitted frame (with
        ``encode``: their JPEG or PNG files, a list of ``bytes``).  With
        ``jpeg``, the int32 decode status [batch] follows; with ``track``, the int64 track ids [batch, P] come last.  ``gathered=True`` (rank 0 of a
        ``gather=True`` pipeline): the records of ALL ranks' batches instead, leading dimension ``world * batch`` (rank-major).
        ``source_coords`` is a construction-time option (the scaling runs on the device); passing a different value here is an
        error."""
        assert source_coords is None or bool(source_coords) == self.source_coords, \
            "source_coords is fixed when the pipeline is built (the scaling runs on the device, before the D2H copy)"
        s = self.slots[ticket]
        assert s["busy"], "no batch in flight for this ticket"
        s["out"].synchronize()
        s["busy"] = False
        flat = s["rec_host"].numpy()
        if copy:
            flat = flat.copy()
        frames = ()
        if self.encode is not None:
            frames = (self._files(s),)
        elif self.overlay:
            fr = s["frames_host"].numpy()
            if self.mixed:
                rows = fr.reshape(self.batch, -1)
                fr = [rows[i, :h * w * 3].reshape(h, w, 3) for i, (h, w) in enumerate(s["shapes"])]
                frames = ([f.copy() for f in fr] if copy else fr,)
            else:
                frames = (fr.copy() if copy else fr,)
        if self.jpeg:
            frames = frames + (s["status_host"].numpy().copy(),)
        if self.track is not None:
            frames = frames + (s["ids_host"].numpy().copy(),)
        if not gathered:
            own = flat[self.rank * self.nrec:(self.rank + 1) * self.nrec] if self.collect_all else flat
            return split_pose_records(own, self.batch, self.P) + frames
        assert self.collect_all, "gathered=True: only rank 0 of a gather=True pipeline reads every rank's records back"
        parts = [split_pose_records(flat[r * self.nrec:(r + 1) * self.nrec], self.batch, self.P) for r in range(self.world)]
        return tuple(np.concatenate([p[j] for p in parts], axis=0) for j in range(4)) + frames

    def _files(self, s):
        """The slot's packed files, copied back on their own stream once the offsets are on the host (the d2h stream would
        queue the copy behind later tickets' copies).  Returns only when the copy is done: the next step of this slot rewrites
        the packed buffer."""
        off = s["offsets_host"].numpy().copy()
        n = int(off[-1])
        if n > s["files_host"].numel():
            s["files_host"] = torch.empty(n, dtype=torch.uint8).pin_memory()
        if n:
            with torch.cuda.device(self.dev), torch.cuda.stream(self.files_stream):
                s["files_host"][:n].copy_(s["enc"].out[:n], non_blocking=True)
            self.files_stream.synchronize()
        self.last_file_bytes = n
        data = s["files_host"].numpy()
        count = len(s["shapes"]) if self.mixed else self.batch
        return [data[off[i]:off[i + 1]].tobytes() for i in range(count)]

    def time_gather(self, reps=20):
        """Device time (ms) of one all-gather of a step's record buffer, measured alone with CUDA events."""
        import torch.distributed as dist
        assert self.gather
        s = self.slots[0]
        with torch.cuda.device(self.dev), torch.cuda.stream(self.d2h):
            for _ in range(3):
                dist.all_gather_into_tensor(s["rec_all"], s["rec"], group=self.group)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(self.d2h)
            for _ in range(reps):
                dist.all_gather_into_tensor(s["rec_all"], s["rec"], group=self.group)
            e1.record(self.d2h)
            self.d2h.synchronize()
        return e0.elapsed_time(e1) / reps

    def run(self, batches, copy=True, source_coords=None):
        """Generator: yields the pose records of every batch of ``batches`` in order, keeping ``depth`` batches in flight.
        Items are uint8 batches, or ``(batch, shapes)`` pairs for a ``mixed=True`` pipeline, ``(batch, shapes, streams)`` for
        a ``track=`` one (``shapes`` None unless mixed)."""
        pending = []
        for hb in batches:
            if len(pending) == len(self.slots):
                yield self.result(pending.pop(0), copy=copy, source_coords=source_coords)
            pending.append(self.submit(*hb) if isinstance(hb, (tuple, list)) else self.submit(hb))
        while pending:
            yield self.result(pending.pop(0), copy=copy, source_coords=source_coords)
