"""Pose tracking across the frames of video streams on the GPU (``pn_track_poses``): the bounding-box tracker of TF.js
pose-detection (``BoundingBoxTracker``), run on the records ``decode_multiple_poses_batch`` leaves on the device, so that pose k
of frame t keeps its id in frame t + 1 without a host round trip.

    tracker = posenet.PoseTracker(n_streams=4)
    ps, ks, kc, ko, _ = posenet.decode_multiple_poses_batch(*heads, output_stride=16)
    ids = tracker.update(ps, ks, kc, stream_ids=[0, 1, 2, 3, 0, 1, 2, 3])     # CUDA int64 [N, P], no synchronisation

``BatchPipeline(..., track=tracker)`` runs it inside the step's graph (``posenet.pipeline``).

With ``smoothing=OneEuro(...)`` the tracker also smooths each tracked pose's keypoints across frames with a One Euro filter
(``pn_smooth_keypoints``, after the tracking), the filter TF.js pose-detection runs per tracked pose:

    tracker = posenet.PoseTracker(n_streams=4, smoothing=posenet.OneEuro(fps=30.0))
    ids, coords = tracker.update(ps, ks, kc, stream_ids)     # coords: new CUDA float64 [N, P, 17, 2], kc is not modified

Semantics (tests/test_track_cpu.py restates them in numpy):
- A stream is a video source with an id in ``0 .. n_streams-1``.  Each stream holds up to ``max_tracks`` tracks (an id, a box,
  the stream frame at which it was last matched), a frame counter and a ``next_id`` that starts at 1.
- Frames are processed in submission order, and the rows of one stream within a batch in row order.  Rows of stream -1 are
  not tracked: all their ids are -1.
- A detection is a record with ``pose_score > 0``.  Its box is the min / max of y and x over its keypoints with
  ``keypoint_score >= min_part_score``, in the coordinates the records hold (frame pixels in a ``source_coords`` pipeline).  No
  such keypoint: an empty box.  One keypoint: a box of zero area, whose IoU with every box is 0.
- For each frame of stream s: (1) s's frame counter becomes t; (2) tracks with ``t - last > max_age`` are dropped, stably;
  (3) the IoU of each detection with each remaining track is computed in float64: ``iy = min(ymax) - max(ymin)``,
  ``ix = min(xmax) - max(xmin)``; 0 if ``iy <= 0`` or ``ix <= 0`` or either box is empty; otherwise ``inter = iy * ix``,
  ``union = area_a + area_b - inter`` with ``area = (ymax - ymin) * (xmax - xmin)``, and the IoU is ``inter / union`` (0 when
  ``union <= 0``); (4) walking the detections in record order, each takes the unmatched track with the largest IoU among those
  with ``IoU >= min_similarity`` (a tie goes to the first such track); the track takes the detection's box and ``last = t`` and
  keeps its id.  A detection without such a track gets a new track, appended with ``id = next_id++``; (5) the tracks are
  stably sorted by ``last``, descending, and the first ``max_tracks`` kept.
- The result: int64 ``[N, P]`` ids aligned with ``pose_scores``; -1 for records that are not detections and for untracked rows.

IoU and not OKS: it needs only ``+ - * /`` and min / max, so the device (float64, no FMA contraction) is bit-exact with a numpy
restatement, and no last-ulp difference of ``exp`` can flip a ``>= min_similarity`` test.  Ages count stream frames, not
milliseconds (TF.js counts 1000 ms): the pipeline knows frames, not wall time.

Smoothing semantics (tests/test_smooth_cpu.py restates them in numpy; Casiez et al., "1€ Filter", CHI 2012):
- ``OneEuro(fps=30.0, min_cutoff=1.0, beta=0.0, d_cutoff=1.0)``: the starting point of the paper's tuning procedure.  ``fps``
  converts stream frames to seconds; ``beta`` is in 1/pixel of the coordinates the records hold (frame pixels with
  ``source_coords=True``, network-input pixels otherwise).  ``fps``, ``min_cutoff``, ``d_cutoff`` finite and > 0, ``beta``
  finite and >= 0: ValueError otherwise.
- Each stream holds a smoothing frame counter, which advances on every row of the stream as the tracker's does, and a table
  of up to ``max_tracks`` entries: a track id, ``last`` (the stream frame of its last update) and, per coordinate (17 x 2),
  the previous raw value ``x_prev``, previous filtered value ``x_hat`` and previous filtered derivative ``dx_hat`` (float64).
- For each frame of stream s, rows in order: (1) ``t += 1``; entries with ``t - last > max_age`` are removed, stably (the
  tracker drops a track under the same condition, so a live id keeps its filter); (2) the detections (records with id >= 1)
  are walked in record order: an id with an entry updates it; otherwise a fresh entry is appended while the table has room;
  otherwise the entry with the smallest ``last < t`` is replaced in place (the first in table order on a tie; only when more
  than ``max_tracks`` ids compete); a record for which every entry was updated in this frame, or whose id was already met in
  this frame, keeps its raw coordinates and no state; (3) a fresh entry outputs x unchanged and stores ``x_prev = x_hat = x``,
  ``dx_hat = 0``, ``last = t``.  An existing entry computes per coordinate, in float64 without FMA and in this order:
  ``rate = fps / (t - last)``, ``dx = (x - x_prev) * rate``, ``a_d = 1 / (1 + rate / (TWO_PI * d_cutoff))``,
  ``dx_hat = a_d * dx + (1 - a_d) * dx_hat``, ``cutoff = min_cutoff + beta * |dx_hat|``,
  ``a = 1 / (1 + rate / (TWO_PI * cutoff))``, ``x_hat = a * x + (1 - a) * x_hat``, with ``TWO_PI = 2 * math.pi``; the output
  is ``x_hat``, and ``x_prev`` becomes the raw x (as the paper's reference code and TF.js's ``OneEuroFilter`` do), ``last = t``.
- All 17 keypoints are filtered whatever their score, as TF.js does.  Scores, pose scores and offsets are never changed;
  untracked rows and records that are not detections are left as they are.  The boxes and ids come from the raw coordinates:
  smoothing runs after the tracking.
Only ``+ - * /`` and ``|x|``: the device is bit-exact with the numpy restatement.
"""
import ctypes as C
from typing import NamedTuple

import numpy as np
import torch

from posenet import _native as nat
from posenet.constants import NUM_KEYPOINTS

DECODE_SCORE_THRESHOLD = 0.5            # decode_multiple_poses(_batch)'s default score_threshold


class _OneEuro(NamedTuple):
    fps: float
    min_cutoff: float
    beta: float
    d_cutoff: float


class OneEuro(_OneEuro):
    """Parameters of the One Euro filter ``PoseTracker(smoothing=...)`` runs on each tracked pose: ``fps`` (stream frames per
    second), ``min_cutoff`` and ``d_cutoff`` (Hz), ``beta`` (1/pixel).  ValueError unless ``fps``, ``min_cutoff`` and
    ``d_cutoff`` are finite and > 0 and ``beta`` is finite and >= 0."""
    __slots__ = ()

    def __new__(cls, fps=30.0, min_cutoff=1.0, beta=0.0, d_cutoff=1.0):
        vals = []
        for name, v, lo_open in (("fps", fps, True), ("min_cutoff", min_cutoff, True), ("beta", beta, False),
                                 ("d_cutoff", d_cutoff, True)):
            try:
                f = float(v)
            except (TypeError, ValueError):
                raise ValueError("%s=%r is not a number" % (name, v)) from None
            if isinstance(v, bool) or not np.isfinite(f) or (f <= 0 if lo_open else f < 0):
                raise ValueError("%s=%r: a finite number %s 0" % (name, v, ">" if lo_open else ">="))
            vals.append(f)
        return super().__new__(cls, *vals)


class PoseTracker:
    def __init__(self, n_streams, max_tracks=18, max_age=30, min_similarity=0.15, min_part_score=None, device=None,
                 smoothing=None):
        """Device state for ``n_streams`` streams of at most ``max_tracks`` tracks (1..256) each; TF.js's defaults, with
        ``max_age`` in stream frames.  ``min_part_score``: the keypoint score a box takes in; None for the decode's
        ``score_threshold`` (0.5 unless a ``BatchPipeline``'s decode arguments set another).  ``smoothing``: a ``OneEuro``
        to also smooth each tracked pose's keypoints (``update`` then returns ``(ids, coords)``); None: no smoothing."""
        if smoothing is not None and not isinstance(smoothing, OneEuro):
            raise ValueError("smoothing= takes a posenet.OneEuro, got %r" % (smoothing,))
        smoothing = None if smoothing is None else OneEuro(*smoothing)          # checked again: _replace skips __new__
        for name, v, lo, hi in (("n_streams", n_streams, 1, 1 << 20), ("max_tracks", max_tracks, 1, nat.TRACK_MAX_TRACKS),
                                ("max_age", max_age, 0, (1 << 31) - 1)):
            if not isinstance(v, (int, np.integer)) or isinstance(v, bool) or not lo <= v <= hi:
                raise ValueError("%s=%r: an integer in %d..%d" % (name, v, lo, hi))
        if not np.isfinite(float(min_similarity)):
            raise ValueError("min_similarity=%r is not a finite number" % (min_similarity,))
        if min_part_score is not None and np.isnan(float(min_part_score)):
            raise ValueError("min_part_score is NaN")
        self.n_streams, self.max_tracks, self.max_age = int(n_streams), int(max_tracks), int(max_age)
        self.min_similarity = float(min_similarity)
        self.min_part_score = None if min_part_score is None else float(min_part_score)
        nat.require_device()
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        nbytes = C.c_size_t()
        nat.check(nat.load().pn_track_state_bytes(self.n_streams, self.max_tracks, C.byref(nbytes)), "pn_track_state_bytes")
        self.stream_bytes = nbytes.value // self.n_streams
        # all zero bytes: every stream at its start (no tracks, frame 0, next id 1)
        self.state = torch.zeros(nbytes.value // 8, dtype=torch.int64, device=self.device)
        self.smoothing = smoothing
        self.smooth_state = None
        if self.smoothing is not None:
            nat.check(nat.load().pn_smooth_state_bytes(self.n_streams, self.max_tracks, C.byref(nbytes)), "pn_smooth_state_bytes")
            self.smooth_stream_bytes = nbytes.value // self.n_streams
            # all zero bytes: every stream at its start (frame 0, no filters)
            self.smooth_state = torch.zeros(nbytes.value // 8, dtype=torch.int64, device=self.device)
        self.stream = None          # the CUDA stream reset() enqueues on: None for the current one; a BatchPipeline sets its own

    def stream_ids(self, streams, n):
        """Host stream ids of n rows as int32 numpy; ValueError for a wrong count or an id outside -1..n_streams-1."""
        a = np.asarray(streams)
        if a.shape != (n,) or not (a.dtype.kind in "iu" or (a.size == 0 and a.dtype.kind == "f")):
            raise ValueError("stream ids: %d integers expected, got %s %s" % (n, a.dtype, a.shape))
        if a.size and (a.min() < -1 or a.max() >= self.n_streams):
            raise ValueError("stream ids must be in -1..%d (-1: not tracked), got %d..%d" % (self.n_streams - 1, a.min(), a.max()))
        return a.astype(np.int32)

    def launch(self, pose_scores, keypoint_scores, keypoint_coords, stream_ids, ids, min_part_score):
        """pn_track_poses on the current stream: float64 CUDA records, CUDA int32 ``stream_ids`` [N], CUDA int64 ``ids`` [N, P]
        out (every buffer contiguous)."""
        n, P = ids.shape
        nat.check(nat.load().pn_track_poses(C.c_void_p(pose_scores.data_ptr()), C.c_void_p(keypoint_scores.data_ptr()),
                                            C.c_void_p(keypoint_coords.data_ptr()), n, P, C.c_void_p(stream_ids.data_ptr()),
                                            C.c_void_p(self.state.data_ptr()), self.n_streams, self.max_tracks, self.max_age,
                                            self.min_similarity, min_part_score, C.c_void_p(ids.data_ptr()), nat.stream_ptr()),
                  "pn_track_poses")

    def launch_smooth(self, ids, keypoint_coords, stream_ids):
        """pn_smooth_keypoints on the current stream: CUDA int64 ``ids`` [N, P] (``launch``'s output), CUDA float64
        ``keypoint_coords`` [N, P, 17, 2] smoothed in place, CUDA int32 ``stream_ids`` [N] (every buffer contiguous)."""
        n, P = ids.shape
        q = self.smoothing
        nat.check(nat.load().pn_smooth_keypoints(C.c_void_p(ids.data_ptr()), C.c_void_p(keypoint_coords.data_ptr()), n, P,
                                                 C.c_void_p(stream_ids.data_ptr()), C.c_void_p(self.smooth_state.data_ptr()),
                                                 self.n_streams, self.max_tracks, self.max_age, q.fps, q.min_cutoff, q.beta,
                                                 q.d_cutoff, nat.stream_ptr()),
                  "pn_smooth_keypoints")

    def update(self, pose_scores, keypoint_scores, keypoint_coords, stream_ids):
        """Track one batch of records (``decode_multiple_poses_batch``'s CUDA float64 ``[N, P]``, ``[N, P, 17]``,
        ``[N, P, 17, 2]``) on the current stream, without synchronising.  ``stream_ids``: N host integers in -1..n_streams-1
        (ValueError otherwise), or a CUDA int32 tensor [N], which is not checked (the device treats an id out of range as -1;
        this form can be captured in a CUDA graph).  Returns CUDA int64 ids [N, P]; with ``smoothing``, ``(ids, coords)``,
        ``coords`` a new CUDA float64 [N, P, 17, 2] tensor of the smoothed coordinates (``keypoint_coords`` is not modified)."""
        ps, ks, kc = pose_scores, keypoint_scores, keypoint_coords
        if ps.dim() != 2 or tuple(ks.shape) != tuple(ps.shape) + (NUM_KEYPOINTS,) or \
                tuple(kc.shape) != tuple(ps.shape) + (NUM_KEYPOINTS, 2):
            raise ValueError("records of shapes [N, P], [N, P, 17], [N, P, 17, 2] expected, got %s %s %s" % (
                tuple(ps.shape), tuple(ks.shape), tuple(kc.shape)))
        if any(t.dtype != torch.float64 or t.device != self.device for t in (ps, ks, kc)):
            raise ValueError("records must be float64 tensors on %s" % self.device)
        n, P = ps.shape
        if not 1 <= P <= nat.TRACK_MAX_POSES:
            raise ValueError("P=%d poses per frame: the tracker takes 1..%d" % (P, nat.TRACK_MAX_POSES))
        with torch.cuda.device(self.device):
            if torch.is_tensor(stream_ids) and stream_ids.is_cuda:
                if stream_ids.dtype != torch.int32 or tuple(stream_ids.shape) != (n,) or stream_ids.device != self.device:
                    raise ValueError("device stream ids: int32 [%d] on %s expected" % (n, self.device))
                sid = stream_ids.contiguous()
            else:
                host = torch.from_numpy(self.stream_ids(stream_ids.numpy() if torch.is_tensor(stream_ids) else stream_ids, n))
                sid = host.pin_memory().to(self.device, non_blocking=True)
            ids = torch.empty((n, P), dtype=torch.int64, device=self.device)
            coords = kc.clone(memory_format=torch.contiguous_format) if self.smoothing is not None else None
            if n:
                mps = DECODE_SCORE_THRESHOLD if self.min_part_score is None else self.min_part_score
                self.launch(ps.contiguous(), ks.contiguous(), kc.contiguous(), sid, ids, mps)
                if coords is not None:
                    self.launch_smooth(ids, coords, sid)
        return ids if coords is None else (ids, coords)

    def reset(self, stream=None):
        """Forget every stream (``stream=None``) or one: its tracks, frame counter and ids start over, and so do its
        filters with ``smoothing``.  Enqueued on the tracker's CUDA stream (a pipeline's step stream: ordered with the steps
        submitted before and after)."""
        if stream is not None and not (isinstance(stream, (int, np.integer)) and 0 <= stream < self.n_streams):
            raise ValueError("stream %r: an integer in 0..%d" % (stream, self.n_streams - 1))
        words = self.stream_bytes // 8
        with torch.cuda.device(self.device), torch.cuda.stream(self.stream or torch.cuda.current_stream(self.device)):
            (self.state if stream is None else self.state[int(stream) * words:(int(stream) + 1) * words]).zero_()
            if self.smooth_state is not None:
                sw = self.smooth_stream_bytes // 8
                (self.smooth_state if stream is None else self.smooth_state[int(stream) * sw:(int(stream) + 1) * sw]).zero_()
