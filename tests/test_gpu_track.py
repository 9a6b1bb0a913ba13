"""Pose tracking on the GPU (pn_track_poses) against the numpy oracle of tests/trackref.py, id for id: PoseTracker.update on
seeded synthetic records at P = 10 and 50, batches of 1, 32 and 512 and 1 to 512 streams; graph replay with new records and
reset; and BatchPipeline(track=...) on a seeded video of moving people (I420 frames at 1280x720, random-init MobileNetV1-50,
OS8) against the oracle fed with the pipeline's own records, with graphs on and off, with overlays and with JPEG files out.  A
track= pipeline's records and frames are those of the same pipeline without it."""
import cv2
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

import posenet  # noqa: E402
from oracle import net as onet  # noqa: E402
from oracle import synth  # noqa: E402
from trackref import Oracle, interleave, synth_stream  # noqa: E402

DEV = "cuda"


def cuda(*arrays):
    return [torch.from_numpy(np.ascontiguousarray(a)).to(DEV) for a in arrays]


def state_of(tracker, s):
    """(frame, ids issued, [(id, last), ...]) of stream s, read from the device state."""
    words = tracker.stream_bytes // 8
    g = tracker.state[s * words:(s + 1) * words].cpu().numpy()
    n = int(g[2:3].view(np.int32)[0])
    tr = g[4:4 + 6 * n].reshape(n, 6)
    return int(g[0]), int(g[1]), [(int(t[4]), int(t[5])) for t in tr]


@pytest.mark.parametrize("P,batch,n_streams,n_frames,max_tracks,max_age", [
    (10, 1, 1, 200, 18, 30),
    (10, 32, 1, 320, 18, 30),
    (10, 32, 5, 120, 4, 6),
    (50, 32, 3, 100, 18, 10),
    (10, 512, 8, 200, 18, 30),
    (50, 512, 64, 24, 18, 5),
    (10, 512, 512, 6, 18, 2),
])
def test_update_matches_the_oracle(P, batch, n_streams, n_frames, max_tracks, max_age):
    rng = np.random.default_rng(P * 1000 + batch + n_streams)
    recs = [synth_stream(rng, n_frames, int(rng.integers(3, 16)), P, max_age) for _ in range(n_streams)]
    tracker = posenet.PoseTracker(n_streams, max_tracks=max_tracks, max_age=max_age)
    ref = Oracle(n_streams, max_tracks=max_tracks, max_age=max_age)
    for ps, ks, kc, sid in interleave(rng, recs, batch, min_batch=batch):
        ids = tracker.update(*cuda(ps, ks, kc), sid.tolist())
        assert ids.dtype == torch.int64 and ids.is_cuda
        want = ref.batch(ps, ks, kc, sid)
        got = ids.cpu().numpy()
        assert np.array_equal(got, want), np.argwhere(got != want)[:5]
    for s in range(n_streams):
        assert state_of(tracker, s) == ref.tracks(s), s


def test_graph_replay_with_new_records_and_reset():
    rng = np.random.default_rng(11)
    n_streams, P, batch = 3, 10, 8
    recs = [synth_stream(rng, 160, 6, P, 8) for _ in range(n_streams)]
    batches = list(interleave(rng, recs, batch, min_batch=batch))[:-1]      # full batches only
    tracker = posenet.PoseTracker(n_streams, max_age=8)
    ref = Oracle(n_streams, max_age=8)
    ps_d, ks_d, kc_d = cuda(*batches[0][:3])
    sid_d = torch.zeros(batch, dtype=torch.int32, device=DEV)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    g = torch.cuda.CUDAGraph()
    with torch.cuda.stream(side), torch.cuda.graph(g, stream=side):
        ids_d = tracker.update(ps_d, ks_d, kc_d, sid_d)
    torch.cuda.current_stream().wait_stream(side)
    assert state_of(tracker, 0) == (0, 0, [])                               # capturing ran nothing
    for i, (ps, ks, kc, sid) in enumerate(batches):
        if i == len(batches) // 3:
            tracker.reset(1)
            ref.reset(1)
        if i == 2 * len(batches) // 3:
            tracker.reset()
            ref.reset()
        if i % 5 == 4:                                                      # device ids out of range are untracked rows
            sid = sid.copy()
            sid[0], sid[-1] = 7, -3
        for d, h in zip((ps_d, ks_d, kc_d), (ps, ks, kc)):
            d.copy_(torch.from_numpy(h))
        sid_d.copy_(torch.from_numpy(sid))
        g.replay()
        assert np.array_equal(ids_d.cpu().numpy(), ref.batch(ps, ks, kc, sid)), i
    for s in range(n_streams):
        assert state_of(tracker, s) == ref.tracks(s)


def test_update_arguments():
    tracker = posenet.PoseTracker(2)
    ps, ks, kc = cuda(np.zeros((3, 10)), np.zeros((3, 10, 17)), np.zeros((3, 10, 17, 2)))
    for sid in ([0, 1, 2], [0, -2, 1], [0, 1], [0.0, 1.0, 1.0], [[0, 1, 1]]):
        with pytest.raises(ValueError):
            tracker.update(ps, ks, kc, sid)
    with pytest.raises(ValueError):
        tracker.update(ps.float(), ks, kc, [0, 1, 1])
    with pytest.raises(ValueError):
        tracker.update(ps, ks[:, :, :16], kc, [0, 1, 1])
    with pytest.raises(ValueError):
        tracker.update(ps, ks, kc, torch.zeros(3, dtype=torch.int64, device=DEV))
    with pytest.raises(ValueError):
        tracker.reset(2)
    assert tracker.update(ps, ks, kc, np.array([-1, 1, 0])).cpu().numpy().tolist() == [[-1] * 10] * 3


# ---- BatchPipeline(track=...) on a video of moving people

N, H, W, OS = 4, 720, 1280, 8
KW = dict(depth=2, output_stride=OS, source_coords=True, max_pose_detections=10, min_pose_score=0.05, score_threshold=0.3,
          yuv=cv2.COLOR_YUV2BGR_I420)


def model():
    sd = onet.init_params(50, seed=5, scheme="scaled", gain=0.8)
    m = posenet.MobileNetV1(50, output_stride=OS)
    m.load_state_dict(sd)
    return m.cuda().set_compute_dtype("bf16")


def person(img, y, x, s):
    """A stick figure of height ~4s px with its head at (y, x)."""
    c = (230, 220, 210)
    cv2.circle(img, (int(x), int(y)), int(s * 0.4), c, -1)
    cv2.rectangle(img, (int(x - s * 0.4), int(y + s * 0.5)), (int(x + s * 0.4), int(y + s * 2)), c, -1)
    for dx in (-1, 1):
        cv2.line(img, (int(x + dx * s * 0.4), int(y + s * 0.7)), (int(x + dx * s * 1.1), int(y + s * 1.8)), c, max(2, s // 8))
        cv2.line(img, (int(x + dx * s * 0.2), int(y + s * 2)), (int(x + dx * s * 0.4), int(y + s * 3.6)), c, max(2, s // 8))


def video(n_batches, streams):
    """I420 batches of two streams of moving people (stream per row in ``streams``, -1 rows: still frames) and the rows'
    stream ids."""
    bg = [synth.smooth_image(H, W, 900 + s) for s in range(3)]
    t = [0, 0, 0]
    out = []
    for _ in range(n_batches):
        frames = []
        for s in streams:
            f = bg[s].copy()
            k = t[s]
            if s == 0:
                person(f, 200 + 2 * k, 150 + 25 * k, 90)
                person(f, 150, 900 - 10 * k, 110)
            elif s == 1:
                person(f, 100 + 15 * k, 600, 120)
            t[s] += 1
            frames.append(cv2.cvtColor(f, cv2.COLOR_BGR2YUV_I420))
        out.append(torch.from_numpy(np.stack(frames)).pin_memory())
    return out


STREAMS = [0, 1, 0, -1]


@pytest.mark.parametrize("use_graph,extra", [(True, {}), (False, {}), (True, dict(overlay=(0.05, 0.1))),
                                             (True, dict(overlay=(0.05, 0.1), encode=[]))])
def test_pipeline_tracks_a_video_like_the_oracle(use_graph, extra):
    m = model()
    batches = video(6, STREAMS)
    kw = dict(KW, use_graph=use_graph, **extra)
    ref_pipe = posenet.BatchPipeline(m, N, H, W, **kw)
    ref = list(ref_pipe.run(batches))
    tracker = posenet.PoseTracker(2, max_age=3)
    pipe = posenet.BatchPipeline(m, N, H, W, track=tracker, **kw)
    assert pipe.d2h_bytes_per_batch == ref_pipe.d2h_bytes_per_batch + N * 10 * 8
    got = list(pipe.run((b, None, STREAMS) for b in batches))
    oracle = Oracle(2, max_age=3, min_part_score=0.3)               # the tracker takes the decode's score_threshold
    n_det = 0
    for g, r in zip(got, ref):
        assert len(g) == len(r) + 1
        for a, b in zip(g[:-1], r):                                 # records, frames / files: as without track=
            assert (a == b) if isinstance(a, list) else np.array_equal(a, b)
        want = oracle.batch(r[0], r[1], r[2], STREAMS)
        assert g[-1].dtype == np.int64 and np.array_equal(g[-1], want)
        n_det += int((r[0] > 0).sum())
    assert n_det > 0 and (got[-1][-1][3] == -1).all()
    assert max(oracle.tracks(s)[1] for s in range(2)) > 0


def test_pipeline_reset_and_stream_arguments():
    m = model()
    batches = video(4, STREAMS)
    tracker = posenet.PoseTracker(2, min_part_score=0.2)
    pipe = posenet.BatchPipeline(m, N, H, W, track=tracker, **KW)
    with pytest.raises(ValueError):
        pipe.submit(batches[0])
    with pytest.raises(ValueError):
        pipe.submit(batches[0], None, [0, 1, 2, 0])
    with pytest.raises(ValueError):
        pipe.submit(batches[0], None, [0, 1])
    with pytest.raises(ValueError):
        posenet.BatchPipeline(m, N, H, W, **KW).submit(batches[0], None, STREAMS)
    oracle = Oracle(2, min_part_score=0.2)
    for i, b in enumerate(batches):
        if i == 2:
            tracker.reset(0)                                        # ordered with the steps: on the pipeline's stream
            oracle.reset(0)
        r = pipe.result(pipe.submit(b, None, STREAMS))
        assert np.array_equal(r[-1], oracle.batch(r[0], r[1], r[2], STREAMS)), i


def test_gather_with_track_raises():
    m = model()
    with pytest.raises(ValueError):
        posenet.BatchPipeline(m, N, H, W, gather=True, track=posenet.PoseTracker(1), **KW)
    with pytest.raises(ValueError):
        posenet.BatchPipeline(m, N, H, W, track=object(), **KW)
