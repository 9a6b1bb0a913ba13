"""One Euro keypoint smoothing on the GPU (pn_smooth_keypoints) against the numpy oracle of tests/smoothref.py, bit for bit:
PoseTracker(smoothing=...).update on seeded synthetic records at P = 10 and 50, batches of 1, 32 and 512 and 1 to 512 streams
(the input records stay as they were, the ids are those of a tracker without smoothing); graph replay with new records and
reset; and BatchPipeline(track=tracker) with smoothing on test_gpu_track.py's seeded video of moving people (I420 frames at
1280x720), with graphs on and off: its records are the oracle's smoothing of the records and ids of the same pipeline with a
tracker without smoothing, and its drawn frames and JPEG files are cv2's of those records."""
import cv2
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

import posenet  # noqa: E402
from smoothref import NC, SmoothOracle, TrackSmoothOracle  # noqa: E402
from test_gpu_track import KW, H, N, STREAMS, W, cuda, model, video  # noqa: E402
from trackref import interleave, synth_stream  # noqa: E402

DEV = "cuda"


def bits_equal(a, b):
    return np.array_equal(np.asarray(a).view(np.int64), np.asarray(b).view(np.int64))


def table_of(tracker, s):
    """(frame, [(id, last, x_prev, x_hat, dx_hat), ...]) of stream s, read from the device's smoothing state."""
    words = tracker.smooth_stream_bytes // 8
    g = tracker.smooth_state[s * words:(s + 1) * words].cpu().numpy()
    n = int(g[1:2].view(np.int32)[0])
    tab = g[2:2 + 2 * n].reshape(n, 2)
    val = g[2 + 2 * tracker.max_tracks:].view(np.float64).reshape(tracker.max_tracks, 3, NC)
    return int(g[0]), [(int(tab[i, 0]), int(tab[i, 1]), val[i, 0], val[i, 1], val[i, 2]) for i in range(n)]


def same_table(a, b):
    return a[0] == b[0] and len(a[1]) == len(b[1]) and all(
        x[:2] == y[:2] and all(bits_equal(u, v) for u, v in zip(x[2:], y[2:])) for x, y in zip(a[1], b[1]))


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
    q = posenet.OneEuro(fps=30.0, min_cutoff=0.8, beta=0.02, d_cutoff=1.0)
    tracker = posenet.PoseTracker(n_streams, max_tracks=max_tracks, max_age=max_age, smoothing=q)
    plain = posenet.PoseTracker(n_streams, max_tracks=max_tracks, max_age=max_age)
    ref = TrackSmoothOracle(n_streams, max_tracks=max_tracks, max_age=max_age, smoothing=q)
    for ps, ks, kc, sid in interleave(rng, recs, batch, min_batch=batch):
        dev = cuda(ps, ks, kc)
        ids, coords = tracker.update(*dev, sid.tolist())
        assert coords.dtype == torch.float64 and coords.is_cuda and tuple(coords.shape) == kc.shape
        want_ids, want = ref.batch(ps, ks, kc, sid)
        assert np.array_equal(ids.cpu().numpy(), want_ids)
        assert np.array_equal(plain.update(*dev, sid.tolist()).cpu().numpy(), want_ids)
        got = coords.cpu().numpy()
        assert bits_equal(got, want), np.argwhere(got != want)[:5]
        assert bits_equal(dev[2].cpu().numpy(), kc)                        # the caller's records are not modified
    for s in range(n_streams):
        assert same_table(table_of(tracker, s), ref.smooth.table(s)), s
    assert ref.smooth.events["update"] > 0


def test_graph_replay_with_new_records_and_reset():
    rng = np.random.default_rng(12)
    n_streams, P, batch = 3, 10, 8
    recs = [synth_stream(rng, 160, 6, P, 8) for _ in range(n_streams)]
    batches = list(interleave(rng, recs, batch, min_batch=batch))[:-1]      # full batches only
    q = posenet.OneEuro(fps=24.0, beta=0.05)
    tracker = posenet.PoseTracker(n_streams, max_age=8, smoothing=q)
    ref = TrackSmoothOracle(n_streams, max_age=8, smoothing=q)
    ps_d, ks_d, kc_d = cuda(*batches[0][:3])
    sid_d = torch.zeros(batch, dtype=torch.int32, device=DEV)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    g = torch.cuda.CUDAGraph()
    with torch.cuda.stream(side), torch.cuda.graph(g, stream=side):
        ids_d, coords_d = tracker.update(ps_d, ks_d, kc_d, sid_d)
    torch.cuda.current_stream().wait_stream(side)
    assert table_of(tracker, 0) == (0, [])                                  # capturing ran nothing
    for i, (ps, ks, kc, sid) in enumerate(batches):
        if i == len(batches) // 2:
            tracker.reset(0)
            ref.reset(0)
        if i % 5 == 4:                                                      # device ids out of range are untracked rows
            sid = sid.copy()
            sid[0], sid[-1] = 7, -3
        for d, h in zip((ps_d, ks_d, kc_d), (ps, ks, kc)):
            d.copy_(torch.from_numpy(h))
        sid_d.copy_(torch.from_numpy(sid))
        g.replay()
        want_ids, want = ref.batch(ps, ks, kc, sid)
        assert np.array_equal(ids_d.cpu().numpy(), want_ids), i
        assert bits_equal(coords_d.cpu().numpy(), want), i
    for s in range(n_streams):
        assert same_table(table_of(tracker, s), ref.smooth.table(s))
    assert ref.smooth.table(0)[0] < ref.smooth.table(1)[0]


# ---- BatchPipeline(track=tracker) with smoothing, on test_gpu_track.py's video of moving people

SMOOTHING = posenet.OneEuro(fps=30.0, min_cutoff=0.5, beta=0.01, d_cutoff=1.0)


@pytest.mark.parametrize("use_graph,extra", [(True, {}), (False, {}), (True, dict(overlay=(0.05, 0.1))),
                                             (False, dict(overlay=(0.05, 0.1))), (True, dict(overlay=(0.05, 0.1), encode=[]))])
def test_pipeline_smooths_a_video_like_the_oracle(use_graph, extra):
    m = model()
    batches = video(6, STREAMS)
    kw = dict(KW, use_graph=use_graph, **extra)
    items = [(b, None, STREAMS) for b in batches]
    ref_pipe = posenet.BatchPipeline(m, N, H, W, track=posenet.PoseTracker(2, max_age=3), **kw)
    ref = list(ref_pipe.run(items))
    tracker = posenet.PoseTracker(2, max_age=3, smoothing=SMOOTHING)
    pipe = posenet.BatchPipeline(m, N, H, W, track=tracker, **kw)
    assert (pipe.h2d_bytes_per_batch, pipe.d2h_bytes_per_batch) == (ref_pipe.h2d_bytes_per_batch, ref_pipe.d2h_bytes_per_batch)
    got = list(pipe.run(items))
    oracle = SmoothOracle(2, max_age=3, **SMOOTHING._asdict())
    changed = False
    for b, g, r in zip(batches, got, ref):
        assert len(g) == len(r)
        want = oracle.batch(r[-1], r[2], STREAMS)
        assert np.array_equal(g[-1], r[-1])                                 # the ids come from the raw coordinates
        for j in (0, 1, 3):                                                 # scores and offsets are not changed
            assert np.array_equal(g[j], r[j])
        assert bits_equal(g[2], want)
        changed |= not np.array_equal(g[2], r[2])
        if extra:
            i420 = b.numpy()
            for i in range(N):
                bgr = cv2.cvtColor(i420[i], cv2.COLOR_YUV2BGR_I420)
                drawn = posenet.draw_skel_and_kp(bgr, g[0][i], g[1][i], want[i], *extra["overlay"])
                if "encode" in extra:
                    assert g[4][i] == cv2.imencode(".jpg", drawn)[1].tobytes(), i
                else:
                    assert np.array_equal(g[4][i], drawn), i
    assert changed and oracle.events["update"] > 0


def test_pipeline_reset_restarts_the_filters():
    m = model()
    batches = video(4, STREAMS)
    tracker = posenet.PoseTracker(2, smoothing=SMOOTHING)
    pipe = posenet.BatchPipeline(m, N, H, W, track=tracker, **KW)
    plain = posenet.BatchPipeline(m, N, H, W, track=posenet.PoseTracker(2), **KW)
    oracle = SmoothOracle(2, **SMOOTHING._asdict())
    for i, b in enumerate(batches):
        if i == 2:
            tracker.reset(0)                                                # ordered with the steps: on the pipeline's stream
            plain.track.reset(0)
            oracle.reset(0)
        r = plain.result(plain.submit(b, None, STREAMS))
        g = pipe.result(pipe.submit(b, None, STREAMS))
        assert np.array_equal(g[-1], r[-1]), i
        assert bits_equal(g[2], oracle.batch(r[-1], r[2], STREAMS)), i
    assert same_table(table_of(tracker, 0), oracle.table(0)) and same_table(table_of(tracker, 1), oracle.table(1))
