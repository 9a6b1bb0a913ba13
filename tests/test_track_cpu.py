"""Pose tracker arithmetic (csrc/track.cuh) against the numpy oracle of tests/trackref.py, on the host.

The header is compiled into a small host library that runs track_frame with one "lane" per stream over the same state layout
the kernel keeps, row by row as pn_track_poses does.  Seeded synthetic sequences are compared frame by frame: ids, and each
stream's frame counter, issued ids and tracks.  Also exact IoU ties, IoUs exactly at min_similarity, empty and zero-area boxes,
and the argument checks of pn_track_poses / pn_track_state_bytes, which run on the host before any launch.  The kernel's warp
split of the work is covered by tests/test_gpu_track.py."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from posenet import _native as nat
from trackref import Oracle, interleave, synth_stream

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "posenet-pytorch_b200", "csrc")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")

SHIM = r"""
#include <string.h>
#include <vector>
#include "track.cuh"
using namespace pn::track;
extern "C" void t_track(const double *ps, const double *ks, const double *kc, int n_img, int P, const int *sid,
                        unsigned char *state, int n_streams, int max_tracks, long long max_age, double min_similarity,
                        double min_part_score, long long *ids) {
    std::vector<Track> tr(max_tracks + P), out(max_tracks);
    std::vector<Box> box(P);
    std::vector<unsigned char> det(P), taken(max_tracks);
    for (int r = 0; r < n_img; ++r) {
        const int s = sid[r];
        if (s < 0 || s >= n_streams) {
            for (int p = 0; p < P; ++p) ids[(long long)r * P + p] = -1;
            continue;
        }
        unsigned char *g = state + s * stream_bytes(max_tracks);
        Head h;
        memcpy(&h, g, sizeof(Head));
        memcpy(tr.data(), g + sizeof(Head), sizeof(Track) * h.n);
        frame_boxes(SerialTeam(), box.data(), det.data(), 0, P, ps + (long long)r * P, ks + (long long)r * P * KP,
                    kc + (long long)r * P * KP * 2, min_part_score);
        track_frame(SerialTeam(), h, tr.data(), box.data(), det.data(), taken.data(), out.data(), P, max_tracks, max_age,
                    min_similarity, (int64_t *)ids + (long long)r * P);
        memcpy(g, &h, sizeof(Head));
        memcpy(g + sizeof(Head), tr.data(), sizeof(Track) * h.n);
    }
}
"""


@pytest.fixture(scope="module")
def lib(tmp_path_factory):
    d = tmp_path_factory.mktemp("track")
    src, so = d / "track_shim.cu", d / "libtrack_shim.so"
    src.write_text(SHIM)
    cmd = [NVCC, "-O2", "-std=c++17", "-shared", "-Xcompiler", "-fPIC", "-gencode", "arch=compute_100a,code=sm_100a",
           "-I", CSRC, str(src), "-o", str(so)]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    L = C.CDLL(str(so))
    L.t_track.argtypes = [C.c_void_p] * 3 + [C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_longlong,
                                             C.c_double, C.c_double, C.c_void_p]
    L.t_track.restype = None
    return L


STREAM_HEAD, TRACK = 32, 48


class HostTracker:
    """The header on the host, over a state buffer of the kernel's layout."""

    def __init__(self, L, n_streams, max_tracks=18, max_age=30, min_similarity=0.15, min_part_score=0.5):
        self.L, self.n_streams, self.max_tracks, self.max_age = L, n_streams, max_tracks, max_age
        self.min_similarity, self.min_part_score = min_similarity, min_part_score
        self.sb = STREAM_HEAD + TRACK * max_tracks
        self.state = np.zeros(n_streams * self.sb, np.uint8)

    def batch(self, ps, ks, kc, sid):
        ps, ks, kc = (np.ascontiguousarray(a, np.float64) for a in (ps, ks, kc))
        sid = np.ascontiguousarray(sid, np.int32)
        n, P = ps.shape
        ids = np.empty((n, P), np.int64)
        self.L.t_track(ps.ctypes.data, ks.ctypes.data, kc.ctypes.data, n, P, sid.ctypes.data, self.state.ctypes.data,
                       self.n_streams, self.max_tracks, self.max_age, self.min_similarity, self.min_part_score, ids.ctypes.data)
        return ids

    def tracks(self, s):
        g = self.state[s * self.sb:(s + 1) * self.sb]
        frame, issued = (int(v) for v in g[:16].view(np.int64))
        n = int(g[16:20].view(np.int32)[0])
        tr = g[STREAM_HEAD:STREAM_HEAD + TRACK * n].view(np.int64).reshape(n, 6)
        return frame, issued, [(int(t[4]), int(t[5])) for t in tr]


def run_both(L, batches, n_streams, **kw):
    host, ref = HostTracker(L, n_streams, **kw), Oracle(n_streams, **kw)
    n_rows = 0
    for ps, ks, kc, sid in batches:
        got, want = host.batch(ps, ks, kc, sid), ref.batch(ps, ks, kc, sid)
        assert np.array_equal(got, want), (n_rows, np.argwhere(got != want)[:5])
        for s in set(int(v) for v in sid if v >= 0):
            assert host.tracks(s) == ref.tracks(s), (n_rows, s)
        n_rows += len(sid)
    return ref


@pytest.mark.parametrize("seed,n_streams,n_people,max_tracks,max_age,P,batch_max", [
    (0, 1, 6, 18, 30, 10, 1),          # one stream, one frame a batch
    (1, 3, 8, 18, 5, 10, 16),          # short ages: people come back after more and fewer than max_age frames
    (2, 4, 12, 4, 8, 10, 32),          # more people than max_tracks
    (3, 2, 30, 18, 30, 50, 64),        # P = 50, crowded
    (4, 5, 5, 3, 0, 6, 7),             # max_age 0: a track lives one frame unless matched in the next
])
def test_sequences_match_the_oracle(lib, seed, n_streams, n_people, max_tracks, max_age, P, batch_max):
    rng = np.random.default_rng(seed)
    recs = [synth_stream(rng, 160, n_people, P, max(max_age, 2)) for _ in range(n_streams)]
    ref = run_both(lib, interleave(rng, recs, batch_max, untracked=0.08), n_streams, max_tracks=max_tracks, max_age=max_age)
    issued = sum(ref.tracks(s)[1] for s in range(n_streams))
    assert issued > n_people * n_streams, "the sequences should end tracks and start new ones"


def test_ids_follow_people_who_move():
    """The oracle itself on a clean scene: two people who move keep their ids; one who is away for max_age - 1 frames keeps
    its id (t - last = max_age), one away for max_age frames comes back with a new one."""
    ref = Oracle(1, max_age=3)

    def frame(boxes):
        ps = np.zeros(4)
        ks = np.ones((4, 17))
        kc = np.zeros((4, 17, 2))
        for p, (y0, x0, y1, x1) in enumerate(boxes):
            ps[p] = 0.9
            kc[p, :, 0] = np.linspace(y0, y1, 17)
            kc[p, :, 1] = np.linspace(x0, x1, 17)
        return ref.frame(0, ps, ks, kc)[:len(boxes)].tolist()

    assert frame([(0, 0, 10, 10), (0, 50, 10, 60)]) == [1, 2]
    assert frame([(0, 52, 10, 62), (1, 1, 11, 11)]) == [2, 1]
    for _ in range(2):
        assert frame([(1, 1, 11, 11)]) == [1]
    assert frame([(0, 52, 10, 62), (1, 1, 11, 11)]) == [2, 1]
    for _ in range(3):
        assert frame([(1, 1, 11, 11)]) == [1]
    assert frame([(0, 52, 10, 62), (1, 1, 11, 11)]) == [3, 1]


def record(boxes, P=None, scores=None):
    """One frame whose detections have exactly the given boxes (first and last keypoint on the corners)."""
    P = P or len(boxes)
    ps, ks, kc = np.zeros(P), np.zeros((P, 17)), np.zeros((P, 17, 2))
    for p, b in enumerate(boxes):
        ps[p] = 0.9
        ks[p] = 0.9 if scores is None else scores[p]
        kc[p, :, 0] = b[0]
        kc[p, :, 1] = b[1]
        kc[p, -1] = b[2], b[3]
    return ps, ks, kc


def test_exact_ties_and_the_similarity_threshold(lib):
    # frame 1: tracks 1, 2 with the same box; frame 2: one detection equally close to both takes the first track in order
    host = HostTracker(lib, 1)
    for boxes, want in (([(0, 0, 4, 4), (0, 0, 4, 4)], [1, 2]), ([(0, 0, 4, 2)], [1]), ([(0, 0, 4, 4), (0, 0, 4, 4)], [2, 1])):
        ps, ks, kc = record(boxes)
        assert host.batch(ps[None], ks[None], kc[None], [0])[0].tolist() == want
    # IoU exactly at min_similarity matches; the next double above it does not
    for ms, want in ((0.5, [1, 1]), (np.nextafter(0.5, 1), [1, 2])):
        host, ref = HostTracker(lib, 1, min_similarity=ms), Oracle(1, min_similarity=ms)
        got = []
        for b in ((0, 0, 2, 2), (0, 0, 2, 1)):                  # IoU 2 / 4
            ps, ks, kc = record([b])
            got.append(int(host.batch(ps[None], ks[None], kc[None], [0])[0, 0]))
            assert ref.frame(0, ps, ks, kc)[0] == got[-1]
        assert got == want
    # the larger IoU wins over the earlier track, and a matched track is not offered to the next detection
    host = HostTracker(lib, 1)
    ps, ks, kc = record([(0, 0, 4, 4), (0, 2, 4, 6)])
    assert host.batch(ps[None], ks[None], kc[None], [0])[0].tolist() == [1, 2]
    ps, ks, kc = record([(0, 2, 4, 6), (0, 2, 4, 6)])
    assert host.batch(ps[None], ks[None], kc[None], [0])[0].tolist() == [2, 1]


@pytest.mark.parametrize("min_similarity", [0.15, 0.0])
def test_empty_and_zero_area_boxes(lib, min_similarity):
    """All keypoints below min_part_score (empty box) and a single keypoint (zero area): IoU 0 with everything, so they
    never match at min_similarity > 0 and take any unmatched track at 0."""
    low = np.full(17, 0.1)
    one = low.copy()
    one[0] = 0.5
    host, ref = HostTracker(lib, 1, min_similarity=min_similarity), Oracle(1, min_similarity=min_similarity)
    seen = set()
    for t in range(6):
        ps, ks, kc = record([(0, 0, 10, 10), (0, 0, 10, 10), (5, 5, 30, 30)], P=5, scores=[low, one, np.full(17, 0.9)])
        got = host.batch(ps[None], ks[None], kc[None], [0])[0]
        assert got.tolist() == ref.frame(0, ps, ks, kc).tolist()
        assert got[3:].tolist() == [-1, -1]
        if min_similarity == 0:
            assert got[:3].tolist() == [1, 2, 3]
        elif t:
            assert got[2] == 3 and not {int(got[0]), int(got[1])} & seen
        seen |= set(got[:3].tolist())
    assert host.tracks(0) == ref.tracks(0)


def test_untracked_rows_and_one_stream_twice_in_a_batch(lib):
    rng = np.random.default_rng(7)
    recs = [synth_stream(rng, 12, 4, 10, 5) for _ in range(3)]
    # stream 1 on every other row, streams 0 and 2 interleaved, -1 rows between
    order = [(1, 0), (0, 0), (-1, 0), (1, 1), (2, 0), (1, 2), (0, 1), (-1, 0), (2, 1), (1, 3)]
    ps = np.stack([recs[s][0][f] if s >= 0 else np.ones(10) for s, f in order])
    ks = np.stack([recs[s][1][f] if s >= 0 else np.ones((10, 17)) for s, f in order])
    kc = np.stack([recs[s][2][f] if s >= 0 else np.ones((10, 17, 2)) for s, f in order])
    sid = [s for s, _ in order]
    host, ref = HostTracker(lib, 3, max_age=5), Oracle(3, max_age=5)
    got = host.batch(ps, ks, kc, sid)
    assert np.array_equal(got, ref.batch(ps, ks, kc, sid))
    assert (got[[2, 7]] == -1).all()
    # the same frames one at a time give the same ids: rows of a stream are its frames in row order
    host2 = HostTracker(lib, 3, max_age=5)
    one_by_one = np.concatenate([host2.batch(ps[r:r + 1], ks[r:r + 1], kc[r:r + 1], sid[r:r + 1]) for r in range(len(sid))])
    assert np.array_equal(got, one_by_one)


def test_abi_argument_errors():
    lib = nat.load()
    size = C.c_size_t()
    assert lib.pn_track_state_bytes(3, 18, C.byref(size)) == 0 and size.value == 3 * (32 + 48 * 18)
    for n_streams, max_tracks in ((0, 18), (3, 0), (3, 257), (1 << 21, 18)):
        assert lib.pn_track_state_bytes(n_streams, max_tracks, C.byref(size)) == -1
    assert lib.pn_track_state_bytes(1, 1, None) == -1
    A = 1 << 20                                              # aligned fake device pointers: the checks run before any launch
    good = dict(ps=A, ks=A, kc=A, n=4, P=10, sid=A, state=A, ns=2, mt=18, ma=30, msim=0.15, mps=0.5, ids=A)

    def call(**over):
        a = dict(good, **over)
        return lib.pn_track_poses(a["ps"], a["ks"], a["kc"], a["n"], a["P"], a["sid"], a["state"], a["ns"], a["mt"], a["ma"],
                                  a["msim"], a["mps"], a["ids"], None)

    bad = [dict(ps=None), dict(ks=None), dict(kc=None), dict(sid=None), dict(state=None), dict(ids=None), dict(ps=A + 4),
           dict(state=A + 4), dict(ids=A + 2), dict(sid=A + 2), dict(n=0), dict(P=0), dict(P=257), dict(ns=0),
           dict(ns=(1 << 20) + 1), dict(mt=0), dict(mt=257), dict(ma=-1), dict(msim=float("nan")), dict(mps=float("nan"))]
    for over in bad:
        assert call(**over) == -1, over
        assert lib.pn_last_error_string().startswith(b"pn_track_poses")


def test_tracker_arguments_are_checked_before_the_device():
    import posenet
    for kw in (dict(n_streams=0), dict(n_streams=2.0), dict(n_streams=1, max_tracks=0), dict(n_streams=1, max_tracks=257),
               dict(n_streams=1, max_age=-1), dict(n_streams=1, min_similarity=float("nan")),
               dict(n_streams=1, min_part_score=float("nan")), dict(n_streams=True)):
        with pytest.raises(ValueError):
            posenet.PoseTracker(**kw)
