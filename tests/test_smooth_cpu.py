"""One Euro keypoint smoothing (csrc/smooth.cuh) against the numpy oracle of tests/smoothref.py, on the host.

The header is compiled into a small host library that runs smooth_frame with one "lane" per stream over the state layout the
kernel keeps, row by row as pn_smooth_keypoints does.  Seeded sequences are compared bit for bit, batch by batch: the smoothed
coordinates and each stream's frame counter and filter table (ids, last, and the three float64 values of every coordinate).
Covered: interleaved streams with untracked rows and one stream several times in a batch, gaps of several frames, max_age 0,
more ids than max_tracks (eviction, ties on last, records that keep their coordinates because every entry was updated),
reset of one stream and extreme parameters.  Two properties show the filter does its job: it removes most of a still person's
jitter, and beta > 0 shortens the lag behind a moving one.  The argument checks of pn_smooth_keypoints /
pn_smooth_state_bytes, OneEuro and PoseTracker(smoothing=) run before any device is touched.  The kernel's split of the work
over threads is covered by tests/test_gpu_smooth.py."""
import ctypes as C
import math
import os
import subprocess

import numpy as np
import pytest

from posenet import _native as nat
from smoothref import NC, SmoothOracle, TrackSmoothOracle
from trackref import Oracle, interleave, synth_stream

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "posenet-pytorch_b200", "csrc")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")

SHIM = r"""
#include <vector>
#include "smooth.cuh"
using namespace pn::smooth;
extern "C" void t_smooth(const long long *ids, double *kc, int n_img, int P, const int *sid, unsigned char *state, int n_streams,
                         int max_tracks, long long max_age, double fps, double min_cutoff, double beta, double d_cutoff) {
    std::vector<Job> job(P);
    const Params q = {fps, min_cutoff, beta, d_cutoff};
    for (int r = 0; r < n_img; ++r) {
        const int s = sid[r];
        if (s < 0 || s >= n_streams) continue;
        unsigned char *g = state + s * stream_bytes(max_tracks);
        int n_jobs = 0;
        smooth_frame(pn::track::SerialTeam(), *(Head *)g, (Entry *)(g + sizeof(Head)), (Values *)(g + table_bytes(max_tracks)),
                     job.data(), n_jobs, (const int64_t *)ids + (long long)r * P, kc + (long long)r * P * NC, P, max_tracks,
                     max_age, q);
    }
}
"""


@pytest.fixture(scope="module")
def lib(tmp_path_factory):
    d = tmp_path_factory.mktemp("smooth")
    src, so = d / "smooth_shim.cu", d / "libsmooth_shim.so"
    src.write_text(SHIM)
    cmd = [NVCC, "-O2", "-std=c++17", "-shared", "-Xcompiler", "-fPIC,-ffp-contract=off", "-gencode",
           "arch=compute_100a,code=sm_100a", "-I", CSRC, str(src), "-o", str(so)]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    L = C.CDLL(str(so))
    L.t_smooth.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_longlong,
                           C.c_double, C.c_double, C.c_double, C.c_double]
    L.t_smooth.restype = None
    return L


HEAD, ENTRY, VALUES = 16, 16, 3 * NC * 8


class HostSmoother:
    """The header on the host, over a state buffer of the kernel's layout."""

    def __init__(self, L, n_streams, max_tracks=18, max_age=30, fps=30.0, min_cutoff=1.0, beta=0.0, d_cutoff=1.0):
        self.L, self.n_streams, self.max_tracks, self.max_age = L, n_streams, max_tracks, max_age
        self.q = (fps, min_cutoff, beta, d_cutoff)
        self.sb = HEAD + (ENTRY + VALUES) * max_tracks
        self.state = np.zeros(n_streams * self.sb, np.uint8)

    def batch(self, ids, kc, sid):
        ids = np.ascontiguousarray(ids, np.int64)
        out = np.array(kc, np.float64, order="C")
        sid = np.ascontiguousarray(sid, np.int32)
        n, P = ids.shape
        self.L.t_smooth(ids.ctypes.data, out.ctypes.data, n, P, sid.ctypes.data, self.state.ctypes.data, self.n_streams,
                        self.max_tracks, self.max_age, *self.q)
        return out

    def reset(self, s):
        self.state[s * self.sb:(s + 1) * self.sb] = 0

    def table(self, s):
        g = self.state[s * self.sb:(s + 1) * self.sb]
        frame = int(g[:8].view(np.int64)[0])
        n = int(g[8:12].view(np.int32)[0])
        tab = g[HEAD:HEAD + ENTRY * n].view(np.int64).reshape(n, 2)
        val = g[HEAD + ENTRY * self.max_tracks:].view(np.float64).reshape(self.max_tracks, 3, NC)
        return frame, [(int(tab[i, 0]), int(tab[i, 1]), val[i, 0], val[i, 1], val[i, 2]) for i in range(n)]


def same_table(a, b):
    return a[0] == b[0] and len(a[1]) == len(b[1]) and all(
        x[:2] == y[:2] and all(np.array_equal(u, v) for u, v in zip(x[2:], y[2:])) for x, y in zip(a[1], b[1]))


def bits_equal(a, b):
    return np.array_equal(np.asarray(a).view(np.int64), np.asarray(b).view(np.int64))


def run_both(L, batches, n_streams, **kw):
    """batches of (ids, kc, sid); returns the smoothing oracle."""
    host, ref = HostSmoother(L, n_streams, **kw), SmoothOracle(n_streams, **kw)
    n_rows = 0
    for ids, kc, sid in batches:
        got, want = host.batch(ids, kc, sid), ref.batch(ids, kc, sid)
        assert bits_equal(got, want), (n_rows, np.argwhere(got != want)[:5])
        for s in set(int(v) for v in sid if 0 <= v < n_streams):
            assert same_table(host.table(s), ref.table(s)), (n_rows, s)
        n_rows += len(sid)
    return ref


def tracked(rng, n_streams, n_frames, n_people, P, max_tracks, max_age, batch_max, untracked=0.08, **synth):
    """Interleaved batches of synthetic streams with the tracker oracle's ids: (ids, kc, sid)."""
    recs = [synth_stream(rng, n_frames, n_people, P, max(max_age, 2), **synth) for _ in range(n_streams)]
    tr = Oracle(n_streams, max_tracks=max_tracks, max_age=max_age)
    for ps, ks, kc, sid in interleave(rng, recs, batch_max, untracked=untracked):
        yield tr.batch(ps, ks, kc, sid), kc, sid


@pytest.mark.parametrize("seed,n_streams,n_people,max_tracks,max_age,P,batch_max", [
    (0, 1, 6, 18, 30, 10, 1),          # one stream, one frame a batch
    (1, 3, 8, 18, 5, 10, 16),          # short ages: people come back after more and fewer than max_age frames
    (2, 4, 12, 4, 8, 10, 32),          # more people than max_tracks
    (3, 2, 30, 18, 30, 50, 64),        # P = 50, crowded
    (4, 5, 5, 3, 0, 6, 7),             # max_age 0: a filter lives one frame unless updated in the next
])
def test_tracked_sequences_match_the_oracle(lib, seed, n_streams, n_people, max_tracks, max_age, P, batch_max):
    rng = np.random.default_rng(seed)
    ref = run_both(lib, tracked(rng, n_streams, 160, n_people, P, max_tracks, max_age, batch_max), n_streams,
                   max_tracks=max_tracks, max_age=max_age)
    ev = ref.events
    assert ev["fresh"] > n_people and ev["expire"] + ev["evict"] > 0, ev
    if max_age == 0:                                                # every entry expires before the next frame
        assert ev["update"] == 0 and ev["expire"] > 0, ev
    else:
        assert ev["update"] > ev["fresh"] and ev["gap"] > 0, ev    # gap: an update after frames without the id (rate < fps)


def test_untracked_rows_and_one_stream_twice_in_a_batch(lib):
    rng = np.random.default_rng(7)
    recs = [synth_stream(rng, 12, 4, 10, 5) for _ in range(3)]
    order = [(1, 0), (0, 0), (-1, 0), (1, 1), (2, 0), (1, 2), (0, 1), (-1, 0), (2, 1), (1, 3)]
    ps = np.stack([recs[s][0][f] if s >= 0 else np.ones(10) for s, f in order])
    ks = np.stack([recs[s][1][f] if s >= 0 else np.ones((10, 17)) for s, f in order])
    kc = np.stack([recs[s][2][f] if s >= 0 else rng.uniform(0, 400, (10, 17, 2)) for s, f in order])
    sid = np.array([s for s, _ in order])
    ids = Oracle(3, max_age=5).batch(ps, ks, kc, sid)
    ids[2] = 1                                                      # untracked rows are left as they are, whatever their ids
    sid[7] = 3                                                      # a stream id out of range is untracked too
    host, ref = HostSmoother(lib, 3, max_age=5), SmoothOracle(3, max_age=5)
    got = host.batch(ids, kc, sid)
    assert bits_equal(got, ref.batch(ids, kc, sid))
    assert bits_equal(got[[2, 7]], kc[[2, 7]]) and not np.array_equal(got, kc)
    # the same frames one at a time give the same coordinates: rows of a stream are its frames in row order
    host2 = HostSmoother(lib, 3, max_age=5)
    one_by_one = np.concatenate([host2.batch(ids[r:r + 1], kc[r:r + 1], sid[r:r + 1]) for r in range(len(sid))])
    assert bits_equal(got, one_by_one)


def test_more_ids_than_max_tracks(lib):
    """Ids drawn directly (not from the tracker), up to 9 a frame for 3 entries: eviction of the oldest entry, ties on last,
    records that keep their coordinates because every entry was updated in the frame, ids that come back after eviction,
    an id twice in one frame, and non-detection ids (0, -1) among them."""
    rng = np.random.default_rng(21)
    P, n = 9, 400

    def batches():
        for _ in range(n // 8):
            ids = np.full((8, P), -1, np.int64)
            for r in range(8):
                k = int(rng.integers(0, P + 1))
                ids[r, :k] = rng.choice(np.arange(1, 13), k, replace=False)
                if rng.random() < 0.1:
                    ids[r, int(rng.integers(P))] = 0
                if k > 1 and rng.random() < 0.05:
                    ids[r, k - 1] = ids[r, 0]
            yield ids, rng.normal(200, 50, (8, P, 17, 2)), rng.integers(0, 2, 8)

    ref = run_both(lib, batches(), 2, max_tracks=3, max_age=4)
    ev = ref.events
    assert ev["evict"] > 50 and ev["evict_tie"] > 10 and ev["full"] > 50 and ev["gap"] > 0, ev


def test_reset_of_one_stream(lib):
    rng = np.random.default_rng(3)
    batches = list(tracked(rng, 3, 60, 5, 10, 18, 10, 12, untracked=0.0))
    host, ref = HostSmoother(lib, 3, max_age=10), SmoothOracle(3, max_age=10)
    tr_ref = None
    for i, (ids, kc, sid) in enumerate(batches):
        if i == len(batches) // 2:
            host.reset(1)
            ref.reset(1)
            tr_ref = ref.table(0)
            assert host.table(1) == (0, [])
        assert bits_equal(host.batch(ids, kc, sid), ref.batch(ids, kc, sid)), i
    for s in range(3):
        assert same_table(host.table(s), ref.table(s))
    assert tr_ref is not None and ref.table(1)[0] < ref.table(0)[0]


@pytest.mark.parametrize("fps,min_cutoff,beta,d_cutoff", [
    (30.0, 1.0, 1e3, 1.0),             # large beta: the cutoff follows every movement
    (30.0, 1e-6, 0.0, 1.0),            # tiny min_cutoff: a nearly frozen filter
    (1.0, 0.5, 0.3, 3.0),              # 1 fps
    (240.0, 2.0, 0.007, 0.25),         # 240 fps
    (59.94, 1.7, 0.02, 1e-3),
])
def test_extreme_parameters(lib, fps, min_cutoff, beta, d_cutoff):
    rng = np.random.default_rng(int(fps * 100) + int(beta * 10))
    q = dict(fps=fps, min_cutoff=min_cutoff, beta=beta, d_cutoff=d_cutoff)
    run_both(lib, tracked(rng, 2, 80, 5, 10, 18, 6, 9), 2, max_tracks=18, max_age=6, **q)


def still_and_moving(v, n=240, sigma=3.0, seed=0):
    """n frames of one person (id 1) at a fixed or constant-speed position (v px / frame), with Gaussian keypoint jitter."""
    rng = np.random.default_rng(seed)
    base = rng.uniform(100, 300, (17, 2))
    truth = base[None] + v * np.arange(n)[:, None, None, None]
    return truth, truth + rng.normal(0, sigma, truth.shape)


def smooth_one(kc, **q):
    ref = SmoothOracle(1, **q)
    ids = np.ones((len(kc), 1), np.int64)
    return ref.batch(ids, kc[:, None], np.zeros(len(kc), int))[:, 0]


def test_a_still_person_jitters_less():
    truth, raw = still_and_moving(0.0)
    smoothed = smooth_one(raw)
    rms = lambda a: float(np.sqrt(np.mean((a[30:] - truth[30:]) ** 2)))
    assert rms(smoothed) < 0.5 * rms(raw), (rms(smoothed), rms(raw))


def test_beta_shortens_the_lag_of_a_moving_person():
    truth, _ = still_and_moving(np.array([2.0, 5.0]), sigma=0.0)
    lag = {beta: float(np.mean(np.abs(smooth_one(truth, beta=beta)[-60:] - truth[-60:]))) for beta in (0.0, 0.05)}
    assert lag[0.05] < 0.5 * lag[0.0], lag
    assert lag[0.0] > 10.0                                          # the still-person setting trails by ~5 frames


def test_the_oracle_follows_the_formulas():
    """The oracle's first update against the formulas written out once more, and a fresh entry's pass-through."""
    q = dict(fps=25.0, min_cutoff=0.7, beta=0.01, d_cutoff=1.3)
    ref = SmoothOracle(1, **q)
    x0, x1 = 10.0, 13.5
    kc = np.zeros((2, 1, 17, 2))
    kc[0], kc[1] = x0, x1
    out = ref.batch(np.ones((2, 1), np.int64), kc, [0, 0])
    assert (out[0] == x0).all()
    rate = 25.0
    dx = (x1 - x0) * rate
    a_d = 1 / (1 + rate / (2 * math.pi * 1.3))
    dx_hat = a_d * dx
    a = 1 / (1 + rate / (2 * math.pi * (0.7 + 0.01 * abs(dx_hat))))
    assert (out[1] == a * x1 + (1 - a) * x0).all()


def test_abi_argument_errors():
    lib = nat.load()
    size = C.c_size_t()
    assert lib.pn_smooth_state_bytes(3, 18, C.byref(size)) == 0 and size.value == 3 * (HEAD + (ENTRY + VALUES) * 18)
    for n_streams, max_tracks in ((0, 18), (3, 0), (3, 257), (1 << 21, 18)):
        assert lib.pn_smooth_state_bytes(n_streams, max_tracks, C.byref(size)) == -1
    assert lib.pn_smooth_state_bytes(1, 1, None) == -1
    A = 1 << 20                                              # aligned fake device pointers: the checks run before any launch
    good = dict(ids=A, kc=A, n=4, P=10, sid=A, state=A, ns=2, mt=18, ma=30, fps=30.0, mc=1.0, beta=0.0, dc=1.0)

    def call(**over):
        a = dict(good, **over)
        return lib.pn_smooth_keypoints(a["ids"], a["kc"], a["n"], a["P"], a["sid"], a["state"], a["ns"], a["mt"], a["ma"],
                                       a["fps"], a["mc"], a["beta"], a["dc"], None)

    inf, nan = float("inf"), float("nan")
    bad = [dict(ids=None), dict(kc=None), dict(sid=None), dict(state=None), dict(ids=A + 4), dict(kc=A + 4), dict(state=A + 2),
           dict(sid=A + 2), dict(n=0), dict(P=0), dict(P=257), dict(ns=0), dict(ns=(1 << 20) + 1), dict(mt=0), dict(mt=257),
           dict(ma=-1), dict(fps=0.0), dict(fps=-30.0), dict(fps=inf), dict(fps=nan), dict(mc=0.0), dict(mc=inf), dict(mc=nan),
           dict(dc=0.0), dict(dc=-1.0), dict(dc=inf), dict(dc=nan), dict(beta=-1e-9), dict(beta=inf), dict(beta=nan)]
    for over in bad:
        assert call(**over) == -1, over
        assert lib.pn_last_error_string().startswith(b"pn_smooth_keypoints")


def test_one_euro_and_tracker_arguments_are_checked_before_the_device():
    import posenet
    from posenet import track
    assert posenet.OneEuro is track.OneEuro
    q = posenet.OneEuro()
    assert q == (30.0, 1.0, 0.0, 1.0) and (q.fps, q.min_cutoff, q.beta, q.d_cutoff) == (30.0, 1.0, 0.0, 1.0)
    assert posenet.OneEuro(60, beta=0, d_cutoff=2) == (60.0, 1.0, 0.0, 2.0)
    assert isinstance(hash(q), int)
    with pytest.raises(AttributeError):
        q.fps = 60.0
    for kw in (dict(fps=0), dict(fps=-1.0), dict(fps=float("inf")), dict(fps=float("nan")), dict(min_cutoff=0.0),
               dict(min_cutoff=float("inf")), dict(d_cutoff=0.0), dict(d_cutoff=float("nan")), dict(beta=-0.1),
               dict(beta=float("inf")), dict(beta=float("nan")), dict(fps="fast"), dict(fps=None), dict(beta=True)):
        with pytest.raises(ValueError):
            posenet.OneEuro(**kw)
    for smoothing in ((30.0, 1.0, 0.0, 1.0), dict(fps=30.0), 30.0, q._replace(fps=0.0)):
        with pytest.raises(ValueError):
            posenet.PoseTracker(1, smoothing=smoothing)


def test_track_smooth_oracle_keeps_the_tracker_ids():
    """Smoothing runs after the tracking: the ids are the tracker's, and scores are not inputs."""
    rng = np.random.default_rng(5)
    recs = [synth_stream(rng, 40, 5, 10, 8)]
    both, plain = TrackSmoothOracle(1, max_age=8), Oracle(1, max_age=8)
    for ps, ks, kc, sid in interleave(rng, recs, 8, untracked=0.0):
        ids, out = both.batch(ps, ks, kc, sid)
        assert np.array_equal(ids, plain.batch(ps, ks, kc, sid))
        assert bits_equal(out[ids < 1], kc[ids < 1])
