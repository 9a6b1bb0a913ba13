"""numpy restatement of the One Euro keypoint smoothing (posenet.track, csrc/smooth.cuh), for its tests.

The oracle follows the smoothing semantics of posenet/track.py's docstring step by step, with Python floats (IEEE float64, no
FMA).  The ids it smooths come from the tracker's oracle (trackref.Oracle) or are given directly."""
import math

import numpy as np

from trackref import Oracle

NC = 34
TWO_PI = 2 * math.pi


class SmoothOracle:
    def __init__(self, n_streams, max_tracks=18, max_age=30, fps=30.0, min_cutoff=1.0, beta=0.0, d_cutoff=1.0):
        self.n_streams, self.max_tracks, self.max_age = n_streams, max_tracks, max_age
        self.fps, self.min_cutoff, self.beta, self.d_cutoff = float(fps), float(min_cutoff), float(beta), float(d_cutoff)
        self.events = dict(fresh=0, update=0, gap=0, evict=0, evict_tie=0, full=0, expire=0)   # what the sequences covered
        self.reset()

    def reset(self, stream=None):
        fresh = lambda: dict(frame=0, table=[])
        if stream is None:
            self.streams = [fresh() for _ in range(self.n_streams)]
        else:
            self.streams[stream] = fresh()

    def filter(self, e, dt, c, x):
        rate = self.fps / float(dt)
        dx = (x - e["x_prev"][c]) * rate
        a_d = 1.0 / (1.0 + rate / (TWO_PI * self.d_cutoff))
        dx_hat = a_d * dx + (1.0 - a_d) * e["dx_hat"][c]
        cutoff = self.min_cutoff + self.beta * abs(dx_hat)
        a = 1.0 / (1.0 + rate / (TWO_PI * cutoff))
        x_hat = a * x + (1.0 - a) * e["x_hat"][c]
        e["x_prev"][c], e["x_hat"][c], e["dx_hat"][c] = x, x_hat, dx_hat
        return x_hat

    def frame(self, s, ids, kc):
        """One frame of stream s: ids [P], kc [P, 17, 2] -> smoothed kc (a new array)."""
        st = self.streams[s]
        st["frame"] += 1
        t = st["frame"]
        kept = [e for e in st["table"] if not t - e["last"] > self.max_age]
        self.events["expire"] += len(st["table"]) - len(kept)
        table = st["table"] = kept
        out = np.array(kc, np.float64).reshape(len(ids), NC)
        for p in range(len(ids)):
            pid = int(ids[p])
            if not pid >= 1:
                continue
            e = next((e for e in table if e["id"] == pid), None)
            if e is not None:
                if e["last"] == t:                  # the id twice in one frame
                    continue
                dt = t - e["last"]
                e["last"] = t
                self.events["update"] += 1
                self.events["gap"] += dt > 1
                for c in range(NC):
                    out[p, c] = self.filter(e, dt, c, float(out[p, c]))
                continue
            fresh = dict(id=pid, last=t, x_prev=[float(v) for v in out[p]], x_hat=[float(v) for v in out[p]], dx_hat=[0.0] * NC)
            if len(table) < self.max_tracks:
                table.append(fresh)
                self.events["fresh"] += 1
                continue
            old = [i for i, e in enumerate(table) if e["last"] < t]
            if not old:
                self.events["full"] += 1
                continue
            lo = min(table[i]["last"] for i in old)
            i = next(i for i in old if table[i]["last"] == lo)
            self.events["evict"] += 1
            self.events["evict_tie"] += sum(table[j]["last"] == lo for j in old) > 1
            table[i] = fresh
        return out.reshape(np.shape(kc))

    def batch(self, ids, kc, streams):
        """Rows in order; rows of a stream outside 0..n_streams-1 are left as they are."""
        out = np.array(kc, np.float64)
        for r, s in enumerate(streams):
            if 0 <= s < self.n_streams:
                out[r] = self.frame(int(s), ids[r], kc[r])
        return out

    def table(self, s):
        """(frame, [(id, last, x_prev, x_hat, dx_hat), ...]) of stream s, the three values as float64 [34] arrays."""
        st = self.streams[s]
        return st["frame"], [(e["id"], e["last"], np.array(e["x_prev"]), np.array(e["x_hat"]), np.array(e["dx_hat"]))
                             for e in st["table"]]


class TrackSmoothOracle:
    """The tracker's oracle followed by the smoothing oracle, as PoseTracker(smoothing=...).update runs them."""

    def __init__(self, n_streams, max_tracks=18, max_age=30, min_similarity=0.15, min_part_score=0.5, smoothing=(30.0, 1.0, 0.0, 1.0)):
        self.track = Oracle(n_streams, max_tracks, max_age, min_similarity, min_part_score)
        self.smooth = SmoothOracle(n_streams, max_tracks, max_age, *smoothing)

    def reset(self, stream=None):
        self.track.reset(stream)
        self.smooth.reset(stream)

    def batch(self, ps, ks, kc, streams):
        ids = self.track.batch(ps, ks, kc, streams)
        return ids, self.smooth.batch(ids, kc, streams)
