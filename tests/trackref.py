"""numpy restatement of the pose tracker (posenet.track, csrc/track.cuh) and seeded synthetic pose sequences for its tests.

The oracle follows the semantics of posenet/track.py's docstring step by step, with Python floats (IEEE float64, no FMA)."""
import numpy as np

K = 17


def box_of(ks, kc, min_part_score):
    """(ymin, xmin, ymax, xmax) over the keypoints with score >= min_part_score, or None."""
    m = ks >= min_part_score
    if not m.any():
        return None
    y, x = kc[m, 0], kc[m, 1]
    return float(y.min()), float(x.min()), float(y.max()), float(x.max())


def iou(a, b):
    if a is None or b is None:
        return 0.0
    iy = min(a[2], b[2]) - max(a[0], b[0])
    ix = min(a[3], b[3]) - max(a[1], b[1])
    if iy <= 0 or ix <= 0:
        return 0.0
    inter = iy * ix
    union = (a[2] - a[0]) * (a[3] - a[1]) + (b[2] - b[0]) * (b[3] - b[1]) - inter
    return 0.0 if union <= 0 else inter / union


class Oracle:
    def __init__(self, n_streams, max_tracks=18, max_age=30, min_similarity=0.15, min_part_score=0.5):
        self.n_streams, self.max_tracks, self.max_age = n_streams, max_tracks, max_age
        self.min_similarity, self.min_part_score = min_similarity, min_part_score
        self.reset()

    def reset(self, stream=None):
        fresh = lambda: dict(frame=0, next_id=1, tracks=[])
        if stream is None:
            self.streams = [fresh() for _ in range(self.n_streams)]
        else:
            self.streams[stream] = fresh()

    def frame(self, s, ps, ks, kc):
        """One frame of stream s: ps [P], ks [P, 17], kc [P, 17, 2] -> ids [P]."""
        st = self.streams[s]
        st["frame"] += 1
        t = st["frame"]
        tracks = [tr for tr in st["tracks"] if not t - tr["last"] > self.max_age]
        n_old = len(tracks)
        taken = [False] * n_old
        ids = np.full(len(ps), -1, np.int64)
        for p in range(len(ps)):
            if not ps[p] > 0:
                continue
            b = box_of(ks[p], kc[p], self.min_part_score)
            best, bj = 0.0, -1
            for j in range(n_old):
                if taken[j]:
                    continue
                v = iou(b, tracks[j]["box"])
                if v >= self.min_similarity and (bj < 0 or v > best):
                    best, bj = v, j
            if bj >= 0:
                taken[bj] = True
                tracks[bj]["box"], tracks[bj]["last"] = b, t
                ids[p] = tracks[bj]["id"]
            else:
                tracks.append(dict(id=st["next_id"], box=b, last=t))
                ids[p] = st["next_id"]
                st["next_id"] += 1
        tracks.sort(key=lambda tr: -tr["last"])              # stable
        st["tracks"] = tracks[:self.max_tracks]
        return ids

    def batch(self, ps, ks, kc, streams):
        """Rows in order; rows of stream -1 get -1 ids."""
        ids = np.full(ps.shape, -1, np.int64)
        for r, s in enumerate(streams):
            if 0 <= s < self.n_streams:
                ids[r] = self.frame(int(s), ps[r], ks[r], kc[r])
        return ids

    def tracks(self, s):
        """(frame, ids issued, [(id, last), ...]) of stream s."""
        st = self.streams[s]
        return st["frame"], st["next_id"] - 1, [(tr["id"], tr["last"]) for tr in st["tracks"]]


def synth_stream(rng, n_frames, n_people, P, max_age, min_part_score=0.5, size=400.0, quant=0.25):
    """Records of one stream of n_frames frames: people who move, enter, leave and come back after gaps around max_age.
    Returns ps [n, P], ks [n, P, 17], kc [n, P, 17, 2] float64, in the decoder's layout (detections first, zero rows after)
    except for an occasional zero-score row among the detections."""
    ps = np.zeros((n_frames, P))
    ks = np.zeros((n_frames, P, K))
    kc = np.zeros((n_frames, P, K, 2))
    people = []
    for _ in range(n_people):
        vis = np.zeros(n_frames, bool)
        f = int(rng.integers(0, max(1, n_frames // 3)))
        while f < n_frames:
            on = int(rng.integers(3, 3 * max_age + 4))
            vis[f:f + on] = True
            f += on + int(rng.choice([rng.integers(1, max_age + 1), max_age, max_age + 1, rng.integers(max_age + 2, 2 * max_age + 3)]))
        people.append(dict(c=rng.uniform(0, size, 2), v=rng.uniform(-4, 4, 2), hw=rng.uniform(20, 150, 2), vis=vis,
                           kind=rng.choice(4, p=[0.85, 0.05, 0.05, 0.05])))
    q = lambda a: np.round(a / quant) * quant
    for t in range(n_frames):
        order = [i for i in rng.permutation(n_people) if people[i]["vis"][t]][:P]
        row = 0
        for i in order:
            pp = people[i]
            c = pp["c"] + t * pp["v"]
            if row < P - 1 and rng.random() < 0.03:
                kc[t, row] = q(rng.uniform(0, size, (K, 2)))     # a record that is not a detection (pose_score 0)
                ks[t, row] = rng.uniform(0, 1, K)
                row += 1
            ps[t, row] = rng.uniform(0.05, 1.0)
            kc[t, row] = q(c + (rng.uniform(0, 1, (K, 2)) - 0.5) * pp["hw"])
            sc = rng.uniform(0, 1, K)
            if pp["kind"] == 1:                                  # no keypoint above the threshold: an empty box
                sc = rng.uniform(0, min_part_score * 0.999, K)
            elif pp["kind"] == 2:                                # exactly one: a box of zero area
                sc = rng.uniform(0, min_part_score * 0.999, K)
                sc[rng.integers(K)] = min_part_score
            elif pp["kind"] == 3:                                # exact ties: all of its keypoints on its box's corners
                kc[t, row] = q(c + (rng.integers(0, 2, (K, 2)) - 0.5) * pp["hw"])
            ks[t, row] = sc
            row += 1
            if row == P:
                break
    return ps, ks, kc


def interleave(rng, streams_records, batch_max, untracked=0.05, min_batch=1):
    """Batches of rows from several streams' records, each stream's frames in order, streams mixed at random (a stream can
    appear several times in one batch), with some -1 rows of random records.  Yields (ps, ks, kc, stream_ids)."""
    labels = np.repeat(np.arange(len(streams_records)), [len(r[0]) for r in streams_records])
    rng.shuffle(labels)
    seen = [0] * len(streams_records)
    queue = []
    for s in labels:
        queue.append((int(s), seen[s]))
        seen[s] += 1
    P = streams_records[0][0].shape[1]
    i = 0
    while i < len(queue):
        n = int(rng.integers(min_batch, batch_max + 1))
        rows = []
        while len(rows) < n and i < len(queue):
            if rng.random() < untracked:
                rows.append((-1, None))
            else:
                rows.append(queue[i])
                i += 1
        ps = np.zeros((len(rows), P))
        ks = np.zeros((len(rows), P, K))
        kc = np.zeros((len(rows), P, K, 2))
        sid = np.empty(len(rows), np.int32)
        for r, (s, f) in enumerate(rows):
            sid[r] = s
            if s < 0:
                ps[r] = rng.uniform(0, 1, P)
                ks[r] = rng.uniform(0, 1, (P, K))
                kc[r] = rng.uniform(0, 400, (P, K, 2))
            else:
                ps[r], ks[r], kc[r] = (a[f] for a in streams_records[s])
        yield ps, ks, kc, sid
