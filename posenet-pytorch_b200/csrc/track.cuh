// N9: the bounding-box pose tracker of TF.js pose-detection (BoundingBoxTracker, Apache-2.0) -- the per-frame arithmetic,
// shared by the device kernel (track.cu, one warp per stream) and the host test (tests/test_track_cpu.py, one "lane").
//
// Everything is float64 with explicit unfused operations and plain comparisons, so that host and device agree bit for bit with
// a numpy restatement: the IoU needs only + - * / and min / max.  min / max are written as comparisons (not fmin / fmax), the
// same expression on both sides.
#pragma once
#include <math.h>
#include <stdint.h>

#ifdef __CUDACC__
#define PN_TRACK_HD __host__ __device__ __forceinline__
#else
#define PN_TRACK_HD inline
#endif

namespace pn {
namespace track {

constexpr int KP = 17;              // keypoints of a pose record
constexpr int MAX_P = 256;          // poses per frame the kernel's shared memory holds
constexpr int MAX_TRACKS = 256;

PN_TRACK_HD double dadd(double a, double b) {
#ifdef __CUDA_ARCH__
    return __dadd_rn(a, b);
#else
    return a + b;
#endif
}
PN_TRACK_HD double dsub(double a, double b) {
#ifdef __CUDA_ARCH__
    return __dsub_rn(a, b);
#else
    return a - b;
#endif
}
PN_TRACK_HD double dmul(double a, double b) {
#ifdef __CUDA_ARCH__
    return __dmul_rn(a, b);
#else
    return a * b;
#endif
}
PN_TRACK_HD double ddiv(double a, double b) {
#ifdef __CUDA_ARCH__
    return __ddiv_rn(a, b);
#else
    return a / b;
#endif
}
PN_TRACK_HD double dmin(double a, double b) { return b < a ? b : a; }
PN_TRACK_HD double dmax(double a, double b) { return b > a ? b : a; }

// A box is empty when no keypoint passed the threshold: then y0 > y1 (it stays at its +inf / -inf start).
struct Box {
    double y0, x0, y1, x1;
};

// State of one stream, as it lies in the caller's state buffer: a head, then max_tracks tracks, tracks[0 .. n) in use.  All
// zero bytes is the start: no tracks, frame 0, no id issued (the first id is 1).
struct Head {
    int64_t frame;      // frames of this stream seen so far
    int64_t issued;     // ids issued so far
    int32_t n;          // tracks in use
    int32_t pad;
    int64_t pad2;
};
struct Track {
    Box box;
    int64_t id;
    int64_t last;       // the stream frame at which the track was last matched
};
static_assert(sizeof(Head) == 32 && sizeof(Track) == 48, "state layout");

PN_TRACK_HD int64_t stream_bytes(int max_tracks) { return (int64_t)sizeof(Head) + (int64_t)sizeof(Track) * max_tracks; }

PN_TRACK_HD bool empty(const Box &b) { return b.y0 > b.y1 || b.x0 > b.x1; }

// The box of one pose: min / max of y and x over the keypoints with score >= min_part_score, in keypoint order.
PN_TRACK_HD Box box_of(const double *kscores, const double *kcoords, double min_part_score) {
    Box b = {INFINITY, INFINITY, -INFINITY, -INFINITY};
    for (int k = 0; k < KP; ++k) {
        if (!(kscores[k] >= min_part_score)) continue;
        const double y = kcoords[2 * k], x = kcoords[2 * k + 1];
        b.y0 = dmin(b.y0, y); b.y1 = dmax(b.y1, y);
        b.x0 = dmin(b.x0, x); b.x1 = dmax(b.x1, x);
    }
    return b;
}

PN_TRACK_HD double iou(const Box &a, const Box &b) {
    if (empty(a) || empty(b)) return 0.0;
    const double iy = dsub(dmin(a.y1, b.y1), dmax(a.y0, b.y0));
    const double ix = dsub(dmin(a.x1, b.x1), dmax(a.x0, b.x0));
    if (iy <= 0.0 || ix <= 0.0) return 0.0;
    const double inter = dmul(iy, ix);
    const double area_a = dmul(dsub(a.y1, a.y0), dsub(a.x1, a.x0));
    const double area_b = dmul(dsub(b.y1, b.y0), dsub(b.x1, b.x0));
    const double uni = dsub(dadd(area_a, area_b), inter);
    return uni <= 0.0 ? 0.0 : ddiv(inter, uni);
}

// The argmax rule of the greedy step: candidate (v, j) beats (best, bj) when it is the first candidate, has a larger IoU, or
// the same IoU at an earlier track.  bj < 0: no candidate yet.
PN_TRACK_HD bool better(double v, int j, double best, int bj) {
    return j >= 0 && (bj < 0 || v > best || (v == best && j < bj));
}

// Stable removal of the tracks with t - last > max_age; returns the new count.
PN_TRACK_HD int expire(Track *tr, int n, int64_t t, int64_t max_age) {
    int m = 0;
    for (int i = 0; i < n; ++i)
        if (!(t - tr[i].last > max_age)) tr[m++] = tr[i];
    return m;
}

// One host "lane": the team the host test runs the frame with.
struct SerialTeam {
    PN_TRACK_HD int lane() const { return 0; }
    PN_TRACK_HD int size() const { return 1; }
    PN_TRACK_HD void sync() const {}
    PN_TRACK_HD void argmax(double &, int &) const {}
};

// Stable sort of tr [n] by last, descending, keeping the first max_tracks; returns the count kept.  Each lane places its tracks
// at their rank (the tracks with a larger last, or the same last and a smaller index, come first) in out (room for max_tracks),
// and the lanes copy them back.  A serial insertion sort costs a shared-memory round trip per moved track, and after a frame
// the matched tracks move past every unmatched one.
#ifdef __CUDACC__
#pragma nv_exec_check_disable
#endif
template <class Team>
PN_TRACK_HD int sort_truncate(const Team &team, Track *tr, int n, int max_tracks, Track *out) {
    const int lane = team.lane(), nl = team.size();
    for (int i = lane; i < n; i += nl) {
        const int64_t li = tr[i].last;
        int rank = 0;
        for (int j = 0; j < n; ++j) rank += tr[j].last > li || (tr[j].last == li && j < i);
        if (rank < max_tracks) out[rank] = tr[i];
    }
    team.sync();
    const int m = n < max_tracks ? n : max_tracks;
    for (int i = lane; i < m; i += nl) tr[i] = out[i];
    team.sync();
    return m;
}

// Detection flags and boxes of n poses of a frame, written at det + p0 and box + p0: ps [n], ks [n, 17], kc [n, 17, 2] are the
// poses' records (the kernel stages them in shared memory first).  The lanes split the poses.
#ifdef __CUDACC__
#pragma nv_exec_check_disable
#endif
template <class Team>
PN_TRACK_HD void frame_boxes(const Team &team, Box *box, unsigned char *det, int p0, int n, const double *ps, const double *ks,
                             const double *kc, double min_part_score) {
    for (int i = team.lane(); i < n; i += team.size()) {
        det[p0 + i] = ps[i] > 0.0;
        box[p0 + i] = box_of(ks + i * KP, kc + i * KP * 2, min_part_score);
    }
}

// One frame of one stream, once frame_boxes has filled det [P] and box [P].  h and tr (room for max_tracks + P tracks), taken
// and out (room for max_tracks each) are the team's shared scratch; ids [P] receives the track ids (-1 for records that are not
// detections).  Lane 0 does the serial parts; the lanes split the IoUs, and team.argmax combines the lanes' best candidates
// with the rule of `better`.
#ifdef __CUDACC__
#pragma nv_exec_check_disable
#endif
template <class Team>
PN_TRACK_HD void track_frame(const Team &team, Head &h, Track *tr, const Box *box, const unsigned char *det, unsigned char *taken,
                             Track *out, int P, int max_tracks, int64_t max_age, double min_similarity, int64_t *ids) {
    const int lane = team.lane(), nl = team.size();
    if (lane == 0) {
        h.frame += 1;
        h.n = expire(tr, h.n, h.frame, max_age);
    }
    team.sync();
    const int64_t t = h.frame;
    const int n_old = h.n;
    for (int j = lane; j < n_old; j += nl) taken[j] = 0;
    team.sync();
    int n = n_old;                  // lane 0's count: new tracks are appended past the candidates
    for (int p = 0; p < P; ++p) {
        if (!det[p]) {
            if (lane == 0) ids[p] = -1;
            continue;
        }
        double best = 0.0;
        int bj = -1;
        for (int j = lane; j < n_old; j += nl) {
            if (taken[j]) continue;
            const double v = iou(box[p], tr[j].box);
            if (v >= min_similarity && better(v, j, best, bj)) {
                best = v;
                bj = j;
            }
        }
        team.argmax(best, bj);
        if (lane == 0) {
            if (bj >= 0) {
                taken[bj] = 1;
                tr[bj].box = box[p];
                tr[bj].last = t;
                ids[p] = tr[bj].id;
            } else {
                tr[n].box = box[p];
                tr[n].id = ++h.issued;
                tr[n].last = t;
                ids[p] = tr[n].id;
                ++n;
            }
        }
        team.sync();
    }
    if (lane == 0) h.n = n;
    team.sync();
    const int m = sort_truncate(team, tr, h.n, max_tracks, out);
    if (lane == 0) h.n = m;
    team.sync();
}

}  // namespace track
}  // namespace pn
