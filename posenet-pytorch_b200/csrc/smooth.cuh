// N10: One Euro smoothing of tracked keypoints (Casiez et al., CHI 2012; the filter TF.js pose-detection runs per tracked pose)
// -- the per-entry update and the per-frame table step, shared by the device kernel (smooth.cu) and the host test
// (tests/test_smooth_cpu.py, one "lane").
//
// float64 with the unfused helpers of track.cuh and |x| only, so that host and device agree bit for bit with a numpy
// restatement.
#pragma once
#include "track.cuh"

namespace pn {
namespace smooth {

constexpr int NC = 2 * track::KP;   // coordinates of a pose record (y, x per keypoint)
constexpr int NV = 3 * NC;          // filter values of an entry
constexpr double TWO_PI = 6.283185307179586;

// State of one stream, as it lies in the caller's state buffer: a head, max_tracks table entries (entries [0 .. n) in use),
// then max_tracks Values, Values i belonging to entry i.  All zero bytes is the start: frame 0, no entries.
struct Head {
    int64_t frame;      // frames of this stream seen so far
    int32_t n;          // entries in use
    int32_t pad;
};
struct Entry {
    int64_t id;
    int64_t last;       // the stream frame of the entry's last update
};
struct Values {
    double x_prev[NC];  // previous raw coordinate
    double x_hat[NC];   // previous filtered coordinate
    double dx_hat[NC];  // previous filtered derivative
};
static_assert(sizeof(Head) == 16 && sizeof(Entry) == 16 && sizeof(Values) == NV * 8, "state layout");

PN_TRACK_HD int64_t table_bytes(int max_tracks) { return (int64_t)sizeof(Head) + (int64_t)sizeof(Entry) * max_tracks; }
PN_TRACK_HD int64_t stream_bytes(int max_tracks) { return table_bytes(max_tracks) + (int64_t)sizeof(Values) * max_tracks; }

struct Params {
    double fps, min_cutoff, beta, d_cutoff;
};

// One coordinate of an existing entry, dt >= 1 stream frames after its last update: returns the filtered value and updates
// the entry's three values.  The operations and their order are the semantics (posenet/track.py); do not reassociate.
PN_TRACK_HD double filter(const Params &q, int64_t dt, double x, double &x_prev, double &x_hat, double &dx_hat) {
    using track::dadd;
    using track::ddiv;
    using track::dmul;
    using track::dsub;
    const double rate = ddiv(q.fps, (double)dt);
    const double dx = dmul(dsub(x, x_prev), rate);
    const double a_d = ddiv(1.0, dadd(1.0, ddiv(rate, dmul(TWO_PI, q.d_cutoff))));
    dx_hat = dadd(dmul(a_d, dx), dmul(dsub(1.0, a_d), dx_hat));
    const double cutoff = dadd(q.min_cutoff, dmul(q.beta, fabs(dx_hat)));
    const double a = ddiv(1.0, dadd(1.0, ddiv(rate, dmul(TWO_PI, cutoff))));
    x_hat = dadd(dmul(a, x), dmul(dsub(1.0, a), x_hat));
    x_prev = x;
    return x_hat;
}

// A detection the frame filters: record p, table entry e, dt = t - last of an existing entry, 0 for a fresh one.
struct Job {
    int32_t p, e;
    int64_t dt;
};

// The entry a new id takes when the table is full: the smallest last that is < t, the first in table order on a tie; -1 when
// every entry was updated in this frame.
PN_TRACK_HD int evict(const Entry *tab, int n, int64_t t) {
    int e = -1;
    for (int i = 0; i < n; ++i)
        if (tab[i].last < t && (e < 0 || tab[i].last < tab[e].last)) e = i;
    return e;
}

// One frame of one stream.  h and tab (max_tracks entries) and job (room for P) are the team's shared scratch, val
// (max_tracks Values) the stream's filter values; ids [P] are the frame's track ids (>= 1: a detection) and kc [P, 34] its
// coordinates, smoothed in place.  Lane 0 does the table step; the lanes split the expiry's moves of values and the 34
// coordinates of each filtered detection.
#ifdef __CUDACC__
#pragma nv_exec_check_disable
#endif
template <class Team>
PN_TRACK_HD void smooth_frame(const Team &team, Head &h, Entry *tab, Values *val, Job *job, int &n_jobs, const int64_t *ids,
                              double *kc, int P, int max_tracks, int64_t max_age, const Params &q) {
    const int lane = team.lane(), nl = team.size();
    const int64_t t = h.frame + 1;
    // 1. stable removal of the entries with t - last > max_age: each lane moves its words of the kept entries' values
    const int n_old = h.n;
    int m = 0;
    for (int i = 0; i < n_old; ++i) {
        if (t - tab[i].last > max_age) continue;
        if (m != i) {
            const double *src = reinterpret_cast<const double *>(val + i);
            double *dst = reinterpret_cast<double *>(val + m);
            for (int w = lane; w < NV; w += nl) dst[w] = src[w];
        }
        ++m;
    }
    team.sync();
    // 2. lane 0 walks the detections in record order: update, append, evict or pass through
    if (lane == 0) {
        int n = 0;
        for (int i = 0; i < n_old; ++i)
            if (!(t - tab[i].last > max_age)) tab[n++] = tab[i];
        int nj = 0;
        for (int p = 0; p < P; ++p) {
            const int64_t id = ids[p];
            if (!(id >= 1)) continue;
            int e = -1;
            for (int i = 0; i < n; ++i)
                if (tab[i].id == id) {
                    e = i;
                    break;
                }
            int64_t dt = 0;
            if (e >= 0) {
                if (tab[e].last == t) continue;         // the id twice in one frame: its second record keeps its coordinates
                dt = t - tab[e].last;
            } else if (n < max_tracks) {
                e = n++;
            } else {
                e = evict(tab, n, t);
                if (e < 0) continue;
            }
            tab[e].id = id;
            tab[e].last = t;
            job[nj].p = p;
            job[nj].e = e;
            job[nj].dt = dt;
            ++nj;
        }
        h.frame = t;
        h.n = n;
        n_jobs = nj;
    }
    team.sync();
    // 3. the lanes split the coordinates of the filtered detections (each entry has at most one job)
    const int work = n_jobs * NC;
    for (int w = lane; w < work; w += nl) {
        const Job j = job[w / NC];
        const int c = w - (w / NC) * NC;
        Values &v = val[j.e];
        double *xp = kc + (int64_t)j.p * NC + c;
        const double x = *xp;
        if (j.dt == 0) {
            v.x_prev[c] = x;
            v.x_hat[c] = x;
            v.dx_hat[c] = 0.0;
        } else {
            double x_prev = v.x_prev[c], x_hat = v.x_hat[c], dx_hat = v.dx_hat[c];
            *xp = filter(q, j.dt, x, x_prev, x_hat, dx_hat);
            v.x_prev[c] = x_prev;
            v.x_hat[c] = x_hat;
            v.dx_hat[c] = dx_hat;
        }
    }
    team.sync();
}

}  // namespace smooth
}  // namespace pn
