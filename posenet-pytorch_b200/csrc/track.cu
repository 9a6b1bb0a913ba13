// N9: pose tracking across the frames of video streams (the bounding-box tracker of TF.js pose-detection), on the device, after
// the decode (track.cuh holds the arithmetic, shared with the host test).
//
// One warp (one CTA) per stream: the grid depends only on n_streams, so the call can be captured in a CUDA graph.  The warp
// loads its stream's state into shared memory, finds its rows by ballots over stream_ids and runs them in row order (the
// frames of one stream depend on each other), and writes the state back.  Rows of different streams run in parallel.
#include "common.cuh"
#include "track.cuh"

namespace pn {

namespace {

using track::Box;
using track::Head;
using track::Track;

struct WarpTeam {
    __device__ __forceinline__ int lane() const { return threadIdx.x & 31; }
    __device__ __forceinline__ int size() const { return 32; }
    __device__ __forceinline__ void sync() const { __syncwarp(); }
    // every lane ends with the warp's best (IoU, track) under track::better
    __device__ __forceinline__ void argmax(double &best, int &bj) const {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const double ob = __shfl_xor_sync(0xffffffffu, best, o);
            const int oj = __shfl_xor_sync(0xffffffffu, bj, o);
            if (track::better(ob, oj, best, bj)) {
                best = ob;
                bj = oj;
            }
        }
    }
};

struct TrackArgs {
    const double *ps, *ks, *kc;
    const int *stream_ids;
    unsigned char *state;
    int64_t *ids;
    int n_img, P, n_streams, max_tracks;
    int64_t max_age;
    double min_similarity, min_part_score;
};

// Poses whose records a warp stages at a time: their 52 doubles each (pose score, 17 keypoint scores, 34 coordinates) come in
// as coalesced loads, all issued before the first is stored, so a frame costs one memory round trip instead of one per
// keypoint.
constexpr int CHUNK = 32;
constexpr int REC = 1 + 3 * track::KP;
// the staging buffer is free while a frame's tracks are sorted: it holds the sorted ones
static_assert(CHUNK * REC * sizeof(double) >= track::MAX_TRACKS * sizeof(Track), "sort buffer");

__device__ __forceinline__ void stage_records(double *stage, int n, const double *ps, const double *ks, const double *kc) {
    const int lane = threadIdx.x & 31;
    double v[REC];
#pragma unroll
    for (int j = 0; j < REC; ++j) {             // element i of [ps n][ks 17n][kc 34n]
        const int i = lane + 32 * j;
        v[j] = i < n ? ps[i] : i < (1 + track::KP) * n ? ks[i - n] : i < REC * n ? kc[i - (1 + track::KP) * n] : 0.0;
    }
#pragma unroll
    for (int j = 0; j < REC; ++j)
        if (lane + 32 * j < REC * n) stage[lane + 32 * j] = v[j];
}

__global__ void __launch_bounds__(32) track_kernel(TrackArgs a) {
    __shared__ __align__(16) double stage[CHUNK * REC];
    extern __shared__ __align__(16) unsigned char smem[];
    Head &h = *reinterpret_cast<Head *>(smem);
    Track *tr = reinterpret_cast<Track *>(smem + sizeof(Head));
    Box *box = reinterpret_cast<Box *>(tr + a.max_tracks + a.P);
    unsigned char *det = reinterpret_cast<unsigned char *>(box + a.P);
    unsigned char *taken = det + a.P;
    const WarpTeam team;
    const int lane = team.lane(), s = blockIdx.x;
    int64_t *g = reinterpret_cast<int64_t *>(a.state + (int64_t)s * track::stream_bytes(a.max_tracks));
    int64_t *sh = reinterpret_cast<int64_t *>(smem);

    for (int i = lane; i < (int)(sizeof(Head) / 8); i += 32) sh[i] = g[i];
    __syncwarp();
    const int n0 = min(max(h.n, 0), a.max_tracks);     // a state that is not all zero bytes or written here cannot overrun
    const int words = (int)(track::stream_bytes(n0) / 8);
    for (int i = (int)(sizeof(Head) / 8) + lane; i < words; i += 32) sh[i] = g[i];
    __syncwarp();
    if (lane == 0) h.n = n0;
    __syncwarp();

    bool any = false;
    for (int base = 0; base < a.n_img; base += 32) {
        const int r = base + lane;
        const int sid = r < a.n_img ? a.stream_ids[r] : s;
        if (s == 0) {                                   // CTA 0 also writes the ids of the untracked rows
            unsigned bad = __ballot_sync(0xffffffffu, sid < 0 || sid >= a.n_streams);
            while (bad) {
                const int row = base + __ffs(bad) - 1;
                bad &= bad - 1;
                for (int p = lane; p < a.P; p += 32) a.ids[(int64_t)row * a.P + p] = -1;
            }
        }
        unsigned mine = __ballot_sync(0xffffffffu, r < a.n_img && sid == s);
        while (mine) {
            const int64_t row = base + __ffs(mine) - 1;
            mine &= mine - 1;
            for (int p0 = 0; p0 < a.P; p0 += CHUNK) {
                const int n = min(CHUNK, a.P - p0);
                const int64_t first = row * a.P + p0;
                stage_records(stage, n, a.ps + first, a.ks + first * track::KP, a.kc + first * track::KP * 2);
                __syncwarp();
                track::frame_boxes(team, box, det, p0, n, stage, stage + n, stage + (1 + track::KP) * n, a.min_part_score);
                __syncwarp();
            }
            track::track_frame(team, h, tr, box, det, taken, reinterpret_cast<Track *>(stage), a.P, a.max_tracks, a.max_age,
                               a.min_similarity, a.ids + row * a.P);
            any = true;
        }
    }
    if (!any) return;
    const int out_words = (int)(track::stream_bytes(h.n) / 8);
    for (int i = lane; i < out_words; i += 32) g[i] = sh[i];
}

}  // namespace

}  // namespace pn

using namespace pn;

extern "C" int pn_track_state_bytes(int n_streams, int max_tracks, size_t *bytes_host) {
    PN_CHECK_ARG(bytes_host, "pn_track_state_bytes: null pointer");
    PN_CHECK_ARG(n_streams >= 1 && n_streams <= (1 << 20), "pn_track_state_bytes: n_streams %d out of 1..%d", n_streams, 1 << 20);
    PN_CHECK_ARG(max_tracks >= 1 && max_tracks <= track::MAX_TRACKS, "pn_track_state_bytes: max_tracks %d out of 1..%d",
                 max_tracks, track::MAX_TRACKS);
    *bytes_host = (size_t)n_streams * (size_t)track::stream_bytes(max_tracks);
    return PN_OK;
}

extern "C" int pn_track_poses(const double *pose_scores, const double *keypoint_scores, const double *keypoint_coords, int n_img,
                              int P, const int *stream_ids, void *state, int n_streams, int max_tracks, int max_age,
                              double min_similarity, double min_part_score, int64_t *ids, pn_stream_t stream) {
    PN_CHECK_ARG(pose_scores && keypoint_scores && keypoint_coords && stream_ids && state && ids, "pn_track_poses: null pointer");
    const uintptr_t align = (uintptr_t)pose_scores | (uintptr_t)keypoint_scores | (uintptr_t)keypoint_coords | (uintptr_t)state |
                            (uintptr_t)ids;
    PN_CHECK_ARG((align & 7) == 0 && ((uintptr_t)stream_ids & 3) == 0, "pn_track_poses: misaligned pointer");
    PN_CHECK_ARG(n_img >= 1, "pn_track_poses: n_img %d < 1", n_img);
    PN_CHECK_ARG(P >= 1 && P <= track::MAX_P, "pn_track_poses: P %d out of 1..%d", P, track::MAX_P);
    PN_CHECK_ARG(n_streams >= 1 && n_streams <= (1 << 20), "pn_track_poses: n_streams %d out of 1..%d", n_streams, 1 << 20);
    PN_CHECK_ARG(max_tracks >= 1 && max_tracks <= track::MAX_TRACKS, "pn_track_poses: max_tracks %d out of 1..%d", max_tracks,
                 track::MAX_TRACKS);
    PN_CHECK_ARG(max_age >= 0, "pn_track_poses: max_age %d < 0", max_age);
    PN_CHECK_ARG(min_similarity == min_similarity && min_part_score == min_part_score,
                 "pn_track_poses: min_similarity and min_part_score must not be NaN");
    TrackArgs a;
    a.ps = pose_scores; a.ks = keypoint_scores; a.kc = keypoint_coords; a.stream_ids = stream_ids;
    a.state = static_cast<unsigned char *>(state); a.ids = ids;
    a.n_img = n_img; a.P = P; a.n_streams = n_streams; a.max_tracks = max_tracks; a.max_age = max_age;
    a.min_similarity = min_similarity; a.min_part_score = min_part_score;
    const size_t smem = sizeof(Head) + sizeof(Track) * (size_t)(max_tracks + P) + (sizeof(Box) + 1) * (size_t)P + max_tracks;
    track_kernel<<<n_streams, 32, smem, as_stream(stream)>>>(a);
    PN_CHECK_LAUNCH();
    return PN_OK;
}
