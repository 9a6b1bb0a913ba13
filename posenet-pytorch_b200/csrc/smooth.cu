// N10: One Euro smoothing of tracked keypoints across the frames of video streams, on the device, after pn_track_poses
// (smooth.cuh holds the arithmetic, shared with the host test).
//
// One CTA per stream: the grid depends only on n_streams, so the call can be captured in a CUDA graph.  The CTA loads its
// stream's head and id / last table into shared memory, finds its rows by ballots over stream_ids and runs them in row order
// (the frames of one stream depend on each other), and writes the table back.  The filter values (816 bytes per entry, 209 KB
// a stream at max_tracks 256) stay in the global state, where each frame reads them in the same round trip as the records.
#include "common.cuh"
#include "smooth.cuh"

namespace pn {

namespace {

using smooth::Entry;
using smooth::Head;
using smooth::Job;
using smooth::Values;

// 128 threads a stream: 1.5x faster than one warp with one stream and 1.6x with 32 streams a C3 batch (one B200): the
// coordinates of a frame's detections take one pass instead of several.
constexpr int THREADS = 128;

struct CtaTeam {
    __device__ __forceinline__ int lane() const { return threadIdx.x; }
    __device__ __forceinline__ int size() const { return THREADS; }
    __device__ __forceinline__ void sync() const { __syncthreads(); }
};

struct SmoothArgs {
    const int64_t *ids;
    double *kc;
    const int *stream_ids;
    unsigned char *state;
    int n_img, P, n_streams, max_tracks;
    int64_t max_age;
    smooth::Params q;
};

__global__ void __launch_bounds__(THREADS) smooth_kernel(SmoothArgs a) {
    __shared__ Head h;
    __shared__ Entry tab[track::MAX_TRACKS];
    __shared__ Job job[track::MAX_P];
    __shared__ int64_t ids[track::MAX_P];
    __shared__ int n_jobs;
    const CtaTeam team;
    const int tid = threadIdx.x, s = blockIdx.x;
    unsigned char *g = a.state + (int64_t)s * smooth::stream_bytes(a.max_tracks);
    Values *val = reinterpret_cast<Values *>(g + smooth::table_bytes(a.max_tracks));

    if (tid == 0) {
        h = *reinterpret_cast<const Head *>(g);
        h.n = min(max(h.n, 0), a.max_tracks);           // a state that is not all zero bytes or written here cannot overrun
    }
    team.sync();
    const Entry *gtab = reinterpret_cast<const Entry *>(g + sizeof(Head));
    for (int i = tid; i < h.n; i += THREADS) tab[i] = gtab[i];
    team.sync();

    bool any = false;
    for (int base = 0; base < a.n_img; base += 32) {
        const int r = base + (tid & 31);                // every warp takes the same ballot
        const bool mine_r = r < a.n_img && a.stream_ids[r] == s;
        unsigned mine = __ballot_sync(0xffffffffu, mine_r);
        while (mine) {
            const int64_t row = base + __ffs(mine) - 1;
            mine &= mine - 1;
            for (int p = tid; p < a.P; p += THREADS) ids[p] = a.ids[row * a.P + p];
            team.sync();
            smooth::smooth_frame(team, h, tab, val, job, n_jobs, ids, a.kc + row * a.P * smooth::NC, a.P, a.max_tracks,
                                 a.max_age, a.q);
            any = true;
        }
    }
    if (!any) return;
    Entry *gout = reinterpret_cast<Entry *>(g + sizeof(Head));
    for (int i = tid; i < h.n; i += THREADS) gout[i] = tab[i];
    if (tid == 0) *reinterpret_cast<Head *>(g) = h;
}

}  // namespace

}  // namespace pn

using namespace pn;

extern "C" int pn_smooth_state_bytes(int n_streams, int max_tracks, size_t *bytes_host) {
    PN_CHECK_ARG(bytes_host, "pn_smooth_state_bytes: null pointer");
    PN_CHECK_ARG(n_streams >= 1 && n_streams <= (1 << 20), "pn_smooth_state_bytes: n_streams %d out of 1..%d", n_streams,
                 1 << 20);
    PN_CHECK_ARG(max_tracks >= 1 && max_tracks <= track::MAX_TRACKS, "pn_smooth_state_bytes: max_tracks %d out of 1..%d",
                 max_tracks, track::MAX_TRACKS);
    *bytes_host = (size_t)n_streams * (size_t)smooth::stream_bytes(max_tracks);
    return PN_OK;
}

extern "C" int pn_smooth_keypoints(const int64_t *ids, double *keypoint_coords, int n_img, int P, const int *stream_ids,
                                   void *state, int n_streams, int max_tracks, int max_age, double fps, double min_cutoff,
                                   double beta, double d_cutoff, pn_stream_t stream) {
    PN_CHECK_ARG(ids && keypoint_coords && stream_ids && state, "pn_smooth_keypoints: null pointer");
    const uintptr_t align = (uintptr_t)ids | (uintptr_t)keypoint_coords | (uintptr_t)state;
    PN_CHECK_ARG((align & 7) == 0 && ((uintptr_t)stream_ids & 3) == 0, "pn_smooth_keypoints: misaligned pointer");
    PN_CHECK_ARG(n_img >= 1, "pn_smooth_keypoints: n_img %d < 1", n_img);
    PN_CHECK_ARG(P >= 1 && P <= track::MAX_P, "pn_smooth_keypoints: P %d out of 1..%d", P, track::MAX_P);
    PN_CHECK_ARG(n_streams >= 1 && n_streams <= (1 << 20), "pn_smooth_keypoints: n_streams %d out of 1..%d", n_streams, 1 << 20);
    PN_CHECK_ARG(max_tracks >= 1 && max_tracks <= track::MAX_TRACKS, "pn_smooth_keypoints: max_tracks %d out of 1..%d",
                 max_tracks, track::MAX_TRACKS);
    PN_CHECK_ARG(max_age >= 0, "pn_smooth_keypoints: max_age %d < 0", max_age);
    PN_CHECK_ARG(isfinite(fps) && fps > 0 && isfinite(min_cutoff) && min_cutoff > 0 && isfinite(d_cutoff) && d_cutoff > 0,
                 "pn_smooth_keypoints: fps, min_cutoff and d_cutoff must be finite and > 0 (got %g, %g, %g)", fps, min_cutoff,
                 d_cutoff);
    PN_CHECK_ARG(isfinite(beta) && beta >= 0, "pn_smooth_keypoints: beta must be finite and >= 0 (got %g)", beta);
    SmoothArgs a;
    a.ids = ids; a.kc = keypoint_coords; a.stream_ids = stream_ids; a.state = static_cast<unsigned char *>(state);
    a.n_img = n_img; a.P = P; a.n_streams = n_streams; a.max_tracks = max_tracks; a.max_age = max_age;
    a.q.fps = fps; a.q.min_cutoff = min_cutoff; a.q.beta = beta; a.q.d_cutoff = d_cutoff;
    smooth_kernel<<<n_streams, THREADS, 0, as_stream(stream)>>>(a);
    PN_CHECK_LAUNCH();
    return PN_OK;
}
