// Pose smoothing of a tracked video on the device (see pnp_math.cuh): one thread per lane projects the box corners with
// the lane's pose, pushes them into the lane's history ring (the count lives on the device too, so a captured graph
// replays frame after frame with no host input), averages the recent projections and solves PnP for the average.
// The *_host entry point runs the same code on host memory (unit tests against OpenCV, no GPU needed).
#include "common.cuh"
#include "pnp_math.cuh"

namespace g6d {

constexpr int kTrackMaxLanes = 64;

__global__ void __launch_bounds__(32) track_smooth_kernel(const float* bbox, const double* poses, const g6d_glue_camera* cams,
                                                          const double* weights, const double* wsum, int lanes, int num, float* hist,
                                                          int* count, float* corners, double* wpts, double* smoothed) {
    const int l = blockIdx.x * blockDim.x + threadIdx.x;
    if (l < lanes) pnp::track_smooth_lane(l, bbox, poses, cams, weights, wsum, num, hist, count, corners, wpts, smoothed);
}

}  // namespace g6d

using namespace g6d;

#define G6D_TRACK_ARGS_OK                                                                                                  \
    (bbox && poses && cams && weights && wsum && hist && count && corners && wpts && smoothed && lanes > 0 &&              \
     lanes <= kTrackMaxLanes && num > 0)

extern "C" int g6d_track_smooth(const float* bbox, const double* poses, const g6d_glue_camera* cams, const double* weights,
                                const double* wsum, int lanes, int num, float* hist, int* count, float* corners, double* wpts,
                                double* smoothed, g6d_stream_t stream) {
    G6D_REQUIRE(G6D_TRACK_ARGS_OK, "g6d_track_smooth: bad args (1 <= lanes <= %d, num >= 1)", kTrackMaxLanes);
    track_smooth_kernel<<<ceil_div(lanes, 32), 32, 0, as_stream(stream)>>>(bbox, poses, cams, weights, wsum, lanes, num, hist, count,
                                                                          corners, wpts, smoothed);
    G6D_CHECK_LAUNCH("g6d_track_smooth");
    return G6D_OK;
}

extern "C" int g6d_track_smooth_host(const float* bbox, const double* poses, const g6d_glue_camera* cams, const double* weights,
                                     const double* wsum, int lanes, int num, float* hist, int* count, float* corners, double* wpts,
                                     double* smoothed) {
    G6D_REQUIRE(G6D_TRACK_ARGS_OK, "g6d_track_smooth_host: bad args (1 <= lanes <= %d, num >= 1)", kTrackMaxLanes);
    for (int l = 0; l < lanes; ++l) pnp::track_smooth_lane(l, bbox, poses, cams, weights, wsum, num, hist, count, corners, wpts, smoothed);
    return G6D_OK;
}
