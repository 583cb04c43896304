// Rectification on the device, in front of BICOS::match (extension; the reference expects rectified stacks).
//
// This applies rectification maps the caller already has: CV_32FC1 device images of the rectified size, e.g. the
// two maps cv::initUndistortRectifyMap writes per camera with m1type = CV_32FC1, uploaded once per rig. Computing
// them from a calibration (K, D, R, P) stays a host step outside this library.
//
//  * remap: dst(y, x) = src(map_y(y, x), map_x(y, x)) for every image of `src`, bit for bit OpenCV's CPU
//    cv::remap(src, dst, map_x, map_y, INTER_LINEAR, BORDER_CONSTANT, 0): coordinates rounded to 1/32 px
//    (half to even), bilinear weights in int32 fixed point for 8U and in float32 for 16U, taps outside the
//    source read 0, a NaN / infinite / huge (|m| >= 2^25) map value gives 0. include/bicos_b200.h states the
//    arithmetic. `dst` is resized to one image per source image, of the maps' size and the sources' type
//    (allocated by the callee, like match's disparity). Sources: 8U or 16U, all of one size, type and pitch.
//  * match_rectified: match(remap(stack0, maps.map_x0, maps.map_y0), remap(stack1, maps.map_x1, maps.map_y1), ...)
//    in one call: both remaps are one kernel launch into a workspace of the calling thread's per-device handle,
//    followed by the same match. The results are bit-identical to that composition; disparity and corrmap have
//    the maps' size. Output, exception and stream conventions are those of match (match.hpp).
//
// Sizes: sources and maps have at most 32767 rows and columns; the maps of both cameras share one size and pitch.
#pragma once

#include "match.hpp"

namespace BICOS {

struct RectifyMaps {
    Image map_x0, map_y0; // camera 0 (stack0): CV_32FC1, rectified size
    Image map_x1, map_y1; // camera 1 (stack1)
};

void remap(const std::vector<Image>& src, const Image& map_x, const Image& map_y, std::vector<Image>& dst, void* stream = nullptr);

#ifdef BICOS_WITH_OPENCV
// raw-stream form; the defaulted seventh parameter belongs to the cv::cuda::Stream overload below
void match_rectified(
    const std::vector<Image>& stack0,
    const std::vector<Image>& stack1,
    const RectifyMaps& maps,
    Image& disparity,
    Config cfg,
    Image* corrmap,
    void* stream
);

inline void match_rectified(
    const std::vector<Image>& stack0,
    const std::vector<Image>& stack1,
    const RectifyMaps& maps,
    Image& disparity,
    Config cfg = Config {},
    Image* corrmap = nullptr,
    cv::cuda::Stream& stream = cv::cuda::Stream::Null()
) {
    match_rectified(stack0, stack1, maps, disparity, cfg, corrmap, static_cast<void*>(cv::cuda::StreamAccessor::getStream(stream)));
}
#else
void match_rectified(
    const std::vector<Image>& stack0,
    const std::vector<Image>& stack1,
    const RectifyMaps& maps,
    Image& disparity,
    Config cfg = Config {},
    Image* corrmap = nullptr,
    void* stream = nullptr
);
#endif

} // namespace BICOS
