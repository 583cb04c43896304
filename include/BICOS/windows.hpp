// Per-pixel disparity windows (extension; the reference searches the whole row, Config::disparity_range one interval).
//
//  * match_windows: match() with the search of left pixel (r, i) bounded to the right columns j with
//    windows.min(r, i) <= i - j <= windows.max(r, i), clipped to the row. min > max is an empty window: the pixel is
//    invalid and nothing is searched or refined for it (use it for pixels outside a region of interest). The reverse
//    search of the Consistency check covers exactly the pairs the forward windows define. Constant maps (m, M) give bit
//    for bit the result of Config::disparity_range = {m, M}; maps that cover the row give the unranged match.
//    cfg.disparity_range must be unset. include/bicos_b200.h states the semantics in full. Output, exception and stream
//    conventions are those of match (match.hpp).
//  * windows_from_disparity: window maps from a prior disparity (CV_16SC1 or CV_32FC1, e.g. the previous frame's
//    match): a valid prior d gives [floor(d) - margin, ceil(d) + margin] clamped to int16; an invalid one (int16
//    -32768; float32 NaN, -32768.0f or +-inf) gives `fallback`, std::nullopt = the whole row. margin: 0..32767.
//    `windows` is (re)allocated by the callee to the prior's size.
#pragma once

#include "match.hpp"

namespace BICOS {

struct DisparityWindows {
    Image min, max; // CV_16SC1 device images of the disparity's size, one pitch for both
};

void windows_from_disparity(const Image& prior, int margin, std::optional<DisparityRange> fallback, DisparityWindows& windows,
                            void* stream = nullptr);

#ifdef BICOS_WITH_OPENCV
// raw-stream form; the defaulted sixth parameter belongs to the cv::cuda::Stream overload below
void match_windows(
    const std::vector<Image>& stack0,
    const std::vector<Image>& stack1,
    const DisparityWindows& windows,
    Image& disparity,
    Config cfg,
    Image* corrmap,
    void* stream
);

inline void match_windows(
    const std::vector<Image>& stack0,
    const std::vector<Image>& stack1,
    const DisparityWindows& windows,
    Image& disparity,
    Config cfg = Config {},
    Image* corrmap = nullptr,
    cv::cuda::Stream& stream = cv::cuda::Stream::Null()
) {
    match_windows(stack0, stack1, windows, disparity, cfg, corrmap, static_cast<void*>(cv::cuda::StreamAccessor::getStream(stream)));
}

inline void windows_from_disparity(const Image& prior, int margin, std::optional<DisparityRange> fallback, DisparityWindows& windows,
                                   cv::cuda::Stream& stream) {
    windows_from_disparity(prior, margin, fallback, windows, static_cast<void*>(cv::cuda::StreamAccessor::getStream(stream)));
}
#else
void match_windows(
    const std::vector<Image>& stack0,
    const std::vector<Image>& stack1,
    const DisparityWindows& windows,
    Image& disparity,
    Config cfg = Config {},
    Image* corrmap = nullptr,
    void* stream = nullptr
);
#endif

} // namespace BICOS
