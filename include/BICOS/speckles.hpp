// Speckle removal on the device, after BICOS::match (extension; OpenCV users know it as cv::filterSpeckles).
//
// Sets every small connected blob of a disparity image to `new_value`, in place. Two 4-neighbours belong to one
// blob when both are valid disparities other than `new_value` and differ by at most `max_diff`; a blob of at most
// `max_speckle_size` pixels is a speckle. Invalid disparities (int16 -32768; float32 NaN or -32768.0f) never
// belong to a blob. include/bicos_b200.h states the semantics bit for bit (bicos_b200_filter_speckles): for an
// int16 disparity with new_value = -32768, or without -32768 pixels, the result is exactly
// cv::filterSpeckles(disparity, new_value, max_speckle_size, max_diff); float32 disparities (what every match with a
// threshold returns) are supported as well.
//
// disparity: IMG_16S or IMG_32F device image (what match returns) of at most 32767 rows and columns. The filter is
// enqueued on `stream` and runs on the calling thread's per-device handle, like match. With `counts` the call
// synchronises `stream` to return how many pixels were set and how many speckles were removed; without it the call
// does not synchronise. Errors throw BICOS::Exception.
#pragma once

#include "common.hpp"

#include <cstddef>

#ifdef BICOS_WITH_OPENCV
    #include <opencv2/core/cuda.hpp>
    #include <opencv2/core/cuda_stream_accessor.hpp>
#endif

namespace BICOS {

struct SpeckleCounts {
    size_t pixels; // pixels set to new_value
    size_t speckles; // speckles removed
};

#ifdef BICOS_WITH_OPENCV
// raw-stream form; the defaulted last parameters belong to the cv::cuda::Stream overload below
void filter_speckles(Image& disparity, double new_value, int max_speckle_size, double max_diff, SpeckleCounts* counts, void* stream);

inline void filter_speckles(Image& disparity, double new_value, int max_speckle_size, double max_diff, SpeckleCounts* counts = nullptr,
                            cv::cuda::Stream& stream = cv::cuda::Stream::Null()) {
    filter_speckles(disparity, new_value, max_speckle_size, max_diff, counts,
                    static_cast<void*>(cv::cuda::StreamAccessor::getStream(stream)));
}
#else
void filter_speckles(Image& disparity, double new_value, int max_speckle_size, double max_diff, SpeckleCounts* counts = nullptr,
                     void* stream = nullptr);
#endif

} // namespace BICOS
