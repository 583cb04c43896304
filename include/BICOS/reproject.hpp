// Reprojection on the device, after BICOS::match (extension; the reference does it on the host in its CLI).
//
// Turns a disparity image into 3D points through the 4x4 reprojection matrix Q of the rectified rig, e.g. the Q
// cv::stereoRectify returns (computing Q stays a host step outside this library). Per disparity pixel (row r,
// column c), with the arithmetic include/bicos_b200.h states bit for bit (bicos_b200_reproject):
//   invalid disparities (int16 -32768; float32 NaN or -32768.0f) are skipped;
//   [X Y Z W] = Q [c r d 1] in double without FMA contraction, point = (float)(X / W), (float)(Y / W), (float)(Z / W);
//   points with a non-finite coordinate are skipped, and so are points with Z < 0 unless allow_negative_z.
// This is not cv::reprojectImageTo3D's arithmetic (which multiplies by 1 / W and writes Z = 10000 for missing
// values); where both keep a point they agree within a few float ULPs.
//
//  * reproject: the dense map. `xyz` is (re)allocated as rows x cols IMG_32FC3 (CV_32FC3), X Y Z per pixel, NaN NaN
//    NaN where a pixel is skipped. Enqueued, not synchronised.
//  * reproject_points: the kept points only, in row-major pixel order (the content and order of bicos-cli's .xyz
//    file). `points` is (re)allocated as 1 x rows*cols IMG_32FC3 and `pixel_index`, if given, as 1 x rows*cols
//    IMG_32S (CV_32SC1, r * cols + c per point); only the first ReprojectCounts::points entries are written. The
//    call synchronises `stream` to return the counts, which sum to rows * cols.
//
// disparity: IMG_16S or IMG_32F device image (what match returns) of at most 32767 rows and columns. Both run on
// the calling thread's per-device handle, like match; errors throw BICOS::Exception.
#pragma once

#include "common.hpp"

#include <array>
#include <cstddef>

#ifdef BICOS_WITH_OPENCV
    #include <opencv2/core/cuda.hpp>
    #include <opencv2/core/cuda_stream_accessor.hpp>
#endif

namespace BICOS {

struct ReprojectCounts {
    size_t points; // kept
    size_t invalid_disparity;
    size_t non_finite;
    size_t negative_z;
};

#ifdef BICOS_WITH_OPENCV
// raw-stream forms; the defaulted last parameters belong to the cv::cuda::Stream overloads below
void reproject(const Image& disparity, const std::array<double, 16>& Q, Image& xyz, bool allow_negative_z, void* stream);
ReprojectCounts reproject_points(const Image& disparity, const std::array<double, 16>& Q, Image& points, Image* pixel_index,
                                 bool allow_negative_z, void* stream);

inline void reproject(const Image& disparity, const std::array<double, 16>& Q, Image& xyz, bool allow_negative_z = false,
                      cv::cuda::Stream& stream = cv::cuda::Stream::Null()) {
    reproject(disparity, Q, xyz, allow_negative_z, static_cast<void*>(cv::cuda::StreamAccessor::getStream(stream)));
}

inline ReprojectCounts reproject_points(const Image& disparity, const std::array<double, 16>& Q, Image& points,
                                        Image* pixel_index = nullptr, bool allow_negative_z = false,
                                        cv::cuda::Stream& stream = cv::cuda::Stream::Null()) {
    return reproject_points(disparity, Q, points, pixel_index, allow_negative_z,
                            static_cast<void*>(cv::cuda::StreamAccessor::getStream(stream)));
}
#else
void reproject(const Image& disparity, const std::array<double, 16>& Q, Image& xyz, bool allow_negative_z = false,
               void* stream = nullptr);
ReprojectCounts reproject_points(const Image& disparity, const std::array<double, 16>& Q, Image& points,
                                 Image* pixel_index = nullptr, bool allow_negative_z = false, void* stream = nullptr);
#endif

} // namespace BICOS
