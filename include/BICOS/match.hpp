// BICOS::match -- the reference's one public entry point (reference include/match.hpp:31-41,
// src/lib.cpp:31-49), implemented on hand-written sm_100a kernels through the C ABI in
// include/bicos_b200.h.
//
//  * stack0 / stack1: n >= 2 rectified single-channel device images per side, all of one
//    size and depth (8U or 16U). Borrowed, never modified.
//  * disparity: (re)allocated by the callee. int16 (-32768 = invalid) when
//    cfg.nxcorr_threshold is unset; float32 otherwise: integer mode keeps -32768.0f as the
//    invalid marker, subpixel mode uses NaN -- the reference CPU backend's convention
//    (src/impl/cpu.cpp:77-95), which is the parity oracle of this implementation.
//  * corrmap: only touched when cfg.nxcorr_threshold is set; float32 (SINGLE) or float64
//    (DOUBLE), NaN where no correlation was evaluated.
//  * stream: a cudaStream_t (nullptr = default stream); with -DBICOS_WITH_OPENCV a cv::cuda::Stream&, exactly
//    the reference's signature. Work is enqueued, not synchronised. Matches issued by one host thread on one
//    device share a workspace (descriptors, search keys): a match enqueued on another stream than the
//    thread's previous one first waits, on the device, for that previous match (the reference allocates per
//    call instead and so never overlaps either: its destructors synchronise, src/impl/cuda.cu:79-94). For
//    matches that really run side by side use one host thread per stream.
//
// Errors: BICOS::Exception for n < 2, bad depths and CUDA failures; std::invalid_argument
// when the stack needs more than 256 descriptor bits -- as in the reference
// (src/impl/cpu.cpp:110-114,154-155; include/impl/cuda/cutil.cuh:32-41). Deviations:
// mismatching image sizes/types inside a stack throw (undefined behaviour in the reference).
// A negative nxcorr_threshold is honoured as a threshold here (the NXC is evaluated, nothing is
// rejected); only the Python C ABI keeps the reference's "negative = unset" (src/pybicos_c.cpp:59-69).
// Extension: cfg.disparity_range (common.hpp) bounds the search of match and match_sharded to
// min <= x_left - x_right <= max; left pixels without a right column in range are invalid, and
// min > max throws BICOS::Exception.
#pragma once

#include "common.hpp"

#include <vector>

#ifdef BICOS_WITH_OPENCV
    #include <opencv2/core/cuda.hpp>
    #include <opencv2/core/cuda_stream_accessor.hpp>
#endif

namespace BICOS {

#ifdef BICOS_WITH_OPENCV
// raw-stream form; the defaulted sixth parameter belongs to the cv::cuda::Stream overload below
void match(
    const std::vector<Image>& stack0,
    const std::vector<Image>& stack1,
    Image& disparity,
    Config cfg,
    Image* corrmap,
    void* stream
);

// the reference's signature (include/match.hpp:31-41)
inline void match(
    const std::vector<Image>& stack0,
    const std::vector<Image>& stack1,
    Image& disparity,
    Config cfg = Config {},
    Image* corrmap = nullptr,
    cv::cuda::Stream& stream = cv::cuda::Stream::Null()
) {
    match(stack0, stack1, disparity, cfg, corrmap, static_cast<void*>(cv::cuda::StreamAccessor::getStream(stream)));
}
#else
void match(
    const std::vector<Image>& stack0,
    const std::vector<Image>& stack1,
    Image& disparity,
    Config cfg = Config {},
    Image* corrmap = nullptr,
    void* stream = nullptr
);
#endif

// Row-sharded match over several GPUs of one node from a single process: device g handles
// rows [g*H/G, (g+1)*H/G) and writes its rows of `disparity` / `corrmap` (allocated on
// devices[0]) over NVLink peer access. Inputs must be resident on devices[0] and peer
// access between devices[0] and the others must be available.
void match_sharded(
    const std::vector<Image>& stack0,
    const std::vector<Image>& stack1,
    Image& disparity,
    const std::vector<int>& devices,
    Config cfg = Config {},
    Image* corrmap = nullptr
);

} // namespace BICOS
