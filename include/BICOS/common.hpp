// Public types of the B200-native BICOS matcher. Same names, fields, defaults and
// meaning as the reference's include/common.hpp:34-90 (Config, TransformMode, Precision,
// Variant::NoDuplicates / Variant::Consistency, SearchVariant, INVALID_DISP, is_invalid,
// Exception), so that code written against libBICOS compiles against this header.
// This build is always a CUDA build (there is no CPU fallback), hence Precision exists.
#pragma once

#include <cmath>
#include <exception>
#include <limits>
#include <optional>
#include <string>
#include <type_traits>
#include <variant>

#if defined(BICOS_WITH_OPENCV)
    #include <opencv2/core.hpp>
    #include <opencv2/core/cuda.hpp>
#else
    #include "image.hpp"
#endif

#ifndef BICOS_CUDA
    #define BICOS_CUDA 1
#endif

namespace BICOS {

using uint128_t = __uint128_t;

// ---- invalid-disparity markers -------------------------------------------------------------
// Floating point results mark "no match" with NaN, integer results with the lowest value of the
// type (-32768 for the int16 disparities of a run without NXC threshold). One exception,
// inherited from the reference's CPU backend which this library follows: integer-mode runs
// WITH a threshold return float32 whose invalid marker is -32768.0f (src/impl/cpu.cpp:88-94).
template<typename T>
constexpr T INVALID_DISP =
    std::numeric_limits<T>::has_quiet_NaN ? std::numeric_limits<T>::quiet_NaN() : std::numeric_limits<T>::lowest();

template<typename T>
constexpr bool is_invalid(T disparity) {
    if constexpr (std::is_floating_point_v<T>)
        return disparity != disparity; // NaN
    else
        return disparity == INVALID_DISP<T>;
}

#if defined(BICOS_WITH_OPENCV)
using Image = cv::cuda::GpuMat;
#endif

// ---- what to compute -------------------------------------------------------------------------

// Which temporal descriptor is built per pixel from the n images of a stack:
//   LIMITED  neighbour, mean and neighbouring pair-sum comparisons: 4n-6 bits, n <= 65
//   FULL     additionally all pair-sum against pair-sum comparisons: n^2-2n+3 bits, n <= 16
// (descriptors are held in 32 / 64 / 128 / 256 bits; wider stacks are rejected unless
// Config::wide_descriptors allows 384 / 512 bits, FULL n <= 23)
enum class TransformMode { LIMITED, FULL };

// Arithmetic of the normalised cross correlation; the correlation map is float32 or float64
// accordingly, the disparity stays float32 / int16.
enum class Precision { SINGLE, DOUBLE };

namespace Variant {
    // A left pixel matches only if exactly one right pixel of its row attains the minimal
    // Hamming distance.
    struct NoDuplicates {};
    // Left-right check: the best match of the matched right pixel, searched back over the left
    // row, must lie within max_lr_diff columns of the left pixel; the disparity is measured from
    // the midpoint of the two. no_dupes additionally demands unique minima in both directions.
    struct Consistency {
        int max_lr_diff = 1;
        bool no_dupes = false;
    };
} // namespace Variant

using SearchVariant = std::variant<Variant::NoDuplicates, Variant::Consistency>;

// Bounds of the disparity x_left - x_right a match may have, both inclusive; min may be negative.
struct DisparityRange {
    int min;
    int max;
};

struct Config {
    // Matches whose normalised cross correlation over the stack is below this are dropped.
    // Unset: no correlation stage at all, the result is the raw int16 disparity. A negative
    // value is a valid threshold ("evaluate the correlation, drop nothing").
    std::optional<float> nxcorr_threshold = 0.5f;
    // Set: the right pixel is interpolated (parabola through its two neighbours) at
    // x = -1, -1 + step, ... <= 1 and the x with the highest correlation refines the disparity;
    // results are float32 with NaN as the invalid marker. Must not be 0.
    std::optional<float> subpixel_step = std::nullopt;
    // Set: pixels whose intensity variance over the stack (either side) is below this get
    // correlation -1, i.e. are dropped by any threshold above -1.
    std::optional<float> min_variance = std::nullopt;
    TransformMode mode = TransformMode::LIMITED;
    Precision precision = Precision::SINGLE;
    SearchVariant variant = Variant::NoDuplicates {};
    // Extension beyond the reference (leave false for its behaviour): descriptors of 384 and 512
    // bits, i.e. FULL stacks of 17..23 images, which the reference rejects as "too large".
    bool wide_descriptors = false;
    // Extension beyond the reference (leave unset for its behaviour, the search over the whole row):
    // search only the pairs (left column i, right column j) with min <= i - j <= max. The forward
    // search of i runs over right columns [i - max, i - min], the reverse search of the Consistency
    // check from right column b over left columns [b + min, b + max], both clipped to the image;
    // ties are decided as without a range. A left pixel with no right column in range is invalid.
    // Fewer wrong matches outside the rig's working volume, and D = max - min + 1 instead of W
    // candidates per pixel. The range bounds the search, not the refined value: the subpixel
    // refinement still looks at the two neighbours of the match, so a subpixel disparity may lie up
    // to 1 px outside [min, max]. min > max throws BICOS::Exception; other values are accepted: bounds
    // beyond +-(cols - 1) select no further pairs, and a range that covers the whole row is the same as unset.
    std::optional<DisparityRange> disparity_range = std::nullopt;
};

// Thrown for invalid input (fewer than two images, unsupported depth, mismatching stacks) and
// for CUDA failures; stacks that need more than 256 descriptor bits raise std::invalid_argument,
// as in the reference.
class Exception: public std::exception {
    std::string message_;

public:
    explicit Exception(const std::string& message): message_(message) {}
    const char* what() const noexcept override {
        return message_.c_str();
    }
};

} // namespace BICOS
