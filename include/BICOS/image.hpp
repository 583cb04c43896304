// BICOS::Image for builds without OpenCV: a reference-counted, pitched
// device matrix exposing the members of cv::cuda::GpuMat that callers of BICOS::match use
// (rows, cols, step, data, type(), depth(), create(), upload(), download(), empty()).
//
// The reference's public signature uses cv::cuda::GpuMat for its CUDA build
// (reference include/common.hpp:50-56). OpenCV is a container type there, not part of the
// matching arithmetic; define BICOS_WITH_OPENCV to alias the real type instead
// (include/BICOS/common.hpp).
#pragma once

#include <cstddef>
#include <cstdint>
#include <memory>

namespace BICOS {

// OpenCV type codes, so that code written against cv::Mat::type() keeps working: single channel, plus the int32
// pixel indices and the interleaved float32 X Y Z points of BICOS::reproject (reproject.hpp)
constexpr int IMG_8U = 0, IMG_16U = 2, IMG_16S = 3, IMG_32S = 4, IMG_32F = 5, IMG_64F = 6;
constexpr int IMG_32FC3 = 21; // CV_32FC3: depth IMG_32F, three channels (channel count - 1 in bits 3 and up)

size_t image_elem_size(int type);

// Non-owning view of a dense or pitched host image (what cv::Mat is to the reference's CPU build).
struct HostImage {
    int rows = 0, cols = 0, type_code = IMG_8U;
    void* data = nullptr;
    size_t step = 0; // bytes per row; 0 = dense

    HostImage() = default;
    HostImage(int r, int c, int type, void* ptr, size_t stepb = 0):
        rows(r),
        cols(c),
        type_code(type),
        data(ptr),
        step(stepb ? stepb : (size_t)c * image_elem_size(type)) {}
    int type() const {
        return type_code;
    }
};

class Image {
public:
    int rows = 0, cols = 0;
    size_t step = 0; // bytes per row
    unsigned char* data = nullptr; // device pointer

    Image() = default;
    Image(int r, int c, int type) {
        create(r, c, type);
    }
    // borrow caller-owned device memory (no copy, no ownership)
    Image(int r, int c, int type, void* device_ptr, size_t stepb);
    // allocate + upload, like cv::cuda::GpuMat(const cv::Mat&)
    explicit Image(const HostImage& host) {
        upload(host);
    }

    int type() const {
        return type_;
    }
    int depth() const {
        return type_ & 7;
    }
    int channels() const {
        return (type_ >> 3) + 1;
    }
    size_t elemSize() const {
        return image_elem_size(type_);
    }
    bool empty() const {
        return data == nullptr || rows == 0 || cols == 0;
    }

    // (re)allocates only if shape or type differ, like cv::cuda::GpuMat::create
    void create(int r, int c, int type);
    void release();
    void upload(const HostImage& host, void* stream = nullptr);
    void download(const HostImage& host, void* stream = nullptr) const; // host must be preallocated

private:
    int type_ = IMG_8U;
    std::shared_ptr<void> owner_;
};

} // namespace BICOS
