// Host side of the C++ API: BICOS::Image and BICOS::match on top of the C ABI
// (include/bicos_b200.h). Mirrors the validation and error behaviour of the reference's
// drivers (src/lib.cpp:31-49, src/impl/cpu.cpp:100-159, src/impl/cuda.cu:465-524).

#include "../../include/BICOS/match.hpp"
#include "../../include/BICOS/rectify.hpp"
#include "../../include/BICOS/reproject.hpp"
#include "../../include/BICOS/speckles.hpp"
#include "../../include/BICOS/windows.hpp"
#include "../../include/bicos_b200.h"

#include <cuda_runtime.h>

#include <map>
#include <mutex>
#include <stdexcept>
#include <string>

namespace BICOS {

namespace {

void cuda_check(cudaError_t err, const char* what) {
    if (err != cudaSuccess)
        throw Exception(std::string(what) + ": " + cudaGetErrorString(err));
}

[[noreturn]] void rethrow_last(int status) {
    const std::string msg = bicos_b200_last_error();
    // the reference throws std::invalid_argument for ">256 bits" and BICOS::Exception otherwise
    if (status == BICOS_B200_ERR_INVALID && msg.rfind("input stacks too large", 0) == 0)
        throw std::invalid_argument(msg);
    throw Exception(msg);
}

// one workspace per (thread, device): BICOS::match is re-entrant across threads like the
// reference (which has no global mutable state), and repeated calls reuse their buffers.
struct HandleCache {
    std::map<int, bicos_b200_handle> handles;
    std::map<int, unsigned long long*> counts; // device counters: four of reproject_points, two of filter_speckles
    ~HandleCache() {
        for (auto& kv: counts) {
            cudaSetDevice(kv.first);
            cudaFree(kv.second);
        }
        for (auto& kv: handles)
            bicos_b200_destroy(kv.second);
    }
    bicos_b200_handle get(int device) {
        auto it = handles.find(device);
        if (it != handles.end())
            return it->second;
        bicos_b200_handle h = nullptr;
        const int rc = bicos_b200_create(&h, device);
        if (rc != 0)
            rethrow_last(rc);
        handles[device] = h;
        return h;
    }
};

thread_local HandleCache t_handles;

// the device counters of reproject_points and filter_speckles on `device` (current)
unsigned long long* counts_buffer(int device) {
    auto it = t_handles.counts.find(device);
    if (it != t_handles.counts.end())
        return it->second;
    void* p = nullptr;
    cuda_check(cudaMalloc(&p, 4 * sizeof(unsigned long long)), "cudaMalloc");
    t_handles.counts[device] = static_cast<unsigned long long*>(p);
    return static_cast<unsigned long long*>(p);
}

bicos_b200_config to_c_config(const Config& cfg) {
    bicos_b200_config c {};
    c.nxcorr_threshold = cfg.nxcorr_threshold.value_or(-1.f);
    c.negative_threshold_is_set = cfg.nxcorr_threshold.has_value() && !(*cfg.nxcorr_threshold >= 0) ? 1 : 0;
    c.subpixel_step = cfg.subpixel_step.value_or(-1.f);
    c.min_variance = cfg.min_variance.value_or(-1.f);
    c.mode = cfg.mode == TransformMode::FULL ? 1 : 0;
    c.precision = cfg.precision == Precision::DOUBLE ? 1 : 0;
    c.wide_descriptors = cfg.wide_descriptors ? 1 : 0;
    if (cfg.disparity_range) {
        c.has_disparity_range = 1;
        c.min_disparity = cfg.disparity_range->min;
        c.max_disparity = cfg.disparity_range->max;
    }
    if (std::holds_alternative<Variant::Consistency>(cfg.variant)) {
        const auto& v = std::get<Variant::Consistency>(cfg.variant);
        c.variant_type = 1;
        c.max_lr_diff = v.max_lr_diff;
        c.no_dupes = v.no_dupes ? 1 : 0;
    } else {
        c.variant_type = 0;
        c.max_lr_diff = 1;
        c.no_dupes = 0;
    }
    return c;
}

struct StackView {
    std::vector<const void*> planes;
    int rows = 0, cols = 0, depth = 0;
    size_t step = 0;
};

StackView view_of(const std::vector<Image>& stack, const char* name) {
    StackView v;
    if (stack.size() < 2)
        throw Exception("need at least two images");
    const Image& first = stack.front();
    v.rows = first.rows;
    v.cols = first.cols;
    v.depth = first.depth();
    v.step = first.step;
    if (first.type() != IMG_8U && first.type() != IMG_16U)
        throw Exception("bad input depths, only CV_8UC1 and CV_16UC1 are supported");
    v.planes.reserve(stack.size());
    for (const Image& im: stack) {
        if (im.rows != v.rows || im.cols != v.cols || im.type() != first.type() || im.step != v.step || im.empty())
            throw Exception(std::string("images of ") + name + " differ in size, type or pitch");
        v.planes.push_back(im.data);
    }
    return v;
}

int device_of(const void* ptr) {
    cudaPointerAttributes attr {};
    cuda_check(cudaPointerGetAttributes(&attr, ptr), "cudaPointerGetAttributes");
    if (attr.type != cudaMemoryTypeDevice && attr.type != cudaMemoryTypeManaged)
        throw Exception("input images must live in device memory");
    return attr.device;
}

// checks a map pair of the rectified size: CV_32FC1 device images of one size and pitch
void check_maps(const Image& map_x, const Image& map_y, const Image& like) {
    for (const Image* m: { &map_x, &map_y })
        if (m->empty() || m->type() != IMG_32F || m->rows != like.rows || m->cols != like.cols || m->step != like.step)
            throw Exception("rectification maps must be non-empty CV_32FC1 images of one size and pitch");
}

// makes `device` current for the scope's lifetime
struct DeviceScope {
    int prev = 0, device = 0;
    explicit DeviceScope(int dev): device(dev) {
        cuda_check(cudaGetDevice(&prev), "cudaGetDevice");
        if (prev != device)
            cuda_check(cudaSetDevice(device), "cudaSetDevice");
    }
    ~DeviceScope() {
        if (prev != device)
            cudaSetDevice(prev);
    }
};

} // namespace

size_t image_elem_size(int type) {
    if (type == IMG_32FC3)
        return 3 * sizeof(float);
    switch (type & 7) {
        case IMG_8U:
        case 1:
            return 1;
        case IMG_16U:
        case IMG_16S:
            return 2;
        case 4:
        case IMG_32F:
            return 4;
        case IMG_64F:
            return 8;
    }
    throw Exception("unsupported image type");
}

Image::Image(int r, int c, int type, void* device_ptr, size_t stepb):
    rows(r),
    cols(c),
    step(stepb ? stepb : (size_t)c * image_elem_size(type)),
    data(static_cast<unsigned char*>(device_ptr)),
    type_(type) {}

void Image::create(int r, int c, int type) {
    if (data && r == rows && c == cols && type == type_)
        return;
    release();
    if (r <= 0 || c <= 0)
        throw Exception("cannot create an empty image");
    void* ptr = nullptr;
    size_t pitch = 0;
    cuda_check(cudaMallocPitch(&ptr, &pitch, (size_t)c * image_elem_size(type), (size_t)r), "cudaMallocPitch");
    owner_ = std::shared_ptr<void>(ptr, [](void* p) { cudaFree(p); });
    data = static_cast<unsigned char*>(ptr);
    rows = r;
    cols = c;
    step = pitch;
    type_ = type;
}

void Image::release() {
    owner_.reset();
    data = nullptr;
    rows = cols = 0;
    step = 0;
}

void Image::upload(const HostImage& host, void* stream) {
    create(host.rows, host.cols, host.type());
    cuda_check(
        cudaMemcpy2DAsync(data, step, host.data, host.step, (size_t)cols * elemSize(), (size_t)rows,
                          cudaMemcpyHostToDevice, static_cast<cudaStream_t>(stream)),
        "upload"
    );
    if (!stream)
        cuda_check(cudaStreamSynchronize(nullptr), "upload sync");
}

void Image::download(const HostImage& host, void* stream) const {
    if (host.rows != rows || host.cols != cols || host.type() != type_ || !host.data)
        throw Exception("download target does not match the image");
    cuda_check(
        cudaMemcpy2DAsync(host.data, host.step, data, step, (size_t)cols * elemSize(), (size_t)rows,
                          cudaMemcpyDeviceToHost, static_cast<cudaStream_t>(stream)),
        "download"
    );
    if (!stream)
        cuda_check(cudaStreamSynchronize(nullptr), "download sync");
}

void match(
    const std::vector<Image>& stack0,
    const std::vector<Image>& stack1,
    Image& disparity,
    Config cfg,
    Image* corrmap,
    void* stream
) {
    const StackView v0 = view_of(stack0, "stack0");
    const StackView v1 = view_of(stack1, "stack1");
    if (stack0.size() != stack1.size() || v0.rows != v1.rows || v0.cols != v1.cols || v0.depth != v1.depth || v0.step != v1.step)
        throw Exception("stack0 and stack1 differ in length, size, type or pitch");

    const bicos_b200_config c = to_c_config(cfg);
    const int device = device_of(v0.planes.front());
    bicos_b200_handle h = t_handles.get(device);

    int prev = 0;
    cuda_check(cudaGetDevice(&prev), "cudaGetDevice");
    if (prev != device)
        cuda_check(cudaSetDevice(device), "cudaSetDevice");
    try {
        disparity.create(v0.rows, v0.cols, bicos_b200_disparity_type(&c));
        const bool want_corr = corrmap && cfg.nxcorr_threshold.has_value(); // cpu.cpp:77-81
        if (want_corr)
            corrmap->create(v0.rows, v0.cols, bicos_b200_corrmap_type(&c));
        const int rc = bicos_b200_match(
            h, v0.planes.data(), v1.planes.data(), (int)stack0.size(), v0.rows, v0.cols, v0.step, v0.depth, &c,
            disparity.data, disparity.step, want_corr ? corrmap->data : nullptr, want_corr ? corrmap->step : 0, stream
        );
        if (rc != 0)
            rethrow_last(rc);
    } catch (...) {
        if (prev != device)
            cudaSetDevice(prev);
        throw;
    }
    if (prev != device)
        cudaSetDevice(prev);
}

void remap(const std::vector<Image>& src, const Image& map_x, const Image& map_y, std::vector<Image>& dst, void* stream) {
    if (src.empty())
        throw Exception("no images to remap");
    const Image& first = src.front();
    if (first.type() != IMG_8U && first.type() != IMG_16U)
        throw Exception("bad input depths, only CV_8UC1 and CV_16UC1 are supported");
    std::vector<const void*> planes;
    for (const Image& im: src) {
        if (im.empty() || im.rows != first.rows || im.cols != first.cols || im.type() != first.type() || im.step != first.step)
            throw Exception("images to remap differ in size, type or pitch");
        planes.push_back(im.data);
    }
    check_maps(map_x, map_y, map_x);
    const int device = device_of(planes.front());
    bicos_b200_handle h = t_handles.get(device);
    DeviceScope scope(device);
    dst.resize(src.size());
    std::vector<void*> out;
    for (Image& im: dst) {
        im.create(map_x.rows, map_x.cols, first.type());
        out.push_back(im.data);
    }
    for (const Image& im: dst)
        if (im.step != dst.front().step)
            throw Exception("remap outputs differ in pitch");
    const int rc = bicos_b200_remap(h, planes.data(), (int)planes.size(), first.rows, first.cols, first.step, first.depth(),
                                    reinterpret_cast<const float*>(map_x.data), reinterpret_cast<const float*>(map_y.data),
                                    map_x.step, map_x.rows, map_x.cols, out.data(), dst.front().step, stream);
    if (rc != 0)
        rethrow_last(rc);
}

void match_rectified(
    const std::vector<Image>& stack0,
    const std::vector<Image>& stack1,
    const RectifyMaps& maps,
    Image& disparity,
    Config cfg,
    Image* corrmap,
    void* stream
) {
    const StackView v0 = view_of(stack0, "stack0");
    const StackView v1 = view_of(stack1, "stack1");
    if (stack0.size() != stack1.size() || v0.rows != v1.rows || v0.cols != v1.cols || v0.depth != v1.depth || v0.step != v1.step)
        throw Exception("stack0 and stack1 differ in length, size, type or pitch");
    check_maps(maps.map_x0, maps.map_y0, maps.map_x0);
    check_maps(maps.map_x1, maps.map_y1, maps.map_x0);
    const bicos_b200_config c = to_c_config(cfg);
    const int device = device_of(v0.planes.front());
    bicos_b200_handle h = t_handles.get(device);
    DeviceScope scope(device);
    const int rows = maps.map_x0.rows, cols = maps.map_x0.cols;
    disparity.create(rows, cols, bicos_b200_disparity_type(&c));
    const bool want_corr = corrmap && cfg.nxcorr_threshold.has_value();
    if (want_corr)
        corrmap->create(rows, cols, bicos_b200_corrmap_type(&c));
    const bicos_b200_rectify_maps m { reinterpret_cast<const float*>(maps.map_x0.data), reinterpret_cast<const float*>(maps.map_y0.data),
                                      reinterpret_cast<const float*>(maps.map_x1.data), reinterpret_cast<const float*>(maps.map_y1.data),
                                      maps.map_x0.step };
    const int rc = bicos_b200_match_rectified(h, v0.planes.data(), v1.planes.data(), (int)stack0.size(), v0.rows, v0.cols, v0.step,
                                              v0.depth, &m, rows, cols, &c, disparity.data, disparity.step,
                                              want_corr ? corrmap->data : nullptr, want_corr ? corrmap->step : 0, stream);
    if (rc != 0)
        rethrow_last(rc);
}

namespace {

// a window pair of the disparity's size: CV_16SC1 device images of one pitch
bicos_b200_disparity_windows windows_of(const DisparityWindows& w, int rows, int cols) {
    for (const Image* m: { &w.min, &w.max })
        if (m->empty() || m->type() != IMG_16S || m->rows != rows || m->cols != cols || m->step != w.min.step)
            throw Exception("disparity windows must be non-empty CV_16SC1 images of the stacks' size and one pitch");
    return bicos_b200_disparity_windows { reinterpret_cast<const int16_t*>(w.min.data), reinterpret_cast<const int16_t*>(w.max.data),
                                          w.min.step };
}

} // namespace

void match_windows(
    const std::vector<Image>& stack0,
    const std::vector<Image>& stack1,
    const DisparityWindows& windows,
    Image& disparity,
    Config cfg,
    Image* corrmap,
    void* stream
) {
    const StackView v0 = view_of(stack0, "stack0");
    const StackView v1 = view_of(stack1, "stack1");
    if (stack0.size() != stack1.size() || v0.rows != v1.rows || v0.cols != v1.cols || v0.depth != v1.depth || v0.step != v1.step)
        throw Exception("stack0 and stack1 differ in length, size, type or pitch");
    const bicos_b200_disparity_windows w = windows_of(windows, v0.rows, v0.cols);
    const bicos_b200_config c = to_c_config(cfg);
    const int device = device_of(v0.planes.front());
    bicos_b200_handle h = t_handles.get(device);
    DeviceScope scope(device);
    disparity.create(v0.rows, v0.cols, bicos_b200_disparity_type(&c));
    const bool want_corr = corrmap && cfg.nxcorr_threshold.has_value();
    if (want_corr)
        corrmap->create(v0.rows, v0.cols, bicos_b200_corrmap_type(&c));
    const int rc = bicos_b200_match_windows(h, v0.planes.data(), v1.planes.data(), (int)stack0.size(), v0.rows, v0.cols, v0.step,
                                            v0.depth, &c, &w, disparity.data, disparity.step, want_corr ? corrmap->data : nullptr,
                                            want_corr ? corrmap->step : 0, stream);
    if (rc != 0)
        rethrow_last(rc);
}

void windows_from_disparity(const Image& prior, int margin, std::optional<DisparityRange> fallback, DisparityWindows& windows,
                            void* stream) {
    if (prior.empty() || (prior.type() != IMG_16S && prior.type() != IMG_32F))
        throw Exception("windows_from_disparity needs a non-empty CV_16SC1 or CV_32FC1 prior");
    const int device = device_of(prior.data);
    bicos_b200_handle h = t_handles.get(device);
    DeviceScope scope(device);
    windows.min.create(prior.rows, prior.cols, IMG_16S);
    windows.max.create(prior.rows, prior.cols, IMG_16S);
    if (windows.max.step != windows.min.step)
        throw Exception("disparity windows differ in pitch");
    const DisparityRange fb = fallback.value_or(DisparityRange { -32768, 32767 });
    const int rc = bicos_b200_windows_from_disparity(h, prior.data, prior.type(), prior.step, prior.rows, prior.cols, margin, fb.min,
                                                     fb.max, reinterpret_cast<int16_t*>(windows.min.data),
                                                     reinterpret_cast<int16_t*>(windows.max.data), windows.min.step, stream);
    if (rc != 0)
        rethrow_last(rc);
}

namespace {

void check_disparity(const Image& disparity) {
    if (disparity.empty() || (disparity.type() != IMG_16S && disparity.type() != IMG_32F))
        throw Exception("reprojection needs a non-empty CV_16SC1 or CV_32FC1 disparity image");
}

} // namespace

void reproject(const Image& disparity, const std::array<double, 16>& Q, Image& xyz, bool allow_negative_z, void* stream) {
    check_disparity(disparity);
    const int device = device_of(disparity.data);
    bicos_b200_handle h = t_handles.get(device);
    DeviceScope scope(device);
    xyz.create(disparity.rows, disparity.cols, IMG_32FC3);
    const int rc = bicos_b200_reproject(h, disparity.data, disparity.type(), disparity.step, disparity.rows, disparity.cols, Q.data(),
                                        allow_negative_z ? BICOS_B200_REPROJECT_ALLOW_NEGATIVE_Z : 0,
                                        reinterpret_cast<float*>(xyz.data), xyz.step, nullptr, nullptr, nullptr, stream);
    if (rc != 0)
        rethrow_last(rc);
}

ReprojectCounts reproject_points(const Image& disparity, const std::array<double, 16>& Q, Image& points, Image* pixel_index,
                                 bool allow_negative_z, void* stream) {
    check_disparity(disparity);
    const int device = device_of(disparity.data);
    bicos_b200_handle h = t_handles.get(device);
    DeviceScope scope(device);
    if (disparity.rows > 32767 || disparity.cols > 32767)
        throw Exception("reprojection: the disparity has more than 32767 rows or columns");
    const int capacity = disparity.rows * disparity.cols; // < 2^30
    points.create(1, capacity, IMG_32FC3);
    if (pixel_index)
        pixel_index->create(1, capacity, IMG_32S);
    unsigned long long* counts = counts_buffer(device);
    const int rc = bicos_b200_reproject(h, disparity.data, disparity.type(), disparity.step, disparity.rows, disparity.cols, Q.data(),
                                        allow_negative_z ? BICOS_B200_REPROJECT_ALLOW_NEGATIVE_Z : 0, nullptr, 0,
                                        reinterpret_cast<float*>(points.data),
                                        pixel_index ? reinterpret_cast<int32_t*>(pixel_index->data) : nullptr, counts, stream);
    if (rc != 0)
        rethrow_last(rc);
    unsigned long long host[4] = { 0, 0, 0, 0 };
    const cudaStream_t s = static_cast<cudaStream_t>(stream);
    cuda_check(cudaMemcpyAsync(host, counts, sizeof host, cudaMemcpyDeviceToHost, s), "download counts");
    cuda_check(cudaStreamSynchronize(s), "cudaStreamSynchronize");
    return ReprojectCounts { (size_t)host[0], (size_t)host[1], (size_t)host[2], (size_t)host[3] };
}

void filter_speckles(Image& disparity, double new_value, int max_speckle_size, double max_diff, SpeckleCounts* counts, void* stream) {
    if (disparity.empty() || (disparity.type() != IMG_16S && disparity.type() != IMG_32F))
        throw Exception("speckle filtering needs a non-empty CV_16SC1 or CV_32FC1 disparity image");
    const int device = device_of(disparity.data);
    bicos_b200_handle h = t_handles.get(device);
    DeviceScope scope(device);
    unsigned long long* dev_counts = counts ? counts_buffer(device) : nullptr;
    const int rc = bicos_b200_filter_speckles(h, disparity.data, disparity.type(), disparity.step, disparity.rows, disparity.cols,
                                              new_value, max_speckle_size, max_diff, dev_counts, stream);
    if (rc != 0)
        rethrow_last(rc);
    if (!counts)
        return;
    unsigned long long host[2] = { 0, 0 };
    const cudaStream_t s = static_cast<cudaStream_t>(stream);
    cuda_check(cudaMemcpyAsync(host, dev_counts, sizeof host, cudaMemcpyDeviceToHost, s), "download counts");
    cuda_check(cudaStreamSynchronize(s), "cudaStreamSynchronize");
    *counts = SpeckleCounts { (size_t)host[0], (size_t)host[1] };
}

void match_sharded(
    const std::vector<Image>& stack0,
    const std::vector<Image>& stack1,
    Image& disparity,
    const std::vector<int>& devices,
    Config cfg,
    Image* corrmap
) {
    if (devices.empty())
        throw Exception("no devices given");
    const StackView v0 = view_of(stack0, "stack0");
    const StackView v1 = view_of(stack1, "stack1");
    if (stack0.size() != stack1.size() || v0.rows != v1.rows || v0.cols != v1.cols || v0.depth != v1.depth || v0.step != v1.step)
        throw Exception("stack0 and stack1 differ in length, size, type or pitch");
    const int home = devices.front();
    if (device_of(v0.planes.front()) != home)
        throw Exception("inputs must be resident on devices[0]");

    const bicos_b200_config c = to_c_config(cfg);
    int prev = 0;
    cuda_check(cudaGetDevice(&prev), "cudaGetDevice");

    cuda_check(cudaSetDevice(home), "cudaSetDevice");
    disparity.create(v0.rows, v0.cols, bicos_b200_disparity_type(&c));
    const bool want_corr = corrmap && cfg.nxcorr_threshold.has_value();
    if (want_corr)
        corrmap->create(v0.rows, v0.cols, bicos_b200_corrmap_type(&c));
    cuda_check(cudaDeviceSynchronize(), "sync home device"); // inputs and outputs visible to the peers

    const int G = (int)devices.size();
    std::string error;
    for (int g = 0; g < G && error.empty(); ++g) {
        const int dev = devices[g];
        cuda_check(cudaSetDevice(dev), "cudaSetDevice");
        if (dev != home) {
            int can = 0;
            cuda_check(cudaDeviceCanAccessPeer(&can, dev, home), "cudaDeviceCanAccessPeer");
            if (!can)
                throw Exception("no peer access from device " + std::to_string(dev) + " to " + std::to_string(home));
            const cudaError_t e = cudaDeviceEnablePeerAccess(home, 0);
            if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled)
                cuda_check(e, "cudaDeviceEnablePeerAccess");
            cudaGetLastError();
        }
        const int rb = (int)((long long)v0.rows * g / G), re = (int)((long long)v0.rows * (g + 1) / G);
        if (rb >= re)
            continue;
        bicos_b200_handle h = t_handles.get(dev);
        const int rc = bicos_b200_match_rows(
            h, v0.planes.data(), v1.planes.data(), (int)stack0.size(), v0.rows, v0.cols, v0.step, v0.depth, &c, rb, re,
            disparity.data, disparity.step, want_corr ? corrmap->data : nullptr, want_corr ? corrmap->step : 0, nullptr
        );
        if (rc != 0)
            error = bicos_b200_last_error();
    }
    for (int g = 0; g < G; ++g) {
        cudaSetDevice(devices[g]);
        cudaDeviceSynchronize();
    }
    cudaSetDevice(prev);
    if (!error.empty())
        throw Exception(error);
}

} // namespace BICOS
