// Per-pixel disparity windows from a prior disparity (bicos_b200_windows_from_disparity): one thread per pixel.
// A valid prior d gives [clamp(floor(d) - margin), clamp(ceil(d) + margin)] to int16, computed in double, where every
// step is exact for |d| < 2^53 and anything larger clamps anyway; an invalid one (the markers bicos_b200_reproject
// skips, or +-inf) gives the fallback window.

#include "kernels.cuh"

namespace bicos_b200 {
namespace {

constexpr int WT = 256;

__device__ __forceinline__ int16_t clamp16(double v) {
    return (int16_t)fmin(32767.0, fmax(-32768.0, v));
}

template<bool FLOAT>
__global__ void __launch_bounds__(WT) windows_kernel(const WindowsParams p) {
    const int c = blockIdx.x * WT + threadIdx.x;
    const int r = blockIdx.y;
    if (c >= p.cols)
        return;
    const char* const row = static_cast<const char*>(p.prior) + (size_t)r * p.prior_pitch;
    double lo, hi;
    bool ok;
    if constexpr (FLOAT) {
        const float d = reinterpret_cast<const float*>(row)[c];
        ok = isfinite(d) && d != -32768.0f;
        lo = floor((double)d);
        hi = ceil((double)d);
    } else {
        const int d = reinterpret_cast<const int16_t*>(row)[c];
        ok = d != -32768;
        lo = hi = (double)d;
    }
    const size_t at = (size_t)r * p.out_pitch + c;
    p.min_out[at] = ok ? clamp16(lo - (double)p.margin) : (int16_t)p.fallback_min;
    p.max_out[at] = ok ? clamp16(hi + (double)p.margin) : (int16_t)p.fallback_max;
}

} // namespace

cudaError_t launch_windows_from_disparity(const WindowsParams& p, int is_float, cudaStream_t stream) {
    const dim3 grid((unsigned)((p.cols + WT - 1) / WT), (unsigned)p.rows);
    if (is_float)
        windows_kernel<true><<<grid, WT, 0, stream>>>(p);
    else
        windows_kernel<false><<<grid, WT, 0, stream>>>(p);
    return cudaGetLastError();
}

} // namespace bicos_b200
