// Rectification stage in front of the match: dst(y, x) = src(map_y(y, x), map_x(y, x)), bilinear, with the
// conventions of OpenCV's CPU cv::remap(..., INTER_LINEAR, BORDER_CONSTANT, 0) on CV_32FC1 maps, bit for bit
// (DESIGN.md §3.7; restated in numpy by tests/test_rectify.py):
//   X = RNE(mx * 32), Y = RNE(my * 32); x0 = X >> 5, y0 = Y >> 5 (floor); fx = X & 31, fy = Y & 31
//   taps v00 = src(y0, x0), v01 = src(y0, x0 + 1), v10 = src(y0 + 1, x0), v11 = src(y0 + 1, x0 + 1); 0 outside the source
//   8U:  ((32-fx)(32-fy) v00 + fx(32-fy) v01 + (32-fx)fy v10 + fx fy v11 + 512) >> 10 in int32
//   16U: float weights w00 = (1-ay)(1-ax) ... (ax = fx/32, ay = fy/32, all exact), the sum
//        ((v00 w00 + v01 w01) + v10 w10) + v11 w11 with every product and sum rounded on its own (no FMA
//        contraction: it moves rounding ties), then RNE and saturation to 16 bits
//   a map value that is NaN, +-inf or of magnitude >= 2^25 gives 0
//
// HBM-bound: each output pixel reads its two map values once and n x 4 source taps, and writes n pixels. A thread owns
// 4 (u8) or 2 (u16) consecutive output pixels, so that its stores are 32-bit; it computes the taps and weights of its
// pixels once and then loops over the n planes. A tap outside the source is read at a clamped address with weight 0,
// which contributes exactly 0 in both depths, so the plane loop has no branches. Rectification maps are smooth: a
// warp's taps lie in a few source rows of each plane, and the read-only path (L1) serves the reuse between
// neighbouring pixels and rows. blockIdx.z selects the side, so both stacks of a match are one launch.

#include "kernels.cuh"

namespace bicos_b200 {
namespace {

constexpr int THREADS = 128;
constexpr float MAP_LIMIT = 33554432.0f; // 2^25: beyond it m * 32 leaves the int range cv::remap rounds into

template<typename T>
struct Depth;
template<>
struct Depth<uint8_t> {
    static constexpr int PX = 4;
    using Weight = int;
};
template<>
struct Depth<uint16_t> {
    static constexpr int PX = 2;
    using Weight = float;
};

template<typename T>
struct Taps {
    size_t off[4]; // byte offsets of v00, v01, v10, v11 in a plane (clamped into the source)
    typename Depth<T>::Weight w[4]; // 0 for a tap outside the source
};

template<typename T>
__device__ __forceinline__ void make_taps(Taps<T>& t, float mx, float my, int src_rows, int src_cols, size_t src_pitch) {
    int x0 = -2, y0 = -2, fx = 0, fy = 0; // -2: every tap outside
    if (fabsf(mx) < MAP_LIMIT && fabsf(my) < MAP_LIMIT) { // false for NaN
        const int X = __float2int_rn(mx * 32.0f); // exact product
        const int Y = __float2int_rn(my * 32.0f);
        x0 = X >> 5;
        y0 = Y >> 5;
        fx = X & 31;
        fy = Y & 31;
    }
    const bool cx0 = x0 >= 0 && x0 < src_cols, cx1 = x0 + 1 >= 0 && x0 + 1 < src_cols;
    const bool ry0 = y0 >= 0 && y0 < src_rows, ry1 = y0 + 1 >= 0 && y0 + 1 < src_rows;
    const size_t es = sizeof(T);
    const size_t c0 = (size_t)min(max(x0, 0), src_cols - 1) * es, c1 = (size_t)min(max(x0 + 1, 0), src_cols - 1) * es;
    const size_t r0 = (size_t)min(max(y0, 0), src_rows - 1) * src_pitch, r1 = (size_t)min(max(y0 + 1, 0), src_rows - 1) * src_pitch;
    t.off[0] = r0 + c0;
    t.off[1] = r0 + c1;
    t.off[2] = r1 + c0;
    t.off[3] = r1 + c1;
    if constexpr (sizeof(T) == 1) {
        t.w[0] = (32 - fx) * (32 - fy);
        t.w[1] = fx * (32 - fy);
        t.w[2] = (32 - fx) * fy;
        t.w[3] = fx * fy;
    } else {
        const float ax = (float)fx * (1.0f / 32.0f), ay = (float)fy * (1.0f / 32.0f);
        t.w[0] = __fmul_rn(1.0f - ay, 1.0f - ax);
        t.w[1] = __fmul_rn(1.0f - ay, ax);
        t.w[2] = __fmul_rn(ay, 1.0f - ax);
        t.w[3] = __fmul_rn(ay, ax);
    }
    const bool in[4] = { ry0 && cx0, ry0 && cx1, ry1 && cx0, ry1 && cx1 };
#pragma unroll
    for (int k = 0; k < 4; ++k)
        if (!in[k])
            t.w[k] = 0;
}

template<typename T>
__device__ __forceinline__ uint32_t interpolate(const Taps<T>& t, const unsigned char* plane) {
    const uint32_t v00 = __ldg(reinterpret_cast<const T*>(plane + t.off[0]));
    const uint32_t v01 = __ldg(reinterpret_cast<const T*>(plane + t.off[1]));
    const uint32_t v10 = __ldg(reinterpret_cast<const T*>(plane + t.off[2]));
    const uint32_t v11 = __ldg(reinterpret_cast<const T*>(plane + t.off[3]));
    if constexpr (sizeof(T) == 1) {
        return (uint32_t)((t.w[0] * (int)v00 + t.w[1] * (int)v01 + t.w[2] * (int)v10 + t.w[3] * (int)v11 + 512) >> 10);
    } else {
        float s = __fmul_rn((float)v00, t.w[0]);
        s = __fadd_rn(s, __fmul_rn((float)v01, t.w[1]));
        s = __fadd_rn(s, __fmul_rn((float)v10, t.w[2]));
        s = __fadd_rn(s, __fmul_rn((float)v11, t.w[3]));
        return (uint32_t)min(max(__float2int_rn(s), 0), 65535);
    }
}

template<typename T>
__global__ void __launch_bounds__(THREADS) remap_kernel(const RemapParams prm) {
    constexpr int PX = Depth<T>::PX;
    const RemapSide& side = prm.side[blockIdx.z];
    const int y = blockIdx.y;
    const int x = (blockIdx.x * THREADS + threadIdx.x) * PX;
    if (x >= prm.cols)
        return;
    const int count = min(PX, prm.cols - x);
    const float* mxr = reinterpret_cast<const float*>(reinterpret_cast<const char*>(side.map_x) + (size_t)y * prm.map_pitch) + x;
    const float* myr = reinterpret_cast<const float*>(reinterpret_cast<const char*>(side.map_y) + (size_t)y * prm.map_pitch) + x;
    Taps<T> taps[PX];
#pragma unroll
    for (int q = 0; q < PX; ++q) {
        const float mx = q < count ? __ldg(mxr + q) : 0.f;
        const float my = q < count ? __ldg(myr + q) : 0.f;
        make_taps(taps[q], mx, my, prm.src_rows, prm.src_cols, prm.src_pitch);
    }
    const size_t dst_off = (size_t)y * prm.dst_pitch + (size_t)x * sizeof(T);
#pragma unroll 4
    for (int t = 0; t < prm.n; ++t) {
        const unsigned char* src = static_cast<const unsigned char*>(side.src.p[t]);
        uint32_t word = 0;
#pragma unroll
        for (int q = 0; q < PX; ++q)
            word |= interpolate(taps[q], src) << (8 * sizeof(T) * q);
        unsigned char* dst = static_cast<unsigned char*>(const_cast<void*>(side.dst.p[t])) + dst_off; // output planes, filled by fill_table
        if (count == PX && (reinterpret_cast<uintptr_t>(dst) & 3) == 0) {
            *reinterpret_cast<uint32_t*>(dst) = word;
        } else {
            for (int q = 0; q < count; ++q)
                reinterpret_cast<T*>(dst)[q] = (T)(word >> (8 * sizeof(T) * q));
        }
    }
}

} // namespace

cudaError_t launch_remap(const RemapParams& prm, int sides, int is_u16, cudaStream_t stream) {
    if (sides < 1 || sides > 2 || prm.n < 1 || prm.n > MAX_IMAGES || prm.rows <= 0 || prm.cols <= 0 || prm.rows > 32767 ||
        prm.cols > 32767 || prm.src_rows <= 0 || prm.src_cols <= 0)
        return cudaErrorInvalidValue;
    const int px = is_u16 ? Depth<uint16_t>::PX : Depth<uint8_t>::PX;
    const dim3 grid((unsigned)((prm.cols + THREADS * px - 1) / (THREADS * px)), (unsigned)prm.rows, (unsigned)sides);
    if (is_u16)
        remap_kernel<uint16_t><<<grid, THREADS, 0, stream>>>(prm);
    else
        remap_kernel<uint8_t><<<grid, THREADS, 0, stream>>>(prm);
    return cudaGetLastError();
}

} // namespace bicos_b200
